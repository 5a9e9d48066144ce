/* b2h264_wels_api.h — layer 3: the reference's own public entry points, exported by
 * openh264_b200/libopenh264_b200_wels.so so that an application built against the reference's headers can
 * load this library in place of libopenh264.so for the supported encoder configuration.
 *
 * The objects handed out are C++ objects whose vtable has the slot order of `class ISVCEncoder`
 * (codec/api/wels/codec_api.h:272-339: Initialize, InitializeExt, GetDefaultParams, Uninitialize, EncodeFrame,
 * EncodeParameterSets, ForceIntraFrame, SetOption, GetOption, destructor).  The structures and vtables are declared
 * with the layout of the reference's public headers in include/b2h264_wels_abi.h, which the shim is compiled
 * against.  C callers see the same pointer-to-vtable layout (codec_api.h:475-536).
 *
 * Types below are only forward-declared; include/b2h264_wels_abi.h (or the reference's codec_api.h) defines them.
 *
 * Supported configuration (InitializeExt returns cmUnsupportedData = 4 for anything else, with the reason on
 * stderr; nothing is silently approximated and there is no CPU fallback):
 *   iUsageType CAMERA_VIDEO_REAL_TIME, iSpatialLayerNum 1, iTemporalLayerNum 1, iRCMode RC_OFF_MODE,
 *   SM_SINGLE_SLICE, iEntropyCodingModeFlag 0, iNumRefFrame 1 or AUTO, uiIntraPeriod 0, iLoopFilterDisableIdc 0
 *   with zero offsets, iComplexityMode MEDIUM/HIGH, bEnableDenoise / BackgroundDetection / AdaptiveQuant /
 *   SceneChangeDetect / LongTermReference / FrameSkip all false, bEnableFrameCroppingFlag true,
 *   profile baseline/unknown, no SSEI / simulcast / prefix NAL, eSpsPpsIdStrategy CONSTANT_ID or INCREASING_ID
 *   (every IDR's parameter sets take the next id, as in the reference), width % 4 == 0, height % 2 == 0.
 * Initialize(SEncParamBase*) implies RC on (the reference's default RC_QUALITY_MODE): unsupported unless
 *   iRCMode == RC_OFF_MODE.
 */
#ifndef B2H264_WELS_API_H
#define B2H264_WELS_API_H
#ifdef __cplusplus
class ISVCEncoder;
class ISVCDecoder;
extern "C" {
#else
typedef const struct ISVCEncoderVtbl* ISVCEncoder;
typedef const struct ISVCDecoderVtbl* ISVCDecoder;
#endif
struct TagDecoderCapability;
struct _tagVersion;

/* codec_api.h:551 — creates an encoder object; 0 on success, 1 on failure (no CUDA device / library). */
int  WelsCreateSVCEncoder (ISVCEncoder** ppEncoder);
/* codec_api.h:558 */
void WelsDestroySVCEncoder (ISVCEncoder* pEncoder);
/* codec_api.h:566-580 — the decoder is not part of this round (SURVEY §8f / DESIGN.md §9): WelsCreateDecoder
 * returns 1 and stores NULL, WelsGetDecoderCapability returns 1.  They exist so that the export list of
 * libopenh264 (openh264.def) resolves; they fail loudly rather than decode on the CPU. */
int  WelsGetDecoderCapability (struct TagDecoderCapability* pDecCapability);
long WelsCreateDecoder (ISVCDecoder** ppDecoder);
void WelsDestroyDecoder (ISVCDecoder* pDecoder);
/* codec_api.h:584-590 — reports the API version of the headers the shim was compiled against. */
void WelsGetCodecVersionEx (struct _tagVersion* pVersion);
#ifdef __cplusplus
}
#endif
#endif
