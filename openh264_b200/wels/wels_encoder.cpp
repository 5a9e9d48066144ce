// wels_encoder.cpp — layer 3: an ISVCEncoder (codec/api/wels/codec_api.h:272-339) over the layer-2 C ABI
// (include/b2h264_codec.h).  One object = one stream, but NOT one private GPU encoder: objects of equal configuration
// are streams of a shared batched encoder and their EncodeFrame calls are coded together (broker.h).  The vtable slot
// order and the parameter / bitstream-info structures are the reference's own (include/b2h264_wels_abi.h,
// include/b2h264_wels_api.h).  Behavioural model: CWelsH264SVCEncoder (codec/encoder/plus/src/welsEncoderExt.cpp):
// Initialize* validate and (re)create the encoder, EncodeFrame is synchronous and returns encoder-owned bitstream
// memory that stays valid until the next call.  No CPU encoder lives here: every picture goes through
// b2h264_enc_submit / b2h264_enc_collect, i.e. the CUDA macroblock pipeline; creation fails without a device.
#include <cuda_runtime_api.h>
#include <stdio.h>
#include <string.h>

#include <vector>

#include "b2h264_codec.h"
#include "broker.h"
#include "b2h264_wels_abi.h"

namespace {

const int kMaxFps = 60, kMinFps = 1;          // MAX_FRAME_RATE / MIN_FRAME_RATE (codec/encoder/core/inc/wels_const.h:60-61)

void why(const char* msg) { fprintf(stderr, "[b2h264] unsupported encoder configuration: %s\n", msg); }

class B2Encoder : public ISVCEncoder {
 public:
  B2Encoder() { default_params(&par_); }
  ~B2Encoder() override { Uninitialize(); }

  int EXTAPI Initialize(const SEncParamBase* p) override {
    if (!p) return cmInitParaError;
    // SWelsSvcCodingParam::ParamBaseTranscode (codec/encoder/core/inc/param_svc.h:236): the base parameters
    // over the defaults
    SEncParamExt e;
    default_params(&e);
    e.iUsageType = p->iUsageType;
    e.iPicWidth = p->iPicWidth;
    e.iPicHeight = p->iPicHeight;
    e.iTargetBitrate = p->iTargetBitrate;
    e.iRCMode = p->iRCMode;
    e.fMaxFrameRate = p->fMaxFrameRate;
    e.sSpatialLayers[0].iVideoWidth = p->iPicWidth;
    e.sSpatialLayers[0].iVideoHeight = p->iPicHeight;
    e.sSpatialLayers[0].fFrameRate = p->fMaxFrameRate;
    e.sSpatialLayers[0].iSpatialBitrate = p->iTargetBitrate;
    // ParamBaseTranscode keeps FillDefault's tools switched on: scene-change detection (inserts IDRs), background
    // detection (changes the skip decision), adaptive quantisation (per-MB QP even with RC off: WelsRcMbInitDisable,
    // ratectl.cpp:1301), frame skipping, and LOW_COMPLEXITY mode decision.  None of them is a no-op for the output,
    // so this entry point cannot be honoured bit-exactly; it is refused with the reason instead of approximated.
    if (p->iRCMode != RC_OFF_MODE) { why("Initialize(SEncParamBase): rate control is on (only RC_OFF_MODE; needs the on-device bit count)"); return cmUnsupportedData; }
    why("Initialize(SEncParamBase) implies bEnableSceneChangeDetect, bEnableBackgroundDetection, bEnableAdaptiveQuant and "
        "iComplexityMode = LOW_COMPLEXITY, which change the bitstream; use InitializeExt with them off");
    (void)e;
    return cmUnsupportedData;
  }

  int EXTAPI InitializeExt(const SEncParamExt* p) override {
    if (!p) return cmInitParaError;
    if (p->iPicWidth < 16 || p->iPicHeight < 16) return cmInitParaError;
    const SSpatialLayerConfig& l = p->sSpatialLayers[0];
#define REQUIRE(cond, msg) do { if (!(cond)) { why(msg); return cmUnsupportedData; } } while (0)
    REQUIRE(p->iUsageType == CAMERA_VIDEO_REAL_TIME, "iUsageType != CAMERA_VIDEO_REAL_TIME");
    REQUIRE(p->iSpatialLayerNum == 1 && p->iTemporalLayerNum == 1, "more than one spatial/temporal layer");
    REQUIRE(p->iRCMode == RC_OFF_MODE, "iRCMode != RC_OFF_MODE");
    REQUIRE(l.sSliceArgument.uiSliceMode == SM_SINGLE_SLICE, "uiSliceMode != SM_SINGLE_SLICE");
    REQUIRE(p->iNumRefFrame == 1 || p->iNumRefFrame == AUTO_REF_PIC_COUNT, "iNumRefFrame != 1");
    if (p->iLoopFilterDisableIdc < 0 || p->iLoopFilterDisableIdc > 2 || p->iLoopFilterAlphaC0Offset < -6 || p->iLoopFilterAlphaC0Offset > 6 ||
        p->iLoopFilterBetaOffset < -6 || p->iLoopFilterBetaOffset > 6) return cmInitParaError;       // encoder_ext.cpp:316-323
    REQUIRE(p->iComplexityMode == LOW_COMPLEXITY || p->iComplexityMode == MEDIUM_COMPLEXITY || p->iComplexityMode == HIGH_COMPLEXITY,
            "iComplexityMode");
    REQUIRE(!p->bEnableDenoise && !p->bEnableBackgroundDetection && !p->bEnableAdaptiveQuant && !p->bEnableSceneChangeDetect,
            "denoise / background detection / adaptive quant / scene change detection enabled");
    REQUIRE(!p->bEnableLongTermReference && !p->bEnableFrameSkip, "LTR or frame skip enabled");
    REQUIRE(p->bEnableFrameCroppingFlag, "bEnableFrameCroppingFlag false");
    REQUIRE(!p->bEnableSSEI && !p->bSimulcastAVC && !p->bPrefixNalAddingCtrl, "SSEI / simulcast / prefix NAL");
    REQUIRE(p->eSpsPpsIdStrategy == CONSTANT_ID || p->eSpsPpsIdStrategy == INCREASING_ID, "eSpsPpsIdStrategy");
    REQUIRE(l.uiProfileIdc != PRO_SCALABLE_BASELINE && l.uiProfileIdc != PRO_SCALABLE_HIGH, "scalable profile");
    REQUIRE(l.uiLevelIdc == LEVEL_UNKNOWN, "explicit level");
    REQUIRE(!l.bAspectRatioPresent && !l.bVideoSignalTypePresent, "VUI");
    REQUIRE(l.iVideoWidth == p->iPicWidth && l.iVideoHeight == p->iPicHeight, "layer resolution != picture resolution");
    REQUIRE((p->iPicWidth % 4) == 0 && (p->iPicHeight % 2) == 0, "width % 4 or height % 2");
    REQUIRE(l.iDLayerQp >= 0 && l.iDLayerQp <= 51, "iDLayerQp out of range");
    REQUIRE(p->uiMaxNalSize == 0, "uiMaxNalSize");
#undef REQUIRE
    Uninitialize();
    b2wels::PoolKey key;
    key.width = p->iPicWidth;
    key.height = p->iPicHeight;
    key.qp = l.iDLayerQp;
    // level selection inputs exactly as the reference derives them (param_svc.h:409-437, au_set.cpp:526):
    // the layer's frame rate clipped to [MIN_FRAME_RATE, clipped fMaxFrameRate], the layer's bitrate (total as fallback)
    float fmax = p->fMaxFrameRate;                      // WELS_CLIP3 (param_svc.h:238)
    fmax = fmax < kMinFps ? kMinFps : (fmax > kMaxFps ? kMaxFps : fmax);
    float fps = l.fFrameRate;
    fps = fps < kMinFps ? kMinFps : (fps > fmax ? fmax : fps);
    key.fps = fps;
    key.bitrate = l.iSpatialBitrate ? l.iSpatialBitrate : p->iTargetBitrate;
    key.strategy = p->eSpsPpsIdStrategy == INCREASING_ID ? 1 : 0;
    key.complexity_low = p->iComplexityMode == LOW_COMPLEXITY ? 1 : 0;
    // CABAC / CAVLC and the profile: layer 2 resolves the pair as the reference does (Baseline forces CAVLC, anything but
    // Baseline / Main / High counts as unspecified: encoder_ext.cpp:126-141,652-664)
    key.entropy_cabac = p->iEntropyCodingModeFlag != 0 ? 1 : 0;
    key.profile_idc = (int)l.uiProfileIdc;
    key.dbk_idc = p->iLoopFilterDisableIdc; key.dbk_alpha = p->iLoopFilterAlphaC0Offset; key.dbk_beta = p->iLoopFilterBetaOffset;
    key.intra_period = p->uiIntraPeriod == (unsigned int)-1 ? 0 : (int)p->uiIntraPeriod;       // param_svc.h:370-372 (GOP size 1: no rounding)
    pool_ = b2wels::Broker::get().attach(key, &slot_);
    if (!pool_ || slot_ < 0) { pool_.reset(); slot_ = -1; return cmMallocMemeError; }
    par_ = *p;
    // what GetOption(ENCODER_OPTION_SVC_ENCODE_PARAM_EXT) reports is the RESOLVED configuration, as with the reference
    // (param_svc.h:370-372, encoder_ext.cpp:126-141,652-664)
    if (par_.uiIntraPeriod == (unsigned int)-1) par_.uiIntraPeriod = 0;
    {
      EProfileIdc& pr = par_.sSpatialLayers[0].uiProfileIdc;
      if (pr != PRO_BASELINE && pr != PRO_MAIN && pr != PRO_HIGH) pr = PRO_UNKNOWN;
      if (pr == PRO_BASELINE) par_.iEntropyCodingModeFlag = 0;
      if (pr == PRO_UNKNOWN) pr = par_.iEntropyCodingModeFlag ? PRO_HIGH : PRO_BASELINE;
    }
    w_ = key.width; h_ = key.height;
    return cmResultSuccess;
  }

  int EXTAPI GetDefaultParams(SEncParamExt* p) override {
    if (!p) return cmInitParaError;
    default_params(p);
    return cmResultSuccess;
  }

  int EXTAPI Uninitialize() override {
    if (pool_) { b2wels::Broker::get().detach(pool_, slot_); pool_.reset(); slot_ = -1; }
    return cmResultSuccess;
  }

  int EXTAPI EncodeFrame(const SSourcePicture* pic, SFrameBSInfo* info) override {
    if (!pool_ || !pic || !info) return cmInitParaError;            // welsEncoderExt.cpp:376-379
    if (pic->iColorFormat != videoFormatI420) return cmInitParaError;   // :380
    if (pic->iPicWidth != w_ || pic->iPicHeight != h_) return cmInitParaError;
    // the caller may reuse its planes after return: gather them (any stride) into this stream's page-locked staging
    // picture, which the batch DMA reads in place
    uint8_t* d = pool_->staging(slot_);
    for (int pl = 0; pl < 3; pl++) {
      const int pw = pl ? w_ / 2 : w_, ph = pl ? h_ / 2 : h_;
      if (!pic->pData[pl] || pic->iStride[pl] < pw) return cmInitParaError;
      if (pic->iStride[pl] == pw) memcpy(d, pic->pData[pl], (size_t)pw * ph);
      else for (int y = 0; y < ph; y++) memcpy(d + (size_t)y * pw, pic->pData[pl] + (size_t)y * pic->iStride[pl], pw);
      d += (size_t)pw * ph;
    }
    bool idr = false;
    if (pool_->upload(slot_) != 0) return cmUnknownReason;
    if (pool_->encode(slot_, &au_, &idr) != 0) return cmUnknownReason;
    fill_info(info, idr, pic->uiTimeStamp);
    return cmResultSuccess;
  }

  int EXTAPI EncodeParameterSets(SFrameBSInfo*) override {
    why("EncodeParameterSets: parameter sets are emitted with every IDR access unit");
    return cmUnsupportedData;
  }

  int EXTAPI ForceIntraFrame(bool idr, int /*layer*/ = -1) override {
    if (!pool_) return 1;
    if (!idr) return 1;                                            // welsEncoderExt.cpp: nothing to do
    return pool_->force_idr(slot_) == 0 ? 0 : 1;
  }

  int EXTAPI SetOption(ENCODER_OPTION id, void* v) override {
    if (!v) return cmInitParaError;
    switch (id) {
      case ENCODER_OPTION_TRACE_LEVEL:
      case ENCODER_OPTION_TRACE_CALLBACK:
      case ENCODER_OPTION_TRACE_CALLBACK_CONTEXT:
        return cmResultSuccess;                                    // this library does not trace
      case ENCODER_OPTION_DATAFORMAT:
        return *(int*)v == videoFormatI420 ? cmResultSuccess : cmInitParaError;
      case ENCODER_OPTION_IDR_INTERVAL: {
        // the period is part of the shared encoder's configuration: it can be set before InitializeExt (through the parameters),
        // a change on a running stream would need the stream to move to another pool
        const int want = *(int*)v == -1 ? 0 : *(int*)v;
        if (want == (int)par_.uiIntraPeriod) return cmResultSuccess;
        why("ENCODER_OPTION_IDR_INTERVAL: changing uiIntraPeriod of a running stream (set it in InitializeExt)");
        return cmUnsupportedData;
      }
      default:
        why("SetOption: option not supported by the constant-QP single-layer pipeline");
        return cmUnsupportedData;
    }
  }

  int EXTAPI GetOption(ENCODER_OPTION id, void* v) override {
    if (!v) return cmInitParaError;
    if (!pool_) return cmInitExpected;
    switch (id) {
      case ENCODER_OPTION_DATAFORMAT: *(int*)v = videoFormatI420; return cmResultSuccess;
      case ENCODER_OPTION_IDR_INTERVAL: *(int*)v = (int)par_.uiIntraPeriod; return cmResultSuccess;
      case ENCODER_OPTION_SVC_ENCODE_PARAM_EXT: *(SEncParamExt*)v = par_; return cmResultSuccess;
      case ENCODER_OPTION_FRAME_RATE: *(float*)v = par_.fMaxFrameRate; return cmResultSuccess;
      default: return cmInitParaError;
    }
  }

 private:
  // values of SWelsSvcCodingParam::FillDefault (codec/encoder/core/inc/param_svc.h:132-217)
  static void default_params(SEncParamExt* p) {
    memset(p, 0, sizeof(*p));
    p->iUsageType = CAMERA_VIDEO_REAL_TIME;
    p->iNumRefFrame = AUTO_REF_PIC_COUNT;
    p->fMaxFrameRate = (float)kMaxFps;
    p->iComplexityMode = LOW_COMPLEXITY;
    p->iTargetBitrate = p->iMaxBitrate = UNSPECIFIED_BIT_RATE;
    p->iMultipleThreadIdc = 1;
    p->bUseLoadBalancing = true;
    p->iLtrMarkPeriod = 30;
    p->bEnableFrameCroppingFlag = true;
    p->iRCMode = RC_QUALITY_MODE;
    p->bEnableSceneChangeDetect = p->bEnableBackgroundDetection = p->bEnableAdaptiveQuant = p->bEnableFrameSkip = true;
    p->eSpsPpsIdStrategy = INCREASING_ID;
    p->iSpatialLayerNum = p->iTemporalLayerNum = 1;
    p->iMaxQp = 51;
    p->iMinQp = 0;
    p->bFixRCOverShoot = true;
    p->iIdrBitrateRatio = 4 * 100;                       // IDR_BITRATE_RATIO (rc.h:120)
    for (int i = 0; i < MAX_SPATIAL_LAYER_NUM; i++) {
      SSpatialLayerConfig& l = p->sSpatialLayers[i];
      l.uiProfileIdc = PRO_UNKNOWN;
      l.uiLevelIdc = LEVEL_UNKNOWN;
      l.iDLayerQp = 26;                                  // SVC_QUALITY_BASE_QP
      l.fFrameRate = p->fMaxFrameRate;
      l.iMaxSpatialBitrate = UNSPECIFIED_BIT_RATE;
      l.sSliceArgument.uiSliceMode = SM_SINGLE_SLICE;
      l.sSliceArgument.uiSliceSizeConstraint = 1500;
      l.eAspectRatio = ASP_UNSPECIFIED;
      l.uiVideoFormat = VF_UNDEF;
      l.uiColorPrimaries = CP_UNDEF;
      l.uiTransferCharacteristics = TRC_UNDEF;
      l.uiColorMatrix = CM_UNDEF;
    }
  }

  // The access unit is [SPS PPS] slice, each NAL behind a 4-byte start code.  The reference reports an IDR as
  // two layers (parameter sets: NON_VIDEO_CODING_LAYER, then the slice: VIDEO_CODING_LAYER), a P picture as one.
  void fill_info(SFrameBSInfo* info, bool idr, long long ts) {
    memset(info, 0, sizeof(*info));
    nal_len_.clear();
    std::vector<size_t> start;
    for (size_t i = 0; i + 3 < au_.size(); i++)
      if (au_[i] == 0 && au_[i + 1] == 0 && au_[i + 2] == 0 && au_[i + 3] == 1) { start.push_back(i); i += 3; }
    for (size_t k = 0; k < start.size(); k++)
      nal_len_.push_back((int)((k + 1 < start.size() ? start[k + 1] : au_.size()) - start[k]));
    const EVideoFrameType ft = idr ? videoFrameTypeIDR : videoFrameTypeP;
    int layer = 0;
    size_t first_vcl = 0;
    if (idr && nal_len_.size() >= 3) {
      SLayerBSInfo& l = info->sLayerInfo[layer++];
      l.eFrameType = ft;
      l.uiLayerType = NON_VIDEO_CODING_LAYER;
      l.iNalCount = (int)nal_len_.size() - 1;
      l.pNalLengthInByte = nal_len_.data();
      l.pBsBuf = au_.data();
      first_vcl = nal_len_.size() - 1;
    }
    SLayerBSInfo& v = info->sLayerInfo[layer++];
    v.eFrameType = ft;
    v.uiLayerType = VIDEO_CODING_LAYER;
    v.iNalCount = (int)(nal_len_.size() - first_vcl);
    v.pNalLengthInByte = nal_len_.data() + first_vcl;
    v.pBsBuf = au_.data() + (first_vcl ? start[first_vcl] : 0);
    info->iLayerNum = layer;
    info->eFrameType = ft;
    info->iFrameSizeInBytes = (int)au_.size();
    info->uiTimeStamp = ts;
  }

  std::shared_ptr<b2wels::Pool> pool_;
  int slot_ = -1;
  SEncParamExt par_;
  int w_ = 0, h_ = 0;
  std::vector<uint8_t> au_;
  std::vector<int> nal_len_;
};

}  // namespace

extern "C" {

int WelsCreateSVCEncoder(ISVCEncoder** pp) {
  if (!pp) return 1;
  *pp = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
    fprintf(stderr, "[b2h264] WelsCreateSVCEncoder: no CUDA device — this library has no CPU path\n");
    return 1;
  }
  *pp = new B2Encoder();
  return 0;
}

void WelsDestroySVCEncoder(ISVCEncoder* p) { delete static_cast<B2Encoder*>(p); }

// WelsCreateDecoder / WelsDestroyDecoder / WelsGetDecoderCapability: wels_decoder.cpp

OpenH264Version WelsGetCodecVersion(void) {
  OpenH264Version v = {OPENH264_MAJOR, OPENH264_MINOR, OPENH264_REVISION, OPENH264_RESERVED};
  return v;
}
void WelsGetCodecVersionEx(OpenH264Version* v) { if (v) *v = WelsGetCodecVersion(); }

}  // extern "C"
