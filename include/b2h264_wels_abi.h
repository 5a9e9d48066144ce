/* b2h264_wels_abi.h — the binary interface of libopenh264 (API 2.6) that layer 3 implements
 * (openh264_b200/wels) and that the API-level test applications (tests/wels) are written against.
 *
 * An application built for libopenh264 passes these structures by pointer and calls the objects through
 * their vtables, so what has to match is the memory layout (field order and types, LP64) and the slot order
 * of the virtual functions; the names are the API's so that application code reads the same.  Only the part
 * of the interface this project uses is declared: the enumerations list the values the code refers to, and
 * the sizes are pinned below so that a layout change cannot go unnoticed.  C++ only. */
#ifndef B2H264_WELS_ABI_H
#define B2H264_WELS_ABI_H

#define EXTAPI

#define OPENH264_MAJOR (2)
#define OPENH264_MINOR (6)
#define OPENH264_REVISION (0)
#define OPENH264_RESERVED (2502)

#define MAX_SPATIAL_LAYER_NUM 4
#define MAX_LAYER_NUM_OF_FRAME 128
#define MAX_SLICES_NUM_TMP 35          /* (128 NAL units per layer - 21 kept for parameter sets / SEI / padding) / 3 */
#define AUTO_REF_PIC_COUNT -1
#define UNSPECIFIED_BIT_RATE 0

typedef struct _tagVersion {
  unsigned int uMajor, uMinor, uRevision, uReserved;
} OpenH264Version;

/* ---- return values and states ---- */
typedef enum { cmResultSuccess, cmInitParaError, cmUnknownReason, cmMallocMemeError, cmInitExpected, cmUnsupportedData } CM_RETURN;

typedef enum {
  dsErrorFree = 0x00, dsFramePending = 0x01, dsRefLost = 0x02, dsBitstreamError = 0x04, dsDepLayerLost = 0x08,
  dsNoParamSets = 0x10, dsDataErrorConcealed = 0x20, dsRefListNullPtrs = 0x40,
  dsInvalidArgument = 0x1000, dsInitialOptExpected = 0x2000, dsOutOfMemory = 0x4000, dsDstBufNeedExpan = 0x8000
} DECODING_STATE;

typedef enum { videoFormatI420 = 23 } EVideoFormatType;

typedef enum {
  videoFrameTypeInvalid, videoFrameTypeIDR, videoFrameTypeI, videoFrameTypeP, videoFrameTypeSkip, videoFrameTypeIPMixed
} EVideoFrameType;

/* ---- options (only the ids this project sets or answers; the values are the API's) ---- */
typedef enum {
  ENCODER_OPTION_DATAFORMAT = 0,
  ENCODER_OPTION_IDR_INTERVAL = 1,
  ENCODER_OPTION_SVC_ENCODE_PARAM_EXT = 3,
  ENCODER_OPTION_FRAME_RATE = 4,
  ENCODER_OPTION_TRACE_LEVEL = 25,
  ENCODER_OPTION_TRACE_CALLBACK = 26,
  ENCODER_OPTION_TRACE_CALLBACK_CONTEXT = 27
} ENCODER_OPTION;

typedef enum {
  DECODER_OPTION_END_OF_STREAM = 1,
  DECODER_OPTION_VCL_NAL = 2,
  DECODER_OPTION_TEMPORAL_ID = 3,
  DECODER_OPTION_ERROR_CON_IDC = 8,
  DECODER_OPTION_TRACE_LEVEL = 9,
  DECODER_OPTION_TRACE_CALLBACK = 10,
  DECODER_OPTION_TRACE_CALLBACK_CONTEXT = 11,
  DECODER_OPTION_PROFILE = 14,
  DECODER_OPTION_STATISTICS_LOG_INTERVAL = 16,
  DECODER_OPTION_IS_REF_PIC = 17,
  DECODER_OPTION_NUM_OF_FRAMES_REMAINING_IN_BUFFER = 18,
  DECODER_OPTION_NUM_OF_THREADS = 19
} DECODER_OPTION;

enum { WELS_LOG_QUIET = 0 };

/* ---- encoder parameters ---- */
typedef enum { ERROR_CON_DISABLE = 0 } ERROR_CON_IDC;
typedef enum { NON_VIDEO_CODING_LAYER = 0, VIDEO_CODING_LAYER = 1 } LAYER_TYPE;
typedef enum { VIDEO_BITSTREAM_AVC = 0, VIDEO_BITSTREAM_SVC = 1, VIDEO_BITSTREAM_DEFAULT = VIDEO_BITSTREAM_SVC } VIDEO_BITSTREAM_TYPE;
typedef enum { RC_QUALITY_MODE = 0, RC_OFF_MODE = -1 } RC_MODES;
typedef enum {
  PRO_UNKNOWN = 0, PRO_BASELINE = 66, PRO_MAIN = 77, PRO_HIGH = 100, PRO_SCALABLE_BASELINE = 83, PRO_SCALABLE_HIGH = 86
} EProfileIdc;
typedef enum { LEVEL_UNKNOWN = 0 } ELevelIdc;
typedef enum { SM_SINGLE_SLICE = 0 } SliceModeEnum;
typedef enum { CAMERA_VIDEO_REAL_TIME = 0 } EUsageType;
typedef enum { LOW_COMPLEXITY = 0, MEDIUM_COMPLEXITY = 1, HIGH_COMPLEXITY = 2 } ECOMPLEXITY_MODE;
typedef enum { CONSTANT_ID = 0, INCREASING_ID = 1 } EParameterSetStrategy;
typedef enum { ASP_UNSPECIFIED = 0 } ESampleAspectRatio;
enum { VF_UNDEF = 5, CP_UNDEF = 2, TRC_UNDEF = 2, CM_UNDEF = 2 };      /* "unspecified" codes of the VUI fields (H.264 E.2.1) */

typedef struct {
  SliceModeEnum uiSliceMode;
  unsigned int uiSliceNum;
  unsigned int uiSliceMbNum[MAX_SLICES_NUM_TMP];
  unsigned int uiSliceSizeConstraint;
} SSliceArgument;

typedef struct {
  int iVideoWidth, iVideoHeight;
  float fFrameRate;
  int iSpatialBitrate, iMaxSpatialBitrate;
  EProfileIdc uiProfileIdc;
  ELevelIdc uiLevelIdc;
  int iDLayerQp;
  SSliceArgument sSliceArgument;
  bool bVideoSignalTypePresent;
  unsigned char uiVideoFormat;
  bool bFullRange, bColorDescriptionPresent;
  unsigned char uiColorPrimaries, uiTransferCharacteristics, uiColorMatrix;
  bool bAspectRatioPresent;
  ESampleAspectRatio eAspectRatio;
  unsigned short sAspectRatioExtWidth, sAspectRatioExtHeight;
} SSpatialLayerConfig;

typedef struct TagEncParamBase {
  EUsageType iUsageType;
  int iPicWidth, iPicHeight, iTargetBitrate;
  RC_MODES iRCMode;
  float fMaxFrameRate;
} SEncParamBase;

typedef struct TagEncParamExt {
  EUsageType iUsageType;                 /* the SEncParamBase fields first */
  int iPicWidth, iPicHeight, iTargetBitrate;
  RC_MODES iRCMode;
  float fMaxFrameRate;
  int iTemporalLayerNum, iSpatialLayerNum;
  SSpatialLayerConfig sSpatialLayers[MAX_SPATIAL_LAYER_NUM];
  ECOMPLEXITY_MODE iComplexityMode;
  unsigned int uiIntraPeriod;
  int iNumRefFrame;
  EParameterSetStrategy eSpsPpsIdStrategy;
  bool bPrefixNalAddingCtrl, bEnableSSEI, bSimulcastAVC;
  int iPaddingFlag, iEntropyCodingModeFlag;
  bool bEnableFrameSkip;
  int iMaxBitrate, iMaxQp, iMinQp;
  unsigned int uiMaxNalSize;
  bool bEnableLongTermReference;
  int iLTRRefNum;
  unsigned int iLtrMarkPeriod;
  unsigned short iMultipleThreadIdc;
  bool bUseLoadBalancing;
  int iLoopFilterDisableIdc, iLoopFilterAlphaC0Offset, iLoopFilterBetaOffset;
  bool bEnableDenoise, bEnableBackgroundDetection, bEnableAdaptiveQuant, bEnableFrameCroppingFlag, bEnableSceneChangeDetect,
      bIsLosslessLink, bFixRCOverShoot;
  int iIdrBitrateRatio;
  bool bPsnrY, bPsnrU, bPsnrV;
} SEncParamExt;

/* ---- encoder input / output ---- */
typedef struct Source_Picture_s {
  int iColorFormat;
  int iStride[4];
  unsigned char* pData[4];
  int iPicWidth, iPicHeight;
  long long uiTimeStamp;
  bool bPsnrY, bPsnrU, bPsnrV;
} SSourcePicture;

typedef struct {
  unsigned char uiTemporalId, uiSpatialId, uiQualityId;
  EVideoFrameType eFrameType;
  unsigned char uiLayerType;
  int iSubSeqId;
  int iNalCount;
  int* pNalLengthInByte;
  unsigned char* pBsBuf;
  float rPsnr[3];
} SLayerBSInfo;

typedef struct {
  int iLayerNum;
  SLayerBSInfo sLayerInfo[MAX_LAYER_NUM_OF_FRAME];
  EVideoFrameType eFrameType;
  int iFrameSizeInBytes;
  long long uiTimeStamp;
} SFrameBSInfo;

/* ---- decoder ---- */
typedef struct {
  unsigned int size;
  VIDEO_BITSTREAM_TYPE eVideoBsType;
} SVideoProperty;

typedef struct TagSVCDecodingParam {
  char* pFileNameRestructed;
  unsigned int uiCpuLoad;
  unsigned char uiTargetDqLayer;
  ERROR_CON_IDC eEcActiveIdc;
  bool bParseOnly;
  SVideoProperty sVideoProperty;
} SDecodingParam;

typedef struct TagSysMemBuffer {
  int iWidth, iHeight, iFormat;
  int iStride[2];
} SSysMEMBuffer;

typedef struct TagBufferInfo {
  int iBufferStatus;                     /* 1: a picture is handed back in pDst */
  unsigned long long uiInBsTimeStamp, uiOutYuvTimeStamp;
  union {
    SSysMEMBuffer sSystemBuffer;
  } UsrData;
  unsigned char* pDst[3];
} SBufferInfo;

typedef struct TagDecoderCapability {
  int iProfileIdc, iProfileIop, iLevelIdc, iMaxMbps, iMaxFs, iMaxCpb, iMaxDpb, iMaxBr;
  bool bRedPicCap;
} SDecoderCapability;

typedef struct TagParserBsInfo SParserBsInfo;      /* parse-only mode: not supported, passed through by pointer only */

/* LP64 sizes of the API's structures */
static_assert(sizeof(SSliceArgument) == 152 && sizeof(SSpatialLayerConfig) == 200, "SSpatialLayerConfig layout");
static_assert(sizeof(SEncParamBase) == 24 && sizeof(SEncParamExt) == 924, "SEncParamExt layout");
static_assert(sizeof(SSourcePicture) == 80, "SSourcePicture layout");
static_assert(sizeof(SLayerBSInfo) == 56 && sizeof(SFrameBSInfo) == 7192, "SFrameBSInfo layout");
static_assert(sizeof(SDecodingParam) == 32 && sizeof(SBufferInfo) == 72, "decoder structure layout");
static_assert(sizeof(SDecoderCapability) == 36, "SDecoderCapability layout");

/* ---- the objects: virtual functions in vtable slot order ---- */
class ISVCEncoder {
 public:
  virtual int EXTAPI Initialize(const SEncParamBase* pParam) = 0;
  virtual int EXTAPI InitializeExt(const SEncParamExt* pParam) = 0;
  virtual int EXTAPI GetDefaultParams(SEncParamExt* pParam) = 0;
  virtual int EXTAPI Uninitialize() = 0;
  virtual int EXTAPI EncodeFrame(const SSourcePicture* kpSrcPic, SFrameBSInfo* pBsInfo) = 0;
  virtual int EXTAPI EncodeParameterSets(SFrameBSInfo* pBsInfo) = 0;
  virtual int EXTAPI ForceIntraFrame(bool bIDR, int iLayerId = -1) = 0;
  virtual int EXTAPI SetOption(ENCODER_OPTION eOptionId, void* pOption) = 0;
  virtual int EXTAPI GetOption(ENCODER_OPTION eOptionId, void* pOption) = 0;
  virtual ~ISVCEncoder() {}
};

class ISVCDecoder {
 public:
  virtual long EXTAPI Initialize(const SDecodingParam* pParam) = 0;
  virtual long EXTAPI Uninitialize() = 0;
  virtual DECODING_STATE EXTAPI DecodeFrame(const unsigned char* pSrc, const int iSrcLen, unsigned char** ppDst, int* pStride,
                                            int& iWidth, int& iHeight) = 0;
  virtual DECODING_STATE EXTAPI DecodeFrameNoDelay(const unsigned char* pSrc, const int iSrcLen, unsigned char** ppDst,
                                                   SBufferInfo* pDstInfo) = 0;
  virtual DECODING_STATE EXTAPI DecodeFrame2(const unsigned char* pSrc, const int iSrcLen, unsigned char** ppDst,
                                             SBufferInfo* pDstInfo) = 0;
  virtual DECODING_STATE EXTAPI FlushFrame(unsigned char** ppDst, SBufferInfo* pDstInfo) = 0;
  virtual DECODING_STATE EXTAPI DecodeParser(const unsigned char* pSrc, const int iSrcLen, SParserBsInfo* pDstInfo) = 0;
  virtual DECODING_STATE EXTAPI DecodeFrameEx(const unsigned char* pSrc, const int iSrcLen, unsigned char* pDst, int iDstStride,
                                              int& iDstLen, int& iWidth, int& iHeight, int& iColorFormat) = 0;
  virtual long EXTAPI SetOption(DECODER_OPTION eOptionId, void* pOption) = 0;
  virtual long EXTAPI GetOption(DECODER_OPTION eOptionId, void* pOption) = 0;
  virtual ~ISVCDecoder() {}
};

extern "C" {
int WelsCreateSVCEncoder(ISVCEncoder** ppEncoder);
void WelsDestroySVCEncoder(ISVCEncoder* pEncoder);
int WelsGetDecoderCapability(SDecoderCapability* pDecCapability);
long WelsCreateDecoder(ISVCDecoder** ppDecoder);
void WelsDestroyDecoder(ISVCDecoder* pDecoder);
OpenH264Version WelsGetCodecVersion(void);
void WelsGetCodecVersionEx(OpenH264Version* pVersion);
}

#endif
