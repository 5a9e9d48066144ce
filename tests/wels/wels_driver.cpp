// wels_driver.cpp — TEST INFRASTRUCTURE.  An application written against the reference's public API
// (codec/api/wels/codec_api.h) that loads "some libopenh264" with dlopen and encodes a clip through
// WelsCreateSVCEncoder / InitializeExt / EncodeFrame.  The tests require openh264_b200/libopenh264_b200_wels.so to
// give the bitstreams and SFrameBSInfo layouts this binary got from the compiled reference (oracle/_ref/libopenh264_ref.so,
// stored in tests/golden/wels_api.json): that is the drop-in claim of include/b2h264_wels_api.h.
//   wels_driver <lib.so> <in.yuv> <w> <h> <frames> <qp> <force_idr_at|-1> <out.264> <out.layout>
#include <dlfcn.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "b2h264_wels_abi.h"

typedef int (*create_fn)(ISVCEncoder**);
typedef void (*destroy_fn)(ISVCEncoder*);

int main(int argc, char** argv) {
  if (argc < 10) { fprintf(stderr, "usage: see source\n"); return 2; }
  void* lib = dlopen(argv[1], RTLD_NOW | RTLD_LOCAL);
  if (!lib) { fprintf(stderr, "dlopen: %s\n", dlerror()); return 3; }
  create_fn create = (create_fn)dlsym(lib, "WelsCreateSVCEncoder");
  destroy_fn destroy = (destroy_fn)dlsym(lib, "WelsDestroySVCEncoder");
  if (!create || !destroy) { fprintf(stderr, "missing entry points\n"); return 3; }
  const int w = atoi(argv[3]), h = atoi(argv[4]), n = atoi(argv[5]), qp = atoi(argv[6]), idr_at = atoi(argv[7]);
  FILE* fin = fopen(argv[2], "rb");
  FILE* fout = fopen(argv[8], "wb");
  FILE* flay = fopen(argv[9], "w");
  if (!fin || !fout || !flay) { fprintf(stderr, "cannot open files\n"); return 3; }
  ISVCEncoder* enc = NULL;
  if (create(&enc) || !enc) { fprintf(stderr, "WelsCreateSVCEncoder failed\n"); return 4; }
  SEncParamExt p;
  enc->GetDefaultParams(&p);
  fprintf(flay, "defaults rc=%d complexity=%d fps=%.1f scd=%d bgd=%d aq=%d skip=%d qp0=%d strategy=%d\n", (int)p.iRCMode,
          (int)p.iComplexityMode, p.fMaxFrameRate, (int)p.bEnableSceneChangeDetect, (int)p.bEnableBackgroundDetection,
          (int)p.bEnableAdaptiveQuant, (int)p.bEnableFrameSkip, p.sSpatialLayers[0].iDLayerQp, (int)p.eSpsPpsIdStrategy);
  p.iUsageType = CAMERA_VIDEO_REAL_TIME;
  p.iPicWidth = w; p.iPicHeight = h;
  p.iTargetBitrate = 5000000;
  p.iRCMode = RC_OFF_MODE;
  p.fMaxFrameRate = 30.0f;
  p.iComplexityMode = HIGH_COMPLEXITY;
  p.iNumRefFrame = 1;
  p.bEnableFrameSkip = false;
  p.bEnableDenoise = p.bEnableBackgroundDetection = p.bEnableAdaptiveQuant = p.bEnableSceneChangeDetect = false;
  p.sSpatialLayers[0].iVideoWidth = w; p.sSpatialLayers[0].iVideoHeight = h;
  p.sSpatialLayers[0].fFrameRate = 30.0f;
  p.sSpatialLayers[0].iSpatialBitrate = 5000000;
  p.sSpatialLayers[0].iDLayerQp = qp;
  p.sSpatialLayers[0].uiProfileIdc = PRO_BASELINE;
  if (argc > 11) {                       // optional: iEntropyCodingModeFlag and uiProfileIdc (0 = PRO_UNKNOWN)
    p.iEntropyCodingModeFlag = atoi(argv[10]);
    p.sSpatialLayers[0].uiProfileIdc = (EProfileIdc)atoi(argv[11]);
  }
  if (argc > 12) p.uiIntraPeriod = (unsigned int)atoi(argv[12]);   // optional: uiIntraPeriod
  if (argc > 15) {                       // optional: iLoopFilterDisableIdc, iLoopFilterAlphaC0Offset, iLoopFilterBetaOffset
    p.iLoopFilterDisableIdc = atoi(argv[13]); p.iLoopFilterAlphaC0Offset = atoi(argv[14]); p.iLoopFilterBetaOffset = atoi(argv[15]);
  }
  p.sSpatialLayers[0].sSliceArgument.uiSliceMode = SM_SINGLE_SLICE;
  int rc = enc->InitializeExt(&p);
  if (rc) { fprintf(stderr, "InitializeExt -> %d\n", rc); return 5; }
  int lvl = WELS_LOG_QUIET;
  enc->SetOption(ENCODER_OPTION_TRACE_LEVEL, &lvl);
  // an unsupported request must be refused, not approximated (only checked on our library by the test)
  const size_t fsz = (size_t)w * h * 3 / 2;
  std::vector<unsigned char> buf(fsz);
  for (int i = 0; i < n; i++) {
    if (fread(buf.data(), 1, fsz, fin) != fsz) break;
    if (i == idr_at) fprintf(flay, "force_idr -> %d\n", enc->ForceIntraFrame(true));
    SSourcePicture pic;
    memset(&pic, 0, sizeof(pic));
    pic.iColorFormat = videoFormatI420;
    pic.iPicWidth = w; pic.iPicHeight = h;
    pic.iStride[0] = w; pic.iStride[1] = pic.iStride[2] = w / 2;
    pic.pData[0] = buf.data();
    pic.pData[1] = pic.pData[0] + (size_t)w * h;
    pic.pData[2] = pic.pData[1] + (size_t)w * h / 4;
    pic.uiTimeStamp = (long long)(i * 1000.0 / 30.0);
    SFrameBSInfo info;
    memset(&info, 0, sizeof(info));
    rc = enc->EncodeFrame(&pic, &info);
    if (rc) { fprintf(stderr, "EncodeFrame -> %d\n", rc); return 6; }
    fprintf(flay, "frame %d type %d layers %d bytes %d ts %lld:", i, (int)info.eFrameType, info.iLayerNum, info.iFrameSizeInBytes,
            info.uiTimeStamp);
    for (int l = 0; l < info.iLayerNum; l++) {
      const SLayerBSInfo& L = info.sLayerInfo[l];
      fprintf(flay, " [lt %d ft %d t%d s%d q%d nals", (int)L.uiLayerType, (int)L.eFrameType, L.uiTemporalId, L.uiSpatialId, L.uiQualityId);
      int sz = 0;
      for (int k = 0; k < L.iNalCount; k++) { fprintf(flay, " %d", L.pNalLengthInByte[k]); sz += L.pNalLengthInByte[k]; }
      fprintf(flay, "]");
      fwrite(L.pBsBuf, 1, sz, fout);
    }
    fprintf(flay, "\n");
  }
  enc->Uninitialize();
  destroy(enc);
  fclose(fin); fclose(fout); fclose(flay);
  return 0;
}
