// wels_mt_driver.cpp — TEST / BENCH INFRASTRUCTURE.  A multi-threaded application against the reference's public API
// (codec/api/wels/codec_api.h): T threads, each with its OWN ISVCEncoder object (as a conferencing server or a
// transcoding farm would hold them), each coding `frames` pictures of the clip starting `phase * t` pictures in
// (ping-pong order, no scene cuts) through InitializeExt / EncodeFrame.  dlopen()s whichever libopenh264 it is given:
// with the compiled reference every object is a CPU encoder; with libopenh264_b200_wels.so the objects become
// streams of shared batched GPU encoders (openh264_b200/wels/broker.h).  Prints one JSON line with the wall-clock
// frames/s between a start barrier (all encoders initialised and warmed up) and the last EncodeFrame return.
//   wels_mt_driver <lib.so> <clip.yuv> <w> <h> <clip_frames> <qp> <threads> <frames> <warmup> <phase> <out_prefix|->
#include <dlfcn.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <chrono>
#include <condition_variable>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "b2h264_wels_abi.h"

typedef int (*create_fn)(ISVCEncoder**);
typedef void (*destroy_fn)(ISVCEncoder*);

struct Barrier {
  std::mutex m; std::condition_variable cv; int n, count = 0, gen = 0;
  explicit Barrier(int n_) : n(n_) {}
  void wait() {
    std::unique_lock<std::mutex> l(m);
    const int g = gen;
    if (++count == n) { count = 0; gen++; cv.notify_all(); }
    else cv.wait(l, [&] { return gen != g; });
  }
};

int main(int argc, char** argv) {
  if (argc < 12) { fprintf(stderr, "usage: see source\n"); return 2; }
  void* lib = dlopen(argv[1], RTLD_NOW | RTLD_LOCAL);
  if (!lib) { fprintf(stderr, "dlopen: %s\n", dlerror()); return 3; }
  create_fn create = (create_fn)dlsym(lib, "WelsCreateSVCEncoder");
  destroy_fn destroy = (destroy_fn)dlsym(lib, "WelsDestroySVCEncoder");
  if (!create || !destroy) { fprintf(stderr, "missing entry points\n"); return 3; }
  const int w = atoi(argv[3]), h = atoi(argv[4]), clip_n = atoi(argv[5]), qp = atoi(argv[6]), T = atoi(argv[7]);
  const int frames = atoi(argv[8]), warmup = atoi(argv[9]), phase = atoi(argv[10]);
  const std::string prefix = argv[11];
  const size_t fsz = (size_t)w * h * 3 / 2;
  std::vector<unsigned char> clip(fsz * clip_n);
  {
    FILE* f = fopen(argv[2], "rb");
    if (!f || fread(clip.data(), 1, clip.size(), f) != clip.size()) { fprintf(stderr, "cannot read clip\n"); return 3; }
    fclose(f);
  }
  // ping-pong order over the clip: 0 1 .. n-1 n-2 .. 1 0 1 ..
  std::vector<int> seq;
  for (int i = 0; i < clip_n; i++) seq.push_back(i);
  for (int i = clip_n - 2; i > 0; i--) seq.push_back(i);
  Barrier bar(T + 1);
  std::atomic<int> failed(0);
  std::atomic<long long> bytes(0);
  std::vector<std::thread> th;
  for (int t = 0; t < T; t++) {
    th.emplace_back([&, t] {
      ISVCEncoder* enc = NULL;
      bool ok = create(&enc) == 0 && enc;
      if (ok) {
        SEncParamExt p;
        enc->GetDefaultParams(&p);
        p.iUsageType = CAMERA_VIDEO_REAL_TIME;
        p.iPicWidth = w; p.iPicHeight = h;
        p.iTargetBitrate = 5000000;
        p.iRCMode = RC_OFF_MODE;
        p.fMaxFrameRate = 30.0f;
        p.iComplexityMode = HIGH_COMPLEXITY;
        p.iNumRefFrame = 1;
        p.iMultipleThreadIdc = 1;
        p.bEnableFrameSkip = false;
        p.bEnableDenoise = p.bEnableBackgroundDetection = p.bEnableAdaptiveQuant = p.bEnableSceneChangeDetect = false;
        p.sSpatialLayers[0].iVideoWidth = w; p.sSpatialLayers[0].iVideoHeight = h;
        p.sSpatialLayers[0].fFrameRate = 30.0f;
        p.sSpatialLayers[0].iSpatialBitrate = 5000000;
        p.sSpatialLayers[0].iDLayerQp = qp;
        p.sSpatialLayers[0].uiProfileIdc = PRO_BASELINE;
        p.sSpatialLayers[0].sSliceArgument.uiSliceMode = SM_SINGLE_SLICE;
        ok = enc->InitializeExt(&p) == 0;
        int lvl = WELS_LOG_QUIET;
        if (ok) enc->SetOption(ENCODER_OPTION_TRACE_LEVEL, &lvl);
      }
      if (!ok) failed++;
      FILE* fo = (ok && prefix != "-") ? fopen((prefix + "." + std::to_string(t) + ".264").c_str(), "wb") : NULL;
      long long my_bytes = 0;
      for (int i = 0; i < warmup + frames; i++) {
        if (i == warmup) { bar.wait(); bar.wait(); }               // all warmed up -> main takes t0 -> go
        if (!ok) continue;
        const unsigned char* src = clip.data() + fsz * seq[(i + (size_t)phase * t) % seq.size()];
        SSourcePicture pic;
        memset(&pic, 0, sizeof(pic));
        pic.iColorFormat = videoFormatI420;
        pic.iPicWidth = w; pic.iPicHeight = h;
        pic.iStride[0] = w; pic.iStride[1] = pic.iStride[2] = w / 2;
        pic.pData[0] = const_cast<unsigned char*>(src);
        pic.pData[1] = pic.pData[0] + (size_t)w * h;
        pic.pData[2] = pic.pData[1] + (size_t)w * h / 4;
        pic.uiTimeStamp = (long long)(i * 1000.0 / 30.0);
        SFrameBSInfo info;
        memset(&info, 0, sizeof(info));
        if (enc->EncodeFrame(&pic, &info) != 0) { failed++; ok = false; continue; }
        for (int l = 0; l < info.iLayerNum; l++) {
          const SLayerBSInfo& L = info.sLayerInfo[l];
          int sz = 0;
          for (int k = 0; k < L.iNalCount; k++) sz += L.pNalLengthInByte[k];
          if (fo) fwrite(L.pBsBuf, 1, sz, fo);
          if (i >= warmup) my_bytes += sz;
        }
      }
      if (warmup + frames <= warmup) { bar.wait(); bar.wait(); }
      bytes += my_bytes;
      if (fo) fclose(fo);
      bar.wait();                                                 // everybody done -> main takes t1
      if (enc) { enc->Uninitialize(); destroy(enc); }
    });
  }
  bar.wait();
  const auto t0 = std::chrono::steady_clock::now();
  bar.wait();
  bar.wait();
  const double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  for (auto& x : th) x.join();
  printf("{\"threads\": %d, \"frames_per_thread\": %d, \"seconds\": %.6f, \"fps\": %.3f, \"failed\": %d, \"bytes\": %lld}\n", T, frames, secs,
         (double)T * frames / secs, failed.load(), bytes.load());
  return failed.load() ? 6 : 0;
}
