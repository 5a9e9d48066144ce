// wels_mt_dec_driver.cpp — TEST INFRASTRUCTURE.  A multi-stream application written against the reference's public decoder API
// (codec/api/wels/codec_api.h): T threads, each with its OWN ISVCDecoder object, decode Annex-B files NAL by NAL (thread t takes
// file t mod n) and write their pictures to <prefix><t>.yuv.  The tests run the SAME binary with the compiled reference and with
// openh264_b200/libopenh264_b200_wels.so (whose decoder objects of one picture size share ONE batched GPU decoder) and require
// identical pictures; it also reports the aggregate decoded pictures per second.
//   wels_mt_dec_driver <lib.so> <threads> <repeat> <out_prefix | -> <in1.264> [in2.264 ...]
#include <dlfcn.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <chrono>
#include <string>
#include <thread>
#include <vector>

#include "b2h264_wels_abi.h"

typedef long (*create_fn)(ISVCDecoder**);
typedef void (*destroy_fn)(ISVCDecoder*);

int main(int argc, char** argv) {
  if (argc < 6) { fprintf(stderr, "usage: see source\n"); return 2; }
  void* lib = dlopen(argv[1], RTLD_NOW | RTLD_LOCAL);
  if (!lib) { fprintf(stderr, "dlopen: %s\n", dlerror()); return 3; }
  create_fn create = (create_fn)dlsym(lib, "WelsCreateDecoder");
  destroy_fn destroy = (destroy_fn)dlsym(lib, "WelsDestroyDecoder");
  if (!create || !destroy) { fprintf(stderr, "missing entry points\n"); return 3; }
  const int T = atoi(argv[2]), repeat = atoi(argv[3]);
  const std::string prefix = argv[4];
  std::vector<std::vector<unsigned char>> files;
  for (int i = 5; i < argc; i++) {
    FILE* f = fopen(argv[i], "rb");
    if (!f) { fprintf(stderr, "cannot open %s\n", argv[i]); return 3; }
    std::vector<unsigned char> bs;
    unsigned char tmp[65536]; size_t n;
    while ((n = fread(tmp, 1, sizeof(tmp), f)) > 0) bs.insert(bs.end(), tmp, tmp + n);
    fclose(f);
    files.push_back(bs);
  }
  std::vector<ISVCDecoder*> dec(T, nullptr);
  for (int t = 0; t < T; t++) {
    if (create(&dec[t]) || !dec[t]) { fprintf(stderr, "WelsCreateDecoder failed\n"); return 4; }
    SDecodingParam p;
    memset(&p, 0, sizeof(p));
    p.uiTargetDqLayer = (unsigned char)-1;
    p.eEcActiveIdc = ERROR_CON_DISABLE;
    p.sVideoProperty.eVideoBsType = VIDEO_BITSTREAM_DEFAULT;
    if (dec[t]->Initialize(&p)) { fprintf(stderr, "Initialize failed\n"); return 5; }
    int lvl = WELS_LOG_QUIET;
    dec[t]->SetOption(DECODER_OPTION_TRACE_LEVEL, &lvl);
  }
  std::atomic<long> frames(0), failed(0);
  const auto t0 = std::chrono::steady_clock::now();
  std::vector<std::thread> th;
  for (int t = 0; t < T; t++)
    th.emplace_back([&, t] {
      const std::vector<unsigned char>& bs = files[t % files.size()];
      FILE* fout = prefix == "-" ? nullptr : fopen((prefix + std::to_string(t) + ".yuv").c_str(), "wb");
      std::vector<size_t> start;
      for (size_t i = 0; i + 3 < bs.size(); i++)
        if (bs[i] == 0 && bs[i + 1] == 0 && ((bs[i + 2] == 1) || (bs[i + 2] == 0 && bs[i + 3] == 1))) { start.push_back(i); i += bs[i + 2] == 1 ? 2 : 3; }
      for (int r = 0; r < repeat; r++)                                   // the file again from its first (IDR) unit
        for (size_t k = 0; k < start.size(); k++) {
          const size_t a = start[k], b = k + 1 < start.size() ? start[k + 1] : bs.size();
          unsigned char* dst[3] = {nullptr, nullptr, nullptr};
          SBufferInfo info;
          memset(&info, 0, sizeof(info));
          const DECODING_STATE st = dec[t]->DecodeFrameNoDelay(bs.data() + a, (int)(b - a), dst, &info);
          if (st != dsErrorFree) failed++;
          if (info.iBufferStatus == 1) {
            frames++;
            if (fout) {
              const SSysMEMBuffer& m = info.UsrData.sSystemBuffer;
              for (int pl = 0; pl < 3; pl++) {
                const int w = pl ? m.iWidth / 2 : m.iWidth, h = pl ? m.iHeight / 2 : m.iHeight, s = m.iStride[pl ? 1 : 0];
                for (int y = 0; y < h; y++) fwrite(dst[pl] + (size_t)y * s, 1, w, fout);
              }
            }
          }
        }
      if (fout) fclose(fout);
    });
  for (auto& x : th) x.join();
  const double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  for (int t = 0; t < T; t++) { dec[t]->Uninitialize(); destroy(dec[t]); }
  printf("{\"threads\": %d, \"frames\": %ld, \"failed\": %ld, \"seconds\": %.6f, \"fps\": %.3f}\n", T, frames.load(), failed.load(), secs, frames.load() / secs);
  return failed.load() ? 6 : 0;
}
