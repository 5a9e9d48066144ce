// wels_dec_driver.cpp — TEST INFRASTRUCTURE.  An application written against the reference's public decoder API
// (codec/api/wels/codec_api.h) that dlopen()s "some libopenh264" and decodes an Annex-B file the way the reference's
// own console decoder does (codec/console/dec/src/h264dec.cpp): one NAL unit per DecodeFrameNoDelay call, pictures
// written through the strides SBufferInfo reports.  The tests run the SAME binary with the compiled reference and with
// openh264_b200/libopenh264_b200_wels.so and require identical pictures and an identical call log.
//   wels_dec_driver <lib.so> <in.264> <out.yuv> <out.log>
#include <dlfcn.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "b2h264_wels_abi.h"

typedef long (*create_fn)(ISVCDecoder**);
typedef void (*destroy_fn)(ISVCDecoder*);
typedef int (*cap_fn)(SDecoderCapability*);

int main(int argc, char** argv) {
  if (argc < 5) { fprintf(stderr, "usage: see source\n"); return 2; }
  void* lib = dlopen(argv[1], RTLD_NOW | RTLD_LOCAL);
  if (!lib) { fprintf(stderr, "dlopen: %s\n", dlerror()); return 3; }
  create_fn create = (create_fn)dlsym(lib, "WelsCreateDecoder");
  destroy_fn destroy = (destroy_fn)dlsym(lib, "WelsDestroyDecoder");
  cap_fn cap = (cap_fn)dlsym(lib, "WelsGetDecoderCapability");
  if (!create || !destroy || !cap) { fprintf(stderr, "missing entry points\n"); return 3; }
  FILE* fin = fopen(argv[2], "rb");
  FILE* fout = fopen(argv[3], "wb");
  FILE* flog = fopen(argv[4], "w");
  if (!fin || !fout || !flog) { fprintf(stderr, "cannot open files\n"); return 3; }
  std::vector<unsigned char> bs;
  { unsigned char tmp[65536]; size_t n; while ((n = fread(tmp, 1, sizeof(tmp), fin)) > 0) bs.insert(bs.end(), tmp, tmp + n); }
  SDecoderCapability dc;
  const int cap_rc = cap(&dc);
  fprintf(flog, "capability rc=%d profile=%d level=%d\n", cap_rc, dc.iProfileIdc, dc.iLevelIdc);
  ISVCDecoder* dec = NULL;
  if (create(&dec) || !dec) { fprintf(stderr, "WelsCreateDecoder failed\n"); return 4; }
  unsigned char* dst[3] = {NULL, NULL, NULL};
  SBufferInfo info;
  memset(&info, 0, sizeof(info));
  // before Initialize the decoder must refuse (welsDecoderExt.cpp:739-744)
  fprintf(flog, "uninitialised -> %d\n", (int)dec->DecodeFrameNoDelay(bs.data(), 4, dst, &info));
  SDecodingParam p;
  memset(&p, 0, sizeof(p));
  p.uiTargetDqLayer = (unsigned char)-1;
  p.eEcActiveIdc = ERROR_CON_DISABLE;
  p.sVideoProperty.eVideoBsType = VIDEO_BITSTREAM_DEFAULT;
  long rc = dec->Initialize(&p);
  if (rc) { fprintf(stderr, "Initialize -> %ld\n", rc); return 5; }
  int lvl = WELS_LOG_QUIET;
  dec->SetOption(DECODER_OPTION_TRACE_LEVEL, &lvl);
  // NAL boundaries (3- or 4-byte start codes)
  std::vector<size_t> start;
  for (size_t i = 0; i + 3 < bs.size(); i++) {
    if (bs[i] == 0 && bs[i + 1] == 0 && ((bs[i + 2] == 1) || (bs[i + 2] == 0 && bs[i + 3] == 1))) {
      start.push_back(i);
      i += bs[i + 2] == 1 ? 2 : 3;
    }
  }
  int frames = 0;
  for (size_t k = 0; k < start.size(); k++) {
    const size_t a = start[k], b = k + 1 < start.size() ? start[k + 1] : bs.size();
    memset(&info, 0, sizeof(info));
    info.uiInBsTimeStamp = k;
    dst[0] = dst[1] = dst[2] = NULL;
    const DECODING_STATE st = dec->DecodeFrameNoDelay(bs.data() + a, (int)(b - a), dst, &info);
    fprintf(flog, "nal %d type %d -> state %d ready %d", (int)k, bs[a + (bs[a + 2] == 1 ? 3 : 4)] & 31, (int)st, info.iBufferStatus);
    if (info.iBufferStatus == 1) {
      const SSysMEMBuffer& m = info.UsrData.sSystemBuffer;
      fprintf(flog, " %dx%d fmt %d ts %llu", m.iWidth, m.iHeight, m.iFormat, info.uiOutYuvTimeStamp);
      for (int pl = 0; pl < 3; pl++) {
        const int w = pl ? m.iWidth / 2 : m.iWidth, h = pl ? m.iHeight / 2 : m.iHeight, s = m.iStride[pl ? 1 : 0];
        for (int y = 0; y < h; y++) fwrite(dst[pl] + (size_t)y * s, 1, w, fout);
      }
      frames++;
    }
    int left = -1;
    dec->GetOption(DECODER_OPTION_NUM_OF_FRAMES_REMAINING_IN_BUFFER, &left);
    fprintf(flog, " left %d\n", left);
  }
  memset(&info, 0, sizeof(info));
  fprintf(flog, "flush -> %d ready %d\n", (int)dec->FlushFrame(dst, &info), info.iBufferStatus);
  fprintf(flog, "frames %d\n", frames);
  dec->Uninitialize();
  destroy(dec);
  fclose(fin); fclose(fout); fclose(flog);
  return 0;
}
