// wels_decoder.cpp — layer 3: an ISVCDecoder (codec/api/wels/codec_api.h:346-468) over the layer-2 batched decoder
// (include/b2h264_codec.h: b2h264_dec_*).  Behavioural model: CWelsDecoder (codec/decoder/plus/src/welsDecoderExt.cpp):
// Initialize(SDecodingParam*) first (else dsInitialOptExpected, :739-744); DecodeFrameNoDelay / DecodeFrame2 take one
// access unit (or parameter sets alone) with Annex-B start codes and hand back pointers into DECODER-OWNED picture
// memory that stay valid until the next decode call, with the SBufferInfo contract of codec_def.h:197-205; a NULL / 0
// input flushes.  Baseline streams: every access unit with a slice yields its picture in the same call.  Main / High streams
// (B slices reorder the output): pictures are held and released by the reference's own rule (ReorderPicturesInDisplay), copies of
// the held pictures live in this object, NUM_OF_FRAMES_REMAINING_IN_BUFFER counts them, FlushFrame hands them out at the end.
// The picture size comes from the stream: the GPU decoder is (re)created when an SPS announces a new size.
// Stream class: what layer 2 decodes (include/b2h264_codec.h: I, P and B slices with CAVLC or CABAC, 4x4 / 8x8 transform, progressive);
// anything else is refused with dsBitstreamError and a reason on stderr — there is no CPU decoder in this library.
#include <cuda_runtime_api.h>
#include <stdio.h>
#include <string.h>

#include <vector>

#include "b2h264_codec.h"
#include "broker.h"
#include "b2h264_wels_abi.h"

namespace {

class B2Decoder : public ISVCDecoder {
 public:
  ~B2Decoder() override { Uninitialize(); }

  long EXTAPI Initialize(const SDecodingParam* p) override {
    if (!p) return cmInitParaError;
    if (p->bParseOnly) { fprintf(stderr, "[b2h264] ISVCDecoder: bParseOnly is not supported\n"); return cmUnsupportedData; }
    Uninitialize();
    par_ = *p;
    inited_ = true;
    return cmResultSuccess;
  }

  long EXTAPI Uninitialize() override {
    drop_slot();
    w_ = h_ = 0;
    inited_ = false;
    return cmResultSuccess;
  }

  DECODING_STATE EXTAPI DecodeFrame(const unsigned char* src, const int len, unsigned char** dst, int* stride, int& w, int& h) override {
    SBufferInfo bi;
    memset(&bi, 0, sizeof(bi));
    const DECODING_STATE st = DecodeFrame2(src, len, dst, &bi);
    if (bi.iBufferStatus == 1) {
      if (stride) { stride[0] = bi.UsrData.sSystemBuffer.iStride[0]; stride[1] = bi.UsrData.sSystemBuffer.iStride[1]; }
      w = bi.UsrData.sSystemBuffer.iWidth; h = bi.UsrData.sSystemBuffer.iHeight;
    }
    return st;
  }

  DECODING_STATE EXTAPI DecodeFrameNoDelay(const unsigned char* src, const int len, unsigned char** dst, SBufferInfo* info) override {
    // the reference: DecodeFrame2(src) then DecodeFrame2(NULL) OR-ing the results (welsDecoderExt.cpp:720-725); here
    // the first call already delivers the picture and the flush has nothing left
    return DecodeFrame2(src, len, dst, info);
  }

  DECODING_STATE EXTAPI DecodeFrame2(const unsigned char* src, const int len, unsigned char** dst, SBufferInfo* info) override {
    if (!inited_) return dsInitialOptExpected;
    if (!info || !dst) return dsInvalidArgument;
    const unsigned long long ts = info->uiInBsTimeStamp;
    info->iBufferStatus = 0;
    dst[0] = dst[1] = dst[2] = nullptr;
    if (!src || len <= 0) { pending_.clear(); return dsErrorFree; }   // the flushing half of DecodeFrameNoDelay: every access unit is decoded
                                                                      // in the call that completes it; an incomplete one is dropped.  Held
                                                                      // pictures leave through later calls or FlushFrame
    // Applications feed whole access units or, like the reference's console decoder, one NAL unit per call.  A picture may
    // be coded as several slices: units are collected until they cover the picture (layer 2 answers -105 while they do not).
    pending_.insert(pending_.end(), src, src + len);
    int32_t w = 0, h = 0, has_slice = 0;
    int rc = b2h264_dec_probe(pending_.data(), (int32_t)pending_.size(), &w, &h, &has_slice);
    if (rc) { pending_.clear(); return refuse(rc); }
    vcl_ = has_slice;
    if (w > 0 && h > 0 && (w != w_ || h != h_)) {                 // a (new) SPS: a stream slot of the shared decoder of that size
      drop_slot();
      pool_ = b2wels::Broker::get().attach_decoder(w, h, &slot_);
      if (!pool_ || slot_ < 0) { pool_.reset(); slot_ = -1; pending_.clear(); return dsOutOfMemory; }
      pic_ = pool_->picture(slot_);
      w_ = w; h_ = h;
    }
    if (!pool_) { pending_.clear(); return dsNoParamSets; }
    // objects of one picture size are streams of one batched GPU decoder: the units of the callers that arrive together are
    // decoded by one launch (openh264_b200/wels/broker.h); a lone decoder is served at once
    rc = pool_->decode(slot_, pending_.data(), (int32_t)pending_.size());
    const int got0 = rc == 1;
    if (rc >= 0) rc = 0;
    else if (rc <= -1000) rc = -1000 - rc;                       // CUDA error of the call
    if (rc == -105) return dsErrorFree;                           // more slices of this picture to come
    pending_.clear();
    if (rc) return refuse(rc);
    if (got0) {
      frames_++;
      int32_t poc = 0, flags = 0, depth = 0;
      pool_->picture_order(slot_, &poc, &flags, &depth);
      if (flags & 1) seq_++;                                        // an IDR picture starts a new sequence
      if (depth == 0) {                                             // Baseline: decoding order is output order, nothing is held
        hand_out(dst, info, pic_, ts);
        return dsErrorFree;
      }
      // Main / High streams: the reference's output rule (CWelsDecoder::ReorderPicturesInDisplay, welsDecoderExt.cpp:1139): a B
      // picture that continues the run of written pictures leaves at once; everything else is held and the picture with the lowest
      // (sequence, count) leaves when it is known to be next — or, while no B slice has been seen, the earliest decoded one as soon
      // as two are held
      const bool is_b = (flags & 2) != 0;
      if (is_b) has_b_ = true;
      if (is_b && (seq_ == last_out_seq_ ? (have_out_ && poc <= last_out_poc_ + 2) : (seq_ - last_out_seq_ == 1 && poc == 0))) {
        last_out_poc_ = poc; last_out_seq_ = seq_; have_out_ = true;
        hand_out(dst, info, pic_, ts);
        return dsErrorFree;
      }
      Held hp;
      hp.seq = seq_; hp.poc = poc; hp.order = frames_; hp.ts = ts;
      hp.data.assign(pic_, pic_ + (size_t)w_ * h_ * 3 / 2);
      held_.push_back(std::move(hp));
      if (!has_b_ && held_.size() > 1) release_earliest(dst, info);
      else release_reorder(dst, info, false, poc, seq_);
    }
    return dsErrorFree;
  }

  DECODING_STATE EXTAPI FlushFrame(unsigned char** dst, SBufferInfo* info) override {
    if (!inited_) return dsInitialOptExpected;
    if (info) info->iBufferStatus = 0;
    if (dst) dst[0] = dst[1] = dst[2] = nullptr;
    // one held picture per call, as the reference (welsDecoderExt.cpp:926-945: after DECODER_OPTION_END_OF_STREAM)
    if (eos_ && info && dst && !held_.empty()) {
      if (!has_b_) release_earliest(dst, info);
      else release_reorder(dst, info, true, 0, 0);
    }
    return dsErrorFree;
  }

  DECODING_STATE EXTAPI DecodeParser(const unsigned char*, const int, SParserBsInfo*) override {
    fprintf(stderr, "[b2h264] ISVCDecoder::DecodeParser (parse-only mode) is not supported\n");
    return dsInvalidArgument;
  }

  DECODING_STATE EXTAPI DecodeFrameEx(const unsigned char* src, const int len, unsigned char* pdst, int dst_stride, int& dst_len, int& w,
                                      int& h, int& fmt) override {
    // the reference's implementation of this entry point is an empty stub that reports success (welsDecoderExt.cpp)
    (void)src; (void)len; (void)pdst; (void)dst_stride; (void)dst_len; (void)w; (void)h; (void)fmt;
    return dsErrorFree;
  }

  long EXTAPI SetOption(DECODER_OPTION id, void* v) override {
    if (!inited_ && id != DECODER_OPTION_TRACE_LEVEL && id != DECODER_OPTION_TRACE_CALLBACK && id != DECODER_OPTION_TRACE_CALLBACK_CONTEXT)
      return dsInitialOptExpected;
    if (!v) return cmInitParaError;
    switch (id) {
      case DECODER_OPTION_END_OF_STREAM: eos_ = *(bool*)v; return cmResultSuccess;
      case DECODER_OPTION_ERROR_CON_IDC: ec_ = *(int*)v; return cmResultSuccess;      // no concealment here: errors are refused
      case DECODER_OPTION_TRACE_LEVEL:
      case DECODER_OPTION_TRACE_CALLBACK:
      case DECODER_OPTION_TRACE_CALLBACK_CONTEXT:
      case DECODER_OPTION_STATISTICS_LOG_INTERVAL:
        return cmResultSuccess;
      case DECODER_OPTION_NUM_OF_THREADS: return cmResultSuccess;                     // the GPU batch replaces decoder threads
      default: return cmInitParaError;
    }
  }

  long EXTAPI GetOption(DECODER_OPTION id, void* v) override {
    if (!inited_) return dsInitialOptExpected;
    if (!v) return cmInitParaError;
    switch (id) {
      case DECODER_OPTION_END_OF_STREAM: *(int*)v = eos_; return cmResultSuccess;
      case DECODER_OPTION_VCL_NAL: *(int*)v = vcl_; return cmResultSuccess;
      case DECODER_OPTION_TEMPORAL_ID: *(int*)v = 0; return cmResultSuccess;
      case DECODER_OPTION_ERROR_CON_IDC: *(int*)v = ec_; return cmResultSuccess;
      case DECODER_OPTION_NUM_OF_FRAMES_REMAINING_IN_BUFFER: *(int*)v = (int)held_.size(); return cmResultSuccess;
      case DECODER_OPTION_NUM_OF_THREADS: *(int*)v = 0; return cmResultSuccess;
      case DECODER_OPTION_IS_REF_PIC: *(int*)v = 1; return cmResultSuccess;
      case DECODER_OPTION_PROFILE: *(int*)v = 66; return cmResultSuccess;
      default: return cmInitParaError;
    }
  }

 private:
  DECODING_STATE refuse(int rc) {
    const char* what = rc == -101 ? "truncated access unit" : rc == -102 ? "stream feature outside the supported class (I / P / B slices, CAVLC or "
                       "CABAC, 4x4 / 8x8 transform, no scaling lists, progressive, no FMO / ASO)" : rc == -103 ? "invalid syntax"
                       : rc == -104 ? "slice before its parameter sets" : rc == -2 ? "picture size changed without an SPS" : "CUDA / internal error";
    fprintf(stderr, "[b2h264] ISVCDecoder: %s (%d)\n", what, rc);
    return rc == -104 ? dsNoParamSets : rc > 0 ? dsOutOfMemory : dsBitstreamError;
  }

  // ---- output order of Main / High streams (pictures come out of layer 2 in decoding order) ----
  struct Held { int seq, poc; long order; unsigned long long ts; std::vector<uint8_t> data; };
  void hand_out(unsigned char** dst, SBufferInfo* info, uint8_t* pic, unsigned long long ts) {
    info->iBufferStatus = 1;
    info->uiOutYuvTimeStamp = ts;
    info->UsrData.sSystemBuffer.iWidth = w_;
    info->UsrData.sSystemBuffer.iHeight = h_;
    info->UsrData.sSystemBuffer.iFormat = videoFormatI420;
    info->UsrData.sSystemBuffer.iStride[0] = w_;
    info->UsrData.sSystemBuffer.iStride[1] = w_ / 2;
    dst[0] = info->pDst[0] = pic;
    dst[1] = info->pDst[1] = pic + (size_t)w_ * h_;
    dst[2] = info->pDst[2] = dst[1] + (size_t)(w_ / 2) * (h_ / 2);
  }
  void release(size_t k, unsigned char** dst, SBufferInfo* info) {
    last_out_poc_ = held_[k].poc; last_out_seq_ = held_[k].seq; have_out_ = true;
    out_.swap(held_[k].data);                                       // stays valid until the next call that returns a picture
    const unsigned long long ts = held_[k].ts;
    held_.erase(held_.begin() + (long)k);
    hand_out(dst, info, out_.data(), ts);
  }
  void release_earliest(unsigned char** dst, SBufferInfo* info) {   // ReleaseBufferedReadyPictureNoReorder (:1094)
    size_t k = 0;
    for (size_t i = 1; i < held_.size(); i++) if (held_[i].order < held_[k].order) k = i;
    release(k, dst, info);
  }
  void release_reorder(unsigned char** dst, SBufferInfo* info, bool flush, int cur_poc, int cur_seq) {   // ReleaseBufferedReadyPictureReorder (:1024)
    if (held_.empty()) return;
    size_t k = 0;
    for (size_t i = 1; i < held_.size(); i++)
      if (held_[i].seq == held_[k].seq ? held_[i].poc < held_[k].poc : held_[i].seq < held_[k].seq) k = i;
    const bool ready = flush || (have_out_ && held_[k].poc - last_out_poc_ <= 1) || held_[k].poc < cur_poc || held_[k].seq < cur_seq;
    if (ready) release(k, dst, info);
  }
  std::vector<Held> held_;
  std::vector<uint8_t> out_;
  int seq_ = 0, last_out_poc_ = 0, last_out_seq_ = 0;
  bool has_b_ = false, have_out_ = false;

  SDecodingParam par_;
  bool inited_ = false, eos_ = false;
  int ec_ = 0, vcl_ = 0;
  void drop_slot() {
    if (pool_) { b2wels::Broker::get().detach_decoder(pool_, slot_); pool_.reset(); }
    slot_ = -1; pic_ = nullptr;
    held_.clear(); has_b_ = have_out_ = false; seq_ = last_out_seq_ = last_out_poc_ = 0;
  }
  std::shared_ptr<b2wels::DecPool> pool_;
  int slot_ = -1;
  uint8_t* pic_ = nullptr;                // the slot's page-locked output picture (owned by the pool)
  int w_ = 0, h_ = 0;
  long frames_ = 0;
  std::vector<uint8_t> pending_;         // NAL units of a picture whose slices have not all arrived yet
};

}  // namespace

extern "C" {

long WelsCreateDecoder(ISVCDecoder** pp) {
  if (!pp) return 1;
  *pp = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
    fprintf(stderr, "[b2h264] WelsCreateDecoder: no CUDA device — this library has no CPU path\n");
    return 1;
  }
  *pp = new B2Decoder();
  return 0;
}
void WelsDestroyDecoder(ISVCDecoder* p) { delete static_cast<B2Decoder*>(p); }

int WelsGetDecoderCapability(SDecoderCapability* c) {
  if (!c) return 1;
  memset(c, 0, sizeof(*c));
  // the same report as the reference (welsDecoderExt.cpp:1404-1417: Baseline, level 3.2 limits)
  c->iProfileIdc = 66;
  c->iProfileIop = 0xE0;
  c->iLevelIdc = 32;
  c->iMaxMbps = 216000;
  c->iMaxFs = 5120;
  c->iMaxCpb = 20000;
  c->iMaxDpb = 20480;
  c->iMaxBr = 20000;
  c->bRedPicCap = 0;
  return 0;
}

}  // extern "C"
