"""Layer 3 (include/b2h264_wels_api.h): the reference's own entry points exported by libopenh264_b200_wels.so.
tests/wels/wels_driver.cpp is an application against the binary interface of libopenh264 (include/b2h264_wels_abi.h)
that dlopen()s the library it is given.  What the same applications produced with the unmodified reference library is
stored in tests/golden/wels_api.json (tests/golden/make_wels_api_golden.py); our library must reproduce it exactly."""
import ctypes as C
import hashlib
import json
import os
import subprocess

import numpy as np
import pytest

import h264lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
APPS = os.path.join(ROOT, "tests", "wels", "build")                  # built by build() (tests/wels/Makefile)
DRIVER = os.path.join(APPS, "wels_driver")
REFLIB = os.path.join(ROOT, "oracle", "_ref", "libopenh264_ref.so")
OURLIB = os.path.join(ROOT, "openh264_b200", "libopenh264_b200_wels.so")
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden", "wels_api")
need_ref = pytest.mark.skipif(not os.path.exists(REFLIB), reason="the compiled reference (oracle/_ref) is not on this machine")


def golden(key):
    """what the test application produced with the unmodified reference library for this case"""
    return json.load(open(os.path.join(ROOT, "tests", "golden", "wels_api.json")))[key]


def sha1(b):
    return hashlib.sha1(b).hexdigest()


def enc_key(tag, *params):
    return "_".join(["enc", tag] + [str(p) for p in params])


def drive(lib, clip, w, h, n, qp, idr_at, tmp, tag, entropy=None, intra_period=None, loop_filter=None):
    yuv = os.path.join(tmp, "in.yuv")
    with open(yuv, "wb") as f:
        f.write(clip.tobytes())
    out, lay = os.path.join(tmp, tag + ".264"), os.path.join(tmp, tag + ".layout")
    extra = [str(entropy[0]), str(entropy[1])] if entropy else []
    if intra_period is not None:
        extra = (extra or ["0", "66"]) + [str(intra_period)]
    if loop_filter is not None:
        extra = (extra + ["0"] if len(extra) == 2 else extra or ["0", "66", "0"]) + [str(v) for v in loop_filter]
    r = subprocess.run([DRIVER, lib, yuv, str(w), str(h), str(n), str(qp), str(idr_at), out, lay] + extra, capture_output=True, text=True,
                       timeout=300)
    return r, (open(out, "rb").read() if os.path.exists(out) else b""), (open(lay).read() if os.path.exists(lay) else "")


def test_exports():
    syms = subprocess.run(["nm", "-D", "--defined-only", OURLIB], capture_output=True, text=True).stdout
    for s in ("WelsCreateSVCEncoder", "WelsDestroySVCEncoder", "WelsCreateDecoder", "WelsDestroyDecoder", "WelsGetDecoderCapability",
              "WelsGetCodecVersion", "WelsGetCodecVersionEx"):           # openh264.def
        assert (" T " + s) in syms, s


@need_ref
def test_driver_with_reference_matches_golden(tmp_path):
    """pins the driver itself: through the reference it reproduces the bitstream ref_encode() gives (encoder.json source)"""
    w, h, n, qp = 176, 144, 5, 26
    clip = h264lib.synth_clip(w, h, n)
    r, bs, lay = drive(REFLIB, clip, w, h, n, qp, -1, str(tmp_path), "ref")
    assert r.returncode == 0, r.stderr
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    from make_encoder_golden import ref_encode
    ref_bs, _, _ = ref_encode(clip, w, h, n, qp, 30.0)
    assert len(ref_bs) > 0 and hashlib.sha1(bs).hexdigest() == hashlib.sha1(bytes(ref_bs)).hexdigest()
    assert "frame 0 type 1 layers 2" in lay and "frame 1 type 3 layers 1" in lay


def test_no_device_fails_loudly(tmp_path):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    clip = h264lib.synth_clip(176, 144, 1)
    r, bs, _ = drive(OURLIB, clip, 176, 144, 1, 26, -1, str(tmp_path), "b2")
    assert r.returncode != 0 and "no CUDA device" in r.stderr and bs == b""


# ---- ISVCEncoder: our library must give what the same application got from the reference (tests/golden/wels_api.json) ----
def encode_case(lib, tmp, clip, w, h, n, qp, idr_at, **kw):
    r, bs, lay = drive(lib, clip, w, h, n, qp, idr_at, tmp, "out", **kw)
    assert r.returncode == 0, r.stderr
    return {"sha1": sha1(bs), "bytes": len(bs), "layout": lay}


DROP_IN = [(176, 144, 6, 26, 3), (320, 192, 5, 32, -1), (640, 368, 4, 22, 2)]
LOOP_FILTER = [(1, 0, 0), (0, 2, -3), (2, -6, 6)]
ENTROPY_PROFILE = [(1, 0), (1, 77), (1, 66), (0, 77), (0, 100)]


def case_drop_in(lib, tmp, w, h, n, qp, idr_at):
    return encode_case(lib, tmp, h264lib.synth_clip(w, h, n, seed=7), w, h, n, qp, idr_at)


def case_loop_filter(lib, tmp, lf):
    w, h, n, qp = 176, 144, 5, 33
    return encode_case(lib, tmp, h264lib.synth_clip(w, h, n, seed=17, noise=6), w, h, n, qp, -1, loop_filter=lf)


def case_intra_period(lib, tmp):
    w, h, n, qp = 176, 144, 9, 29
    return encode_case(lib, tmp, h264lib.synth_clip(w, h, n, seed=13), w, h, n, qp, 4, intra_period=3)


def case_entropy_profile(lib, tmp, cabac, profile):
    w, h, n, qp = 320, 192, 5, 27
    return encode_case(lib, tmp, h264lib.synth_clip(w, h, n, seed=11, noise=5), w, h, n, qp, 3, entropy=(cabac, profile))


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,n,qp,idr_at", DROP_IN)
def test_drop_in_same_driver_two_libraries(tmp_path, w, h, n, qp, idr_at):
    """bitstream and SFrameBSInfo layout / defaults through ISVCEncoder equal the reference's"""
    assert case_drop_in(OURLIB, str(tmp_path), w, h, n, qp, idr_at) == golden(enc_key("drop_in", w, h, n, qp, idr_at))


@pytest.mark.gpu
@pytest.mark.parametrize("lf", LOOP_FILTER)
def test_drop_in_loop_filter_control(tmp_path, lf):
    assert case_loop_filter(OURLIB, str(tmp_path), lf) == golden(enc_key("loop_filter", *lf))


@pytest.mark.gpu
def test_drop_in_intra_period(tmp_path):
    """uiIntraPeriod through ISVCEncoder (with a forced IDR in between, which restarts the period)"""
    assert case_intra_period(OURLIB, str(tmp_path)) == golden(enc_key("intra_period"))


@pytest.mark.gpu
@pytest.mark.parametrize("cabac,profile", ENTROPY_PROFILE)
def test_drop_in_entropy_mode_and_profile(tmp_path, cabac, profile):
    """iEntropyCodingModeFlag / uiProfileIdc through ISVCEncoder: CABAC slice data (High by default, Main on request), Baseline
    forcing CAVLC, Main / High parameter sets over CAVLC"""
    assert case_entropy_profile(OURLIB, str(tmp_path), cabac, profile) == golden(enc_key("entropy_profile", cabac, profile))


# ---- ISVCDecoder object and the batching broker behind ISVCEncoder -------------------------------------------------------
DEC_DRIVER = os.path.join(APPS, "wels_dec_driver")
MT_DRIVER = os.path.join(APPS, "wels_mt_driver")


def drive_dec(lib, bs, tmp, tag):
    src = os.path.join(tmp, tag + ".264")
    with open(src, "wb") as f:
        f.write(bs)
    out, log = os.path.join(tmp, tag + ".yuv"), os.path.join(tmp, tag + ".log")
    r = subprocess.run([DEC_DRIVER, lib, src, out, log], capture_output=True, text=True, timeout=300)
    return r, (open(out, "rb").read() if os.path.exists(out) else b""), (open(log).read() if os.path.exists(log) else "")


def decode_case(lib, tmp, bs):
    """pictures and call log (states, ready flags, sizes, timestamps, frames left) of one stream through ISVCDecoder"""
    r, yuv, log = drive_dec(lib, bs, tmp, "out")
    assert r.returncode == 0, r.stderr
    return {"sha1": sha1(yuv), "bytes": len(yuv), "log": log}


DEC_DROP_IN = [(176, 144, 6, 26), (640, 360, 4, 34), (180, 148, 3, 20)]


def dec_input(w, h, n, qp):
    """the reference encoder's bitstream of synth_clip(w, h, n, seed=21) at constant QP qp (tests/golden/make_wels_api_golden.py)"""
    return os.path.join(GOLDEN_DIR, "ref_%dx%d_n%d_qp%d.264" % (w, h, n, qp))


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,n,qp", DEC_DROP_IN)
def test_decoder_drop_in_same_driver_two_libraries(tmp_path, w, h, n, qp):
    """ISVCDecoder (Initialize / DecodeFrameNoDelay / GetOption / FlushFrame, SBufferInfo contract): the application, NAL by NAL
    like the reference's h264dec, on a stream of the reference encoder — identical pictures and identical call log as with the
    reference library."""
    got = decode_case(OURLIB, str(tmp_path), open(dec_input(w, h, n, qp), "rb").read())
    want = golden("dec_drop_in_%dx%d_n%d_qp%d" % (w, h, n, qp))
    assert want["bytes"] == n * w * h * 3 // 2
    assert got == want


BROKER_ENC = [(6, 0), (5, 2)]


def case_broker_enc(lib, tmp, threads, slots):
    w, h, n, qp, frames = 320, 192, 8, 27, 7
    clip = h264lib.synth_clip(w, h, n, seed=31)
    yuv = os.path.join(tmp, "clip.yuv")
    open(yuv, "wb").write(clip.tobytes())
    env = dict(os.environ)
    if slots:
        env["B2H264_BROKER_SLOTS"] = str(slots)
    r = subprocess.run([MT_DRIVER, lib, yuv, str(w), str(h), str(n), str(qp), str(threads), str(frames), "0", "3",
                        os.path.join(tmp, "out")], capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stderr + r.stdout
    outs = [open(os.path.join(tmp, "out.%d.264" % t), "rb").read() for t in range(threads)]
    return {"sha1": [sha1(o) for o in outs], "bytes": [len(o) for o in outs]}


@pytest.mark.gpu
@pytest.mark.parametrize("threads,slots", BROKER_ENC)
def test_broker_many_encoder_objects_one_batch(tmp_path, threads, slots):
    """T application threads, each with its own ISVCEncoder object, different phases of the clip: behind the API the
    objects are streams of shared batched encoders (B2H264_BROKER_SLOTS = 2 forces several pools).  Every thread's
    stream must equal what the reference's API produces for the same pictures."""
    want = golden("broker_enc_%d" % threads)
    assert all(b > 0 for b in want["bytes"])
    assert case_broker_enc(OURLIB, str(tmp_path), threads, slots) == want


DEC_CONFORMANCE = ["BA_MW_D.264", "SVA_Base_B.264", "MR1_MW_A.264"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", DEC_CONFORMANCE)
def test_decoder_drop_in_on_conformance_streams(tmp_path, name):
    """the reference's test vectors through ISVCDecoder, one NAL unit per DecodeFrameNoDelay call (several slices per
    picture: the picture appears with its last slice; multiple reference frames): identical pictures and call log as with the
    reference library.  BA_MW_D.264 is BASELINE.json configs[0]."""
    bs = open(os.path.join(ROOT, "tests", "golden", "conformance", name), "rb").read()
    want = golden("dec_conformance_" + name)
    assert want["bytes"] > 0
    assert decode_case(OURLIB, str(tmp_path), bs) == want


MT_DEC_DRIVER = os.path.join(APPS, "wels_mt_dec_driver")
QCIF_STREAMS = ["BA_MW_D.264", "SVA_Base_B.264", "MR1_MW_A.264", "BANM_MW_D.264", "MIDR_MW_D.264", "NRF_MW_E.264"]


def drive_mt_dec(lib, names, threads, outdir, tag, slots=None):
    env = dict(os.environ)
    if slots:
        env["B2H264_BROKER_SLOTS"] = str(slots)
    files = [os.path.join(ROOT, "tests", "golden", "conformance", n) for n in names]
    prefix = os.path.join(outdir, tag + "_")
    r = subprocess.run([MT_DEC_DRIVER, lib, str(threads), "1", prefix] + files, capture_output=True, text=True, env=env, timeout=600)
    pics = [open(prefix + "%d.yuv" % t, "rb").read() if os.path.exists(prefix + "%d.yuv" % t) else b"" for t in range(threads)]
    return r, pics


@need_ref
def test_mt_decoder_driver_with_reference(tmp_path):
    """the multi-object decoder application itself, with the compiled reference: every thread reproduces the published pictures"""
    r, pics = drive_mt_dec(REFLIB, QCIF_STREAMS[:2], 3, str(tmp_path), "ref")
    assert r.returncode == 0, r.stderr
    gold = {os.path.basename(k): v for k, v in json.load(open(os.path.join(ROOT, "tests", "golden", "reference_decoder_hashes.json")))["pairs"]}
    for t, p in enumerate(pics):
        assert hashlib.sha1(p).hexdigest() == gold[QCIF_STREAMS[t % 2]]


BROKER_DEC = [(6, None), (7, 4), (12, 16)]


def case_broker_dec(lib, tmp, threads, slots):
    r, pics = drive_mt_dec(lib, QCIF_STREAMS, threads, tmp, "out", slots)
    assert r.returncode == 0, r.stderr
    return {"sha1": [sha1(p) for p in pics], "bytes": [len(p) for p in pics]}


@pytest.mark.gpu
@pytest.mark.parametrize("threads,slots", BROKER_DEC)
def test_broker_many_decoder_objects_one_batch(tmp_path, threads, slots):
    """T application threads, each with its own ISVCDecoder, decode six different QCIF conformance streams NAL by NAL: the objects
    are streams of shared batched GPU decoders (one pool per picture size, several pools when the slots run out); every thread
    must get exactly the pictures the reference gives it — streams of different length, slice structure and reference-frame
    count in ONE batch, objects dropping out as their files end."""
    want = golden("broker_dec_%d" % threads)
    assert all(b > 0 for b in want["bytes"])
    assert case_broker_dec(OURLIB, str(tmp_path), threads, slots) == want
