"""CPU-side check of the encoder's macroblock pipeline SOURCE: the host emulation build (tests/emu, the same
enc_*.cuh code compiled as a 1-lane warp and run in raster order) must reproduce the reference encoder's
bitstream bit for bit — against the golden SHA-1s generated from the reference (tests/golden/encoder.json) and,
where oracle/_ref exists, against the reference run side by side, and against the reference's bitstreams of its own
res/*.yuv clips (BASELINE.json config 2 among them; stored samples, tests/golden/make_reference_res_golden.py).  The GPU build of the same source is
checked by tests/test_gpu_encoder.py."""
import ctypes as C
import hashlib
import json
import os
import subprocess

import numpy as np
import pytest

import h264lib

ROOT = h264lib.ROOT
GOLD = json.load(open(os.path.join(ROOT, "tests", "golden", "encoder.json")))


@pytest.fixture(scope="module")
def emu():
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "tests", "emu")])
    E = C.CDLL(os.path.join(ROOT, "tests", "emu", "libb2h264_emu.so"))
    E.emu_encode.restype = C.c_long
    E.emu_encode.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_long, C.c_void_p, C.c_void_p]
    return E


def emu_encode(E, yuv, w, h, n, qp, fps, low=False, entropy=(0, 66), intra_period=0, loop_filter=(0, 0, 0)):
    E.emu_set_complexity_low(1 if low else 0)
    E.emu_set_entropy(*entropy)
    E.emu_set_intra_period(intra_period)
    E.emu_set_loop_filter(*loop_filter)
    cap = 32 << 20
    out, fb = np.zeros(cap, np.uint8), np.zeros(n, np.int32)
    tot = E.emu_encode(yuv.ctypes.data, w, h, n, qp, fps, out.ctypes.data, cap, fb.ctypes.data, None)
    assert tot > 0
    return out[:tot].tobytes(), fb.tolist()


@pytest.mark.parametrize("key", [k for k in sorted(GOLD) if not k.startswith("1920") and not k.startswith("1280")])
def test_emu_matches_golden(emu, key):
    w, h = map(int, key.split("_")[0].split("x"))
    n, qp, fps = int(key.split("_n")[1].split("_")[0]), int(key.split("_qp")[1].split("_")[0]), float(key.split("_fps")[1])
    yuv = h264lib.synth_clip(w, h, n)
    assert hashlib.sha1(yuv.tobytes()).hexdigest() == GOLD[key]["yuv_sha1"]
    bs, fb = emu_encode(emu, yuv, w, h, n, qp, fps)
    assert fb == GOLD[key]["frame_bytes"]
    assert hashlib.sha1(bs).hexdigest() == GOLD[key]["sha1"]


RES_ENCODE = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_res.json")))["encode"]


def check_reference_clip(emu, key):
    """the host build on one of the reference's own clips against the reference encoder's bitstream of it"""
    g = RES_ENCODE[key]
    w, h, n = g["w"], g["h"], g["n"]
    path = os.path.join(ROOT, "tests", "golden", "reference_res", g["clip"])                 # n pictures and the next
    yuv = np.load(path) if path.endswith(".npy") else np.fromfile(path, dtype=np.uint8)
    bs, fb = emu_encode(emu, yuv, w, h, n, g["qp"], g["fps"], entropy=tuple(g["entropy"]))
    assert fb == g["frame_bytes"] and hashlib.sha1(bs).hexdigest() == g["sha1"], key


def test_emu_matches_reference_on_its_own_clip(emu):
    for qp in (26, 34):
        check_reference_clip(emu, "own_clip_qp%d" % qp)


EDGE_CASES = [
    # (w, h, n, qp, seed): QP extremes, pictures that need cropping in one or both directions, the smallest
    # picture the encoder accepts, a wide flat one (long rows: long top-right chains), level-1.0 vector limit (qcif)
    (176, 144, 4, 0, 3), (176, 144, 4, 51, 3), (176, 144, 4, 12, 4), (176, 144, 4, 45, 4),
    (180, 148, 4, 26, 5), (164, 130, 4, 30, 6), (16, 16, 4, 26, 7), (32, 18, 4, 20, 8),
    (480, 32, 4, 28, 9), (64, 256, 4, 33, 10), (352, 288, 3, 38, 11),
]


@pytest.mark.parametrize("case", EDGE_CASES)
def test_emu_matches_reference_edge_cases(emu, case):
    """the same macroblock SOURCE the GPU runs, against the compiled reference, on the edge cases the reference's own
    encoder tests sweep (QP range, odd resolutions: test/api/encoder_test.cpp, test/encoder/EncUT_*.cpp)"""
    if not h264lib.have_ref():
        pytest.skip("reference build not on this machine")
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    from make_encoder_golden import ref_encode
    w, h, n, qp, seed = case
    yuv = h264lib.synth_clip(w, h, n, seed=seed)
    ref_bs, ref_fb, _ = ref_encode(yuv, w, h, n, qp, 30.0)
    bs, fb = emu_encode(emu, yuv, w, h, n, qp, 30.0)
    assert fb == ref_fb and bs == bytes(ref_bs)


def test_emu_matches_reference_on_other_reference_clips(emu):
    """more of the reference's own res/*.yuv clips (first pictures; the 1280x720 one as a 160x96 crop)"""
    for key in ("power_crop_qp30", "vt160_qp24", "static_qp28"):
        check_reference_clip(emu, key)


EDGE = json.load(open(os.path.join(ROOT, "tests", "golden", "encoder_edge.json")))


@pytest.mark.parametrize("key", sorted(EDGE["low"]))
def test_emu_low_complexity_matches_reference_golden(emu, key):
    """LOW_COMPLEXITY (SAD mode costs, VAA-driven partitions, pruned I4x4 search) in the host build of the macroblock source
    against goldens generated from the unmodified reference at iComplexityMode = LOW_COMPLEXITY"""
    import numpy as np
    g = EDGE["low"][key]
    if key.startswith("clip"):
        w, h, n, qp, fps = 320, 192, 9, int(key.split("qp")[1]), 12.0
        yuv = np.fromfile(os.path.join(ROOT, "tests", "golden", "CiscoVT2people_320x192_12fps.yuv"), dtype=np.uint8)
    else:
        w, h = map(int, key.split("_")[0].split("x"))
        n, qp = int(key.split("_n")[1].split("_")[0]), int(key.split("_qp")[1].split("_")[0])
        yuv = h264lib.synth_clip(w, h, n, seed=int(key.split("_seed")[1].split("_")[0]), noise=int(key.split("_noise")[1]))
        fps = 30.0
    bs, fb = emu_encode(emu, yuv, w, h, n, qp, fps, low=True)
    assert fb == g["frame_bytes"] and hashlib.sha1(bs).hexdigest() == g["sha1"]


@pytest.mark.parametrize("key", sorted(EDGE["cabac"]))
def test_emu_cabac_matches_reference_golden(emu, key):
    """iEntropyCodingModeFlag = 1: the host CABAC slice writer (csrc/h264_cabac.cpp; High profile by default, Main on request)
    behind the unchanged macroblock pipeline, against goldens from the unmodified reference with the same setting"""
    g = EDGE["cabac"][key]
    prof = int(key.split("_profile")[1].split("_")[0])
    if key.startswith("clip"):
        w, h, n, qp, fps = 320, 192, 9, int(key.split("qp")[1].split("_")[0]), 12.0
        yuv = np.fromfile(os.path.join(ROOT, "tests", "golden", "CiscoVT2people_320x192_12fps.yuv"), dtype=np.uint8)
    else:
        w, h = map(int, key.split("_")[0].split("x"))
        n, qp = int(key.split("_n")[1].split("_")[0]), int(key.split("_qp")[1].split("_")[0])
        yuv = h264lib.synth_clip(w, h, n, seed=int(key.split("_seed")[1].split("_")[0]), noise=int(key.split("_noise")[1].split("_")[0]))
        fps = 30.0
    bs, fb = emu_encode(emu, yuv, w, h, n, qp, fps, low=key.endswith("_low"), entropy=(1, prof))
    assert fb == g["frame_bytes"] and hashlib.sha1(bs).hexdigest() == g["sha1"]


def test_emu_cabac_matches_reference_side_by_side(emu):
    """the same, against the reference's bitstreams of its own clips, both profiles"""
    for key in ("vt160_n5_qp24_cabac0", "vt160_n5_qp24_cabac77", "static_qp28_cabac0", "static_qp28_cabac77"):
        check_reference_clip(emu, key)


@pytest.mark.parametrize("key", sorted(EDGE["intra_period"]))
def test_emu_intra_period_matches_reference_golden(emu, key):
    """uiIntraPeriod: periodic IDR pictures, each with fresh parameter-set ids (INCREASING_ID), frame_num / idr_pic_id restarts"""
    g = EDGE["intra_period"][key]
    w, h = map(int, key.split("_")[0].split("x"))
    f = {k: int(key.split("_" + k)[1].split("_")[0]) for k in ("n", "qp", "seed", "period", "cabac")}
    yuv = h264lib.synth_clip(w, h, f["n"], seed=f["seed"])
    bs, fb = emu_encode(emu, yuv, w, h, f["n"], f["qp"], 30.0, entropy=(f["cabac"], 0 if f["cabac"] else 66), intra_period=f["period"])
    assert fb == g["frame_bytes"] and hashlib.sha1(bs).hexdigest() == g["sha1"]


def _loop_filter_case(key):
    w, h = map(int, key.split("_")[0].split("x"))
    f = {}
    for k in ("n", "qp", "seed", "idc", "a", "b", "cabac"):
        f[k] = int(key.split("_" + k)[1].split("_")[0])
    return w, h, f


@pytest.mark.parametrize("key", sorted(EDGE["loop_filter"]))
def test_emu_loop_filter_control_matches_reference_golden(emu, key):
    """iLoopFilterDisableIdc (1: the reference pictures stay unfiltered; 2 = 0 with one slice) and the alpha / beta offsets"""
    g = EDGE["loop_filter"][key]
    w, h, f = _loop_filter_case(key)
    yuv = h264lib.synth_clip(w, h, f["n"], seed=f["seed"], noise=6)
    bs, fb = emu_encode(emu, yuv, w, h, f["n"], f["qp"], 30.0, entropy=(f["cabac"], 0 if f["cabac"] else 66), loop_filter=(f["idc"], f["a"], f["b"]))
    assert fb == g["frame_bytes"] and hashlib.sha1(bs).hexdigest() == g["sha1"]
