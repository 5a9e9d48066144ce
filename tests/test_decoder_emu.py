"""Decoder construct path, CPU side (groundwork for the next SURVEY section-8 row): the host build of
openh264_b200/csrc/dec_mb.cuh (prediction + dequant + inverse transform + reconstruction from parsed macroblock
records, then the same deblocking code the encoder path uses) behind the host bitstream parser
(openh264_b200/csrc/h264_parse.cpp) must reproduce the reference decoder's pictures bit for bit
(ISVCDecoder::DecodeFrameNoDelay through oracle/_ref, or its stored picture hashes) on streams the REFERENCE ENCODER produced.
The device kernel that batches this stage does not exist yet; the product decoder entry points still fail loudly."""
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import h264lib

ROOT = h264lib.ROOT


@pytest.fixture(scope="module")
def emu():
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "tests", "emu")])
    E = C.CDLL(os.path.join(ROOT, "tests", "emu", "libb2h264_emu.so"))
    E.emu_decode.restype = C.c_int
    E.emu_decode.argtypes = [C.c_void_p, C.c_long, C.c_void_p, C.c_long, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    E.emu_encode.restype = C.c_long
    E.emu_encode.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_long, C.c_void_p, C.c_void_p]
    return E


def ref_decode(bs):
    R = C.CDLL(h264lib.REFSHIM_SO)
    R.ref_decode.argtypes = [C.c_void_p, C.c_long, C.c_void_p, C.c_long, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_double)]
    out = np.zeros(64 << 20, np.uint8)
    w, h, s = C.c_int(), C.c_int(), C.c_double()
    a = np.frombuffer(bs, np.uint8)
    n = R.ref_decode(a.ctypes.data, len(a), out.ctypes.data, out.size, C.byref(w), C.byref(h), C.byref(s))
    return n, w.value, h.value, out[:max(0, n) * w.value * h.value * 3 // 2]


CASES = [(176, 144, 6, 26, 1), (176, 144, 5, 0, 2), (176, 144, 5, 51, 2), (320, 192, 6, 30, 3), (180, 148, 5, 24, 4),
         (16, 16, 4, 26, 5), (640, 360, 4, 34, 6), (64, 256, 4, 18, 7)]


DEC_GOLD = json.load(open(os.path.join(ROOT, "tests", "golden", "decoder_emu.json")))
RES = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_res.json")))["h264dec"]


def reference_stream(emu, key, yuv, w, h, n, qp, fps):
    """the reference encoder's stream of `yuv` and the SHA-1 of every picture the reference decoder makes of it
    (tests/golden/make_decoder_emu_golden.py).  The stream is rebuilt by the host build of the encoder, which reproduces
    the reference encoder bit for bit (tests/test_encoder_emu.py); its SHA-1 is checked against the reference's."""
    from test_encoder_emu import emu_encode
    bs, _ = emu_encode(emu, yuv, w, h, n, qp, fps)
    assert hashlib.sha1(bs).hexdigest() == DEC_GOLD[key]["stream_sha1"]
    return bs, DEC_GOLD[key]["pictures"]


def decode_and_check(emu, bs, w, h, n, want):
    a = np.frombuffer(bs, np.uint8)
    out = np.zeros(n * w * h * 3 // 2 + 64, np.uint8)
    W, H = C.c_int(), C.c_int()
    got_n = emu.emu_decode(a.ctypes.data, len(a), out.ctypes.data, out.size, C.byref(W), C.byref(H))
    assert got_n == n, got_n
    assert (W.value, H.value) == (w, h)
    fsz = w * h * 3 // 2
    for f in range(n):
        assert hashlib.sha1(out[f * fsz:(f + 1) * fsz].tobytes()).hexdigest() == want[f], "picture %d differs" % f


def case_key(case):
    return "%dx%d_n%d_qp%d_s%d" % case


@pytest.mark.parametrize("case", CASES)
def test_host_decoder_matches_reference_decoder(emu, case):
    w, h, n, qp, seed = case
    bs, want = reference_stream(emu, case_key(case), h264lib.synth_clip(w, h, n, seed=seed), w, h, n, qp, 30.0)
    assert len(want) == n
    decode_and_check(emu, bs, w, h, n, want)


OWN_CLIP = os.path.join(ROOT, "tests", "golden", "CiscoVT2people_320x192_12fps.yuv")


def test_host_decoder_on_the_references_own_clip(emu):
    yuv = np.fromfile(OWN_CLIP, dtype=np.uint8)
    bs, want = reference_stream(emu, "own_clip_320x192_n9_qp28", yuv, 320, 192, 9, 28, 12.0)
    decode_and_check(emu, bs, 320, 192, 9, want)


def test_unsupported_streams_are_rejected_not_guessed(emu):
    """a stream with scaling lists (outside the supported class) must come back as a parse error, never as pictures"""
    a = np.fromfile(os.path.join(ROOT, "tests", "golden", "reference_res", "test_scalinglist_jm.264"), dtype=np.uint8)
    out = np.zeros(1 << 20, np.uint8)
    W, H = C.c_int(), C.c_int()
    assert emu.emu_decode(a.ctypes.data, len(a), out.ctypes.data, out.size, C.byref(W), C.byref(H)) < 0


def test_reference_conformance_table_exact_or_rejected(emu):
    """every bitstream of the reference's decoder golden table (test/api/decoder_test.cpp) either decodes to what the reference
    decoder makes of it or is rejected as outside the supported stream class — never a wrong picture.  The streams are the
    stored ones (tests/golden/reference_res.json): whole streams against their PUBLISHED hash, the first access units of the
    long ones against the compiled reference's pictures of the same units"""
    tab = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_decoder_hashes.json")))["pairs"]
    out = np.zeros(400 << 20, np.uint8)
    exact, wrong = [], []
    for path, sha in tab:
        stored = RES[os.path.basename(path)]
        if not stored["whole"]:
            sha = stored["sha1"]
        a = np.fromfile(os.path.join(ROOT, "tests", "golden", stored["file"]), dtype=np.uint8)
        W, H = C.c_int(), C.c_int()
        n = emu.emu_decode(a.ctypes.data, len(a), out.ctypes.data, out.size, C.byref(W), C.byref(H))
        if n < 0:
            continue
        h = hashlib.sha1(out[:n * W.value * H.value * 3 // 2].tobytes()).hexdigest()
        (exact if h == sha else wrong).append(os.path.basename(path))
    assert not wrong, wrong
    assert {"BA1_Sony_D.jsv", "NL1_Sony_D.jsv", "SVA_BA1_B.264", "SVA_NL1_B.264"} <= set(exact)
    # CABAC (I and P slices, several slices per picture, I_PCM under CABAC) and the CAVLC I_PCM / multi-reference streams
    assert {"test_qcif_cabac.264", "test_cif_P_CABAC_slice.264", "test_cif_I_CABAC_slice.264", "test_cif_I_CABAC_PCM.264",
            "CVPCMNL1_SVA_C.264", "MR2_TANDBERG_E.264"} <= set(exact)
    # B slices (spatial direct, one or two lists per partition, B_8x8, B_Skip; pictures that leave in POC order), CAVLC and CABAC
    assert {"Cisco_Men_whisper_640x320_CABAC_Bframe_9.264", "Cisco_Men_whisper_640x320_CAVLC_Bframe_9.264",
            "Cisco_Adobe_PDF_sample_a_1024x768_CAVLC_Bframe_9.264"} <= set(exact)
    # High profile as x264 writes it: 8x8 transform + Intra_8x8, explicit weighted P prediction, chroma QP offset, B pyramids, temporal
    # direct prediction, implicit weights — BASELINE.json configs[3]'s 1080p CABAC stream among them
    assert {"VID_1920x1080_cabac_temporal_direct.264", "VID_1920x1080_cavlc_temporal_direct.264", "VID_1280x720_cabac_temporal_direct.264",
            "VID_1280x720_cavlc_temporal_direct.264", "VID_1280x544_cabac_temporal_direct.264", "VID_1280x544_cavlc_temporal_direct.264"} <= set(exact)
    assert len(exact) >= 49                      # of 51; rejected: scaling lists, SVC subset SPS


@pytest.mark.parametrize("entropy", [(0, 66), (1, 0)])
def test_parser_survives_corrupted_streams(emu, entropy):
    """bit flips, byte substitutions and deletions: the parser / host construct path must return (a picture or an
    error code), never crash; the same parser guards the GPU decoder's input (run under ASan during development)"""
    if not h264lib.have_ref():
        pytest.skip("reference build not on this machine")
    import random
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    from make_encoder_golden import ref_encode
    clip = h264lib.synth_clip(64, 48, 4, seed=3)
    bs = bytes(ref_encode(clip, 64, 48, 4, 24, 30.0, entropy=entropy)[0])
    out = np.zeros(8 << 20, np.uint8)
    rng = random.Random(7)
    seen_error = 0
    for _ in range(600):
        b = bytearray(bs)
        for _ in range(rng.randint(1, 6)):
            k = rng.randrange(len(b))
            mode = rng.randrange(3)
            if mode == 0:
                b[k] ^= 1 << rng.randrange(8)
            elif mode == 1:
                b[k] = rng.randrange(256)
            else:
                del b[k:k + rng.randint(1, 8)]
        a = np.frombuffer(bytes(b), np.uint8)
        W, H = C.c_int(), C.c_int()
        n = emu.emu_decode(a.ctypes.data, len(a), out.ctypes.data, out.size, C.byref(W), C.byref(H))
        seen_error += n < 0
    assert seen_error > 100


def test_writer_parser_round_trip_on_random_records(emu):
    """random macroblock records (every type, random cbp / modes / vectors, levels up to the Baseline escape range,
    changing QP) through the CAVLC writer and back through the parser"""
    emu.emu_roundtrip_random.argtypes = [C.c_uint, C.c_int]
    bad = [s for s in range(150) if emu.emu_roundtrip_random(s, 6) != 0]
    assert not bad, bad


def test_random_streams_host_decoder_vs_reference_decoder(emu):
    """random but conforming streams (all P partition shapes with vectors that leave the picture, intra macroblocks in P
    pictures, per-macroblock QP changes, escape-coded levels): the host build of the construct path and the reference
    decoder must produce the same pictures — this exercises level decoding, MV clipping and mixed-QP deblocking far
    beyond what the encoders emit"""
    if not h264lib.have_ref():
        pytest.skip("reference build not on this machine")
    emu.emu_random_stream.restype = C.c_long
    emu.emu_random_stream.argtypes = [C.c_uint, C.c_int, C.c_void_p, C.c_long]
    R = C.CDLL(h264lib.REFSHIM_SO)
    R.ref_decode.argtypes = [C.c_void_p, C.c_long, C.c_void_p, C.c_long, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_double)]
    buf, o1, o2 = np.zeros(4 << 20, np.uint8), np.zeros(8 << 20, np.uint8), np.zeros(8 << 20, np.uint8)
    n_pic, sz = 6, 6 * 80 * 64 * 3 // 2
    for seed in range(80):
        n = emu.emu_random_stream(seed, n_pic, buf.ctypes.data, buf.size)
        assert n > 0, (seed, n)
        W, H, W2, H2, sec = C.c_int(), C.c_int(), C.c_int(), C.c_int(), C.c_double()
        a = emu.emu_decode(buf.ctypes.data, n, o1.ctypes.data, o1.size, C.byref(W), C.byref(H))
        b = R.ref_decode(buf.ctypes.data, n, o2.ctypes.data, o2.size, C.byref(W2), C.byref(H2), C.byref(sec))
        assert a == n_pic and b == n_pic, (seed, a, b)
        assert np.array_equal(o1[:sz], o2[:sz]), seed


def test_host_decoder_cabac_streams_of_our_encoder(emu):
    """the host build of the encoder writes the same pictures with CAVLC and with CABAC (High and Main parameter sets): the CABAC
    parser + construct path must give the encoder's own reconstruction, i.e. the same pictures as the CAVLC stream decodes to —
    and what the reference decoder makes of the CABAC stream where it is available"""
    emu.emu_encode.restype = C.c_long
    emu.emu_encode.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_long, C.c_void_p, C.c_void_p]
    emu.emu_decode.argtypes = [C.c_void_p, C.c_long, C.c_void_p, C.c_long, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    for (w, h, n, qp, seed, noise) in [(176, 144, 5, 24, 3, 3), (320, 192, 4, 33, 5, 12), (64, 48, 4, 8, 6, 30), (180, 148, 4, 40, 9, 3)]:
        yuv = h264lib.synth_clip(w, h, n, seed=seed, noise=noise)
        pics = []
        for entropy in ((0, 66), (1, 0), (1, 77)):
            emu.emu_set_complexity_low(0)
            emu.emu_set_entropy(*entropy)
            bs, fb, rec = np.zeros(16 << 20, np.uint8), np.zeros(n, np.int32), np.zeros(yuv.size, np.uint8)
            tot = emu.emu_encode(yuv.ctypes.data, w, h, n, qp, 30.0, bs.ctypes.data, bs.size, fb.ctypes.data, rec.ctypes.data)
            assert tot > 0
            out = np.zeros(yuv.size + 64, np.uint8)
            W, H = C.c_int(), C.c_int()
            assert emu.emu_decode(bs.ctypes.data, tot, out.ctypes.data, out.size, C.byref(W), C.byref(H)) == n
            assert (W.value, H.value) == (w, h) and np.array_equal(out[:yuv.size], rec), entropy
            if entropy[0] and h264lib.have_ref():
                nr, rw, rh, want = ref_decode(bs[:tot].tobytes())
                assert nr == n and np.array_equal(want[:yuv.size], rec)
            pics.append(out[:yuv.size].copy())
        emu.emu_set_entropy(0, 66)
        assert np.array_equal(pics[0], pics[1]) and np.array_equal(pics[0], pics[2])


CONF_DIR = os.path.join(ROOT, "tests", "golden", "conformance")


def conformance_fixtures():
    import json
    tab = dict((p.split("/")[-1], s) for p, s in json.load(open(os.path.join(ROOT, "tests", "golden", "reference_decoder_hashes.json")))["pairs"])
    return sorted((f, tab[f]) for f in os.listdir(CONF_DIR) if f in tab)


@pytest.mark.parametrize("name,sha", conformance_fixtures())
def test_host_decoder_on_committed_conformance_streams(emu, name, sha):
    """the reference's own decoder test vectors (test/api/decoder_test.cpp:90-142; committed under tests/golden/conformance):
    several slices per picture, up to 16 reference frames with list modification, sub-macroblock partitions, constrained
    intra prediction, non-reference pictures, QP wrap, per-slice deblocking control — the PUBLISHED SHA-1 of the pictures"""
    import hashlib
    a = np.fromfile(os.path.join(CONF_DIR, name), dtype=np.uint8)
    out = np.zeros(64 << 20, np.uint8)
    W, H = C.c_int(), C.c_int()
    emu.emu_decode.argtypes = [C.c_void_p, C.c_long, C.c_void_p, C.c_long, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    n = emu.emu_decode(a.ctypes.data, len(a), out.ctypes.data, out.size, C.byref(W), C.byref(H))
    assert n > 0, n
    assert hashlib.sha1(out[:n * W.value * H.value * 3 // 2].tobytes()).hexdigest() == sha


CONF_B_DIR = os.path.join(ROOT, "tests", "golden", "conformance_b")


def conformance_b_fixtures():
    import json
    tab = dict((p.split("/")[-1], s) for p, s in json.load(open(os.path.join(ROOT, "tests", "golden", "reference_decoder_hashes.json")))["pairs"])
    return sorted((f, tab[f]) for f in os.listdir(CONF_B_DIR) if f in tab)


@pytest.mark.parametrize("name,sha", conformance_b_fixtures())
def test_host_decoder_on_committed_b_slice_streams(emu, name, sha):
    """the reference's B-frame vectors (test/api/decoder_test.cpp; committed under tests/golden/conformance_b): Main profile, CAVLC and
    CABAC, B slices with spatial direct prediction, one- and two-list partitions, B_8x8, B_Skip; the pictures leave in POC order
    (the B pictures of these streams PRECEDE the IDR picture they follow in the stream) — the PUBLISHED SHA-1 of the output"""
    import hashlib
    a = np.fromfile(os.path.join(CONF_B_DIR, name), dtype=np.uint8)
    out = np.zeros(64 << 20, np.uint8)
    W, H = C.c_int(), C.c_int()
    emu.emu_decode.argtypes = [C.c_void_p, C.c_long, C.c_void_p, C.c_long, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    n = emu.emu_decode(a.ctypes.data, len(a), out.ctypes.data, out.size, C.byref(W), C.byref(H))
    assert n == 9, n
    assert hashlib.sha1(out[:n * W.value * H.value * 3 // 2].tobytes()).hexdigest() == sha


def high_profile_prefixes():
    import json
    return sorted(json.load(open(os.path.join(ROOT, "tests", "golden", "high_profile_prefix.json"))).items())


@pytest.mark.parametrize("name,gold", high_profile_prefixes())
def test_host_decoder_on_committed_high_profile_prefixes(emu, name, gold):
    """the first 14 access units of two of the reference's High-profile vectors (tests/golden/make_high_profile_fixture.py: 8x8 transform,
    Intra_8x8, weighted P prediction, B pyramid, temporal direct, implicit weights; CABAC and CAVLC) against what the unmodified
    reference decoder makes of the same prefix"""
    import hashlib
    a = np.fromfile(os.path.join(CONF_B_DIR, name), dtype=np.uint8)
    out = np.zeros(64 << 20, np.uint8)
    W, H = C.c_int(), C.c_int()
    emu.emu_decode.argtypes = [C.c_void_p, C.c_long, C.c_void_p, C.c_long, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    n = emu.emu_decode(a.ctypes.data, len(a), out.ctypes.data, out.size, C.byref(W), C.byref(H))
    assert n == gold["pictures"] and (W.value, H.value) == (gold["width"], gold["height"])
    assert hashlib.sha1(out[:n * W.value * H.value * 3 // 2].tobytes()).hexdigest() == gold["sha1"]
