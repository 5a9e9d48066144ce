"""B slices through the GPU decoder (include/b2h264_codec.h b2h264_dec_*; host: h264_parse.cpp + h264_motion.h resolve both reference
lists of every B macroblock, device: dec_mb.cuh predicts from two lists, enc_deblock.cuh filters with the two-list strength rule):
the reference's own B-frame vectors (test/api/decoder_test.cpp:90-142, committed under tests/golden/conformance_b) must give the
PUBLISHED SHA-1 of their pictures in OUTPUT order.  The decoder returns pictures in decoding order together with their picture
order count (b2h264_dec_last_picture_order); the output order is by count inside every IDR period, as layer 3 delivers them.
(File name: runs after the other GPU tests.)"""
import hashlib
import json
import os

import numpy as np
import pytest

import h264lib

pytestmark = pytest.mark.gpu
ROOT = h264lib.ROOT
CONF_B_DIR = os.path.join(ROOT, "tests", "golden", "conformance_b")


def _fixtures():
    tab = dict((p.split("/")[-1], s) for p, s in json.load(open(os.path.join(ROOT, "tests", "golden", "reference_decoder_hashes.json")))["pairs"])
    return sorted((f, tab[f]) for f in os.listdir(CONF_B_DIR) if f in tab)


def _decode_in_output_order(dec, aus, stream=0, n_streams=1):
    pics, seq = [], 0
    for au in aus:
        units = [None] * n_streams
        units[stream] = au
        p = dec.decode2(units)[stream]
        assert p is not None
        poc, idr, depth = dec.picture_order(stream)
        seq += idr & 1
        pics.append((seq, poc, len(pics), p.copy()))
    pics.sort(key=lambda t: t[:3])
    return [t[3] for t in pics], depth


@pytest.mark.parametrize("name,sha", _fixtures())
def test_gpu_decoder_b_slice_vectors(name, sha):
    from openh264_b200.binding import BatchDecoder, probe_access_unit
    aus = h264lib.split_access_units(open(os.path.join(CONF_B_DIR, name), "rb").read())
    w, h = probe_access_unit(aus[0])[:2]
    dec = BatchDecoder(w, h)
    pics, depth = _decode_in_output_order(dec, aus)
    dec.close()
    assert len(pics) == 9 and depth > 0
    hs = hashlib.sha1()
    for p in pics:
        hs.update(p.tobytes())
    assert hs.hexdigest() == sha


def test_gpu_decoder_b_and_p_streams_in_one_batch():
    """a B-frame stream and a Baseline stream of the same size side by side in one batch: the list-1 records travel only for the
    stream that has them, the other stream decodes exactly as alone"""
    from openh264_b200.binding import BatchDecoder, BatchEncoder
    name = "Cisco_Men_whisper_640x320_CAVLC_Bframe_9.264"
    sha = dict(_fixtures())[name]
    aus_b = h264lib.split_access_units(open(os.path.join(CONF_B_DIR, name), "rb").read())
    w, h, n = 640, 320, len(aus_b)
    yuv = h264lib.synth_clip(w, h, n, seed=5, noise=4)
    fsz = w * h * 3 // 2
    enc = BatchEncoder(w, h, qp=27, fps=30.0, n_streams=1)
    aus_p = [enc.encode([yuv[f * fsz:(f + 1) * fsz]])[0][0] for f in range(n)]
    enc.close()
    alone = BatchDecoder(w, h)
    want_p = [alone.decode([au])[0].copy() for au in aus_p]
    alone.close()
    dec = BatchDecoder(w, h, n_streams=2)
    got_b, got_p, seq = [], [], 0
    for k in range(n):
        pb, pp = dec.decode2([aus_b[k], aus_p[k]])
        poc, idr, _ = dec.picture_order(0)
        seq += idr & 1
        got_b.append((seq, poc, k, pb.copy()))
        got_p.append(pp.copy())
        assert dec.picture_order(1)[2] == 0                    # Baseline: no reordering
    dec.close()
    for k in range(n):
        assert np.array_equal(got_p[k], want_p[k]), k
    got_b.sort(key=lambda t: t[:3])
    hs = hashlib.sha1()
    for t in got_b:
        hs.update(t[3].tobytes())
    assert hs.hexdigest() == sha


def _prefixes():
    return sorted(json.load(open(os.path.join(ROOT, "tests", "golden", "high_profile_prefix.json"))).items())


@pytest.mark.parametrize("name,gold", _prefixes())
def test_gpu_decoder_high_profile_prefixes(name, gold):
    """High profile as x264 writes it (the tool set of BASELINE.json configs[3]: 8x8 transform with Intra_8x8, explicit weighted P
    prediction, chroma QP offset, B pyramid, temporal direct prediction, implicit weights; CABAC and CAVLC): the first 14 access units
    of two of the reference's vectors against the unmodified reference decoder's output for the same prefix
    (tests/golden/make_high_profile_fixture.py)"""
    from openh264_b200.binding import BatchDecoder
    aus = h264lib.split_access_units(open(os.path.join(CONF_B_DIR, name), "rb").read())
    assert len(aus) == gold["pictures"]
    dec = BatchDecoder(gold["width"], gold["height"])
    pics, depth = _decode_in_output_order(dec, aus)
    dec.close()
    hs = hashlib.sha1()
    for p in pics:
        hs.update(p.tobytes())
    assert hs.hexdigest() == gold["sha1"]


DEC_ORDER = ["Cisco_Men_whisper_640x320_CAVLC_Bframe_9.264", "Cisco_Men_whisper_640x320_CABAC_Bframe_9.264",
             "VID_1280x544_cabac_temporal_direct_first14.264"]


@pytest.mark.parametrize("name", DEC_ORDER)
def test_isvcdecoder_output_order_same_driver_two_libraries(tmp_path, name):
    """ISVCDecoder on streams whose output order is not the decoding order: the application (tests/wels/wels_dec_driver.cpp,
    NAL by NAL through DecodeFrameNoDelay) with our library gives what it gave with the reference library
    (tests/golden/wels_api.json): identical pictures in identical calls, identical call log (ready flags, time stamps of the pictures
    handed back, DECODER_OPTION_NUM_OF_FRAMES_REMAINING_IN_BUFFER): layer 3 releases pictures by the reference's own rule
    (ReorderPicturesInDisplay, welsDecoderExt.cpp:1139)"""
    from test_wels_api import OURLIB, decode_case, golden
    want = golden("dec_order_" + name)
    assert want["bytes"] > 0
    assert decode_case(OURLIB, str(tmp_path), open(os.path.join(CONF_B_DIR, name), "rb").read()) == want
