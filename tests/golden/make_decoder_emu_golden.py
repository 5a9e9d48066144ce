"""Writes tests/golden/decoder_emu.json for tests/test_decoder_emu.py: for every case, the SHA-1 of the UNMODIFIED reference
encoder's stream (oracle/_ref, make_encoder_golden.ref_encode) and the SHA-1 of every picture the unmodified reference decoder
(ISVCDecoder::DecodeFrameNoDelay, test_decoder_emu.ref_decode) makes of it.  Run where the reference is built:
    python tests/golden/make_decoder_emu_golden.py
"""
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import h264lib  # noqa: E402
from make_encoder_golden import ref_encode  # noqa: E402
from test_decoder_emu import CASES, OWN_CLIP, case_key, ref_decode  # noqa: E402


def entry(yuv, w, h, n, qp, fps):
    bs, _, _ = ref_encode(yuv, w, h, n, qp, fps)
    nr, rw, rh, pics = ref_decode(bs)
    assert nr == n and (rw, rh) == (w, h)
    fsz = w * h * 3 // 2
    return {"stream_sha1": hashlib.sha1(bytes(bs)).hexdigest(),
            "pictures": [hashlib.sha1(pics[i * fsz:(i + 1) * fsz].tobytes()).hexdigest() for i in range(n)]}


if __name__ == "__main__":
    assert h264lib.have_ref(), "build the reference first (make -f oracle/Makefile.ref)"
    gold = {case_key(c): entry(h264lib.synth_clip(c[0], c[1], c[2], seed=c[4]), c[0], c[1], c[2], c[3], 30.0) for c in CASES}
    gold["own_clip_320x192_n9_qp28"] = entry(np.fromfile(OWN_CLIP, dtype=np.uint8), 320, 192, 9, 28, 12.0)
    with open(os.path.join(HERE, "decoder_emu.json"), "w") as f:
        json.dump(gold, f, indent=1, sort_keys=True)
    print("%d streams" % len(gold))
