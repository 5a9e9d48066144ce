"""Writes tests/golden/reference_res/ and tests/golden/reference_res.json: the data from the reference's own res/ directory that
tests/test_reference_build.py, tests/test_decoder_emu.py and tests/test_encoder_emu.py use, shrunk to fit the repository, and what
the UNMODIFIED reference (oracle/_ref) makes of it.
  "h264dec":  every bitstream of the reference's decoder golden table (reference_decoder_hashes.json) as a file of the repository —
              the whole stream where it is committed or small, else its first access units (at most PREFIX_BYTES, at least one) —
              and the SHA-1 of what the compiled reference decoder (h264dec) outputs for that file; it is checked here that the
              compiled reference reproduces the published hash of every whole stream
  "encode":   SHA-1 and frame sizes of the reference encoder's bitstream for the res/*.yuv clips the encoder tests use
              (the first pictures, plus one: the encoders read the picture after the last one they code; the 1280x720 clip as a
              centred 160x96 crop)
Run where the reference sources and its build exist:
    python tests/golden/make_reference_res_golden.py <reference source tree>
"""
import hashlib
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import h264lib  # noqa: E402
from make_encoder_golden import ref_encode  # noqa: E402

OUT = os.path.join(HERE, "reference_res")
H264DEC = os.path.join(h264lib.REF_DIR, "h264dec_ref")
PREFIX_BYTES, WHOLE_BYTES = 8192, 16384
STORED_PREFIX = {"VID_1280x544_cabac_temporal_direct.264": "conformance_b/VID_1280x544_cabac_temporal_direct_first14.264",
                 "VID_1280x544_cavlc_temporal_direct.264": "conformance_b/VID_1280x544_cavlc_temporal_direct_first14.264",
                 "VID_1920x1080_cabac_temporal_direct.264": "conformance_b/VID_1920x1080_cabac_temporal_direct_first10.264"}
C_ONLY_SCALINGLIST = "f690a3af2896a53360215fb5d35016bfd41499b3"     # see tests/test_reference_build.py
CLIPS = {  # name -> (source, w, h, pictures, crop (x, y, w, h) or None)
    "CiscoVT2people_160x96_6fps_first7.npy": ("res/CiscoVT2people_160x96_6fps.yuv", 160, 96, 7, None),
    "Static_152_100_first9.npy": ("res/Static_152_100.yuv", 152, 100, 9, None),
    "Cisco_Absolute_Power_1280x720_crop160x96_first3.npy": ("res/Cisco_Absolute_Power_1280x720_30fps.yuv", 1280, 720, 3, (560, 312, 160, 96)),
}
ENCODE = [  # (key, clip, w, h, n, qp, fps, entropy)
    ("own_clip_qp26", "../CiscoVT2people_320x192_12fps.yuv", 320, 192, 9, 26, 12.0, (0, 66)),
    ("own_clip_qp34", "../CiscoVT2people_320x192_12fps.yuv", 320, 192, 9, 34, 12.0, (0, 66)),
    ("power_crop_qp30", "Cisco_Absolute_Power_1280x720_crop160x96_first3.npy", 160, 96, 2, 30, 30.0, (0, 66)),
    # five pictures: the sixth of this clip codes to a different size from run to run, in the reference encoder as in ours
    ("vt160_qp24", "CiscoVT2people_160x96_6fps_first7.npy", 160, 96, 5, 24, 30.0, (0, 66)),
    ("static_qp28", "Static_152_100_first9.npy", 152, 100, 8, 28, 30.0, (0, 66)),
    ("vt160_n5_qp24_cabac0", "CiscoVT2people_160x96_6fps_first7.npy", 160, 96, 5, 24, 30.0, (1, 0)),
    ("vt160_n5_qp24_cabac77", "CiscoVT2people_160x96_6fps_first7.npy", 160, 96, 5, 24, 30.0, (1, 77)),
    ("static_qp28_cabac0", "Static_152_100_first9.npy", 152, 100, 8, 28, 30.0, (1, 0)),
    ("static_qp28_cabac77", "Static_152_100_first9.npy", 152, 100, 8, 28, 30.0, (1, 77)),
]


def load_clip(path):
    return np.load(path) if path.endswith(".npy") else np.fromfile(path, dtype=np.uint8)


def h264dec_sha1(path):
    with tempfile.TemporaryDirectory() as tmp:
        out = os.path.join(tmp, "out.yuv")
        subprocess.run([H264DEC, path, out], capture_output=True, timeout=600)
        return hashlib.sha1(open(out, "rb").read() if os.path.exists(out) else b"").hexdigest()


def crop(yuv, w, h, n, x, y, cw, ch):
    out = []
    for f in yuv.reshape(n, -1):
        Y, U, V = f[:w * h].reshape(h, w), f[w * h:w * h * 5 // 4].reshape(h // 2, w // 2), f[w * h * 5 // 4:].reshape(h // 2, w // 2)
        out += [Y[y:y + ch, x:x + cw].ravel(), U[y // 2:(y + ch) // 2, x // 2:(x + cw) // 2].ravel(), V[y // 2:(y + ch) // 2, x // 2:(x + cw) // 2].ravel()]
    return np.concatenate(out)


def main(ref):
    assert os.path.exists(H264DEC), "build the reference first (make -f oracle/Makefile.ref)"
    os.makedirs(OUT, exist_ok=True)
    gold = {"h264dec": {}, "encode": {}}
    committed = {f: "conformance/" + f for f in os.listdir(os.path.join(HERE, "conformance"))}
    committed.update({f: "conformance_b/" + f for f in os.listdir(os.path.join(HERE, "conformance_b"))})
    for path, published in json.load(open(os.path.join(HERE, "reference_decoder_hashes.json")))["pairs"]:
        name, src = os.path.basename(path), os.path.join(ref, path)
        full = h264dec_sha1(src)
        assert full == (C_ONLY_SCALINGLIST if name == "test_scalinglist_jm.264" else published), name
        data = open(src, "rb").read()
        if name in committed:
            rel, whole = committed[name], True
        elif len(data) <= WHOLE_BYTES:
            rel, whole = "reference_res/" + name, True
            open(os.path.join(HERE, rel), "wb").write(data)
        elif name in STORED_PREFIX:
            rel, whole = STORED_PREFIX[name], False
        else:
            aus, keep = h264lib.split_access_units(data), b""
            for au in aus:
                if keep and len(keep) + len(au) > PREFIX_BYTES:
                    break
                keep += au
            rel, whole = "reference_res/" + name, False
            open(os.path.join(HERE, rel), "wb").write(keep)
        got = h264dec_sha1(os.path.join(HERE, rel))
        assert not whole or got == full, name
        gold["h264dec"][name] = {"file": rel, "whole": whole, "sha1": got, "bytes": os.path.getsize(os.path.join(HERE, rel))}
    for name, (src, w, h, n, c) in CLIPS.items():
        yuv = np.fromfile(os.path.join(ref, src), dtype=np.uint8, count=n * w * h * 3 // 2)
        if c:
            yuv = crop(yuv, w, h, n, *c)
        np.save(os.path.join(OUT, name), yuv)                   # .npy: stored as a binary file
    for key, clip, w, h, n, qp, fps, entropy in ENCODE:
        yuv = load_clip(os.path.join(OUT, clip))
        bs, fb, _ = ref_encode(yuv, w, h, n, qp, fps, entropy=entropy)
        gold["encode"][key] = {"clip": clip, "w": w, "h": h, "n": n, "qp": qp, "fps": fps, "entropy": list(entropy),
                               "sha1": hashlib.sha1(bytes(bs)).hexdigest(), "frame_bytes": fb}
    with open(os.path.join(HERE, "reference_res.json"), "w") as f:
        json.dump(gold, f, indent=1, sort_keys=True)
    print("%d decoder streams, %d encodes" % (len(gold["h264dec"]), len(gold["encode"])))


if __name__ == "__main__":
    main(sys.argv[1])
