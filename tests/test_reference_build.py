"""Pins oracle/_ref — the reference compiled here by oracle/Makefile.ref — against the reference's OWN golden vectors:
every (bitstream, SHA-1 of decoded YUV) pair of test/api/decoder_test.cpp (BASELINE.json configs[0] is the first of
them run through h264dec).  The decoder exercises the reference's motion compensation, IDCT-add and deblocking C
code — the same functions the oracle restatement and the CUDA kernels are compared with — so a build that
reproduces the hashes is the reference.  Needs the compiled reference (skipped elsewhere).
The bitstreams are stored in the repository (tests/golden/make_reference_res_golden.py): whole where they are small, else their
first access units together with what the compiled reference decoded them to when it reproduced the published hash of the
whole stream.  The exception is res/test_scalinglist_jm.264 (High-profile scaling matrices, not on the Baseline path this repo
replaces): the C-only build (USE_ASM=No, nasm is absent from this image) decodes it to f690a3af..., both through h264dec and
through ISVCDecoder::DecodeFrameNoDelay; the test pins that value and says so."""
import hashlib
import json
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
H264DEC = os.path.join(ROOT, "oracle", "_ref", "h264dec_ref")
TABLE = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_decoder_hashes.json")))["pairs"]
RES = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_res.json")))["h264dec"]
C_ONLY_SCALINGLIST = "f690a3af2896a53360215fb5d35016bfd41499b3"


def test_table_is_complete():
    assert len(TABLE) == 51 and ["res/BA_MW_D.264", "afd7a9765961ca241bb4bdf344b31397bec7465a"] in TABLE


@pytest.mark.parametrize("pair", TABLE, ids=[os.path.basename(p[0]) for p in TABLE])
def test_compiled_reference_reproduces_its_decoder_goldens(pair, tmp_path):
    path, sha = pair
    stored = RES[os.path.basename(path)]
    src = os.path.join(ROOT, "tests", "golden", stored["file"])
    if not os.path.exists(H264DEC):
        pytest.skip("the compiled reference (oracle/_ref) is not on this machine")
    out = str(tmp_path / "out.yuv")
    r = subprocess.run([H264DEC, src, out], capture_output=True, text=True, timeout=300)
    assert os.path.exists(out), r.stderr[-500:]
    h = hashlib.sha1()
    with open(out, "rb") as f:
        for chunk in iter(lambda: f.read(1 << 20), b""):
            h.update(chunk)
    assert h.hexdigest() == stored["sha1"]
    if not stored["whole"]:
        return
    if path == "res/test_scalinglist_jm.264":
        assert h.hexdigest() == C_ONLY_SCALINGLIST, "the known deviation of the C-only build changed"
        pytest.xfail("C-only build decodes the scaling-list stream differently from the published hash (see module docstring)")
    assert h.hexdigest() == sha
