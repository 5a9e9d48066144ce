"""Writes tests/golden/wels_api.json and the decoder inputs under tests/golden/wels_api/: what the API-level test applications
(tests/wels, built by build()) produce with the UNMODIFIED reference library (oracle/_ref/libopenh264_ref.so) for every case of
tests/test_wels_api.py and of the ISVCDecoder output-order test in tests/test_zz_gpu_decoder_bslices.py.  Run where the
reference is built:
    python tests/golden/make_wels_api_golden.py
"""
import json
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import h264lib  # noqa: E402
import test_wels_api as T  # noqa: E402
from make_encoder_golden import ref_encode  # noqa: E402
from test_zz_gpu_decoder_bslices import CONF_B_DIR, DEC_ORDER  # noqa: E402


def main():
    assert os.path.exists(T.REFLIB), "build the reference first (make -f oracle/Makefile.ref)"
    lib, gold = T.REFLIB, {}
    os.makedirs(T.GOLDEN_DIR, exist_ok=True)
    with tempfile.TemporaryDirectory() as tmp:
        for p in T.DROP_IN:
            gold[T.enc_key("drop_in", *p)] = T.case_drop_in(lib, tmp, *p)
        for lf in T.LOOP_FILTER:
            gold[T.enc_key("loop_filter", *lf)] = T.case_loop_filter(lib, tmp, lf)
        gold[T.enc_key("intra_period")] = T.case_intra_period(lib, tmp)
        for p in T.ENTROPY_PROFILE:
            gold[T.enc_key("entropy_profile", *p)] = T.case_entropy_profile(lib, tmp, *p)
        for (w, h, n, qp) in T.DEC_DROP_IN:
            bs, _, _ = ref_encode(h264lib.synth_clip(w, h, n, seed=21), w, h, n, qp, 30.0)
            with open(T.dec_input(w, h, n, qp), "wb") as f:
                f.write(bs)
            gold["dec_drop_in_%dx%d_n%d_qp%d" % (w, h, n, qp)] = T.decode_case(lib, tmp, bs)
        for threads, _ in T.BROKER_ENC:
            gold["broker_enc_%d" % threads] = T.case_broker_enc(lib, tmp, threads, None)
        for name in T.DEC_CONFORMANCE:
            bs = open(os.path.join(HERE, "conformance", name), "rb").read()
            gold["dec_conformance_" + name] = T.decode_case(lib, tmp, bs)
        for threads, _ in T.BROKER_DEC:
            gold["broker_dec_%d" % threads] = T.case_broker_dec(lib, tmp, threads, None)
        for name in DEC_ORDER:
            gold["dec_order_" + name] = T.decode_case(lib, tmp, open(os.path.join(CONF_B_DIR, name), "rb").read())
    with open(os.path.join(HERE, "wels_api.json"), "w") as f:
        json.dump(gold, f, indent=1, sort_keys=True)
    print("%d cases" % len(gold))


if __name__ == "__main__":
    main()
