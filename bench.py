#!/usr/bin/env python
"""bench.py — 1080p H.264 encode throughput of the B200 macroblock pipeline (BASELINE.json metric).

A "step" = one batch-frame: every one of the S independent 1080p streams resident on this GPU advances by
one picture (mode decision + ME + transform/quant + reconstruction + deblocking + border expansion on the
GPU, CAVLC on host threads).  Workload = BASELINE.json configs[2]: synthetic 1920x1080 I420, constant
QP 26, camera mode, single slice, complexity HIGH ("full ME": SATD costs, all partitions), IDR + P...

Three measurements per run, all on the same pictures:
  value        layer 2 (b2h264_enc_submit / collect), sources already resident in HBM
  e2e          THE REFERENCE'S OWN API: S application threads, each with its own ISVCEncoder object, calling
               EncodeFrame with host pictures (tests/wels/wels_mt_driver.cpp against libopenh264_b200_wels.so; the
               objects are streams of shared batched encoders, openh264_b200/wels/broker.h); host->device and
               device->host copies inside the timed region
  e2e_layer2   layer 2 with pinned host pictures (what round 1 reported as e2e)
After the timed regions the access units of EVERY stream of every mode are hashed and compared with the unmodified
reference encoder (oracle/_ref) run on the same picture order: "parity_checked" = number of streams compared; a
mismatch fails the run.  A second workload point ("workload_hard": +-8 noise, few skipped macroblocks, ~27x the bits) is reported
next to the headline.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--streams S] [--impl reference] [--dump-outputs DIR]

--dump-outputs DIR writes what the headline (resident) path handed back in its last timed step as DIR/*.npy (see
dump_outputs); the pictures are the same from run to run, so two builds can be compared output for output.

N > 1: one process per GPU under torch.distributed (launched by the driver with torchrun); streams are
independent, there is no data-path collective ("scaling": "weak"); NCCL is used only for the barrier and the
max-over-ranks of the timed interval.
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

W, H, QP, FPS = 1920, 1080, 26, 30.0
CLIP_FRAMES = 16                      # distinct synthetic pictures; played forward/backward (no scene cuts)
PHASE_STEP = 2                        # stream s starts PHASE_STEP * s pictures into the ping-pong order: 15 distinct sequences
HARD_NOISE, HARD_FRAMES = 8, 8        # second workload point: +-8 per-frame noise (~130 KB per P picture = 31 Mbit/s at 30 fps; +-12 gives 400 KB)
ALG_BYTES_PER_MB = 2016               # SURVEY.md §8(d): cur 384 + ref 384 + recon 384 + levels 768 + MVs 64 + meta 32
MBS_PER_FRAME = 120 * 68
FSZ = W * H * 3 // 2
WORKLOAD = "encode synthetic 1920x1080 I420, constant QP 26, camera, single slice, complexity HIGH, CAVLC (BASELINE.json configs[2])"


def ping_pong(n_clip):
    return list(range(n_clip)) + list(range(n_clip - 2, 0, -1))


def stream_frame(seq, s, i):
    """index into the clip of picture i of stream s"""
    return seq[(i + PHASE_STEP * s) % len(seq)]


def host_cores():
    """cores this process may really use: the affinity mask, capped by the cgroup CPU quota"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    for path in ("/sys/fs/cgroup/cpu.max",):
        try:
            q, p = open(path).read().split()[:2]
            if q != "max":
                n = min(n, max(1, int(float(q) / float(p))))
        except Exception:
            pass
    try:
        q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        if q > 0 and p > 0:
            n = min(n, max(1, q // p))
    except Exception:
        pass
    return max(1, n)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)).get("hbm_gbs", 6650.0), "measured"
    return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                o = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                   capture_output=True, text=True, timeout=5).stdout.strip()
                if o:
                    self.rows.append([x.strip() for x in o.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows if len(r) > 2 + i)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(self.rows[0][1]) if self.rows[0][1].isdigit() else None,
                "reasons": reasons}


def make_clip(noise=3, frames=CLIP_FRAMES):
    import h264lib
    return h264lib.synth_clip(W, H, frames, noise=noise)


def ref_shim():
    import h264lib
    R = C.CDLL(h264lib.REFSHIM_SO)
    R.ref_enc_open.restype = C.c_void_p
    R.ref_enc_open.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float]
    R.ref_enc_frames.restype = C.c_long
    R.ref_enc_frames.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_longlong)]
    R.ref_enc_close.argtypes = [C.c_void_p]
    return R


# ---------------------------------------------------------------------------------------------------------------
def ref_threads_fps(R, clip, seq, cores, steps, warmup):
    """`cores` single-threaded reference encoders, one stream each (same phases as the GPU arm), `steps` timed pictures"""
    encs = [R.ref_enc_open(W, H, QP, 2, 1, FPS) for _ in range(cores)]
    ts = [C.c_longlong(0) for _ in range(cores)]
    nbytes = [0] * cores

    def run_steps(lo, hi, count):
        def worker(i):
            for st in range(lo, hi):
                f = stream_frame(seq, i, st)
                n = R.ref_enc_frames(encs[i], clip[f * FSZ:].ctypes.data, W, H, 1, C.byref(ts[i]))
                if count:
                    nbytes[i] += max(0, int(n))
        th = [threading.Thread(target=worker, args=(i,)) for i in range(cores)]
        [t.start() for t in th]
        [t.join() for t in th]

    run_steps(0, warmup, False)
    t0 = time.perf_counter()
    run_steps(warmup, warmup + steps, True)
    dt = time.perf_counter() - t0
    for e in encs:
        R.ref_enc_close(e)
    return cores * steps / dt, dt, sum(nbytes) / max(1, cores * steps)


def reference_arm(args, rank, world):
    """The reference's own CPU encoder (oracle/_ref, unmodified, public API) on the box's host cores: one
    single-threaded encoder instance per usable host core, each coding its own 1080p stream — the same batched
    independent-stream workload as the GPU arm.  A step = 1 picture per stream."""
    if rank != 0:
        return
    import h264lib
    if not h264lib.have_ref():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref not built on this machine"}))
        return
    R = ref_shim()
    cores = min(host_cores(), args.ref_threads or host_cores())
    clip = make_clip()
    seq = ping_pong(CLIP_FRAMES)
    fps, dt, kb = ref_threads_fps(R, clip, seq, cores, args.steps, args.warmup)
    hard = None
    if not args.no_hard:
        hclip = make_clip(HARD_NOISE, HARD_FRAMES)
        hfps, _, hkb = ref_threads_fps(R, hclip, ping_pong(HARD_FRAMES), cores, max(2, args.steps // 4), 2)
        hard = {"generator": "same synthetic generator, +-%d per-frame noise" % HARD_NOISE, "value": hfps, "unit": "frames/s",
                "bitstream_kbytes_per_frame": hkb / 1e3}
    asm = "C-only build (USE_ASM=No: nasm / yasm are absent from this image, the reference's x86 assembly cannot be assembled)"
    print(json.dumps({
        "impl": "reference", "metric": "1080p_encode_fps", "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": WORKLOAD + "; %d independent streams, 1 picture per stream per step" % cores,
                   "streams": cores, "workload_hard": hard},
        "bitstream_kbytes_per_frame": kb / 1e3,
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "reference",
                         "cores_source": "sched_getaffinity capped by the cgroup quota (os.cpu_count() = %d)" % (os.cpu_count() or 0),
                         "sample": "%d single-thread reference encoders, %s, x %d pictures each" % (cores, asm, args.steps)},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def cpu_baseline_sample():
    """reference encoder, 1 thread, bounded sample of the same workload (rank 0, N=1)."""
    import h264lib
    if not h264lib.have_ref():
        return None
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    from make_encoder_golden import ref_encode
    clip = make_clip()
    seq = ping_pong(CLIP_FRAMES)
    n = 24
    yuv = np.concatenate([clip[stream_frame(seq, 0, i) * FSZ:(stream_frame(seq, 0, i) + 1) * FSZ] for i in range(n)])
    _, _, secs = ref_encode(yuv, W, H, n, QP, FPS, complexity=2, threads=1)
    return {"value": n / secs, "unit": "frames/s", "cores": 1, "kind": "reference",
            "sample": "%d pictures of the bench clip through the reference's ISVCEncoder::EncodeFrame, 1 thread, "
                      "C-only build (USE_ASM=No: nasm absent, the SSE2/AVX2 assembly cannot be built here)" % n}


def reference_hashes(clip, seq, n_pictures, classes):
    """SHA-1 of the unmodified reference's bitstream for every phase class (first picture of the stream -> hash)"""
    import h264lib
    if not h264lib.have_ref():
        return None
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    from make_encoder_golden import ref_encode
    out = {}
    for c in classes:
        yuv = np.concatenate([clip[seq[(i + c) % len(seq)] * FSZ:(seq[(i + c) % len(seq)] + 1) * FSZ] for i in range(n_pictures)])
        bs, _, _ = ref_encode(yuv, W, H, n_pictures, QP, FPS, complexity=2, threads=1)
        out[c] = hashlib.sha1(bytes(bs)).hexdigest()
    return out


def ncu_traffic(kernel):
    """per-launch DRAM bytes of `kernel` from the committed ncu capture (profiles/ncu_traffic.json), or None"""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).get(kernel)
    except Exception:
        return None


def mc_sad_roofline(L, local, peak):
    """BASELINE metric 2: the MC+SAD unit (b2h264_k_mc_sad, layer 1) against the HBM roofline.  64 stacked 1080p
    planes (cur + padded ref = 302 MB, larger than L2); algorithmic bytes per MB = 256 cur + 256 ref + 4 K vector +
    4 K cost (SURVEY.md section 8d).  Three points: K = 1 integer vectors, K = 1 quarter-sample vectors, K = 9 mixed."""
    import torch
    from openh264_b200.binding import check
    S, stride, rows_per = 64, 2048, 1152                      # 1088 + 2 x 32 rows of padding per picture
    g = torch.Generator(device="cuda"); g.manual_seed(264)
    cur = torch.randint(0, 256, (S * rows_per, stride), dtype=torch.uint8, device="cuda", generator=g)
    ref = torch.randint(0, 256, (S * rows_per, stride), dtype=torch.uint8, device="cuda", generator=g)
    mbw, mbh = 120, (S * rows_per) // 16 - 4                  # skip two MB rows at either end: the halo stays inside
    o0 = 32 * stride + 32
    n = mbw * mbh
    out = {}
    st = torch.cuda.current_stream().cuda_stream
    for name, k, frac in (("integer", 1, 0), ("quarter", 1, 1), ("mixed9", 9, 2)):
        mv = torch.randint(-8, 9, (n, k, 2), dtype=torch.int16, device="cuda", generator=g) * 4
        if frac == 1:
            mv += torch.randint(0, 4, (n, k, 2), dtype=torch.int16, device="cuda", generator=g)
        elif frac == 2:                                        # candidate 0 integer, the others quarter-sample neighbours of it
            mv = mv[:, :1, :].repeat(1, k, 1)
            mv[:, 1:, :] += torch.randint(-3, 4, (n, k - 1, 2), dtype=torch.int16, device="cuda", generator=g)
        mv = mv.contiguous()
        cost = torch.empty((n, k), dtype=torch.int32, device="cuda")
        run = lambda: check(L.b2h264_k_mc_sad(cur.data_ptr() + o0, stride, ref.data_ptr() + o0, stride, mbw, mbh,
                                              mv.data_ptr(), k, cost.data_ptr(), st))
        for _ in range(3):
            run()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        iters = 10
        e0.record()
        for _ in range(iters):
            run()
        e1.record()
        torch.cuda.synchronize()
        sec = e0.elapsed_time(e1) / 1e3 / iters
        alg = 512 + 8 * k
        gbs = n * alg / sec / 1e9
        out[name] = {"achieved": gbs, "frac": gbs / peak, "us_per_launch": sec * 1e6, "mb_per_launch": n, "candidates_per_mb": k,
                     "alg_bytes_per_mb": alg}
    t = ncu_traffic("k_mc_sad_tma")
    return {"kernel": "k_mc_sad_tma (b2h264_k_mc_sad: 8x4-MB tiles staged by TMA bulk tensor copies, separable half-sample planes per tile)",
            "bound": "hbm", "unit": "GB/s",
            "traffic": t["dram_bytes"] if t and t.get("mb_per_launch") == n else None,
            "peak": peak, "alg_bytes_per_mb": 520, "candidates_per_mb": 1, "achieved": out["integer"]["achieved"],
            "frac": out["integer"]["frac"], "integer_mv": out["integer"], "quarter_pel_mv": out["quarter"], "mixed_9_candidates": out["mixed9"],
            "note": "64 stacked padded 1080p planes per launch (302 MB of pixels, larger than L2)"}


def decode_bench(local, clip, seq, peak, S=256, n_pictures=8):
    """Decoder construct path (b2h264_dec_*: host parse, GPU prediction + residual + deblocking + padding): S copies of a
    1080p stream produced by this library's encoder (IDR + P, the bench clip), one access unit per stream per call.
    fps = pictures per second through b2h264_dec_decode with host bitstreams in and host pictures out (synchronous).
    Algorithmic bytes per macroblock (SURVEY 8d): 2,500 (levels 768, meta ~200, reference 384, write 384, deblock rw 768)."""
    from openh264_b200.binding import BatchEncoder, BatchDecoder
    enc = BatchEncoder(W, H, qp=QP, fps=FPS, n_streams=1, device=local)
    aus = []
    for i in range(n_pictures):
        f = stream_frame(seq, 0, i)
        bs, _ = enc.encode([clip[f * FSZ:(f + 1) * FSZ]])
        aus.append(bytes(bs[0]))
    enc.close()
    dec = BatchDecoder(W, H, n_streams=S, device=local, pinned_output=True)      # pictures into page-locked memory (b2h264_host_alloc)
    dec.decode([aus[0]] * S)                                       # IDR (warm-up)
    dec.decode([aus[1]] * S)
    t0 = time.perf_counter()
    for au in aus[2:]:
        dec.decode([au] * S)
    dt = time.perf_counter() - t0
    dec.close()
    n = (n_pictures - 2) * S
    fps = n / dt
    gbs = fps * MBS_PER_FRAME * 2500 / 1e9
    # CPU reference beside it: the reference decoder, one thread, the same stream
    ref = None
    try:
        import h264lib
        if h264lib.have_ref():
            R = C.CDLL(h264lib.REFSHIM_SO)
            R.ref_decode.argtypes = [C.c_void_p, C.c_long, C.c_void_p, C.c_long, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_double)]
            a = np.frombuffer(b"".join(aus), np.uint8)
            out = np.zeros(n_pictures * FSZ + 64, np.uint8)
            w_, h_, secs = C.c_int(), C.c_int(), C.c_double()
            nf = R.ref_decode(a.ctypes.data, len(a), out.ctypes.data, out.size, C.byref(w_), C.byref(h_), C.byref(secs))
            if nf == n_pictures and secs.value > 0:
                ref = {"value": nf / secs.value, "unit": "frames/s", "cores": 1, "kind": "reference",
                       "sample": "%d pictures through ISVCDecoder::DecodeFrameNoDelay, 1 thread, C-only build" % nf}
    except Exception:
        pass
    return {"metric": "1080p_decode_fps", "value": fps, "unit": "frames/s", "streams": S, "pictures": n, "path": "b2h264_dec_decode (host access units -> host pictures in page-locked memory, synchronous)",
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak, "alg_bytes_per_mb": 2500}, "cpu_baseline": ref}


def api_run(args, local, clip_path, out_prefix, S):
    """S threads x S ISVCEncoder objects through libopenh264_b200_wels.so (the reference's API), timed inside the driver"""
    drv = os.path.join(ROOT, "tests", "wels", "build", "wels_mt_driver")
    lib = os.path.join(ROOT, "openh264_b200", "libopenh264_b200_wels.so")
    if not (os.path.exists(drv) and os.path.exists(lib)):
        return None
    env = dict(os.environ)
    env.setdefault("B2H264_BROKER_SLOTS", str(S))                    # all objects are streams of ONE shared encoder: the kernels are the more
                                                                     # efficient the more streams a launch carries (S / 2 per launch costs ~35 %)
    env["B2H264_DEVICE"] = str(local)
    r = subprocess.run([drv, lib, clip_path, str(W), str(H), str(CLIP_FRAMES), str(QP), str(S), str(args.steps), str(args.warmup),
                        str(PHASE_STEP), out_prefix], capture_output=True, text=True, env=env, timeout=1800)
    if r.returncode != 0:
        return {"error": (r.stderr + r.stdout)[-400:]}
    res = json.loads(r.stdout.strip().splitlines()[-1])
    res["broker_slots"] = int(env["B2H264_BROKER_SLOTS"])
    return res


def dump_outputs(out_dir, aus, frame_types, limit=64_000_000):
    """The access units of one step (one per stream) and their frame types, as float arrays: bitstream.npy = the bytes of the
    dumped streams' access units one after the other, au_bytes.npy = their lengths, streams.npy = the stream indices,
    frame_type.npy = EVideoFrameType per dumped stream.  Streams are taken in a fixed seeded order while their bytes fit
    into `limit` as float32 (at 1080p a step of 256 streams is larger than that)."""
    os.makedirs(out_dir, exist_ok=True)
    pick, total = [], 0
    for s in np.random.RandomState(264).permutation(len(aus)):
        if total + 4 * len(aus[s]) > limit - 1_000_000:        # 1 MB left for the small arrays
            break
        pick.append(int(s))
        total += 4 * len(aus[s])
    pick.sort()
    np.save(os.path.join(out_dir, "bitstream.npy"), np.frombuffer(b"".join(aus[s] for s in pick), np.uint8).astype(np.float32))
    np.save(os.path.join(out_dir, "au_bytes.npy"), np.array([len(aus[s]) for s in pick], np.float64))
    np.save(os.path.join(out_dir, "streams.npy"), np.array(pick, np.float64))
    np.save(os.path.join(out_dir, "frame_type.npy"), np.array([frame_types[s] for s in pick], np.float64))


# ---------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=16)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--streams", type=int, default=256, help="independent 1080p streams per GPU")
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--ref-threads", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-hard", action="store_true", help="skip the second (hard content) workload point")
    ap.add_argument("--no-api", action="store_true", help="skip the run through ISVCEncoder::EncodeFrame")
    ap.add_argument("--no-decode", action="store_true", help="skip the decoder throughput block")
    ap.add_argument("--no-parity", action="store_true", help="skip the reference comparison of the produced bitstreams")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the access units of the last timed step as DIR/*.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from openh264_b200.binding import BatchEncoder, lib
    from openh264_b200 import shard
    torch.cuda.set_device(local)
    shard.init("nccl", torch.device("cuda", local))        # one process per GPU; replicas only (DESIGN.md section 8)
    S = args.streams
    L = lib(local)
    clip_h = make_clip()
    seq = ping_pong(CLIP_FRAMES)
    clip_d = torch.from_numpy(clip_h).cuda()
    clip_pinned = torch.from_numpy(clip_h).pin_memory()
    stream = torch.cuda.Stream()
    n_pictures = args.warmup + args.steps
    ent_threads = min(S, max(8, host_cores() // max(1, min(world, torch.cuda.device_count()))))

    def srcs(step, on_dev, clip_dev=None, clip_pin=None, sq=None):
        cd, cp, q = clip_dev if clip_dev is not None else clip_d, clip_pin if clip_pin is not None else clip_pinned, sq or seq
        if on_dev:
            base = cd.data_ptr()
            return [base + stream_frame(q, s, step) * FSZ for s in range(S)]
        a = cp.numpy()
        return [a[stream_frame(q, s, step) * FSZ:(stream_frame(q, s, step) + 1) * FSZ] for s in range(S)]

    def timed_run(enc, on_dev, warmup, steps, keep, **kw):
        """pipelined submit/collect (two batches in flight); returns timing + per-stream access units (if keep)"""
        aus = [[] for _ in range(S)] if keep else None
        last = None
        kern, d2h, coded_mbs = [], [], []
        nb = 0

        def loop(first, count, timed):
            nonlocal nb, last
            enc.submit(srcs(first, on_dev, **kw), on_device=on_dev)
            for i in range(1, count + 1):
                if i < count:
                    enc.submit(srcs(first + i, on_dev, **kw), on_device=on_dev)
                bs, ft = enc.collect()
                if keep:
                    for s in range(S):
                        aus[s].append(bs[s])
                if timed:
                    last = (bs, ft)
                    nb += sum(len(b) for b in bs)
                    kern.append(enc.timing_us())
                    d2h.append(enc.d2h_bytes())
                    coded_mbs.append(enc.coded_mbs())
        loop(0, warmup, False)                                     # warm-up (includes the IDR pictures)
        torch.cuda.synchronize()
        shard.barrier()
        sampler = ClockSampler(local)
        sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        with torch.cuda.stream(stream):
            e0.record(stream)
        t0 = time.perf_counter()
        loop(warmup, steps, True)                                  # timed region: exactly `steps` batch-frames
        with torch.cuda.stream(stream):
            e1.record(stream)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        dev = e0.elapsed_time(e1) / 1e3
        sampler.stop_flag = True
        sampler.join(timeout=2)
        dt, pics = shard.job_totals(max(wall, dev), S * steps, device="cuda")   # MAX over ranks / SUM over ranks
        return {"dt": dt, "pictures": pics, "wall": wall, "dev": dev, "bytes": nb, "clocks": sampler.summary(), "kern": kern, "d2h": d2h,
                "coded": coded_mbs, "aus": aus, "last": last}

    results = {}
    launches0 = L.b2h264_launch_count()
    keep = not args.no_parity
    for mode in ("resident", "e2e_layer2"):
        enc = BatchEncoder(W, H, qp=QP, fps=FPS, n_streams=S, device=local, entropy_threads=ent_threads)
        enc.set_stream(stream.cuda_stream)
        results[mode] = timed_run(enc, mode == "resident", args.warmup, args.steps, keep)
        enc.close()
    launches = L.b2h264_launch_count() - launches0

    # ---- the same workload through the reference's API (ISVCEncoder objects behind the batching broker) ----
    api = None
    tmpdir = tempfile.mkdtemp(prefix="b2h264_bench_")
    if not args.no_api:
        clip_path = os.path.join(tmpdir, "clip.yuv")
        clip_h.tofile(clip_path)
        shard.barrier()
        api = api_run(args, local, clip_path, os.path.join(tmpdir, "api") if keep else "-", S)
        ok = bool(api) and "fps" in api
        dt, pics = shard.job_totals(api["seconds"] if ok else 1e9, S * args.steps, device="cuda")   # every rank takes part
        if ok and dt < 1e8:
            api["job_fps"] = pics / dt

    # ---- parity at bench scale: every stream of every mode against the unmodified reference (outside the timed regions) ----
    parity = {"parity_checked": 0, "note": "skipped (--no-parity)"}
    if keep and rank == 0:
        classes = sorted({(PHASE_STEP * s) % len(seq) for s in range(S)})
        want = reference_hashes(clip_h, seq, n_pictures, classes)
        if want is None:
            parity = {"parity_checked": 0, "note": "oracle/_ref not present on this machine"}
        else:
            checked, bad = 0, []
            for mode in ("resident", "e2e_layer2"):
                for s in range(S):
                    got = hashlib.sha1(b"".join(results[mode]["aus"][s])).hexdigest()
                    checked += 1
                    if got != want[(PHASE_STEP * s) % len(seq)]:
                        bad.append((mode, s))
            if api and "fps" in api:
                for s in range(S):
                    got = hashlib.sha1(open(os.path.join(tmpdir, "api.%d.264" % s), "rb").read()).hexdigest()
                    checked += 1
                    if got != want[(PHASE_STEP * s) % len(seq)]:
                        bad.append(("api", s))
            if bad:
                print(json.dumps({"error": "bitstream differs from the reference", "streams": bad[:16], "n_bad": len(bad)}))
                sys.exit(1)
            parity = {"parity_checked": checked, "distinct_sequences": len(classes), "pictures_per_stream": n_pictures,
                      "note": "SHA-1 of all access units of every stream (resident, e2e_layer2%s) == the unmodified reference encoder "
                              "on the same picture order" % (", EncodeFrame API" if api and "fps" in api else "")}
    try:
        for f in os.listdir(tmpdir):
            os.unlink(os.path.join(tmpdir, f))
        os.rmdir(tmpdir)
    except Exception:
        pass

    # ---- second workload point: hard content ----
    hard = None
    if not args.no_hard:
        hclip = make_clip(HARD_NOISE, HARD_FRAMES)
        hd = torch.from_numpy(hclip).cuda()
        enc = BatchEncoder(W, H, qp=QP, fps=FPS, n_streams=S, device=local, entropy_threads=ent_threads)
        enc.set_stream(stream.cuda_stream)
        hsteps = max(4, args.steps // 2)
        r = timed_run(enc, True, 3, hsteps, False, clip_dev=hd, sq=ping_pong(HARD_FRAMES))
        enc.close()
        coded = float(np.mean(r["coded"]))                       # coded (not P_SKIP) macroblocks per step, counted by the host writer
        hard = {"generator": "same synthetic generator, +-%d per-frame noise" % HARD_NOISE, "value": r["pictures"] / r["dt"], "unit": "frames/s",
                "steps": hsteps, "skip_ratio": 1.0 - coded / (S * MBS_PER_FRAME), "bitstream_kbytes_per_frame": r["bytes"] / (S * hsteps) / 1e3,
                "encode_kernel_ms": float(np.mean([k[0] for k in r["kern"]])) * 1e-3, "host_entropy_ms": float(np.mean([k[2] for k in r["kern"]])) * 1e-3}

    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, *results["resident"]["last"])

    if rank == 0:
        res, l2 = results["resident"], results["e2e_layer2"]
        value = res["pictures"] / res["dt"]
        e2e_l2 = l2["pictures"] / l2["dt"]
        peak, peak_kind = measured_peaks()
        k_enc = float(np.mean([k[0] for k in res["kern"]])) * 1e-6        # seconds per launch of pad + macroblock wavefront kernel
        k_dbk = float(np.mean([k[1] for k in res["kern"]])) * 1e-6
        ent = float(np.mean([k[2] for k in res["kern"]])) * 1e-6
        alg = S * MBS_PER_FRAME * ALG_BYTES_PER_MB
        achieved = alg / k_enc / 1e9
        coded = float(np.mean(l2["coded"]))
        d2h = int(world * np.mean(l2["d2h"]))
        if api and "job_fps" in api:
            e2e = {"value": api["job_fps"], "unit": "frames/s", "h2d_bytes_per_step": world * S * FSZ, "d2h_bytes_per_step": d2h,
                   "path": "ISVCEncoder::EncodeFrame (the reference's API): %d application threads, one encoder object each, host "
                           "pictures; objects share batched GPU encoders of %d streams (openh264_b200/wels/broker.h)" % (S, api["broker_slots"]),
                   "d2h_note": "index table + records of the coded macroblocks only, written by the GPU into mapped pinned memory (figure of the "
                               "layer-2 run on the same pictures)"}
        else:
            e2e = {"value": e2e_l2, "unit": "frames/s", "h2d_bytes_per_step": world * S * FSZ, "d2h_bytes_per_step": d2h,
                   "path": "layer 2 (b2h264_enc_submit / collect) with pinned host pictures; the EncodeFrame run was not possible: %s"
                           % (api or "driver or layer-3 library not built")}
        out = {
            "metric": "1080p_encode_fps", "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": res["dt"] / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": WORKLOAD + "; %d independent streams per GPU (%d distinct picture sequences), 1 picture per stream per step"
                                   % (S, len({(PHASE_STEP * s) % len(seq) for s in range(S)})),
                       "streams_per_gpu": S, "parallelism": "replica x%d (independent streams, no collective)" % world,
                       "l2": "inputs larger than L2 (%.0f MB of source pictures per step, %.0f MB of reference pictures)" % (S * FSZ / 1e6, S * 3.43),
                       "skip_ratio": 1.0 - coded / (S * MBS_PER_FRAME), "workload_hard": hard},
            "e2e": e2e,
            "e2e_layer2": {"value": e2e_l2, "unit": "frames/s", "path": "b2h264_enc_submit / collect, pinned host pictures, two batches in flight"},
            "gpu_launches": int(launches),
            "clocks": res["clocks"],
            "roofline": {"bound": "hbm", "kernel": "k_encode_mbs (macroblock wavefront, all streams)", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak,
                         "traffic": (ncu_traffic("k_encode_mbs") or {}).get("dram_bytes") if S == (ncu_traffic("k_encode_mbs") or {}).get("streams") else None,
                         "peak_source": peak_kind,
                         "note": "wavefront kernel is dependency/latency-bound by construction (SURVEY.md §8d); "
                                 "alg bytes = %d B/MB x %d MB/launch" % (ALG_BYTES_PER_MB, S * MBS_PER_FRAME)},
            "breakdown_ms_per_step": {"encode_kernel": k_enc * 1e3, "deblock_expand": k_dbk * 1e3, "host_entropy": ent * 1e3,
                                      "wall_resident": res["wall"] / args.steps * 1e3, "wall_e2e_layer2": l2["wall"] / args.steps * 1e3},
            "bitstream_kbytes_per_frame": res["bytes"] / (S * args.steps) / 1e3,
            "host_cores": host_cores(),
        }
        out.update({"parity_checked": parity["parity_checked"], "parity": parity})
        if world == 1:
            out["roofline_mc_sad"] = mc_sad_roofline(L, local, peak)
            if not args.no_decode:
                out["decode"] = decode_bench(local, clip_h, seq, peak)
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline_sample()
        print(json.dumps(out))
    if world > 1:
        shard.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
