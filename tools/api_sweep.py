"""ISVCEncoder-API throughput for several (threads, broker pool size) combinations (profiling aid, not the bench)."""
import json, os, subprocess, sys, tempfile
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench
clip = bench.make_clip()
with tempfile.TemporaryDirectory() as d:
    p = os.path.join(d, "clip.yuv"); clip.tofile(p)
    for threads, slots in [(256, 256), (256, 128), (512, 256), (512, 512)]:
        env = dict(os.environ, B2H264_BROKER_SLOTS=str(slots), B2H264_DEVICE="0")
        r = subprocess.run([os.path.join(ROOT, "tests/wels/build/wels_mt_driver"), os.path.join(ROOT, "openh264_b200/libopenh264_b200_wels.so"), p,
                            "1920", "1080", str(bench.CLIP_FRAMES), "26", str(threads), "10", "3", str(bench.PHASE_STEP), "-"],
                           capture_output=True, text=True, env=env, timeout=900)
        print(threads, slots, r.stdout.strip().splitlines()[-1] if r.returncode == 0 else ("FAILED " + (r.stderr + r.stdout)[-300:]), flush=True)
