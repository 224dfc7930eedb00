"""GPU probe: fused MA-LLM compression (rtk_mallm_compress) vs the reference's torch op loop on the same GPU.

Shapes: the model shapes (Qwen2-VL 256 / 1024 frames, LLaVA-OneVision 64 frames; soft / hard x sync 0 / 1) and the long
videos at C = 8192: per-patch mode at T = 7944 and 7945 (the last T with two row buffers in shared memory and the first
with one) and T = 8192, sync mode at T = C = 8192.  Each call is timed with CUDA events over windows of at least
--window-s seconds (back-to-back calls on the same bank: a bank under the 126 MB L2, LLaVA's 107 MB, is read from L2
after the first call); the median window and every window are reported.  The reference loop runs once per shape for the
speedup and the bit-identity check: always for the model shapes unless --no-ref, for the long videos only with --long-ref.

    python tests/probes/prof_mallm.py [--out FILE] [--window-s 0.3] [--windows 3] [--no-ref] [--long-ref]
"""
import argparse, json, os, statistics, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "video-retake_b200")):
    sys.path.insert(0, p)
import torch
from retake import visual_compression as vc
from oracle import reference_ops as ro

ap = argparse.ArgumentParser()
ap.add_argument("--out", help="also write the results to this JSON file")
ap.add_argument("--window-s", type=float, default=0.3)
ap.add_argument("--windows", type=int, default=3)
ap.add_argument("--no-ref", action="store_true", help="skip the reference loop everywhere")
ap.add_argument("--long-ref", action="store_true", help="also run the reference loop for the long videos")
args = ap.parse_args()


def ev_windows(fn):
    """ms per call in each of args.windows windows of at least args.window_s seconds"""
    fn(); torch.cuda.synchronize()
    t0 = time.perf_counter(); fn(); torch.cuda.synchronize()
    reps = max(1, int(args.window_s / max(time.perf_counter() - t0, 1e-6)) + 1)
    out = []
    for _ in range(args.windows):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record(); torch.cuda.synchronize()
        out.append(a.elapsed_time(b) / reps)
    return out, reps


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


MODEL = [("qwen_256f", 128, 256, 3584, 64), ("qwen_1024f", 512, 256, 3584, 256), ("llava_64f", 64, 729, 1152, 32)]
LONG = [(f"long_T{T}", T, 3, 8192, T - 256, syncs) for T, syncs in ((7944, (False,)), (7945, (False,)), (8192, (False, True)))]
cases = [(name, T, N, C, t, (False, True), False) for name, T, N, C, t in MODEL] + \
        [(name, T, N, C, t, syncs, True) for name, T, N, C, t, syncs in LONG]

out = {"card": card()}
print(out["card"], flush=True)
g = torch.Generator(device="cuda").manual_seed(0)
for name, T, N, C, t, syncs, long_video in cases:
    x = torch.randn(1, T, N, C, generator=g, device="cuda").to(torch.bfloat16)
    run_ref = not args.no_ref and (args.long_ref or not long_video)
    for sync in syncs:
        for hard in (False, True):
            windows, reps = ev_windows(lambda: vc.mallm_compress(x, t, sync=sync, hard=hard))
            ours = statistics.median(windows)
            rec = {"T": T, "N": N, "C": C, "t": t, "rounds": T - t, "ours_ms": ours, "windows_ms": windows, "reps": reps,
                   "bank_bytes": 2 * T * N * C}
            if run_ref:
                torch.cuda.synchronize(); t0 = time.perf_counter()
                want, ws = ro.mallm_compress(x.clone(), t, sync, hard)
                torch.cuda.synchronize()
                ref = (time.perf_counter() - t0) * 1e3
                got, gs = vc.mallm_compress(x, t, sync=sync, hard=hard)
                rec.update(torch_cuda_ops_ms=ref, speedup=ref / ours,
                           bit_identical=bool(torch.equal(got, want)) and (hard or bool(torch.equal(gs, ws))))
                del want, ws, got, gs
            out[f"{name}_sync{int(sync)}_hard{int(hard)}"] = rec
            print(name, sync, hard, rec, flush=True)
    del x
print(json.dumps(out))
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    json.dump(out, open(args.out, "w"), indent=1)
