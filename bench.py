#!/usr/bin/env python
"""bench.py - 2048-frame DPSelect + PivotKV throughput (frames/s) on B200.

A "step" is one pass of the hot path over one synthetic 2048-frame Qwen2-VL-7B-shape video:
  DPSelect  memory_bank_compress_keyframe on X[1, T=1024, N=256, C=3584] bf16 (per-patch mode)
  PivotKV   PivotKVCache.update for 64 prefill chunks x 28 layers, L = 4096 tokens per chunk, H = 28, KVH = 4, D = 128
with the shipped recipe of the reference (configs/qwen2_vl/retake_qwen2-vl_mlvu.yaml): visual ratio 1.0 (mask only,
identity compaction), dynamic KV ratio 32000 / 262144 = 0.122 (keep 499 of 4096), pos_embed_reforge on.

  value  frames / s with every input already resident in HBM, through the public operators
  e2e    the same through the same operators with the inputs in pinned HOST memory: the H2D copy of the step's
         inputs and a D2H read of the step's result are inside the timed region
  roofline      the tcgen05 scoring launches (the dominant kernels), CUDA-event timed inside the timed region
  cpu_baseline  the reference's own torch-op sequence (oracle/reference_ops.py) on the host cores, bounded sample

--impl reference times that CPU op sequence alone (rank 0 only).  N > 1: one video per rank (weak scaling, no
data-path collective), torchrun launch.  --dump-outputs DIR writes what the last timed step computed as .npy files
(dump_outputs()); the inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "video-retake_b200"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

# stdout carries exactly ONE JSON line: whatever libraries print while the run is in progress (NCCL's version banner,
# transformers' notices ...) is sent to stderr by pointing fd 1 at fd 2 until the line is ready (emit()).
_REAL_STDOUT = None


def quiet_stdout():
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(obj):
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.dup2(_REAL_STDOUT, 1)
    print(json.dumps(obj), flush=True)
    if _REAL_STDOUT is not None:
        os.dup2(2, 1)


import torch  # noqa: E402

METRIC = "2048-frame DPSelect+PivotKV frames/s"
UNIT = "frames/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--frames", type=int, default=2048)
    ap.add_argument("--shape", default="qwen2vl", choices=["qwen2vl", "llava"],
                    help="qwen2vl: Qwen2-VL-7B @448px (headline); llava: LLaVA-Video-Qwen2-7B, SigLIP-so400m grid (config 4)")
    ap.add_argument("--visual-ratio", type=float, default=1.0)
    ap.add_argument("--kv-ratio", type=float, default=-1.0, help="-1: dynamic, 32000 / video tokens (shipped recipe)")
    ap.add_argument("--no-reforge", action="store_true")
    ap.add_argument("--pool", type=int, default=28, help="distinct Q/K/V sets cycled through the layer-chunks")
    ap.add_argument("--immediate", action="store_true",
                    help="compress inside every update() (one rtk_pivot_update per layer) instead of one batched call per chunk")
    ap.add_argument("--layers", type=int, default=28)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-immediate-ab", action="store_true", help="skip the extra timing with deferred compression off")
    ap.add_argument("--no-parity", action="store_true", help="skip the kept-index parity self-check before the timed region")
    ap.add_argument("--no-sharded", action="store_true", help="N > 1: skip the within-video split record (config 3)")
    ap.add_argument("--only-sharded", action="store_true", help="N > 1: print only the within-video split record")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed (rank 0) to DIR/<name>.npy")
    return ap.parse_args()


class Shape:
    """Qwen2-VL-7B shape at 448x448, or LLaVA-Video-Qwen2-7B with the SigLIP-so400m token grid (SURVEY.md section 8)."""

    def __init__(self, a):
        self.name = a.shape
        self.frames = a.frames
        self.H, self.KVH, self.D = 28, 4, 128
        self.layers = a.layers
        self.reforge = not a.no_reforge
        self.deferred = not a.immediate      # compression of a chunk's layers batched at after_forward() (SURVEY.md 8 f2)
        if a.shape == "qwen2vl":
            self.T = a.frames // 2            # temporal_patch_size 2
            self.N, self.C = 256, 3584        # DPSelect runs on the LLM-side embeddings
            self.tok_per_grid = 256
            self.L = min(32, self.T) * 1024 // 8            # chunked_prefill_frames 32 -> 4096 tokens
            self.mrope, budget = [16, 24, 24], 32000
        else:
            self.T = a.frames
            self.N, self.C = 729, 1152        # DPSelect runs on the SigLIP features before the projector
            self.tok_per_grid = 196           # after projector + 2x bilinear pooling
            self.L = min(32, self.T) * 196    # 6272
            self.mrope, budget = None, 40000
        self.t = max(1, round(a.visual_ratio * self.T))
        self.tokens = self.t * self.tok_per_grid           # (the newline slot is dropped with visual compression on)
        self.chunks = (self.tokens + self.L - 1) // self.L
        self.kv_ratio = a.kv_ratio if a.kv_ratio > 0 else min(1.0, budget / self.tokens)
        self.keep = max(1, int(self.kv_ratio * self.L))


def make_rotary(device, shape="qwen2vl"):
    if shape == "llava":
        from transformers.models.qwen2.configuration_qwen2 import Qwen2Config
        from transformers.models.qwen2.modeling_qwen2 import Qwen2RotaryEmbedding
        tc = Qwen2Config(hidden_size=3584, num_attention_heads=28, num_key_value_heads=4, num_hidden_layers=28,
                         max_position_embeddings=32768,
                         rope_parameters={"rope_type": "yarn", "factor": 4.0, "beta_fast": 32.0, "beta_slow": 1.0,
                                          "rope_theta": 1e6, "original_max_position_embeddings": 32768})
        return Qwen2RotaryEmbedding(tc).to(device)
    from transformers.models.qwen2_vl.configuration_qwen2_vl import Qwen2VLTextConfig
    from transformers.models.qwen2_vl.modeling_qwen2_vl import Qwen2VLRotaryEmbedding
    tc = Qwen2VLTextConfig(hidden_size=3584, num_attention_heads=28, num_key_value_heads=4, num_hidden_layers=28,
                           max_position_embeddings=32768,
                           rope_parameters={"rope_type": "yarn", "factor": 4.0, "beta_fast": 32.0, "beta_slow": 1.0,
                                            "rope_theta": 1e6, "mrope_section": [16, 24, 24],
                                            "original_max_position_embeddings": 32768})
    return Qwen2VLRotaryEmbedding(tc).to(device)


def cache_config(s):
    import types
    cfg = types.SimpleNamespace(hidden_size=s.H * s.D, num_hidden_layers=s.layers, num_attention_heads=s.H,
                                num_key_value_heads=s.KVH)
    cfg.longvideo_kwargs = {"kvcache_compression": True,
                            "kvcache_compression_kwargs": {"compression_ratio": s.kv_ratio, "compression_method": "pivotkv",
                                                           "pos_embed_reforge": s.reforge,
                                                           "deferred_compression": s.deferred}}
    return cfg


def synth_host(s, pool, seed):
    """pinned host inputs: scene-structured embeddings + a pool of Q/K/V sets in the attention layout [1, L, heads, D]"""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.set_num_threads(max(1, (os.cpu_count() or 1) // world))      # ranks share the host cores while generating
    g = torch.Generator().manual_seed(seed)
    x = torch.empty(s.T, s.N, s.C, dtype=torch.bfloat16)
    t = 0
    while t < s.T:                                         # x[t] = scene + 0.3 * noise, scenes of 3..40 grids
        run = int(torch.randint(3, 41, (1,), generator=g))
        scene = torch.randn(s.N, s.C, generator=g)
        for _ in range(run):
            if t >= s.T:
                break
            x[t] = (scene + 0.3 * torch.randn(s.N, s.C, generator=g)).to(torch.bfloat16)
            t += 1
    q = torch.randn(pool, s.L, s.H, s.D, generator=g).to(torch.bfloat16)
    k = torch.randn(pool, s.L, s.KVH, s.D, generator=g).to(torch.bfloat16)
    v = torch.randn(pool, s.L, s.KVH, s.D, generator=g).to(torch.bfloat16)
    if torch.cuda.is_available():
        return [t_.pin_memory() for t_ in (x, q, k, v)]
    return [x, q, k, v]


def synth_device(s, pool, seed, dev):
    """the same synthetic inputs generated ON the GPU (seconds instead of a minute of host randn for the 3.4 GB LLaVA video),
    plus pinned host copies for the end-to-end leg: -> ([x, q, k, v] on dev, [x, q, k, v] pinned)"""
    g = torch.Generator(device=dev).manual_seed(seed)
    gc = torch.Generator().manual_seed(seed)
    x = torch.empty(s.T, s.N, s.C, dtype=torch.bfloat16, device=dev)
    t = 0
    while t < s.T:                                         # x[t] = scene + 0.3 * noise, scenes of 3..40 grids
        run = min(int(torch.randint(3, 41, (1,), generator=gc)), s.T - t)
        scene = torch.randn(s.N, s.C, generator=g, device=dev)
        x[t:t + run] = (scene[None] + 0.3 * torch.randn(run, s.N, s.C, generator=g, device=dev)).to(torch.bfloat16)
        t += run
    q = torch.randn(pool, s.L, s.H, s.D, generator=g, device=dev).to(torch.bfloat16)
    k = torch.randn(pool, s.L, s.KVH, s.D, generator=g, device=dev).to(torch.bfloat16)
    v = torch.randn(pool, s.L, s.KVH, s.D, generator=g, device=dev).to(torch.bfloat16)
    host = []
    for t_ in (x, q, k, v):
        h = torch.empty(t_.shape, dtype=t_.dtype, pin_memory=True)
        h.copy_(t_)
        host.append(h)
    torch.cuda.synchronize()
    return [x, q, k, v], host


class ScoreTimer:
    """CUDA-event pairs recorded by the library around a sample of the scoring launches (rtk_pivot_score inside
    rtk_pivot_update) in the timed region; the events live on the stream the kernels are launched on."""

    def __init__(self, every=8, calls_per_pair=1):
        self.every, self.n, self.pairs, self.on = every, 0, [], False
        self.calls_per_pair = calls_per_pair      # scoring calls between the two events (a batched flush scores every layer)
        self.dpselect = []

    def arm(self, cache):
        self.n += 1
        if not self.on or self.n % self.every:
            return
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()                      # forces creation of the underlying cudaEvent_t; re-recorded by the library
        b.record()
        cache.score_events = (a.cuda_event, b.cuda_event)
        self.pairs.append((a, b))

    def mean_ms(self):
        return sum(a.elapsed_time(b) for a, b in self.pairs) / max(1, len(self.pairs)) / self.calls_per_pair


def run_step(s, x, q, k, v, rotary, lc, vc, pos_grid, timer=None, outputs=None):
    """one video through the public operators; returns a small device tensor standing for the step's result.  A dict
    passed as ``outputs`` receives everything the step computed: the DPSelect output and mask, and the KV cache."""
    if timer is not None and timer.on:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
    out, mask = vc.memory_bank_compress_keyframe(x[None], s.t, 3, sync=False)
    if timer is not None and timer.on:
        b.record()
        timer.dpselect.append((a, b))
    cache = lc.build_kvcache(cache_config(s))
    pool = q.shape[0]
    it = 0

    for c in range(s.chunks):
        ss, ee = c * s.L, min((c + 1) * s.L, s.tokens)
        Lc = ee - ss
        cache.kvcache_compression = True
        cache.keypatches_mask_chunk = mask[ss:ee]            # (LLaVA: only the first t*196 of the t*729 entries land on tokens)
        # the caller's re-basing of the temporal ids (the attention forward continues them after each layer's compacted
        # cache, qwen2_vl.py:68-73) for all layers of the chunk at once - what this repo's model glue does as well
        if s.reforge:
            pos_all = cache.rebased_position_ids(pos_grid[..., :Lc], s.layers)
        else:
            pos_all = pos_grid[..., :Lc].unsqueeze(0).repeat(s.layers, *([1] * pos_grid.dim()))
            pos_all[:, 0] += c * (s.L // s.tok_per_grid if s.mrope else s.L)
        for layer in range(s.layers):
            j = it % pool
            it += 1
            pos = pos_all[layer]
            if timer is not None and not s.deferred:
                timer.arm(cache)
            cache.update(k[j:j + 1, :Lc].transpose(1, 2), v[j:j + 1, :Lc].transpose(1, 2), layer,
                         {"query_states": q[j:j + 1, :Lc].transpose(1, 2), "position_ids": pos, "rotary_emb": rotary,
                          "mrope_section": s.mrope, "position_ids_owned": True})      # a per-layer buffer, rewritten next chunk
        if timer is not None and s.deferred:
            timer.arm(cache)
        cache.after_forward()                                # the chunk loop's hook (qwen2_vl.py:715-716)
    if outputs is not None:
        outputs.update(dpselect_out=out, dpselect_mask=mask, cache=cache)
    return cache.last_keep_indices, cache.get_seq_length(0)


def dump_outputs(d, s, res):
    """``res`` (run_step's ``outputs``) as ``d/<name>.npy``, float32, 64 MB at most: the DPSelect key-patch mask and
    ``dpselect_out`` rows (of the output viewed as [t * N, C]); the compressed KV cache of every layer at a set of token
    slots - ``kv_keys`` / ``kv_values`` [layers, KVH, slots, D], ``kv_positions`` [layers, 3 or 1, slots] with reforge -
    and the kept indices of the last update, ``kv_last_keep_indices``.  An array larger than SAMPLE_BYTES is a fixed seeded
    sample (sorted; its indices, float64, in ``*_rows`` / ``kv_slots``), so the files of two runs with the same arguments
    compare element for element."""
    import numpy as np
    SAMPLE_BYTES = 14 << 20

    def pick(n, row_bytes, seed):
        k = max(1, SAMPLE_BYTES // row_bytes)
        if n <= k:
            return None
        return torch.randperm(n, generator=torch.Generator().manual_seed(seed))[:k].sort().values

    arrays = {}
    mask = res["dpselect_mask"].reshape(-1)
    rows = pick(mask.numel(), 4 + 8, 1)
    if rows is not None:
        arrays["dpselect_mask_rows"] = rows
        mask = mask[rows.to(mask.device)]
    arrays["dpselect_mask"] = mask
    out = res["dpselect_out"].reshape(-1, s.C)
    rows = pick(out.shape[0], 4 * s.C, 2)
    if rows is not None:
        arrays["dpselect_out_rows"] = rows
        out = out[rows.to(out.device)]
    arrays["dpselect_out"] = out
    cache = res["cache"]
    n_layers = len(cache.layers)
    slots = pick(cache.get_seq_length(0), 8 * n_layers * s.KVH * s.D, 3)
    if slots is None:
        slots = torch.arange(cache.get_seq_length(0))
    arrays["kv_slots"] = slots
    sl = slots.to(cache.layers[0].keys.device)
    arrays["kv_keys"] = torch.stack([cache.layers[i].keys[0].index_select(1, sl) for i in range(n_layers)])
    arrays["kv_values"] = torch.stack([cache.layers[i].values[0].index_select(1, sl) for i in range(n_layers)])
    if s.reforge:
        arrays["kv_positions"] = torch.stack([cache.position_cache[i].reshape(-1, cache.position_cache[i].shape[-1])
                                              .index_select(1, sl) for i in range(n_layers)])
    arrays["kv_last_keep_indices"] = cache.last_keep_indices
    arrays = {name: (t.double() if name.endswith(("_rows", "_slots")) else t.float()).cpu().numpy()
              for name, t in arrays.items()}
    total = sum(a_.nbytes for a_ in arrays.values())
    assert total <= 64 << 20, f"{total} bytes of outputs"
    os.makedirs(d, exist_ok=True)
    for name, arr in arrays.items():
        np.save(os.path.join(d, name + ".npy"), arr)


def measured_traffic(s):
    """profiles/ncu_score_traffic.json: [{"score_source_sha", "L", "deferred", "bytes_per_layer", "source"}] from an
    `ncu --set full` capture of the scoring launches; used only when the capture was taken from the scoring source in this
    tree (SHA-256 of csrc/pivot_score.cu) at this shape - never a stale constant"""
    import hashlib
    try:
        rec = json.load(open(os.path.join(ROOT, "profiles", "ncu_score_traffic.json")))
        sha = hashlib.sha256(open(os.path.join(ROOT, "video-retake_b200", "csrc", "pivot_score.cu"), "rb").read()).hexdigest()[:16]
    except Exception:
        return None
    for r in rec if isinstance(rec, list) else [rec]:
        if r.get("score_source_sha") == sha and r.get("L") == s.L and bool(r.get("deferred")) == bool(s.deferred):
            return r.get("bytes_per_layer")
    return None


def torch_ops_keep(q, k, v, ratio, keymask, position_ids, rotary, sections, reforge):
    """Parity self-check, OUTSIDE the timed region: the reference's op sequence for one compressing update issued as stock
    torch-CUDA calls (cuBLAS bf16 matmul, ATen softmax / sum / mean / topk; ``longvideo_cache.py:244-277``) - "the reference
    executed with torch-CUDA ops" on this GPU.  -> (kept indices int64 ascending, bf16 score after the key-patch fill)"""
    import math
    _, H, L, D = q.shape
    KVH = k.shape[1]
    if reforge:
        cos, sin = rotary(v, position_ids)

        def pick(tab):
            if not sections:
                return tab.unsqueeze(1)
            parts = tab.split(list(sections) * 2, dim=-1)
            return torch.cat([p_[i % 3] for i, p_ in enumerate(parts)], dim=-1).unsqueeze(1)

        def half_turn(t):
            h = t.shape[-1] // 2
            return torch.cat((-t[..., h:], t[..., :h]), dim=-1)
        c, sn = pick(cos), pick(sin)
        sc2 = rotary.attention_scaling ** 2
        q = ((q * c) - (half_turn(q) * sn)) / sc2
        k = ((k * c) - (half_turn(k) * sn)) / sc2
    kr = k[:, :, None].expand(1, KVH, H // KVH, L, D).reshape(1, H, L, D)
    w = torch.matmul(q, kr.transpose(2, 3)) / math.sqrt(D)
    w = torch.nn.functional.softmax(w, dim=-1, dtype=torch.float32).to(q.dtype)
    score = w[0].sum(1).reshape(KVH, -1, L).mean(1).mean(0)
    if keymask is not None:
        score.masked_fill_(keymask, 1.0)
    keep = max(1, int(ratio * L))
    return score.topk(keep)[1].sort().values, score


def parity_record(s, q, k, v, rotary, lc, pos_grid, mask, trials=6):
    """kept-index parity of this run's own update (same shapes, ratio, mask and rotary as the timed steps) against
    torch_ops_keep: how many trials are exactly equal, and whether every other one differs only on the cut"""
    from helpers import index_parity
    n = min(trials, q.shape[0])
    identical, justified = 0, True
    for j in range(n):
        qq, kk, vv = q[j:j + 1].transpose(1, 2), k[j:j + 1].transpose(1, 2), v[j:j + 1].transpose(1, 2)
        pos = pos_grid.clone()
        km = mask[j * 17:j * 17 + s.L] if mask is not None and mask.numel() >= j * 17 + s.L else None
        _, _, _, idx, _ = lc.pivot_update(qq, kk, vv, s.keep, km, pos, rotary, s.mrope, s.reforge)
        idx_ref, score_ref = torch_ops_keep(qq, kk, vv, s.kv_ratio, km, pos, rotary, s.mrope, s.reforge)
        same, ok, _ = index_parity(idx, idx_ref, score_ref, s.keep)
        identical += int(same)
        justified = justified and ok
    return {"trials": n, "identical": identical, "others_differ_only_within_1_bf16_ulp_of_the_kth_score": justified,
            "against": "the reference's op sequence with stock torch-CUDA ops (cuBLAS + ATen) on this GPU, L=%d keep=%d" % (s.L, s.keep)}


def _native_lib():
    from retake import _native
    return _native.lib()


def sharded_within_video(dev, dist, rank, world, steps=3):
    """BASELINE config 3 - ONE 1024-frame Qwen2-VL-7B-shape video split over the GPUs of a box (SURVEY.md 8e): PivotKV by KV
    head (KVH = 4: groups of min(world, 4) ranks, every group its own video), DPSelect by frame range with a one-frame halo.
    Timed with CUDA events, max over ranks, against the single-GPU operators run by the same process on the same inputs;
    rank 0 of every group checks that the split gives bit-identical kept indices, K / V rows and embeddings."""
    from retake import distributed as rd
    from retake import longvideo_cache as lc
    from retake import visual_compression as vc
    H, KVH, D, L, layers, mrope = 28, 4, 128, 4096, 28, [16, 24, 24]
    frames, T, N, C = 1024, 512, 256, 3584
    gsz = min(world, KVH)
    n_groups = world // gsz
    groups = [dist.new_group(list(range(g * gsz, (g + 1) * gsz))) for g in range(n_groups)]
    if rank >= n_groups * gsz:
        return None
    group = groups[rank // gsz]
    grank = rank % gsz
    tokens = T * 256
    chunks = tokens // L                                   # 32
    r_kv = min(1.0, 32000 / tokens)                        # 0.244: the shipped dynamic ratio at 1024 frames
    keep = max(1, int(r_kv * L))
    rotary = make_rotary(dev, "qwen2vl")
    g = torch.Generator(device=dev).manual_seed(777 + rank // gsz)          # the ranks of a group hold the same video
    pool = 4
    q = torch.randn(pool, L, H, D, generator=g, device=dev).to(torch.bfloat16)
    k = torch.randn(pool, L, KVH, D, generator=g, device=dev).to(torch.bfloat16)
    v = torch.randn(pool, L, KVH, D, generator=g, device=dev).to(torch.bfloat16)
    x = torch.randn(T, N, C, generator=g, device=dev).to(torch.bfloat16)
    ar = torch.arange(L, device=dev)
    pos = torch.stack([ar // 256, (ar % 256) // 16, ar % 16])[:, None]
    per = [KVH // gsz] * gsz
    g0, G = grank * per[0], H // KVH
    t = T // 2
    t0, t1 = rd.split_range(T, gsz)[grank]
    xl = x[t0 - int(t0 > 0):t1].contiguous()

    def single(j):                                          # the single-GPU fused update: one rtk_pivot_update call
        return lc.pivot_update(q[j:j + 1].transpose(1, 2), k[j:j + 1].transpose(1, 2), v[j:j + 1].transpose(1, 2), keep, None,
                               pos, rotary, mrope, True)

    def sharded(j, transport):
        return rd.pivot_update_kv_sharded(q[j:j + 1, :, g0 * G:(g0 + per[0]) * G].transpose(1, 2),
                                          k[j:j + 1, :, g0:g0 + per[0]].transpose(1, 2),
                                          v[j:j + 1, :, g0:g0 + per[0]].transpose(1, 2), keep, per, None, pos, rotary, mrope,
                                          True, group, transport)

    def timed(fn, n, sync_group=True):
        for i in range(3):
            fn(i)
        torch.cuda.synchronize()
        if sync_group:
            dist.barrier(group)
            torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(n):
            fn(i)
        b.record()
        torch.cuda.synchronize()
        ms = torch.tensor([a.elapsed_time(b) / n], device=dev)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)          # max over ALL ranks of the job
        return float(ms)

    out = {"config": f"1024 frames Qwen2-VL-7B shape, L={L}, keep={keep} (r_kv={r_kv:.3f}), reforge on; KV heads split over "
                     f"{gsz} GPUs per video ({n_groups} video(s) in flight); DPSelect T={T} -> t={t} split by frame range",
           "gpus_per_video": gsz, "videos": n_groups}
    # ---- bit-equality self-check against the single-GPU operators (every rank checks its own heads / frames)
    # (the kept set of the split equals the single-GPU one unless a score sits on the cut: a unit split between CTAs folds
    #  its fp32 partials in another order when the launch holds other heads - then the rule of tests/test_gpu_index_parity.py)
    from helpers import index_parity
    ok = cut_ok = True
    for j in range(pool):
        sk, sv, sp, sidx, shs = single(j)
        for transport in ("p2p", "nccl"):
            kk, vv, pp, idx, hs = sharded(j, transport)
            same, justified, _ = index_parity(idx, sidx, shs.float().mean(0).to(torch.bfloat16), keep)
            cut_ok = cut_ok and justified
            ok = ok and same and bool(torch.equal(kk, sk[:, g0:g0 + per[0]])) and bool(torch.equal(vv, sv[:, g0:g0 + per[0]])) \
                and bool(torch.equal(pp, sp))
    want_out, want_mask, want_idx = vc.memory_bank_compress_keyframe(x[None], t, 3, sync=False, return_indices=True)
    dps_out = torch.zeros((1, t, N, C), dtype=torch.bfloat16, device=dev)      # the split writes its own slots into it
    part, mask2, idx2 = rd.dpselect_frame_sharded_fused(xl, t0, t1, T, t, False, group, dps_out)
    own = ((idx2.long() >= t0) & (idx2.long() < t1))[None, :, :, None].expand_as(want_out)
    ok = ok and bool(torch.equal(mask2, want_mask)) and bool(torch.equal(idx2.long(), want_idx)) \
        and bool(torch.equal(part[own], want_out[own]))
    okt = torch.tensor([int(ok), int(cut_ok)], device=dev)
    dist.all_reduce(okt, op=dist.ReduceOp.MIN)
    out["bit_identical_to_single_gpu"] = bool(int(okt[0]))
    out["kept_indices_differ_only_on_the_cut_if_at_all"] = bool(int(okt[1]))
    del want_out
    # ---- one compressing update (the judge's unit): single GPU, split with NVLink peer stores, split with one NCCL collective
    n = 40
    out["update_ms_single_gpu"] = timed(lambda i: single(i % pool), n, False)
    out["update_ms_split_p2p"] = timed(lambda i: sharded(i % pool, "p2p"), n)
    out["update_ms_split_nccl"] = timed(lambda i: sharded(i % pool, "nccl"), n)
    out["update_speedup_p2p"] = out["update_ms_single_gpu"] / out["update_ms_split_p2p"]
    out["update_speedup_nccl"] = out["update_ms_single_gpu"] / out["update_ms_split_nccl"]
    out["transport"] = rd.ScoreExchange.get(group, dev, KVH, L, "p2p").transport
    # ---- all 28 layers of a chunk in one batched call (deferred compression, what the headline run uses): per layer
    def batch_single(_):
        arr = [(q[i % pool:i % pool + 1].transpose(1, 2), k[i % pool:i % pool + 1].transpose(1, 2),
                v[i % pool:i % pool + 1].transpose(1, 2)) for i in range(layers)]
        return rd_single_batch(arr)

    def rd_single_batch(arr):
        # single GPU: the same batched entry point with one rank's worth of everything (no exchange)
        import ctypes as C
        n_l = len(arr)
        args = (lc._UpdateArgs * n_l)()
        keepalive = []
        for i, (qq, kk, vv) in enumerate(arr):
            a_, outs_, ka, _, _ = lc.fill_update_args(None, True, lc._inv_freq_on_device, qq, kk, vv, pos, rotary, mrope, keep)
            args[i] = a_
            keepalive.append((outs_, ka))
        lib = _native_lib()
        ws = lc._workspace(dev, int(lib.rtk_pivot_update_batch_workspace_bytes(H, KVH, L, D, n_l)) + 256)
        wp = (ws.data_ptr() + 255) & ~255
        from retake import _native as N_
        N_.check(lib.rtk_pivot_update_batch(args, n_l, wp, ws.numel() - (wp - ws.data_ptr()), N_.stream_ptr(dev)),
                 "rtk_pivot_update_batch")
        return keepalive

    def batch_split(_, transport="p2p"):
        return rd.pivot_update_batch_kv_sharded(
            [(q[i % pool:i % pool + 1, :, g0 * G:(g0 + per[0]) * G].transpose(1, 2),
              k[i % pool:i % pool + 1, :, g0:g0 + per[0]].transpose(1, 2),
              v[i % pool:i % pool + 1, :, g0:g0 + per[0]].transpose(1, 2), None, pos) for i in range(layers)],
            keep, per, rotary, mrope, True, group, transport)
    out["batched_update_ms_per_layer_single_gpu"] = timed(batch_single, 6, False) / layers
    out["batched_update_ms_per_layer_split_p2p"] = timed(batch_split, 6) / layers
    out["batched_update_ms_per_layer_split_nccl"] = timed(lambda i: batch_split(i, "nccl"), 6) / layers
    out["batched_update_speedup_p2p"] = out["batched_update_ms_per_layer_single_gpu"] / out["batched_update_ms_per_layer_split_p2p"]
    out["batched_update_speedup_nccl"] = out["batched_update_ms_per_layer_single_gpu"] / out["batched_update_ms_per_layer_split_nccl"]
    # ---- DPSelect operator
    out["dpselect_ms_single_gpu"] = timed(lambda i: vc.memory_bank_compress_keyframe(x[None], t, 3, sync=False), 10, False)
    out["dpselect_ms_split"] = timed(lambda i: rd.dpselect_frame_sharded_fused(xl, t0, t1, T, t, False, group, dps_out), 10)
    out["dpselect_speedup"] = out["dpselect_ms_single_gpu"] / out["dpselect_ms_split"]
    # ---- the whole video: DPSelect + chunks x layers updates, as frames/s (aggregate over the videos in flight)
    def video_split(_):
        rd.dpselect_frame_sharded_fused(xl, t0, t1, T, t, False, group, dps_out)
        for c in range(chunks):
            batch_split(c)

    def video_single(_):
        vc.memory_bank_compress_keyframe(x[None], t, 3, sync=False)
        for c in range(chunks):
            batch_single(c)
    ms_split = timed(video_split, steps)
    ms_single = timed(video_single, steps, False)
    out["video_ms_split"], out["video_ms_single_gpu"] = ms_split, ms_single
    out["frames_per_s_split"] = n_groups * frames / (ms_split * 1e-3)
    out["frames_per_s_one_video_single_gpu"] = frames / (ms_single * 1e-3)
    out["video_latency_speedup"] = ms_single / ms_split
    return out


def clocks_sampler(dev_index):
    try:
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        return subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200",
                                 "-i", str(dev_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    except Exception:
        return None


def clocks_summary(proc):
    if proc is None:
        return None
    proc.terminate()
    try:
        text, _ = proc.communicate(timeout=5)
    except Exception:
        return None
    sm, mx, reasons = [], 0.0, set()
    for line in text.strip().splitlines():
        f = [z.strip() for z in line.split(",")]
        if len(f) < 9:
            continue
        try:
            sm.append(float(f[1]))
            mx = max(mx, float(f[2]))
        except ValueError:
            continue
        for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
            if val.lower().startswith("active"):
                reasons.add(name)
    if not sm:
        return None
    sm.sort()
    return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def cpu_reference_step(s, sample_T, host, it):
    """bounded sample of the reference's CPU path: DPSelect on sample_T grids + ONE compressing update at the real chunk
    length; returns (seconds extrapolated to the whole video - cost is linear in grids and in layer-chunks -, DPSelect
    seconds, update seconds, kind).  kind "reference": the UNMODIFIED reference functions (oracle/real_reference.py finds
    them in $RETAKE_REFERENCE or baseline/_ref - never in /root/reference at run time); kind "port": oracle/reference_ops.py, the same torch op
    sequence (bit-identical on CPU, tests/test_oracle_golden.py) when no reference tree is around."""
    from helpers import TableRotary
    from oracle import real_reference
    x, q, k, v = host
    real = real_reference.load()
    tt = max(1, round(sample_T * s.t / s.T))
    j = it % q.shape[0]
    rot = TableRotary(s.D, mrope=s.mrope is not None)
    if s.mrope:
        pos = torch.stack([torch.arange(s.L) // s.N, (torch.arange(s.L) % s.N) // 16, torch.arange(s.L) % 16])[:, None]
    else:
        pos = torch.arange(s.L)[None]
    qj, kj, vj = q[j:j + 1].transpose(1, 2), k[j:j + 1].transpose(1, 2), v[j:j + 1].transpose(1, 2)
    if real is not None:
        vc_ref, cache_cls, _ = real
        t0 = time.perf_counter()
        out, mask = vc_ref.memory_bank_compress_keyframe(x[None, :sample_T], tt, 3, sync=False)
        t1 = time.perf_counter()
        cache = cache_cls(real_reference.llm_config(s.H, s.KVH, s.D, 1, s.kv_ratio, s.reforge))
        cache.kvcache_compression = True
        cache.keypatches_mask_chunk = mask[:s.L] if mask.numel() >= s.L else None
        cache.update(kj, vj, 0, {"query_states": qj, "position_ids": pos, "rotary_emb": rot, "mrope_section": s.mrope})
        t2 = time.perf_counter()
        kind = "reference"
    else:
        from oracle import reference_ops as ro
        t0 = time.perf_counter()
        out, mask, _ = ro.dpselect(x[None, :sample_T], tt, False)
        t1 = time.perf_counter()
        ro.pivot_update(qj, kj, vj, s.kv_ratio, mask[:s.L] if mask.numel() >= s.L else None, pos, rot, s.mrope, s.reforge)
        t2 = time.perf_counter()
        kind = "port"
    return (t1 - t0) * (s.T / sample_T) + (t2 - t1) * s.chunks * s.layers, (t1 - t0), (t2 - t1), kind


def main():
    a = parse()
    quiet_stdout()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    s = Shape(a)
    model = "Qwen2-VL-7B-shape" if s.name == "qwen2vl" else "LLaVA-Video-Qwen2-7B-shape (SigLIP-so400m grid)"
    workload = (f"{model} {s.frames} frames @448px: DPSelect X[1,{s.T},{s.N},{s.C}] r_v={s.t / s.T:.3g} "
                f"patch_sync=False + PivotKV {s.chunks} chunks x {s.layers} layers, L={s.L}, H={s.H}, KVH={s.KVH}, "
                f"D={s.D}, r_kv={s.kv_ratio:.4g} (keep {s.keep}), reforge={s.reforge}")
    config = {"workload": workload, "frames": s.frames, "visual_ratio": s.t / s.T, "kv_ratio": s.kv_ratio,
              "pos_embed_reforge": s.reforge, "qkv_pool": a.pool,
              "deferred_compression": s.deferred,
              "l2_policy": f"inputs larger than L2 (X {2 * s.T * s.N * s.C / 1e9:.2f} GB; Q/K/V pool cycled, reuse distance > 126 MB)",
              "parallelism": f"dp{world} (one video per GPU, no data-path collective)"}

    if a.impl == "reference":
        if rank != 0:
            return
        host = synth_host(s, 2, 1234)
        # rank 0 alone runs the CPU arm and may use every host core: torchrun exports OMP_NUM_THREADS=1 and synth_host
        # divides the cores among the ranks - both would throttle this arm as N grows (VERDICT r1)
        torch.set_num_threads(os.cpu_count())
        sample_T = 64
        times = []
        kind = "port"
        for i in range(a.warmup + a.steps):
            t, td, tu, kind = cpu_reference_step(s, sample_T, host, i)
            if i >= a.warmup:
                times.append(t)
        sec = sum(times) / len(times)
        val = s.frames / sec
        sample = (f"per step: DPSelect on {sample_T} of {s.T} temporal grids + 1 of {s.chunks * s.layers} compressing updates "
                  f"at L={s.L}, scaled linearly to the whole video (extrapolated); threads {torch.get_num_threads()}")
        emit(({"metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
                          "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                          "dtype": "bf16", "data": "synthetic", "impl": "reference", "config": config,
                          "cpu_baseline": {"value": val, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind, "sample": sample},
                          "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                          "gpu_launches": 0}))
        return

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU path for --impl b200)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    from retake import _native
    from retake import longvideo_cache as lc
    from retake import visual_compression as vc
    if a.only_sharded:
        assert world > 1, "--only-sharded needs torchrun with at least 2 ranks"
        rec = sharded_within_video(dev, dist, rank, world)
        if rank == 0:
            emit({"sharded_within_video": rec, "n_gpus": world, "build_id": _native.build_id()})
        dist.destroy_process_group()
        return
    timer = ScoreTimer(every=2, calls_per_pair=s.layers) if s.deferred else ScoreTimer()
    rotary = make_rotary(dev, s.name)
    (x, q, k, v), host = synth_device(s, a.pool, 1234 + rank, dev)
    ar = torch.arange(s.L, device=dev)
    pos_grid = torch.stack([ar // s.N, (ar % s.N) // 16, ar % 16])[:, None] if s.mrope else ar[None]
    torch.cuda.synchronize()

    def sync_all():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    # kept-index parity self-check and the r_v = 0.5 DPSelect figure: BEFORE the warm-up, so that the warm-up steps leave
    # the caching allocator in the state the timed steps find
    parity = dps_half = None
    key_patch_share = None
    if rank == 0:
        _, kp_mask = vc.memory_bank_compress_keyframe(x[None], s.t, 3, sync=False)
        key_patch_share = float(kp_mask[:s.tokens].float().mean())       # the keys pass 2 of the scoring skips
        del kp_mask
    if rank == 0 and not a.no_parity:
        _, kp_mask = vc.memory_bank_compress_keyframe(x[None], s.t, 3, sync=False)
        parity = parity_record(s, q, k, v, rotary, lc, pos_grid, kp_mask)
        del kp_mask
        th = max(1, s.T // 2)
        for _ in range(2):
            vc.memory_bank_compress_keyframe(x[None], th, 3, sync=False)
        h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        h0.record()
        for _ in range(5):
            vc.memory_bank_compress_keyframe(x[None], th, 3, sync=False)
        h1.record()
        torch.cuda.synchronize()
        dps_half = (h0.elapsed_time(h1) / 5, 2.0 * s.T * s.N * s.C + 4.0 * s.T * s.N + 4.0 * th * s.N * s.C)
        torch.cuda.empty_cache()
    for _ in range(a.warmup):
        run_step(s, x, q, k, v, rotary, lc, vc, pos_grid)
    sync_all()
    sampler = clocks_sampler(local_rank) if rank == 0 else None
    launches0 = _native.launch_count()
    timer.on = True
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    marks = []
    e0.record()
    host_s = []
    last = {} if a.dump_outputs and rank == 0 else None
    for i in range(a.steps):
        h0 = time.perf_counter()
        res = run_step(s, x, q, k, v, rotary, lc, vc, pos_grid, timer, last if i == a.steps - 1 else None)
        host_s.append(time.perf_counter() - h0)          # the host's time to ENQUEUE a step (no synchronisation inside)
        marks.append(torch.cuda.Event(enable_timing=True))
        marks[-1].record()
    e1.record()
    sync_all()
    timer.on = False
    per_step = [p0.elapsed_time(p1) for p0, p1 in zip([e0] + marks[:-1], marks)]       # this rank's steps, device time
    launches = _native.launch_count() - launches0
    clocks = clocks_summary(sampler)
    if last:
        dump_outputs(a.dump_outputs, s, last)
        del last
    ms = e0.elapsed_time(e1)
    if dist is not None:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
    ms_per_step = ms / a.steps
    value = world * s.frames / (ms_per_step * 1e-3)

    # ---- A/B inside the same process: the reference's call order (compression inside every update(), one rtk_pivot_update
    #      per layer) on the same inputs; reported next to `value`, never instead of it
    immediate = None
    if s.deferred and not a.no_immediate_ab:
        import copy
        s_imm = copy.copy(s)
        s_imm.deferred = False
        run_step(s_imm, x, q, k, v, rotary, lc, vc, pos_grid)
        sync_all()
        i0, i1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        i0.record()
        for _ in range(a.steps):
            run_step(s_imm, x, q, k, v, rotary, lc, vc, pos_grid)
        i1.record()
        sync_all()
        ims = i0.elapsed_time(i1)
        if dist is not None:
            t = torch.tensor([ims], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ims = float(t)
        immediate = {"value": world * s.frames / (ims / a.steps * 1e-3), "unit": UNIT, "ms_per_step": ims / a.steps,
                     "what": "deferred_compression off: compression inside every update(), bit-identical results"}

    # ---- A/B inside the same process: key elision off (pass 2 of the scoring visits every key, like round 1); the kept
    #      indices are the same, only the time differs - reported next to `value`, never instead of it
    no_elision = None
    if not a.no_immediate_ab:
        lib_ = _native.lib()
        prev = lib_.rtk_debug_key_elision(0)
        try:
            run_step(s, x, q, k, v, rotary, lc, vc, pos_grid)
            sync_all()
            n0, n1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n0.record()
            for _ in range(a.steps):
                run_step(s, x, q, k, v, rotary, lc, vc, pos_grid)
            n1.record()
            sync_all()
        finally:
            lib_.rtk_debug_key_elision(prev)
        nms = n0.elapsed_time(n1)
        if dist is not None:
            t = torch.tensor([nms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            nms = float(t)
        no_elision = {"value": world * s.frames / (nms / a.steps * 1e-3), "unit": UNIT, "ms_per_step": nms / a.steps,
                      "what": "rtk_debug_key_elision(0): pass 2 of the scoring also visits the key patches (whose score the "
                              "reference overwrites with 1.0 before the top-k); same kept indices"}

    # ---- end to end: inputs in pinned host memory, H2D + D2H inside the timed region
    e2e = None
    if not a.no_e2e:
        h2d = sum(h.numel() * h.element_size() for h in host)
        # two device input sets: the H2D copy of step i+1 runs on a copy stream while step i computes (a serving loop
        # would do the same); every step still copies all of its inputs from pinned host memory and reads its result back
        bufs = [[torch.empty_like(h, device=dev) for h in host] for _ in range(2)]
        copy_stream = torch.cuda.Stream(device=dev)
        ready = [torch.cuda.Event(), torch.cuda.Event()]
        freed = [torch.cuda.Event(), torch.cuda.Event()]

        def enqueue_copy(i):
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(freed[i % 2])
                for dst, src in zip(bufs[i % 2], host):
                    dst.copy_(src, non_blocking=True)
                ready[i % 2].record(copy_stream)

        sync_all()
        for ev in freed:
            ev.record()
        e0.record()
        d2h = 0
        results = []
        enqueue_copy(0)
        for i in range(a.steps):
            if i + 1 < a.steps:
                enqueue_copy(i + 1)
            torch.cuda.current_stream().wait_event(ready[i % 2])
            xd, qd, kd, vd = bufs[i % 2]
            keep_idx, seq = run_step(s, xd, qd, kd, vd, rotary, lc, vc, pos_grid)
            freed[i % 2].record()
            # the step's result goes back to pinned host memory on the compute stream, without stalling the host: the copy
            # is ordered before e1, so every step's read-back completes inside the timed region
            back = torch.empty(keep_idx.shape, dtype=keep_idx.dtype, pin_memory=True)
            back.copy_(keep_idx, non_blocking=True)
            results.append(back)
            d2h = back.numel() * back.element_size()
        e1.record()
        sync_all()
        assert all(1 <= int(r.numel()) <= s.keep and 0 <= int(r[-1]) < s.L for r in results)       # the read-backs really arrived
        ems = e0.elapsed_time(e1)
        if dist is not None:
            t = torch.tensor([ems], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ems = float(t)
        e2e = {"value": world * s.frames / (ems / a.steps * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h}
        del bufs

    # ---- N > 1: the within-video split (BASELINE config 3) next to the data-parallel headline
    sharded = None
    if world > 1 and not a.no_sharded:
        sharded = sharded_within_video(dev, dist, rank, world)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (of measured)" if peaks else "fallback 1.4 PFLOP/s sustained (of fallback)"
    score_ms = timer.mean_ms()
    flops = 2.0 * s.H * s.L * s.L * s.D
    achieved = flops / (score_ms * 1e-3) / 1e12 if score_ms > 0 else 0.0
    elide = bool(_native.lib().rtk_debug_key_elision(-1))
    executed = 2.0 - (key_patch_share if (elide and key_patch_share is not None) else 0.0)
    roofline = {"kernel": ("pivot_score_kernel<1> + pivot_score_kernel<2> (the scoring of one layer; timed around the batched "
                           f"scoring of a chunk's {s.layers} layers, divided by {s.layers})") if s.deferred else
                          "pivot_score_kernel<1> + pivot_score_kernel<2> (one rtk_pivot_score call)", "bound": "tensor",
                "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                # pass 1 contracts every (query, key) pair, pass 2 only the keys that are not key patches (their score is
                # overwritten with 1.0 before the top-k, longvideo_cache.py:272-274)
                "key_patch_share": key_patch_share, "executed_over_algorithmic": executed,
                "achieved_executed": executed * achieved, "frac_executed": executed * achieved / peak_tf, "peak_source": peak_src,
                "ms_per_call": score_ms, "calls_timed": len(timer.pairs),
                # dram__bytes_read.sum + dram__bytes_write.sum of both launches per layer from the committed `ncu --set full`
                # capture - used only when that capture was taken from THIS build and shape, else null (never a stale constant)
                "traffic": measured_traffic(s),
                # an exact two-pass softmax needs 2*H*L^2 fp32 ex2; B200 issues 16 MUFU per clock and SM
                "xu_floor_ms": executed * s.H * s.L * s.L / (16.0 * 148 * 1.9e9) * 1e3,
                "frac_of_xu_floor": (executed * s.H * s.L * s.L / (16.0 * 148 * 1.9e9) * 1e3) / score_ms if score_ms > 0 else 0.0,
                "note": ("algorithmic = ONE Q.K^T (2*H*L^2*D); the exact two-pass softmax executes it once for the row statistics and "
                         "once more for the keys that are not key patches, and is bounded by "
                         "MUFU.EX2 throughput and the softmax warps' instruction stream (XU pipe 76-79 % busy; xu_floor_ms = "
                         "executed_over_algorithmic*H*L^2 exps at 16/clk/SM, 1.9 GHz), not by the tensor pipe (37 % busy); the kernel also holds the board at its "
                         "1 kW power cap (clocks.reasons sw_power_cap; profiles/r1_score_power_probe.json: the TMA + MMA feeder alone "
                         "needs 0.245 ms per call at 1 kW) - DESIGN.md section 5")}
    # the first timed step follows a synchronisation: the GPU is idle when its DPSelect is launched, so the host's own
    # latency (event record, output allocation, the ctypes call: 40-70 us) sits inside that pair.  From the second step on
    # the device queue is ahead of the host and the pair brackets the three kernels only - that is the figure reported;
    # the first one is kept next to it
    dps_all = [a.elapsed_time(b) for a, b in timer.dpselect]
    dps_steady = dps_all[1:] if len(dps_all) > 1 else dps_all
    dps_ms = sum(dps_steady) / max(1, len(dps_steady))
    hbm = peaks.get("hbm_gbs", 6650.0)
    dps_bytes = 2.0 * s.T * s.N * s.C + 4.0 * s.T * s.N + 4.0 * s.t * s.N * s.C
    dpselect_roofline = {"kernels": "dpselect_dis + dpselect_select_patch + dpselect_gather: one rtk_dpselect_keyframe call, all three "
                                    "this library's own kernels (r_v = 1 is an identity gather through the same kernel)", "bound": "hbm",
                         "achieved": dps_bytes / (dps_ms * 1e-3) / 1e9 if dps_ms > 0 else 0.0, "peak": hbm, "unit": "GB/s",
                         "frac": (dps_bytes / (dps_ms * 1e-3) / 1e9 / hbm) if dps_ms > 0 else 0.0, "ms_per_call": dps_ms,
                         "algorithmic_bytes": dps_bytes, "calls_averaged": len(dps_steady),
                         "ms_first_call_after_sync": dps_all[0] if dps_all else None}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic", "config": config, "roofline": roofline, "roofline_dpselect": dpselect_roofline,
            "gpu_launches": int(launches),
            "step_ms": {"median": sorted(per_step)[len(per_step) // 2], "min": min(per_step), "max": max(per_step),
                        # host time to enqueue one step (first step, GPU idle, and the median of the rest): when it approaches
                        # the device time the step is bound by the Python host, not by the kernels
                        "host_enqueue_first": host_s[0] * 1e3, "host_enqueue_median": sorted(host_s)[len(host_s) // 2] * 1e3}}
    line["build_id"] = _native.build_id()
    if dps_half is not None:
        hms, hby = dps_half
        line["roofline_dpselect_rv0.5"] = {"bound": "hbm", "achieved": hby / (hms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                                           "frac": hby / (hms * 1e-3) / 1e9 / hbm, "ms_per_call": hms, "algorithmic_bytes": hby,
                                           "what": f"the same operator at t = T/2 = {max(1, s.T // 2)} (five back-to-back calls before the timed region)"}
    if parity is not None:
        line["parity"] = parity
    if sharded is not None:
        line["sharded_within_video"] = sharded
    if immediate is not None:
        line["immediate_compression"] = immediate
    if no_elision is not None:
        line["no_key_elision"] = no_elision
    if e2e is not None:
        line["e2e"] = e2e
    if clocks is not None:
        line["clocks"] = clocks
    if world == 1 and not a.no_cpu_baseline:
        torch.set_num_threads(os.cpu_count())
        cpu_host = [h[:2] if i else h for i, h in enumerate(host)]
        cpu_reference_step(s, 16, cpu_host, 0)                      # warm the CPU path
        sec, td, tu, kind = cpu_reference_step(s, 64, cpu_host, 1)
        line["cpu_baseline"] = {"value": s.frames / sec, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind,
                                "sample": (f"DPSelect on 64 of {s.T} grids ({td:.2f} s) + 1 of {s.chunks * s.layers} compressing "
                                           f"updates at L={s.L} ({tu:.2f} s), scaled linearly (extrapolated)")}
    emit(line)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
