"""GPU parity on special values: DPSelect, MA-LLM and the rotary tables on zero, clamp-window, subnormal, overflowing
and non-finite inputs, and the rotary tables at long-video positions.

Every target is the reference's own torch op sequence run on the same GPU (``F.cosine_similarity``,
``F.max_pool1d_with_indices``, ``torch.topk``, ``oracle/reference_ops.py``, the HF rotary module); the oracle is never
the target.  Every comparison goes through ``same``: equal shapes, equal NaN positions, equal bits everywhere else
(so -0 and +0 differ)."""
import math

import pytest
import torch
import torch.nn.functional as F

from helpers import TableRotary, scene_video
from oracle import pivotkv as op
from oracle import reference_ops as ro

pytestmark = pytest.mark.gpu
BF = torch.bfloat16
NAN, INF = float("nan"), float("inf")


def _vc():
    from retake import visual_compression as vc
    return vc


def _lc():
    from retake import longvideo_cache as lc
    return lc


def same(a, b, what=""):
    """equal shapes and dtypes, NaN where the other is NaN, and bit equality everywhere else"""
    assert a.shape == b.shape, f"{what}: shape {tuple(a.shape)} != {tuple(b.shape)}"
    assert a.dtype == b.dtype, f"{what}: dtype {a.dtype} != {b.dtype}"
    if not a.is_floating_point():
        bad = int((a != b).sum())
        assert bad == 0, f"{what}: {bad}/{a.numel()} entries differ"
        return
    na, nb = torch.isnan(a), torch.isnan(b)
    assert torch.equal(na, nb), f"{what}: NaN at {int((na ^ nb).sum())} differing positions"
    it = {2: torch.int16, 4: torch.int32, 8: torch.int64}[a.element_size()]
    ia, ib = a.masked_fill(na, 0).view(it), b.masked_fill(nb, 0).view(it)
    bad = ia != ib
    if bool(bad.any()):
        k = torch.nonzero(bad)[0].tolist()
        raise AssertionError(f"{what}: {int(bad.sum())}/{a.numel()} values differ in their bits, first at {k}: "
                             f"{a[tuple(k)].item()!r} vs {b[tuple(k)].item()!r}")


# ------------------------------------------------------------------------------------------------ special rows
EPS_BITS = 0x322c                        # bf16(1e-8), the norm clamp of F.cosine_similarity


def _bf16_bits(bits):
    return torch.tensor([bits], dtype=torch.int16).view(BF).float()[0]


def special_row(kind, C, g):
    """one fp32 row [C] whose bf16 rounding is the planted value (bf16-exact where it matters)"""
    r = torch.randn(C, generator=g)
    k = int(torch.randint(0, C, (1,), generator=g))
    if kind == "zero":
        return torch.zeros(C)
    if kind == "clamp_inside":                                # norm ~ 1e-10, well inside the clamp window
        return r * (1e-10 / math.sqrt(C))
    if kind in ("clamp_at", "clamp_below", "clamp_above"):    # norm == bf16(1e-8) exactly, and one bf16 step either side
        bits = EPS_BITS + {"clamp_at": 0, "clamp_below": -1, "clamp_above": 1}[kind]
        row = torch.zeros(C)
        row[k] = _bf16_bits(bits) * (1 if bool(r[0] > 0) else -1)
        return row
    if kind == "subnormal":                                   # every element a bf16 subnormal: the squares underflow
        return r * 2.0 ** -129
    if kind == "some_subnormal":
        row = r.clone()
        row[::5] = r[::5] * 2.0 ** -130
        return row
    if kind == "outlier24":                                   # one channel 2^24 above the rest
        row = r.clone()
        row[k] = 2.0 ** 24
        return row
    if kind == "outlier_deep":                                # the rest ~2^-64 of the norm: products below 2^-126
        row = r * 2.0 ** -70
        row[k] = 2.0 ** -6
        return row
    if kind == "overflow":                                    # elements near 2^64: the fp32 sum of squares is inf
        return r.sign() * 2.0 ** 63 * (1 + 0.9 * torch.rand(C, generator=g))
    if kind == "below_overflow":                              # a sum of squares just below FLT_MAX
        return r.sign() * math.sqrt(2.0 ** 127.6 / C) * (0.9 + 0.1 * torch.rand(C, generator=g))
    if kind in ("pinf", "ninf", "nan"):
        row = r.clone()
        row[k] = {"pinf": INF, "ninf": -INF, "nan": NAN}[kind]
        return row
    if kind == "nan_row":
        return torch.full((C,), NAN)
    if kind == "huge":                                        # near bf16 max: a merge with size >= 2 overflows to inf
        return r.sign() * 2.0 ** 127 * (1 + 0.9 * torch.rand(C, generator=g))
    raise ValueError(kind)


ROW_KINDS = ["zero", "clamp_inside", "clamp_at", "clamp_below", "clamp_above", "subnormal", "some_subnormal", "outlier24",
             "outlier_deep", "overflow", "below_overflow", "pinf", "ninf", "nan", "nan_row"]
# "neg" / "dup": the row is the negated / exact copy of the row before it
NEIGHBOUR_KINDS = ["neg", "dup"]


def plant(x, frames, g, kinds):
    """x fp32 [T, N, C]: at each frame f of `frames`, patch p gets kind (p + f) % len(kinds) in frames f and f + 1 (the
    second copy drawn again, so that pairs of one kind meet pairs of mixed kinds); returns the bf16 bank"""
    T, N, C = x.shape
    for f in frames:
        for p in range(N):
            kind = kinds[(p + f) % len(kinds)]
            for ff in (f, f + 1):
                if ff >= T:
                    continue
                if kind == "neg":
                    x[ff, p] = -x[ff - 1, p] if ff > 0 else x[ff, p]
                elif kind == "dup":
                    x[ff, p] = x[ff - 1, p] if ff > 0 else x[ff, p]
                else:
                    x[ff, p] = special_row(kind, C, g)
    return x.to(BF)


def test_special_rows_are_what_they_claim():
    """the planted rows: exact clamp-window norms, bf16 subnormals, an inf sum of squares, one just below"""
    g = torch.Generator().manual_seed(0)
    C = 256
    for kind, bits in (("clamp_at", EPS_BITS), ("clamp_below", EPS_BITS - 1), ("clamp_above", EPS_BITS + 1)):
        r = special_row(kind, C, g).to(BF)
        n = torch.linalg.vector_norm(r.float())
        assert n.to(BF).view(torch.int16).item() == bits and float(n) == float(n.to(BF))
    s = special_row("subnormal", C, g).to(BF).float()
    assert bool((s.abs() < 2.0 ** -126).all()) and bool((s != 0).sum() > C // 2)
    assert math.isinf(float((special_row("overflow", C, g).to(BF).float() ** 2).sum()))
    ss = float((special_row("below_overflow", C, g).to(BF).float() ** 2).sum())
    assert 2.0 ** 127 < ss < 3.4e38


# ----------------------------------------------------------------------------------------- A: distance kernel
def ref_dis_cuda(x):
    """visual_compression.py:100-106 with stock ATen ops on the GPU"""
    sim = F.cosine_similarity(x[None, :-1], x[None, 1:], dim=-1)[0]
    d = 1 - sim.type(torch.float)
    return torch.cat([torch.ones_like(d[:1]), d], dim=0)


def dis_runs(T, N, C):
    """(run length R, streaming warps per CTA) of launch_dis (dpselect.cu) on this device: run r reads rows
    [r*R, r*R + R] and emits the distances of frames r*R + 1 ..."""
    prop = torch.cuda.get_device_properties(torch.cuda.current_device())
    sms, smem_max = prop.multi_processor_count, prop.shared_memory_per_block_optin
    k4 = (C // 4 + 31) // 32
    K4 = next(k for k in (2, 4, 9, 16, 28, 32, 48, 64) if k4 <= k or k == 64)
    ctas = 2 if K4 <= 16 else 1
    row_bytes = 2 * C
    active = 8
    stages = (smem_max // ctas - 2048) // (active * row_bytes)
    while stages < 2 and active > 2:
        active >>= 1
        stages = (smem_max // ctas - 2048) // (active * row_bytes)
    assert stages >= 2
    frames = T - 1
    R = (frames * N) // (sms * active * ctas * 4)
    R = min(max(R, 4), 32, frames)
    return R, active


DIS_C = [256, 264, 1152, 3584, 8184, 8192]


@pytest.mark.parametrize("C", DIS_C)
@pytest.mark.parametrize("halo", [0, 1])
def test_distance_special_rows(C, halo):
    """rtk_dpselect_dis == F.cosine_similarity on CUDA for banks with special rows planted at frame 0, T-1 and at the
    first rows of the kernel's runs (exact and ragged rows, the two-CTA and the fewer-active-warps instantiations)"""
    vc = _vc()
    T, N = 66, 34
    R, active = dis_runs(T, N, C)
    if C >= 8184:
        assert active < 8, "the long rows are meant to reach the fewer-active-warps path"
    starts = list(range(0, T - 1, R))
    frames = sorted({0, T - 1} | set(starts[1::2]) | {s + 1 for s in starts[2::3]})
    assert 0 in frames and T - 1 in frames and sum(f % R == 0 for f in frames if f) >= 3, (R, frames)
    g = torch.Generator().manual_seed(C + halo)
    x = plant(torch.randn(T, N, C, generator=g), frames, g, ROW_KINDS + NEIGHBOUR_KINDS).cuda()
    got = vc.dpselect_distance(x, halo=bool(halo))
    want = ref_dis_cuda(x)[1:] if halo else ref_dis_cuda(x)
    same(got, want, f"distances C={C} halo={halo} R={R}")
    assert bool(torch.isnan(got).any()) and bool((got == 1.0).any())


# ------------------------------------------------------------------------------- B: selection and operator
def ref_select(dis, t, sync):
    """visual_compression.py:108-135 / 141-169: max_pool1d_with_indices + topk on CUDA (as oracle/reference_ops.py)"""
    T, N = dis.shape
    rows = dis.mean(1)[None] if sync else dis.t().contiguous()
    arg = F.max_pool1d_with_indices(rows[:, None, :], 3, 1, padding=1)[1][:, 0]
    peak = arg == torch.arange(T, device=dis.device)[None]
    keys = torch.where(peak, rows + 2, rows)
    kept = torch.topk(keys, k=t, sorted=False, dim=1)[1].sort(dim=1)[0]
    if sync:
        idx = kept[0]
        return idx, peak[0][idx][:, None].repeat(1, N).flatten(), peak[0]
    idx = kept.t()
    return idx, peak.t().gather(0, idx).flatten(), peak.t()


def special_columns(T, g):
    """distance columns [T, n] (fp32): NaN runs of length 1-3 at the start, the middle and the end, runs of +inf and
    -inf, ties, and the all-NaN / all -inf / all-equal columns"""
    cols = []
    for run in (1, 2, 3):
        for at in (0, T // 2, T - run):
            c = torch.randint(0, 3, (T,), generator=g).float() * 0.5          # ties
            c[at:at + run] = NAN
            cols.append(c)
            c = torch.rand(T, generator=g) * 2
            c[at:at + run] = NAN
            c[(at + 7) % T] = NAN                                            # a second, isolated NaN
            cols.append(c)
    for fill in (INF, -INF):
        for run in (1, 2, 3):
            c = torch.rand(T, generator=g) * 2
            c[0:run] = fill
            c[T // 3:T // 3 + run] = fill
            c[T - run:] = fill
            cols.append(c)
    c = torch.rand(T, generator=g)
    c[4:6] = INF
    c[6:8] = NAN                                                             # +inf run next to a NaN run
    c[8:10] = -INF
    cols.append(c)
    cols += [torch.full((T,), NAN), torch.full((T,), -INF), torch.full((T,), INF), torch.full((T,), 0.25)]
    return torch.stack(cols, 1)


@pytest.mark.parametrize("T,N", [(97, 40), (300, 700)])
def test_select_patch_mode_special_values(T, N):
    """rtk_dpselect_select (per patch) == max_pool1d_with_indices + topk on CUDA, t in {1, #NaN, #NaN + 1, T/2, T}"""
    vc = _vc()
    g = torch.Generator().manual_seed(T)
    cols = special_columns(T, g)
    reps = (N + cols.shape[1] - 1) // cols.shape[1]
    dis = torch.cat([cols] * reps, 1)[:, :N].clone()
    dis[:, ::3] = torch.where(torch.rand(T, 1, generator=g) < 0.5, dis[:, ::3], -dis[:, ::3])   # and negated copies
    dis = dis.cuda()
    nan_max = int(torch.isnan(dis).sum(0).max())
    nan_min = int(torch.isnan(dis).sum(0)[torch.isnan(dis).sum(0) > 0].min())
    for t in sorted({1, nan_min, nan_min + 1, nan_max, nan_max + 1, T // 2, T} & set(range(1, T + 1))):
        idx, mask = vc.dpselect_select(dis, t, False)
        want_idx, want_mask, _ = ref_select(dis, t, False)
        same(idx.long(), want_idx, f"indices t={t}")
        same(mask, want_mask, f"mask t={t}")


@pytest.mark.parametrize("N", [7, 64, 729])
def test_select_sync_mode_special_values(N):
    """sync mode: a single NaN patch makes the frame's mean NaN, +inf and -inf in one frame make it NaN too"""
    vc = _vc()
    T = 120
    g = torch.Generator().manual_seed(N)
    dis = torch.randint(0, 4, (T, N), generator=g).float() * 0.25
    dis[0] = 1.0
    for run, at in ((1, 1), (2, 30), (3, 60), (2, T - 2)):
        for f in range(at, at + run):
            dis[f, int(torch.randint(0, N, (1,), generator=g))] = NAN
    dis[10, 0] = INF
    dis[11:13, N - 1] = INF
    dis[20, 1 % N] = -INF
    dis[40:42, 0] = -INF
    dis[50, 0], dis[50, N - 1] = INF, -INF                                   # mean NaN without a NaN distance
    if N > 1:
        dis[80, 0], dis[80, 1] = NAN, INF
    dis = dis.cuda()
    n_nan = int(torch.isnan(dis.mean(1)).sum())
    assert n_nan >= 9
    for t in sorted({1, n_nan, n_nan + 1, T // 2, T}):
        idx, mask = vc.dpselect_select(dis, t, True)
        want_idx, want_mask, _ = ref_select(dis, t, True)
        same(idx.long(), want_idx, f"indices t={t}")
        same(mask, want_mask, f"mask t={t}")


BAD_FRAME = ["pinf", "nan_row", "overflow"]


@pytest.mark.parametrize("C", [256, 1152])
@pytest.mark.parametrize("sync", [False, True])
@pytest.mark.parametrize("kind", BAD_FRAME)
def test_keyframe_operator_with_one_bad_frame(kind, sync, C):
    """memory_bank_compress_keyframe == reference_ops.dpselect (F.cosine_similarity, max_pool1d, topk on CUDA) on banks
    in which one frame of some patches is bad: indices, mask and the compressed bank, t = T included"""
    vc = _vc()
    T, N = 24, 64
    g = torch.Generator().manual_seed(C + len(kind) + sync)
    x = scene_video(g, T, N, C)
    for p in range(0, N, 5):
        x[(3 + 7 * p) % T, p] = special_row(kind, C, g)
    x = x.to(BF).cuda()
    for t in (1, 5, T // 2, T - 1, T):
        out, mask, idx = vc.memory_bank_compress_keyframe(x[None], t, 3, sync=sync, return_indices=True)
        w_out, w_mask, w_idx = ro.dpselect(x[None], t, sync)
        same(idx, w_idx, f"{kind} t={t} indices")
        same(mask, w_mask, f"{kind} t={t} mask")
        same(out, w_out, f"{kind} t={t} bank")
    if kind != "overflow":
        assert bool(w_mask.any()) and bool(torch.isnan(ref_dis_cuda(x)).any())


# ---------------------------------------------------------------------------------------------------- C: MA-LLM
MALLM_KINDS = ["zero", "clamp_inside", "clamp_at", "clamp_below", "clamp_above", "subnormal", "outlier24", "outlier_deep",
               "overflow", "below_overflow", "pinf", "ninf", "nan", "nan_row", "huge", "neg", "dup"]


def mallm_bank(T, N, C, seed, kinds):
    g = torch.Generator().manual_seed(seed)
    x = scene_video(g, T, N, C)
    plant_frames = list(range(1, T - 1, 5))
    x = plant(x, plant_frames, g, kinds).float()
    # runs of zero frames and of clamp-window frames in every patch
    x[T - 6:T - 3] = 0.0
    x[T - 3:T - 1] = torch.stack([special_row("clamp_inside", C, g) for _ in range(2 * N)]).reshape(2, N, C)
    return x.to(BF)


@pytest.mark.parametrize("C", [264, 1152])
@pytest.mark.parametrize("N", [7, 64, 136])
@pytest.mark.parametrize("hard", [False, True])
@pytest.mark.parametrize("sync", [False, True])
def test_mallm_special_values(sync, hard, N, C):
    """mallm_compress == the reference's MA-LLM loop (reference_ops) on CUDA, for banks with special rows,
    bf16-overflowing merges and runs of zero and clamp-window frames"""
    vc = _vc()
    T, t = 40, 9
    x = mallm_bank(T, N, C, 1000 * N + C, MALLM_KINDS).cuda()
    out, sizes = vc.mallm_compress(x[None], t, sync=sync, hard=hard)
    w_out, w_sizes = ro.mallm_compress(x[None], t, sync=sync, hard=hard)
    same(out, w_out, "bank")
    if not hard:
        same(sizes, w_sizes, "sizes")


def test_mallm_finite_specials_keep_their_merges():
    """without NaN and inf rows the argmax decides on finite similarities only: the zero, clamp-window, subnormal and
    overflow rows drive the merges (and the bf16 overflow of "huge" merges makes inf rows mid-loop)"""
    vc = _vc()
    kinds = ["zero", "clamp_inside", "clamp_at", "clamp_below", "subnormal", "outlier_deep", "overflow", "below_overflow",
             "huge", "neg", "dup"]
    T, N, C = 48, 64, 1152
    x = mallm_bank(T, N, C, 5, kinds).cuda()
    assert bool(torch.isfinite(x.float()).all())
    for sync in (False, True):
        for hard in (False, True):
            out, sizes = vc.mallm_compress(x[None], 12, sync=sync, hard=hard)
            w_out, w_sizes = ro.mallm_compress(x[None], 12, sync=sync, hard=hard)
            same(out, w_out, f"bank sync={sync} hard={hard}")
            if not hard:
                same(sizes, w_sizes, f"sizes sync={sync}")


@pytest.mark.parametrize("sync", [False, True])
def test_mallm_sizes_in(sync):
    """sizes fed back in (compression_size other than ones): 0.5, 1.5, 3.0078125, 255, 4096 and 8192, against the
    reference's mallm_round loop fed the same sizes"""
    vc = _vc()
    T, N, C, t = 32, 64, 264, 6
    g = torch.Generator().manual_seed(9 + sync)
    x = mallm_bank(T, N, C, 11, ["zero", "clamp_at", "subnormal", "huge", "pinf", "nan", "dup"]).cuda()
    vals = torch.tensor([1.0, 0.5, 1.5, 3.0078125, 255.0, 4096.0, 8192.0])
    sizes = vals[torch.randint(0, len(vals), (1, T, N), generator=g)].to(BF).cuda()
    out, s_out = vc.mallm_compress(x[None], t, sizes, sync=sync)
    bank, size = x[None], sizes.clone()
    while bank.shape[1] > t:
        bank, size = ro.mallm_round(bank, size, sync)
    same(out, bank, "bank")
    same(s_out, size, "sizes")


# ---------------------------------------------------------------------------------- D: rotary at long positions
POS_STARTS = [0, 105615, 105616, 2 ** 17, 401408, 2 ** 20, 2 ** 24 - 1, 2 ** 24 + 1]


def _hf(shape):
    import bench
    return bench.make_rotary(torch.device("cuda"), shape)


@pytest.mark.parametrize("module", ["qwen2vl_mrope", "llava_1d", "theta1e6_1d", "table64_1d"])
def test_rope_tables_at_long_video_positions(module):
    """rtk_pivot_rope_tables == the rotary module on CUDA for positions from 0 to past 2^24, across the point (105 615)
    where CUDA's cosf / sinf switch to their slow argument reduction"""
    lc = _lc()
    L = 2048
    ar = torch.arange(L, device="cuda")
    if module == "qwen2vl_mrope":
        rot, D, mrope = _hf("qwen2vl"), 128, [16, 24, 24]
    elif module == "llava_1d":
        rot, D, mrope = _hf("llava"), 128, None
    elif module == "theta1e6_1d":
        rot, D, mrope = TableRotary(128, base=1e6, attention_scaling=1.0, mrope=False), 128, None
        rot.inv_freq = rot.inv_freq.cuda()
    else:
        rot, D, mrope = TableRotary(64, mrope=False), 64, None
        rot.inv_freq = rot.inv_freq.cuda()
    for base in POS_STARTS:
        if mrope:
            pos = torch.stack([base + ar, base + (ar * 7) % L, base + ar // 3])[:, None]
        else:
            pos = (base + ar)[None]
        cos, sin = rot(torch.zeros(1, 2, L, D, dtype=BF, device="cuda"), pos)
        got_c, got_s = lc.pivot_rope_tables(pos, rot.inv_freq, D, mrope, rot.attention_scaling)
        want_c, want_s = (op.select_mrope(cos, mrope)[0], op.select_mrope(sin, mrope)[0]) if mrope else (cos[0], sin[0])
        same(got_c, want_c, f"cos from {base}")
        same(got_s, want_s, f"sin from {base}")


def _cfg(H, KVH, D, ratio, reforge):
    import types
    cfg = types.SimpleNamespace(hidden_size=H * D, num_hidden_layers=1, num_attention_heads=H, num_key_value_heads=KVH)
    cfg.longvideo_kwargs = {"kvcache_compression": True,
                            "kvcache_compression_kwargs": {"compression_ratio": ratio, "compression_method": "pivotkv",
                                                           "pos_embed_reforge": reforge}}
    return cfg


@pytest.mark.parametrize("reforge", [False, True])
def test_update_at_long_video_positions(reforge, monkeypatch):
    """PivotKVCache.update with 1-D positions past 400 000 (LLaVA-Video at 2048 frames): the fused un-rotation
    (RTK_ROTARY_TABLES=0) equals calling the rotary module (=1); with re-forging the kept keys and positions are the
    reference's un-rotation, re-forged positions and rotation at the kernel's own kept indices"""
    lc = _lc()
    H, KVH, L, D, ratio = 28, 4, 1024, 128, 0.25
    keep = int(ratio * L)
    rot = _hf("llava")
    g = torch.Generator().manual_seed(3)
    q = torch.randn(1, L, H, D, generator=g).to(BF).cuda().transpose(1, 2)
    k = torch.randn(1, L, KVH, D, generator=g).to(BF).cuda().transpose(1, 2)
    v = torch.randn(1, L, KVH, D, generator=g).to(BF).cuda().transpose(1, 2)
    pos = (401408 + 3 * torch.arange(L, device="cuda"))[None]
    mask = (torch.rand(L, generator=g) < 0.2).cuda()
    res = []
    for tables in ("0", "1"):
        monkeypatch.setenv("RTK_ROTARY_TABLES", tables)
        cache = lc.PivotKVCache(_cfg(H, KVH, D, ratio, reforge))
        cache.keypatches_mask_chunk = mask
        cache.update(k, v, 0, {"query_states": q, "position_ids": pos.clone(), "rotary_emb": rot, "mrope_section": None})
        res.append((cache.layers[0].keys.clone(), cache.layers[0].values.clone(),
                    cache.position_cache[0].clone() if reforge else None, cache.last_keep_indices.clone()))
    for a, b in zip(*res):
        if a is not None:
            same(a, b, "RTK_ROTARY_TABLES=0 vs 1")
    kk, vv, pp, idx = res[0]
    i = idx.long()
    assert i.numel() == keep and bool((i[1:] > i[:-1]).all())
    same(vv, v[:, :, i], "kept values")
    if not reforge:
        same(kk, k[:, :, i], "kept keys")
        return
    cos, sin = rot(v, pos)
    k_un = op.unrotate(k, cos, sin, rot.attention_scaling)
    want_pos = pos[..., i].clone()
    want_pos[0] = op.reforge_temporal(want_pos[0], keep, L)
    same(pp, want_pos, "re-forged positions")
    assert int(want_pos.max()) > 400000
    cos2, sin2 = rot(v, want_pos)
    same(kk, op.rotate(k_un[:, :, i], cos2, sin2), "re-rotated keys")
