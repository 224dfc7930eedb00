"""The kernels at the edges of their supported sizes (include/rtk_b200.h): DPSelect selection up to T = 8192, MA-LLM up to
T = C = 8192, PivotKV up to L = 16384, the distance kernel at N = 2^20, and the generic row gather.

Between the sizes the other GPU tests run and these limits the host code switches between implementations by shared-memory
size.  Every switch point below is computed from the device's opt-in shared memory per block with the formula the host
code uses, and each test asserts which side of it its shape lands on, so a later change of a constant cannot silently move
a test onto the other path.  References are the ones the rest of the suite trusts: the reference's torch op sequence run
on the same GPU (bit-exact where the kernels replay it) and, for the PivotKV scores, cuBLAS with the 1-ulp tolerance plus an
fp64 anchor."""
import math
import time

import pytest
import torch
import torch.nn.functional as F

from helpers import bf16_round, scene_video
from test_gpu_fuzz import _ref_dpselect_indices
from test_gpu_pivotkv import _cfg, _check_keep, _lc, qkv, ref_head_scores_cuda, ulp_diff

pytestmark = pytest.mark.gpu
BF = torch.bfloat16


def _optin():
    """largest dynamic + static shared memory one block may opt into (232 448 B on a B200)"""
    return torch.cuda.get_device_properties(0).shared_memory_per_block_optin


def _vc():
    from retake import visual_compression as vc
    return vc


@pytest.fixture(scope="module", autouse=True)
def _peak_memory():
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    yield
    _BANK.clear()
    print(f"\ntest_gpu_envelope: peak device memory {torch.cuda.max_memory_allocated() / 1e9:.1f} GB, "
          f"{time.perf_counter() - t0:.0f} s")


# ============================================================================================================ DPSelect
# rtk_dpselect_select, sync = 0: a CTA holds W patch columns of T fp32 distances + T peak flags (5 bytes per frame)
SEL_SPLIT_N = 296                                    # W shrinks while the grid would have fewer CTAs (about two per SM)


def _select_patches_per_cta(T, N):
    W = 8
    while W > 1 and (N + W - 1) // W < SEL_SPLIT_N:
        W //= 2
    while W > 1 and W * T * 5 > _optin():
        W //= 2
    return W


def _select_tstar():
    """first T at which eight patch columns no longer fit into one block's shared memory (5812 on a B200)"""
    return _optin() // (8 * 5) + 1


def _select_T(where):
    return {"below": _select_tstar() - 1, "at": _select_tstar(), "limit": 8192}[where]


def _tied_distances(T, N, seed, negative):
    """distances from a small alphabet (ties at the cut), optionally shifted negative with both signed zeros"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    levels = 7
    dis = torch.randint(0, levels, (T, N), generator=g, device="cuda").float() / levels
    dis[0] = 1.0
    if negative:
        dis = dis - 3.0 / levels
        dis[dis.abs() < 1e-6] = -0.0
        dis[torch.rand(T, N, generator=g, device="cuda") < 0.05] = 0.0
    return dis


def _gpu_scene_video(T, N, C, seed, dup_every):
    """scene-structured bf16 bank [1, T, N, C] generated on the GPU (runs of similar frames, exact repeats every dup_every)"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    sid = (torch.rand(T, generator=g, device="cuda") < 0.3).cumsum(0)
    scenes = torch.randn(int(sid.max()) + 1, N, C, generator=g, device="cuda")
    x = scenes[sid]
    x += 0.3 * torch.randn(T, N, C, generator=g, device="cuda")
    x[dup_every::dup_every] = x[dup_every - 1:-1:dup_every].clone()
    return x.to(BF)[None]


@pytest.mark.parametrize("sync", [False, True])
@pytest.mark.parametrize("N", [7, 729, 1200, 4096])
@pytest.mark.parametrize("where", ["below", "at", "limit"])
def test_dpselect_select_at_the_frame_limit(where, N, sync):
    """both sides of the 8-column switch and the documented limit; N = 7, 729, 1200, 4096 run 1, 2, 4 and 8 columns per
    CTA below the switch (7 and 729 are not multiples of 4: the row mean of sync mode takes its unaligned paths)"""
    T = _select_T(where)
    assert T <= 8192
    W = _select_patches_per_cta(T, N)
    assert (8 * T * 5 <= _optin()) == (where == "below")       # which side of the switch this T is on
    rule = {7: 1, 729: 2, 1200: 4, 4096: 8}[N]                 # columns per CTA the grid-size rule alone asks for
    assert W * T * 5 <= _optin() and W <= rule and (W == rule) == (rule * T * 5 <= _optin())
    vc = _vc()
    for t, negative in ((T // 3 + 1, False), (T - T // 7, True), (1, True)):
        dis = _tied_distances(T, N, seed=T + N + t, negative=negative)
        idx, mask = vc.dpselect_select(dis, t, sync)
        want_idx, want_mask = _ref_dpselect_indices(dis, t, sync)
        assert torch.equal(idx.long(), want_idx), (T, N, t, sync)
        assert torch.equal(mask, want_mask), (T, N, t, sync)


@pytest.mark.parametrize("sync", [False, True])
@pytest.mark.parametrize("N", [7, 729])
def test_dpselect_operator_at_the_frame_limit(N, sync):
    """memory_bank_compress_keyframe at T = 8192: distances, kept indices, mask and compacted bank against the reference's
    op sequence on the GPU"""
    from oracle import reference_ops as ro
    vc = _vc()
    T, C = 8192, 256
    assert 8 * T * 5 > _optin()
    x = _gpu_scene_video(T, N, C, seed=N + int(sync), dup_every=11)
    dis = vc.dpselect_distance(x[0])
    sim = F.cosine_similarity(x[0, :-1], x[0, 1:], dim=-1)
    assert torch.equal(dis, torch.cat([torch.ones_like(sim[:1], dtype=torch.float32), 1 - sim.float()], dim=0))
    del sim
    for t in (T // 4, T - 1):
        out, mask, idx = vc.memory_bank_compress_keyframe(x, t, 3, sync=sync, return_indices=True)
        want_out, want_mask, want_idx = ro.dpselect(x, t, sync)
        assert torch.equal(idx, want_idx) and torch.equal(mask, want_mask), (N, t, sync)
        assert torch.equal(out, want_out), (N, t, sync)


def test_dpselect_distance_at_the_patch_limit():
    """T = 2, N = 2^20 patches (the largest N the distance kernel accepts), C = 256: a 1 GB bank"""
    vc = _vc()
    T, N, C = 2, 1 << 20, 256
    g = torch.Generator(device="cuda").manual_seed(5)
    x = torch.randn(T, N, C, generator=g, device="cuda").to(BF)
    x[1, ::97] = x[0, ::97]                                       # exact repeats: sim == 1
    x[1, 1::89] = -x[0, 1::89]
    got = vc.dpselect_distance(x)
    sim = F.cosine_similarity(x[:-1], x[1:], dim=-1)
    want = torch.cat([torch.ones_like(sim[:1], dtype=torch.float32), 1 - sim.float()], dim=0)
    assert torch.equal(got, want)


# ============================================================================================================== MA-LLM
# rtk_mallm_compress, sync = 0: the per-patch state (25 bytes per frame) stays in shared memory together with two row
# buffers while 25*T + 4*C + 32 bytes (+ 1 KB for the kernel's static shared memory) fit, and with one row buffer
# beyond that.  `where` names the side of that switch: "smem" = two buffers, "global" and "limit" = one buffer.
def _mallm_smem_fits(T, C):
    """two row buffers fit"""
    return 25 * T + 4 * C + 32 + 1024 <= _optin()


def _mallm_tg(C):
    """first T at which two row buffers no longer fit (7945 at C = 8192 on a B200)"""
    return (_optin() - 4 * C - 32 - 1024) // 25 + 1


def _mallm_T(where, C):
    return {"smem": _mallm_tg(C) - 1, "global": _mallm_tg(C), "limit": 8192}[where]


_BANK = {}


def _mallm_bank(T, N, C):
    """scene-structured bank with exact repeats (equal similarities: the lowest-index rule decides); one kept at a time"""
    key = (T, N, C)
    if key not in _BANK:
        _BANK.clear()
        g = torch.Generator().manual_seed(T * 7 + N)
        _BANK[key] = scene_video(g, T, N, C, dup_every=6).to(BF)[None].cuda()
    return _BANK[key]


def _mallm_check(x, t, sync, hard):
    from oracle import reference_ops as ro
    vc = _vc()
    keep = x.clone()
    got, got_size = vc.mallm_compress(x, t, sync=sync, hard=hard)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    want, want_size = ro.mallm_compress(x.clone(), t, sync, hard)
    torch.cuda.synchronize()
    ref_s = time.perf_counter() - t0
    assert torch.equal(x, keep), "the input bank must not be modified"
    assert got.shape == want.shape and torch.equal(got, want)
    assert (got_size is None) if hard else torch.equal(got_size, want_size)
    return ref_s


MALLM_EDGE = [(where, N, hard, dt) for where in ("smem", "global", "limit") for N in (1, 3) for hard in (False, True)
              for dt in (1, 40)]


@pytest.mark.parametrize("where,N,hard,dt", MALLM_EDGE)
def test_mallm_patch_mode_around_the_shared_memory_switch(where, N, hard, dt):
    C = 8192
    T = _mallm_T(where, C)
    assert T <= 8192 and _mallm_smem_fits(T, C) == (where == "smem")
    assert 25 * 8192 + 2 * 8192 + 32 + 1024 <= _optin()        # one buffer fits up to the limit: the host never refuses
    _mallm_check(_mallm_bank(T, N, C), T - dt, False, hard)


@pytest.mark.parametrize("hard", [False, True])
def test_mallm_patch_mode_thousands_of_rounds(hard):
    """N = 1, t = T/2 with one row buffer: about 4000 merges of one patch column"""
    C = 8192
    T = _mallm_tg(C)
    assert not _mallm_smem_fits(T, C)
    ref_s = _mallm_check(_mallm_bank(T, 1, C), T // 2, False, hard)
    print(f"\nMA-LLM reference loop, {T - T // 2} rounds (hard={hard}): {ref_s:.1f} s")


@pytest.mark.parametrize("hard", [False, True])
def test_mallm_sync_mode_at_the_limit(hard):
    """T = C = 8192, 16 rounds: the shared argmax scans 8*T = 64 KB of shared memory"""
    T, C = 8192, 8192
    assert 8 * T > 48 * 1024
    _mallm_check(_mallm_bank(T, 3, C), T - 16, True, hard)


# ============================================================================================================= PivotKV
def test_head_scores_fp64_anchor_at_the_length_limit():
    """Two query heads on one KV head at L = 16384 against the reference's chain with exact dot products: fp64 Q.K^T (exact
    for bf16 inputs with D = 128 terms), rounded to bf16 where the reference rounds (QK^T, / sqrt(D), softmax, sum, mean),
    softmax and sums in fp64.  The kernel has to stay within the same 1-ulp bound as against cuBLAS; cuBLAS' own distance
    from the anchor is printed next to it."""
    lc = _lc()
    H, KVH, L, D = 2, 1, 16384, 128
    q, k, _ = qkv(H, KVH, L, D, 1.0, seed=4242)
    got = lc.pivot_head_scores(q, k)
    cublas = ref_head_scores_cuda(q, k)
    kd = k[0, 0].double()
    s = torch.empty(H, L, dtype=torch.float64, device="cuda")
    for h in range(H):                                                               # one [L, L] fp64 plane at a time
        w = bf16_round(torch.matmul(q[0, h].double(), kd.t()))
        w = (w.to(BF) / math.sqrt(D)).double()                                       # the reference's bf16 / python float
        w = bf16_round(torch.softmax(w, dim=-1))
        s[h] = bf16_round(w.sum(0))                                                 # sum over the queries
        del w
    anchor = bf16_round(s.reshape(KVH, H // KVH, L).mean(1)).to(BF)
    d_kernel = ulp_diff(got, anchor)
    d_cublas = ulp_diff(cublas, anchor)
    print(f"\nfp64 anchor, L={L}: kernel max {int(d_kernel.max())} ulp on {float((d_kernel > 0).float().mean()):.4%}, "
          f"cuBLAS max {int(d_cublas.max())} ulp on {float((d_cublas > 0).float().mean()):.4%}")
    rel = ((got.float() - anchor.float()).abs() / anchor.float().abs().clamp_min(1e-6)).max()
    assert float(rel) <= 1e-2
    assert int(d_kernel.max()) <= 1 and float((d_kernel > 0).float().mean()) < 0.02


@pytest.mark.parametrize("reforge", [False, True])
@pytest.mark.parametrize("deferred", [False, True])
def test_update_at_the_length_limit(deferred, reforge):
    """L = 16384, two chunks, 3-D mrope positions, 30 % key patches: kept set against the reference's scores, kept V / K /
    positions exact; immediate (rtk_pivot_update) and deferred (rtk_pivot_update_batch) compression"""
    from helpers import TableRotary
    from oracle import pivotkv as op
    lc = _lc()
    H, KVH, L, D, ratio = 28, 4, 16384, 128, 0.25
    rot = TableRotary(D)
    rot.inv_freq = rot.inv_freq.cuda()
    mrope = [16, 24, 24]
    cfg = _cfg(H, KVH, D, 1, ratio, reforge)
    cfg.longvideo_kwargs["kvcache_compression_kwargs"]["deferred_compression"] = deferred
    cache = lc.PivotKVCache(cfg)
    keep = int(ratio * L)
    past = 0
    for chunk in range(2):
        q, k, v = qkv(H, KVH, L, D, 1.0, seed=700 + chunk)
        mask = (torch.rand(L, generator=torch.Generator().manual_seed(70 + chunk)) < 0.3).cuda()
        cache.kvcache_compression = True
        cache.keypatches_mask_chunk = mask
        base = int(cache.get_prev_temporal_idx(0)) + 1 if reforge else 64 * chunk
        ar = torch.arange(L)
        pos = torch.stack([base + ar // 256, (ar % 256) // 16, ar % 16])[:, None].cuda()
        ko, vo = cache.update(k, v, 0, {"query_states": q, "position_ids": pos, "rotary_emb": rot, "mrope_section": mrope})
        assert ko.shape == (1, KVH, past + L, D) and torch.equal(ko[:, :, past:], k) and torch.equal(vo[:, :, past:], v)
        cache.after_forward()
        idx = cache.last_keep_indices.long()
        assert idx.numel() == keep and bool((idx[1:] > idx[:-1]).all())
        qq, kk = q, k
        if reforge:
            cos, sin = rot(v, pos)
            c1, s1 = op.select_mrope(cos, mrope), op.select_mrope(sin, mrope)
            qq = op.unrotate(q, c1, s1, rot.attention_scaling, "cuda")
            kk = op.unrotate(k, c1, s1, rot.attention_scaling, "cuda")
        ref_hs = ref_head_scores_cuda(qq, kk)
        _check_keep(cache.last_keep_indices, cache.last_head_scores.mean(0), ref_hs.mean(0), mask, keep)
        assert torch.equal(cache.layers[0].values[:, :, past:], v[:, :, idx])
        if not reforge:
            assert torch.equal(cache.layers[0].keys[:, :, past:], k[:, :, idx])
        else:
            want_pos = pos[..., idx].clone()
            want_pos[0] = op.reforge_temporal(want_pos[0], keep, L)
            assert torch.equal(cache.position_cache[0][..., past:], want_pos)
            cos, sin = rot(v, want_pos)
            want_k = op.rotate(kk[:, :, idx], op.select_mrope(cos, mrope), op.select_mrope(sin, mrope))
            assert torch.equal(cache.layers[0].keys[:, :, past:], want_k)
        past += keep
        assert cache.get_seq_length(0) == past and cache.num_evicted_tokens[0] == (chunk + 1) * (L - keep)


# ==================================================================================================== rtk_gather_rows
@pytest.mark.parametrize("rows", [0, 1, 100_000])
@pytest.mark.parametrize("row_bytes", [16, 7168, 16400])
def test_gather_rows_bit_exact(row_bytes, rows):
    """out[i] = x[src_row[i]] for 16-byte multiples of row length (16400 B: a ragged tail behind the 8-vector batches),
    unsorted and repeated source rows; zero rows write nothing"""
    from retake import _native
    n_src = 5000
    g = torch.Generator(device="cuda").manual_seed(row_bytes + rows)
    x = torch.randint(0, 256, (n_src, row_bytes), generator=g, device="cuda", dtype=torch.uint8)
    src = torch.randint(0, n_src, (max(rows, 1),), generator=g, device="cuda", dtype=torch.int64)
    if rows > 2:
        src[:3] = torch.tensor([n_src - 1, 0, n_src - 1])                    # both ends, and a repeat
    out = torch.full((max(rows, 1), row_bytes), 0xA5, dtype=torch.uint8, device="cuda")
    before = out.clone()
    rc = _native.lib().rtk_gather_rows(x.data_ptr(), row_bytes, src.data_ptr(), rows, out.data_ptr(),
                                       _native.stream_ptr(x.device))
    assert rc == 0
    if rows == 0:
        assert torch.equal(out, before)
    else:
        assert torch.equal(out, x.index_select(0, src))
