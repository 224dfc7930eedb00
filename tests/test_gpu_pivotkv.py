"""GPU parity: PivotKV kernels (through the C ABI) against the oracle and against the reference's own
torch-op sequence executed on the same B200."""
import math
import types

import pytest
import torch

from helpers import TableRotary, load_golden
from oracle import pivotkv as op

pytestmark = pytest.mark.gpu
BF = torch.bfloat16


def _lc():
    from retake import longvideo_cache as lc
    return lc


def qkv(H, KVH, L, D, alpha, seed, transposed=True):
    """bf16 q/k/v as the attention forward hands them over: [1, heads, L, D] views of [1, L, heads, D]."""
    g = torch.Generator().manual_seed(seed)
    def mk(h, a):
        t = (torch.randn(1, L, h, D, generator=g) * a).to(BF).cuda()
        return t.transpose(1, 2) if transposed else t.transpose(1, 2).contiguous()
    return mk(H, alpha), mk(KVH, alpha), mk(KVH, 1.0)


def ref_head_scores_cuda(q, k):
    """longvideo_cache.py:260-269 with stock ATen/cuBLAS ops on the GPU (the reference as it runs on CUDA).  Beyond
    L = 6272 the [H, L, L] logits of one call would take tens of GB: there one KV-head group is scored at a time."""
    H, KVH, L, D = q.shape[1], k.shape[1], q.shape[2], q.shape[3]
    if L > 6272 and KVH > 1:
        G = H // KVH
        return torch.cat([ref_head_scores_cuda(q[:, g * G:(g + 1) * G], k[:, g:g + 1]) for g in range(KVH)])
    kr = k[:, :, None].expand(1, KVH, H // KVH, L, D).reshape(1, H, L, D)
    w = torch.matmul(q, kr.transpose(2, 3)) / math.sqrt(D)
    w = torch.nn.functional.softmax(w, dim=-1, dtype=torch.float32).to(q.dtype)
    w = w[0].sum(1)
    return w.reshape(KVH, -1, L).mean(1)


def ulp_diff(a, b):
    """difference in bf16 ulps for positive bf16 tensors"""
    ia = a.view(torch.int16).int()
    ib = b.view(torch.int16).int()
    return (ia - ib).abs()


SCORE_SHAPES = [(4, 2, 128, 64, 1.0), (4, 2, 1024, 64, 1.0), (14, 2, 96, 64, 3.0), (28, 4, 256, 128, 1.0),
                (28, 4, 1000, 128, 3.0), (8, 8, 130, 128, 1.0), (28, 4, 4096, 128, 1.0), (4, 1, 1, 128, 1.0),
                (28, 4, 2304, 128, 3.0),
                # the length and head limits (rtk_b200.h): 12289 = 96 full tiles and one ragged one, H = 256
                (28, 4, 8192, 128, 1.0), (28, 4, 12289, 128, 1.0), (28, 4, 16384, 128, 1.0), (16, 2, 16384, 64, 1.0),
                (256, 32, 1024, 128, 1.0)]


@pytest.mark.parametrize("H,KVH,L,D,alpha", SCORE_SHAPES)
def test_head_scores_vs_reference_ops_on_cuda(H, KVH, L, D, alpha):
    lc = _lc()
    q, k, _ = qkv(H, KVH, L, D, alpha, seed=L + H)
    got = lc.pivot_head_scores(q, k)
    want = ref_head_scores_cuda(q, k)
    assert got.shape == (KVH, L) and got.dtype == BF
    rel = ((got.float() - want.float()).abs() / want.float().abs().clamp_min(1e-6)).max()
    assert float(rel) <= 1e-2, f"max relative score error {float(rel):.4f} > 1e-2 (north_star tolerance)"
    d = ulp_diff(got, want)
    frac = float((d > 0).float().mean())
    assert int(d.max()) <= 1 and frac < 0.02, f"{frac:.4%} of bf16 scores differ, max {int(d.max())} ulp"
    # every query row sums to one, so scores average G-independently to exactly ~1 per key
    assert abs(float(got.float().mean()) - 1.0) < 5e-3


@pytest.mark.parametrize("H,KVH,L,D,alpha", SCORE_SHAPES[:6])
def test_head_scores_vs_oracle(H, KVH, L, D, alpha):
    lc = _lc()
    q, k, _ = qkv(H, KVH, L, D, alpha, seed=7 * L + H)
    got = lc.pivot_head_scores(q, k)
    _, _, b = op.pivot_scores(q.contiguous(), k.contiguous(), "cuda", return_partials=True)
    d = ulp_diff(got, b)
    assert int(d.max()) <= 1 and float((d > 0).float().mean()) < 0.02


def test_head_scores_layout_independent():
    lc = _lc()
    q, k, _ = qkv(28, 4, 384, 128, 1.0, seed=3)
    a = lc.pivot_head_scores(q, k)
    b = lc.pivot_head_scores(q.contiguous(), k.contiguous())
    assert torch.equal(a, b)


@pytest.mark.parametrize("L,keep", [(16, 8), (1024, 512), (4096, 1024), (4096, 499), (6272, 1568), (2304, 2304),
                                    (1, 1), (130, 1), (16384, 4096), (16384, 16384), (16383, 1)])
def test_select_bit_exact_vs_torch_on_cuda(L, keep):
    lc = _lc()
    g = torch.Generator().manual_seed(L + keep)
    KVH = 4
    # few distinct bf16 values -> heavy ties at the boundary (SURVEY.md 8a: ~33 distinct scores at L=1024)
    hs = (0.75 + torch.randint(0, 24, (KVH, L), generator=g).float() / 64).to(BF).cuda()
    for with_mask in (False, True):
        mask = (torch.rand(L, generator=g) < 0.2).cuda() if with_mask else None
        idx, score = lc.pivot_select(hs, keep, mask, return_scores=True)
        want_score = hs.mean(0)                                              # ATen-CUDA mean
        assert torch.equal(score, want_score)
        s = want_score.clone()
        if mask is not None:
            s.masked_fill_(mask, 1.0)
        want = s.topk(keep).indices.sort().values                            # reference lines 276-277 on CUDA
        assert torch.equal(idx.long(), want)


def test_select_matches_reference_on_reference_scores():
    """bit-exact kept indices when fed the reference's own per-head scores"""
    lc = _lc()
    q, k, _ = qkv(28, 4, 2048, 128, 1.0, seed=5)
    hs = ref_head_scores_cuda(q, k)
    g = torch.Generator().manual_seed(1)
    mask = (torch.rand(2048, generator=g) < 0.3).cuda()
    for keep in (1, 250, 512, 1024, 2048):
        idx = lc.pivot_select(hs, keep, mask)
        s = hs.mean(0)
        s.masked_fill_(mask, 1.0)
        assert torch.equal(idx.long(), s.topk(keep).indices.sort().values)


@pytest.mark.parametrize("mrope", [[16, 24, 24], None])
def test_rope_bit_exact_vs_reference_ops_on_cuda(mrope):
    lc = _lc()
    H, KVH, L, D = 28, 4, 333, 128
    q, k, _ = qkv(H, KVH, L, D, 1.0, seed=9)
    rot = TableRotary(D, mrope=mrope is not None)
    tt = torch.arange(L) // 16
    pos = torch.stack([tt, (torch.arange(L) % 16) // 4, torch.arange(L) % 4])[:, None] if mrope else torch.arange(L)[None] + 5
    pos = pos.cuda()
    rot.inv_freq = rot.inv_freq.cuda()
    cos, sin = rot(k, pos)
    c1, s1 = op.select_mrope(cos, mrope), op.select_mrope(sin, mrope)

    def rh(x):
        return torch.cat((-x[..., D // 2:], x[..., :D // 2]), dim=-1)
    for x in (q, k):
        want = ((x * c1.unsqueeze(1)) - (rh(x) * s1.unsqueeze(1))) / rot.attention_scaling ** 2     # reverse=True
        got = lc.pivot_rope(x, cos, sin, mrope, rot.attention_scaling, forward=False)
        assert torch.equal(got, want)
        want_f = (x * c1.unsqueeze(1)) + (rh(x) * s1.unsqueeze(1))
        got_f = lc.pivot_rope(x, cos, sin, mrope, 1.0, forward=True)
        assert torch.equal(got_f, want_f)
        assert torch.equal(op.unrotate(x, c1, s1, rot.attention_scaling, "cuda"), want)            # oracle == ATen-CUDA


@pytest.mark.parametrize("reforge", [False, True])
def test_compact_bit_exact(reforge):
    lc = _lc()
    H, KVH, L, D = 28, 4, 1000, 128
    _, k, v = qkv(H, KVH, L, D, 1.0, seed=11)
    g = torch.Generator().manual_seed(2)
    keep = 377
    idx = torch.randperm(L, generator=g)[:keep].sort().values.cuda()
    pos = torch.stack([100 + torch.arange(L) // 32, (torch.arange(L) % 32) // 8, torch.arange(L) % 8])[:, None].cuda()
    for p in (pos, pos[0]):
        ko, vo, po = lc.pivot_compact(k, v, idx.int(), p, reforge=reforge)
        assert torch.equal(ko, k[:, :, idx]) and torch.equal(vo, v[:, :, idx])
        want = p[..., idx].clone()
        if reforge:
            want[0] = op.reforge_temporal(want[0], keep, L)                 # torch ops on CUDA (lines 293-295)
        assert torch.equal(po, want)


def _cfg(H, KVH, D, layers, ratio, reforge):
    cfg = types.SimpleNamespace(hidden_size=H * D, num_hidden_layers=layers, num_attention_heads=H, num_key_value_heads=KVH)
    cfg.longvideo_kwargs = {"kvcache_compression": True,
                            "kvcache_compression_kwargs": {"compression_ratio": ratio, "compression_method": "pivotkv",
                                                           "pos_embed_reforge": reforge}}
    return cfg


def _check_keep(idx, score, score_ref, keymask, keep):
    """tie/ulp-aware comparison of a kept index set against reference scores (SURVEY.md 8a note N4)."""
    s = score.clone().float()
    r = score_ref.clone().float()
    if keymask is not None:
        s[keymask] = 1.0
        r[keymask] = 1.0
    # self-consistent with the documented rule on the kernel's own scores: exact
    want_self = torch.sort(s, descending=True, stable=True).indices[:keep].sort().values
    assert torch.equal(idx.long(), want_self)
    # against the reference scores: everything clearly above the threshold is kept, nothing clearly below
    kth = torch.sort(r, descending=True).values[keep - 1]
    ulp = kth.abs() * 2 ** -7
    kept = torch.zeros_like(r, dtype=torch.bool)
    kept[idx.long()] = True
    assert bool(kept[r > kth + ulp].all()) and not bool(kept[r < kth - ulp].any())


def test_update_replays_golden_steps_bf16():
    """frozen reference runs (CPU, bf16) replayed through the CUDA cache: shapes, bookkeeping, values as gathers,
    kept sets tie/ulp-aware against the oracle's CUDA-semantics scores."""
    lc = _lc()
    cases = [c for c in load_golden("pivotkv_reference")
             if c["name"] in ("chunks_bf16_reforge", "chunks_bf16_noreforge")]
    assert len(cases) == 2
    for case in cases:
        rot = TableRotary(**case["rotary"])
        rot.inv_freq = rot.inv_freq.cuda()
        cache = lc.PivotKVCache(_cfg(case["H"], case["KVH"], case["D"], 2, case["ratio"], case["reforge"]))
        orc = op.OraclePivotKVCache(case["H"], case["KVH"], case["D"], case["ratio"], case["reforge"], "cuda", "lowest")
        for st in case["steps"]:
            cache.kvcache_compression = True
            cache.keypatches_mask_chunk = st["mask"].cuda()
            orc.keypatches_mask_chunk = st["mask"].cuda()
            q, k, v, pos = st["q"].cuda(), st["k"].cuda(), st["v"].cuda(), st["pos"].cuda()
            ko, vo = cache.update(k, v, st["layer"], {"query_states": q, "position_ids": pos.clone(), "rotary_emb": rot,
                                                      "mrope_section": case["mrope"]})
            oko, ovo = orc.update(k, v, st["layer"], query_states=q, position_ids=pos.clone(), rotary_emb=rot,
                                  mrope_section=case["mrope"])
            assert tuple(ko.shape) == st["k_out_shape"] and torch.equal(ko, oko) and torch.equal(vo, ovo)
            L = case["L"]
            keep = max(1, int(case["ratio"] * L))
            score = cache.last_head_scores.float().mean(0).to(BF)
            _check_keep(cache.last_keep_indices, score, orc.last_scores, st["mask"].cuda(), keep)
            assert cache.layers[st["layer"]].keys.shape == st["key_cache"].shape
            assert cache.num_evicted_tokens[st["layer"]] == st["evicted"]
            if torch.equal(cache.last_keep_indices.long(), orc.last_keep):
                assert torch.equal(cache.layers[st["layer"]].values, orc.value_cache[st["layer"]])
                assert torch.equal(cache.layers[st["layer"]].keys, orc.key_cache[st["layer"]])
                if case["reforge"]:
                    assert torch.equal(cache.position_cache[st["layer"]], orc.position_cache[st["layer"]])
            # keep both caches in lock-step for the next chunk
            orc.key_cache[st["layer"]] = cache.layers[st["layer"]].keys
            orc.value_cache[st["layer"]] = cache.layers[st["layer"]].values
            if case["reforge"]:
                orc.position_cache[st["layer"]] = cache.position_cache[st["layer"]]


@pytest.mark.parametrize("reforge", [False, True])
def test_update_full_size_chunk(reforge):
    """7B shape, L = 4096, two chunks: cache growth, passthrough mode, index parity on reference scores"""
    lc = _lc()
    H, KVH, L, D, ratio = 28, 4, 4096, 128, 0.25
    rot = TableRotary(D)
    rot.inv_freq = rot.inv_freq.cuda()
    mrope = [16, 24, 24]
    cache = lc.PivotKVCache(_cfg(H, KVH, D, 1, ratio, reforge))
    keep = int(ratio * L)
    past = 0
    for chunk in range(2):
        q, k, v = qkv(H, KVH, L, D, 1.0, seed=100 + chunk)
        g = torch.Generator().manual_seed(chunk)
        mask = (torch.rand(L, generator=g) < 0.15).cuda()
        cache.kvcache_compression = True
        cache.keypatches_mask_chunk = mask
        base = int(cache.get_prev_temporal_idx(0)) + 1 if reforge else 16 * chunk
        pos = torch.stack([base + torch.arange(L) // 256, (torch.arange(L) % 256) // 16, torch.arange(L) % 16])[:, None].cuda()
        ko, vo = cache.update(k, v, 0, {"query_states": q, "position_ids": pos, "rotary_emb": rot, "mrope_section": mrope})
        assert ko.shape == (1, KVH, past + L, D) and torch.equal(ko[:, :, past:], k) and torch.equal(vo[:, :, past:], v)
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
            pc = cache.position_cache[0]
            assert pc.shape == (3, 1, past + keep)
            want_pos = pos[..., idx].clone()
            want_pos[0] = op.reforge_temporal(want_pos[0], keep, L)
            assert torch.equal(pc[..., past:], want_pos)
            cos, sin = rot(v, want_pos)
            want_k = op.rotate(kk[:, :, idx], op.select_mrope(cos, mrope), op.select_mrope(sin, mrope))
            assert torch.equal(cache.layers[0].keys[:, :, past:], want_k)
        past += keep
        assert cache.get_seq_length(0) == past and cache.num_evicted_tokens[0] == (chunk + 1) * (L - keep)
    # text segment / decode: compression off -> plain append
    cache.kvcache_compression = False
    cache.keypatches_mask_chunk = None
    q, k, v = qkv(H, KVH, 7, D, 1.0, seed=5)
    pos = torch.arange(7)[None, None].repeat(3, 1, 1).cuda() + 1000
    ko, vo = cache.update(k, v, 0, {"position_ids": pos})
    assert ko.shape[2] == past + 7 and cache.get_seq_length(0) == past + 7
    if reforge:
        assert cache.position_cache[0].shape[-1] == past + 7


def _hf_rotary():
    import bench
    return bench.make_rotary(torch.device("cuda"))


def test_rope_tables_bit_exact_vs_hf_rotary_module():
    """in-library cos/sin tables == stock HF Qwen2-VL rotary module (YaRN x4) + mrope row selection"""
    lc = _lc()
    rot = _hf_rotary()
    L, D, mrope = 4096, 128, [16, 24, 24]
    ar = torch.arange(L, device="cuda")
    for base in (0, 777, 31000):
        pos = torch.stack([base + ar // 256, (ar % 256) // 16, ar % 16])[:, None]
        x = torch.zeros(1, 4, L, D, dtype=BF, device="cuda")
        cos, sin = rot(x, pos)
        got_c, got_s = lc.pivot_rope_tables(pos, rot.inv_freq, D, mrope, rot.attention_scaling)
        assert torch.equal(got_c, op.select_mrope(cos, mrope)[0]) and torch.equal(got_s, op.select_mrope(sin, mrope)[0])
    r1 = TableRotary(64, mrope=False)
    r1.inv_freq = r1.inv_freq.cuda()
    pos = (torch.arange(300, device="cuda") * 7 + 3)[None]
    cos, sin = r1(torch.zeros(1, 2, 300, 64, dtype=BF, device="cuda"), pos)
    got_c, got_s = lc.pivot_rope_tables(pos, r1.inv_freq, 64, None, r1.attention_scaling)
    assert torch.equal(got_c, cos[0]) and torch.equal(got_s, sin[0])


def test_fused_rotary_path_equals_table_path(monkeypatch):
    """rtk_pivot_update with inv_freq (tables computed in the library) == calling the rotary module like the reference"""
    lc = _lc()
    H, KVH, L, D, mrope = 28, 4, 1024, 128, [16, 24, 24]
    rot = _hf_rotary()
    q, k, v = qkv(H, KVH, L, D, 1.0, seed=77)
    ar = torch.arange(L, device="cuda")
    pos = torch.stack([5 + ar // 256, (ar % 256) // 16, ar % 16])[:, None]
    mask = (torch.rand(L, generator=torch.Generator().manual_seed(1)) < 0.2).cuda()
    res = []
    for tables in ("0", "1"):
        monkeypatch.setenv("RTK_ROTARY_TABLES", tables)
        cache = lc.PivotKVCache(_cfg(H, KVH, D, 1, 0.25, True))
        cache.keypatches_mask_chunk = mask
        cache.update(k, v, 0, {"query_states": q, "position_ids": pos.clone(), "rotary_emb": rot, "mrope_section": mrope})
        res.append((cache.layers[0].keys.clone(), cache.layers[0].values.clone(), cache.position_cache[0].clone(),
                    cache.last_head_scores.clone(), cache.last_keep_indices.clone()))
    for a, b in zip(*res):
        assert torch.equal(a, b)


def test_cache_storage_semantics():
    """in-place append + deferred tail overwrite: what callers can observe"""
    lc = _lc()
    H, KVH, L, D = 4, 2, 256, 64
    cache = lc.PivotKVCache(_cfg(H, KVH, D, 2, 0.5, False))
    q, k, v = qkv(H, KVH, L, D, 1.0, seed=1)
    pos = torch.arange(L, device="cuda")[None]
    ko, vo = cache.update(k, v, 0, {"query_states": q, "position_ids": pos})
    # the returned views hold the UNcompressed chunk until the next cache operation ...
    assert torch.equal(ko, k) and torch.equal(vo, v) and cache.get_seq_length(0) == L // 2
    idx = cache.last_keep_indices.long()
    # ... which a read of the cache itself is: it sees [kept]
    assert torch.equal(cache.key_cache[0], k[:, :, idx]) and torch.equal(cache.layers[0].values, v[:, :, idx])
    assert cache.key_cache[0].shape[2] == L // 2
    # second chunk: past = kept rows of chunk 1, returned view = [kept | chunk 2]
    q2, k2, v2 = qkv(H, KVH, L, D, 1.0, seed=2)
    ko2, vo2 = cache.update(k2, v2, 0, {"query_states": q2, "position_ids": pos + L})
    assert ko2.shape[2] == L // 2 + L and torch.equal(ko2[:, :, :L // 2], k[:, :, idx]) and torch.equal(ko2[:, :, L // 2:], k2)
    # another layer's update settles layer 0 (its attention is already on the stream in a real forward)
    cache.update(k, v, 1, {"query_states": q, "position_ids": pos})
    idx2 = cache.last_keep_indices
    assert cache.layers[0]._pending is None and cache.get_seq_length(0) == L and cache.get_seq_length(1) == L // 2
    # 4.48-style assignment and DynamicCache housekeeping still work
    cache.key_cache[0] = cache.key_cache[0][:, :, :10].clone()
    cache.value_cache[0] = cache.value_cache[0][:, :, :10].clone()
    assert cache.get_seq_length(0) == 10
    cache.kvcache_compression = False
    ko3, _ = cache.update(k[:, :, :3], v[:, :, :3], 0, {"position_ids": pos[:, :3]})
    assert ko3.shape[2] == 13 and cache.get_seq_length(0) == 13
    cache.after_forward()
    assert cache.num_evicted_tokens == [L, L // 2]


@pytest.mark.parametrize("reforge", [False, True])
def test_update_single_token_tail_chunk(reforge):
    """LLaVA-Video has frames * 196 + 1 video tokens, so the last prefill chunk can be ONE token: keep = max(1, int(r)) = 1"""
    lc = _lc()
    H, KVH, D = 28, 4, 128
    rot = TableRotary(D, mrope=False)
    rot.inv_freq = rot.inv_freq.cuda()
    cache = lc.PivotKVCache(_cfg(H, KVH, D, 1, 0.25, reforge))
    total = 0
    for L, base in ((256, 0), (1, 256)):
        q, k, v = qkv(H, KVH, L, D, 1.0, seed=L)
        pos = (torch.arange(L, device="cuda") + (int(cache.get_prev_temporal_idx(0)) + 1 if reforge else base))[None]
        cache.keypatches_mask_chunk = torch.zeros(L, dtype=torch.bool, device="cuda")
        ko, vo = cache.update(k, v, 0, {"query_states": q, "position_ids": pos, "rotary_emb": rot, "mrope_section": None})
        assert ko.shape[2] == total + L and torch.equal(ko[:, :, total:], k)
        total += max(1, int(0.25 * L))
        assert cache.get_seq_length(0) == total
    assert cache.last_keep_indices.tolist() == [0] and cache.layers[0].keys.shape[2] == 65
    if reforge:
        assert cache.position_cache[0].shape == (1, 65)


@pytest.mark.parametrize("mrope", [[16, 24, 24], None])
@pytest.mark.parametrize("reverse", [False, True])
def test_reference_named_rotary_helpers(mrope, reverse):
    """`apply_multimodal_rotary_pos_emb` / `apply_rotary_pos_emb` keep the reference's signatures (longvideo_cache.py:36-116)
    and its bf16 expression, bit for bit, in both tensor layouts."""
    from retake import longvideo_cache as lc
    g = torch.Generator().manual_seed(17)
    H, KVH, L, D = 6, 2, 300, 128
    q = torch.randn(1, H, L, D, generator=g).to(torch.bfloat16).cuda()
    k = torch.randn(1, KVH, L, D, generator=g).to(torch.bfloat16).cuda()
    rot = TableRotary(D, mrope=mrope is not None)
    rot.inv_freq = rot.inv_freq.cuda()
    ar = torch.arange(L, device="cuda")
    pos = torch.stack([3 + ar // 64, (ar % 64) // 8, ar % 8])[:, None] if mrope else ar[None]
    cos, sin = rot(k, pos)
    scaling = rot.attention_scaling

    def want(x):
        if mrope:
            parts_c, parts_s = cos.split(mrope * 2, dim=-1), sin.split(mrope * 2, dim=-1)
            c = torch.cat([m[i % 3] for i, m in enumerate(parts_c)], dim=-1).unsqueeze(1)
            s = torch.cat([m[i % 3] for i, m in enumerate(parts_s)], dim=-1).unsqueeze(1)
        else:
            c, s = cos.unsqueeze(1), sin.unsqueeze(1)
        if reverse:
            return ((x * c) - (lc.rotate_half(x) * s)) / scaling ** 2
        return (x * c) + (lc.rotate_half(x) * s)

    if mrope:
        gq, gk = lc.apply_multimodal_rotary_pos_emb(q, k, cos, sin, mrope, reverse=reverse, attention_scaling=scaling)
        tq, tk = lc.apply_multimodal_rotary_pos_emb(q.transpose(1, 2), k.transpose(1, 2), cos, sin, mrope, unsqueeze_dim=2,
                                                    reverse=reverse, attention_scaling=scaling)
    else:
        gq, gk = lc.apply_rotary_pos_emb(q, k, cos, sin, reverse=reverse, attention_scaling=scaling)
        tq, tk = lc.apply_rotary_pos_emb(q.transpose(1, 2), k.transpose(1, 2), cos, sin, unsqueeze_dim=2, reverse=reverse,
                                         attention_scaling=scaling)
    assert torch.equal(gq, want(q)) and torch.equal(gk, want(k))
    assert torch.equal(tq.transpose(1, 2), gq) and torch.equal(tk.transpose(1, 2), gk)
    if not reverse:
        only_k = (lc.apply_multimodal_rotary_pos_emb(None, k, cos, sin, mrope) if mrope
                  else lc.apply_rotary_pos_emb(None, k, cos, sin))
        assert only_k[0] is None and torch.equal(only_k[1], gk)


@pytest.mark.parametrize("reforge", [False, True])
def test_update_full_size_llava_shape(reforge):
    """LLaVA-Video shape: L = 6272 tokens per chunk (32 frames x 196), 1-D rotary positions ([1, L], no mrope), then the
    one-token tail chunk the reference produces when frames % 32 == 0 (llava_onevision.py:157-160)."""
    lc = _lc()
    H, KVH, L, D, ratio = 28, 4, 6272, 128, 0.2
    rot = TableRotary(D, mrope=False)
    rot.inv_freq = rot.inv_freq.cuda()
    cache = lc.PivotKVCache(_cfg(H, KVH, D, 1, ratio, reforge))
    past = 0
    for Lc, seed in ((L, 300), (1, 301)):
        keep = max(1, int(ratio * Lc))
        q, k, v = qkv(H, KVH, Lc, D, 2.0, seed=seed)
        g = torch.Generator().manual_seed(seed)
        mask = (torch.rand(Lc, generator=g) < 0.15).cuda()
        cache.kvcache_compression = True
        cache.keypatches_mask_chunk = mask
        base = int(cache.get_prev_temporal_idx(0)) + 1 if reforge else past
        pos = (base + torch.arange(Lc))[None].cuda()
        ko, vo = cache.update(k, v, 0, {"query_states": q, "position_ids": pos, "rotary_emb": rot, "mrope_section": None})
        assert ko.shape == (1, KVH, past + Lc, D) and torch.equal(ko[:, :, past:], k)
        idx = cache.last_keep_indices.long()
        assert idx.numel() == keep and (keep == 1 or bool((idx[1:] > idx[:-1]).all()))
        qq, kk = q, k
        if reforge:
            cos, sin = rot(v, pos)
            qq = op.unrotate(q, cos, sin, rot.attention_scaling, "cuda")
            kk = op.unrotate(k, cos, sin, rot.attention_scaling, "cuda")
        ref_hs = ref_head_scores_cuda(qq, kk)
        _check_keep(cache.last_keep_indices, cache.last_head_scores.mean(0), ref_hs.mean(0), mask, keep)
        assert torch.equal(cache.layers[0].values[:, :, past:], v[:, :, idx])
        if reforge:
            want_pos = pos[..., idx].clone()
            want_pos[0] = op.reforge_temporal(want_pos[0], keep, Lc)
            assert torch.equal(cache.position_cache[0][..., past:], want_pos)
            cos, sin = rot(v, want_pos)
            assert torch.equal(cache.layers[0].keys[:, :, past:], op.rotate(kk[:, :, idx], cos, sin))
        else:
            assert torch.equal(cache.layers[0].keys[:, :, past:], k[:, :, idx])
        past += keep
