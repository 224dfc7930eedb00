"""Pin the oracle against outputs frozen from the unmodified reference (tests/golden/make_golden.py).

CPU only.  ``tie="torch"`` replays ``torch.topk`` on the same device the reference ran on, so
everything must be bit-identical; ``tie="lowest"`` (the CUDA rule the kernels implement) must agree
wherever the selection boundary is tie-free and be tie-consistent otherwise.
"""

import pytest
import torch

from helpers import TableRotary, load_golden
from oracle import dpselect as od
from oracle import pivotkv as op

DP = load_golden("dpselect_reference")
PK = load_golden("pivotkv_reference")


def _id(c):
    return f"{c['name']}-t{c['t']}-{'sync' if c['sync'] else 'patch'}"


@pytest.mark.parametrize("case", DP, ids=_id)
def test_dpselect_matches_reference_exactly(case):
    out, mask = od.memory_bank_compress_keyframe(case["x"], case["t"], 3, sync=case["sync"], tie="torch")
    assert out.dtype == case["out"].dtype and out.shape == case["out"].shape
    assert torch.equal(mask, case["mask"])
    assert torch.equal(out, case["out"])


@pytest.mark.parametrize("case", DP, ids=_id)
def test_dpselect_lowest_tie_rule_is_consistent(case):
    x, t, sync = case["x"], case["t"], case["sync"]
    out, mask, idx, dis = od.memory_bank_compress_keyframe(x, t, 3, sync=sync, tie="lowest", return_indices=True)
    d = dis.mean(1, keepdim=True) if sync else dis
    keys = d + 2.0 * od.peak_mask(d).float()
    idx2 = idx.reshape(t, -1)
    kth = keys.gather(0, idx2).min(0).values                      # smallest kept key per column
    kept = torch.zeros_like(keys, dtype=torch.bool).scatter_(0, idx2, True)
    assert bool((kept | (keys <= kth)).all())                     # nothing above the threshold is dropped
    assert bool((~kept | (keys >= kth)).all())
    # among keys equal to the threshold the lowest indices are the ones kept
    eq = keys == kth
    for p in range(keys.shape[1]):
        e = torch.nonzero(eq[:, p])[:, 0]
        ke = kept[e, p]
        n = int(ke.sum())
        assert bool(ke[:n].all()) and not bool(ke[n:].any())
    # if the boundary is tie-free the result equals the reference's
    if bool((eq.sum(0) == 1).all()):
        assert torch.equal(mask, case["mask"])
        assert torch.equal(out, case["out"])


def test_kat_d1_known_answers():
    """SURVEY.md 8c KAT-D1 literal values."""
    c = [c for c in DP if c["name"] == "kat_d1"][0]
    dis = od.adjacent_cosine_distance(c["x"][0])
    want0 = [1, .015192, .00060910, .62539, .00060910, .0013704, .57738, .00015223]
    want1 = [1, .00015229, .98255, .00015229, .00015223, .53053, .00015235, .64163]
    assert torch.allclose(dis[:, 0], torch.tensor(want0), rtol=2e-3, atol=2e-7)
    assert torch.allclose(dis[:, 1], torch.tensor(want1), rtol=2e-3, atol=2e-7)
    pk = od.peak_mask(dis)
    assert torch.nonzero(pk[:, 0])[:, 0].tolist() == [0, 3, 6]
    assert torch.nonzero(pk[:, 1])[:, 0].tolist() == [0, 2, 5, 7]
    assert torch.nonzero(od.peak_mask(dis.mean(1)))[:, 0].tolist() == [0, 2, 7]
    x = c["x"]
    _, m, idx, _ = od.memory_bank_compress_keyframe(x, 5, sync=False, return_indices=True)
    assert idx.tolist() == [[0, 0], [1, 2], [3, 5], [5, 6], [6, 7]]
    assert m.int().tolist() == [1, 1, 0, 1, 1, 1, 0, 0, 1, 1]
    _, m, idx, _ = od.memory_bank_compress_keyframe(x, 3, sync=False, return_indices=True)
    assert idx.tolist() == [[0, 0], [3, 2], [6, 7]] and bool(m.all())
    _, m = od.memory_bank_compress_keyframe(x, 8, sync=False)
    assert m.int().tolist() == [1, 1, 0, 0, 0, 1, 1, 0, 0, 0, 0, 1, 1, 0, 0, 1]
    _, m, idx, _ = od.memory_bank_compress_keyframe(x, 5, sync=True, return_indices=True)
    assert idx.tolist() == [0, 2, 3, 6, 7] and m.int().tolist() == [1, 1, 1, 1, 0, 0, 0, 0, 1, 1]
    _, m = od.memory_bank_compress_keyframe(x, 8, sync=True)
    assert m.int().tolist() == [1, 1, 0, 0, 1, 1, 0, 0, 0, 0, 0, 0, 0, 0, 1, 1]
    assert od.memory_bank_compress_keyframe(x, 3, sync=True, return_indices=True)[2].tolist() == [0, 2, 7]
    assert od.memory_bank_compress_keyframe(x, 2, sync=True, return_indices=True)[2].tolist() == [0, 2]


def _aten_peaks(rows):
    """the reference's peak rule on rows [R, T] (visual_compression.py:121-123): max_pool1d_with_indices, CPU"""
    import torch.nn.functional as F
    arg = F.max_pool1d_with_indices(rows[:, None, :], 3, 1, padding=1)[1][:, 0]
    return arg == torch.arange(rows.shape[1])[None]


def test_peak_mask_equals_max_pool_on_nan_and_inf_patterns():
    """oracle peak rule == ATen's max_pool1d_with_indices on every pattern of {NaN, +inf, -inf, 0, 1, 2} over 5 frames,
    NaN runs of length 1-3 at the start, middle and end of long columns, and the sync layout (one row)"""
    vals = torch.tensor([float("nan"), float("inf"), float("-inf"), 0.0, 1.0, 2.0])
    T = 5
    codes = torch.cartesian_prod(*[torch.arange(len(vals))] * T)                     # [6^5, 5]
    rows = vals[codes]
    want = _aten_peaks(rows)
    assert torch.equal(od.peak_mask(rows.t().contiguous()).t(), want)
    for r in range(0, rows.shape[0], 997):                                            # the 1-D (sync) form
        assert torch.equal(od.peak_mask(rows[r]), want[r])
    g = torch.Generator().manual_seed(8)
    cols = []
    for run in (1, 2, 3):
        for at in (0, 20, 40 - run):
            c = torch.rand(40, generator=g)
            c[at:at + run] = float("nan")
            cols.append(c)
    for fill in (float("inf"), float("-inf")):
        c = torch.rand(40, generator=g)
        c[5:8] = fill
        c[30:32] = fill
        cols.append(c)
    rows = torch.stack(cols)
    assert torch.equal(od.peak_mask(rows.t()).t(), _aten_peaks(rows))
    # the pattern of one bad bank element: two adjacent NaN distances; the second one is the peak
    d = torch.tensor([1.0, .95, .96, .97, .95, float("nan"), float("nan"), .95, 1.04, 1.0])
    assert torch.nonzero(od.peak_mask(d))[:, 0].tolist() == [0, 3, 6, 8]
    assert torch.equal(od.peak_mask(d), _aten_peaks(d[None])[0])


def test_aten_cuda_rowsum_agrees_with_plain_sum():
    g = torch.Generator().manual_seed(3)
    x = torch.randn(64, 1152, generator=g)
    for vec in (4, 8):
        a = od.aten_cuda_rowsum(x, vec)
        assert torch.allclose(a, x.sum(-1), rtol=1e-5, atol=1e-4)
        b = od.aten_cuda_rowsum(x, vec, square=True)
        assert torch.allclose(b, (x * x).sum(-1), rtol=1e-5)


# ----------------------------------------------------------------------------- PivotKV
def _kat(c):
    return f"{c['name']}-{str(c['q'].dtype).split('.')[-1]}-{'mask' if c['mask'] is not None else 'nomask'}"


KAT = [c for c in PK if c["name"] == "kat_p1"]
REPLAY = [c for c in PK if c["name"] != "kat_p1"]


@pytest.mark.parametrize("case", KAT, ids=_kat)
def test_kat_p1(case):
    q, k, v = case["q"], case["k"], case["v"]
    cache = op.OraclePivotKVCache(4, 2, 8, 0.5, False, semantics="cpu", tie="torch")
    cache.keypatches_mask_chunk = case["mask"]
    ko, vo = cache.update(k, v, 0, query_states=q, position_ids=case["pos"], mrope_section=case["mrope"])
    assert torch.equal(ko, case["k_out"]) and torch.equal(vo, case["v_out"])
    want = [1, 2, 7, 8, 10, 12, 13, 15] if case["mask"] is not None else [1, 2, 5, 7, 8, 10, 12, 13]
    assert cache.last_keep.tolist() == want                      # SURVEY.md 8c literal
    assert torch.equal(cache.key_cache[0], case["key_cache"])
    assert torch.equal(cache.value_cache[0], case["value_cache"])
    assert cache.num_evicted_tokens == case["evicted"]
    # the CUDA tie rule: identical without the mask; with it the four mask-filled 1.0 scores tie at the
    # boundary (CPU topk kept {10, 15}, an arbitrary pick) and the lowest-index rule keeps {0, 5}
    c2 = op.OraclePivotKVCache(4, 2, 8, 0.5, False, semantics="cuda", tie="lowest")
    c2.keypatches_mask_chunk = case["mask"]
    c2.update(k, v, 0, query_states=q, position_ids=case["pos"], mrope_section=case["mrope"])
    if case["mask"] is None:
        assert c2.last_keep.tolist() == want
    else:
        assert c2.last_keep.tolist() == [0, 1, 2, 5, 7, 8, 12, 13]


def _replay(case, semantics, tie):
    rot = TableRotary(**case["rotary"])
    cache = op.OraclePivotKVCache(case["H"], case["KVH"], case["D"], case["ratio"], case["reforge"],
                                  semantics=semantics, tie=tie)
    res = []
    for st in case["steps"]:
        cache.keypatches_mask_chunk = st["mask"]
        ko, vo = cache.update(st["k"], st["v"], st["layer"], query_states=st["q"], position_ids=st["pos"].clone(),
                              rotary_emb=rot, mrope_section=case["mrope"])
        res.append((tuple(ko.shape), cache.key_cache[st["layer"]].clone(), cache.value_cache[st["layer"]].clone(),
                    cache.position_cache[st["layer"]].clone() if case["reforge"] else None,
                    cache.num_evicted_tokens[st["layer"]], cache.last_scores.clone(), cache.last_keep.clone()))
    return res


@pytest.mark.parametrize("case", [c for c in REPLAY if c["dtype"] == torch.float32], ids=lambda c: c["name"])
def test_replay_fp32_exact(case):
    for st, r in zip(case["steps"], _replay(case, "cpu", "torch")):
        assert r[0] == st["k_out_shape"]
        assert r[4] == st["evicted"]
        assert torch.equal(r[2], st["value_cache"])
        if case["reforge"]:
            assert torch.equal(r[3], st["position_cache"])
        torch.testing.assert_close(r[1], st["key_cache"], rtol=2e-6, atol=2e-6)


@pytest.mark.parametrize("case", [c for c in REPLAY if c["dtype"] == torch.bfloat16], ids=lambda c: c["name"])
def test_replay_bf16(case):
    """bf16: the oracle's fp32-matmul-then-round equals the reference's bf16 matmul up to
    accumulation order, so compare exactly where it is exact and count the rest."""
    steps = case["steps"]
    res = _replay(case, "cpu", "torch")
    same_v = sum(torch.equal(r[2], st["value_cache"]) for st, r in zip(steps, res))
    for st, r in zip(steps, res):
        assert r[0] == st["k_out_shape"] and r[4] == st["evicted"]
        assert r[1].shape == st["key_cache"].shape
    # values are pure gathers: identical whenever the kept index set is identical
    assert same_v == len(steps), f"only {same_v}/{len(steps)} steps reproduced the reference's kept set"
    for st, r in zip(steps, res):
        torch.testing.assert_close(r[1].float(), st["key_cache"].float(), rtol=1e-2, atol=1e-2)
        if case["reforge"]:
            assert torch.equal(r[3], st["position_cache"])


def test_cuda_and_cpu_semantics_differ_only_in_last_bit():
    c = [c for c in REPLAY if c["name"] == "chunks_bf16_noreforge"][0]
    st = c["steps"][0]
    a = op.pivot_scores(st["q"], st["k"], "cpu").float()
    b = op.pivot_scores(st["q"], st["k"], "cuda").float()
    assert float(((a - b).abs() / a.abs().clamp_min(1e-6)).max()) <= 2 ** -7
    assert abs(float(a.mean()) - 1.0) < 0.02                      # scores average 1 per key (note N3)


# ------------------------------------------------------------- second oracle form: the reference's own op sequence
from oracle import reference_ops as ro  # noqa: E402


@pytest.mark.parametrize("case", DP, ids=_id)
def test_reference_ops_dpselect_bit_identical(case):
    out, mask, _ = ro.dpselect(case["x"], case["t"], case["sync"])
    assert torch.equal(mask, case["mask"]) and torch.equal(out, case["out"])


@pytest.mark.parametrize("case", REPLAY, ids=lambda c: c["name"])
def test_reference_ops_pivot_update_bit_identical(case):
    """first chunk of every layer (empty past): cache == kept K/V/positions, all dtypes incl. bf16"""
    rot = TableRotary(**case["rotary"])
    n = 0
    for st in case["steps"]:
        if st["chunk"] != 0:
            continue
        kk, vv, pos, idx, _ = ro.pivot_update(st["q"], st["k"], st["v"], case["ratio"], st["mask"], st["pos"].clone(),
                                              rot, case["mrope"], case["reforge"])
        assert torch.equal(kk, st["key_cache"]) and torch.equal(vv, st["value_cache"])
        if case["reforge"]:
            assert torch.equal(pos, st["position_cache"])
        n += 1
    assert n >= 1


# ------------------------------------------------------------------------------------------- MA-LLM compressors
from oracle import mallm as om  # noqa: E402

ML = load_golden("mallm_reference")


def _replay_mallm(case, soft_round, hard_round):
    bank, size = case["x"].clone(), torch.ones_like(case["x"][:, :, :, 0])
    hard = case["x"].clone()
    for r in range(case["n_rounds"]):
        bank, size = soft_round(bank, size, case["sync"])
        hard = hard_round(hard, case["sync"])
        if r in case["rounds"]:
            want = case["rounds"][r]
            assert torch.equal(bank, want["bank"]) and torch.equal(size, want["size"]), f"soft round {r}"
            assert torch.equal(hard, want["hard"]), f"hard round {r}"
    assert bank.shape[1] == case["t"]


@pytest.mark.parametrize("case", ML, ids=lambda c: f"{c['name']}-{'sync' if c['sync'] else 'patch'}")
def test_mallm_explicit_oracle_matches_reference_every_round(case):
    def soft(b, s, sync):
        o, z, _ = om.mallm_round(b[0], s[0], sync)
        return o[None], z[None]
    _replay_mallm(case, soft, lambda b, sync: om.mallm_hard_round(b[0], sync)[0][None])


@pytest.mark.parametrize("case", ML, ids=lambda c: f"{c['name']}-{'sync' if c['sync'] else 'patch'}")
def test_mallm_reference_ops_match_reference_every_round(case):
    _replay_mallm(case, ro.mallm_round, ro.mallm_hard_round)


def test_mallm_rescale_map_is_idempotent():
    """x -> rd(rd(x * s) / s) reaches a fixed point after ONE application for every bf16 mantissa and every size the
    kernels can meet - the property the incremental CUDA implementation leans on (it still re-checks dynamically)."""
    m = torch.arange(128, dtype=torch.float32) / 128 + 1
    x = torch.cat([m * 2.0 ** e for e in (-3, 0, 2)]).to(torch.bfloat16)
    for s in range(1, 1025):
        sb = torch.tensor(float(s)).to(torch.bfloat16)
        if float(sb) != s:
            continue
        once = (x * sb) / sb
        assert torch.equal((once * sb) / sb, once)


def test_aten_cuda_rowmean_model_is_a_mean():
    g = torch.Generator().manual_seed(2)
    for n in (24, 96, 128, 136, 256, 729):
        v = torch.randn(11, n, generator=g).to(torch.bfloat16).float()
        got = om.aten_cuda_bf16_rowmean(v)
        want = v.double().mean(-1).float()
        assert torch.allclose(got, want, rtol=2 ** -7, atol=1e-3)
