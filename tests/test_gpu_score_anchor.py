"""The PivotKV scores held to an exact fp64 replay of the reference's rounding chain, on inputs whose logits do not depend on
the accumulation order, at the scoring kernel's tile and split edges.

Q entries come from ``a * {-2, ..., 2}`` and K entries from ``b * {-1, 0, 1}`` with ``a``, ``b`` powers of two and D <= 128: every
partial sum of every accumulation order is a multiple of ``ab`` of magnitude <= 256 ab, exact in bf16 and fp32.  The tcgen05
accumulator, cuBLAS and fp64 then give the same bf16 logit (asserted for every input), and what is left to differ is the
softmax formula (``exp2(s log2e - c_q)`` against ``exp(s - m) / sum``) and fp32 summation orders.  The anchor replays
``P = bf16(softmax(s))``, ``a_h = bf16(sum_q P)``, ``score = bf16(mean over the G heads)`` in fp64 and carries, next to every
rounding, the interval of values a correct implementation may round:

* P: ``z (1 -+ delta_P)`` with ``delta_P = 2^-19 + (|s| log2e + |c_q|) 2^-23`` per element.  The kernel's exponent
  ``s log2e - c_q`` is an fp32 FMA of magnitude up to ``|s| log2e + |c_q|`` (rounding 2^-24 of that, times ln 2 in z) and c_q
  carries the fp32 row sum, ``lg2.approx`` and ``ex2.approx`` errors (each about 2^-22); 2^-19 is their sum with a margin.
  Intervals, not flips counted one by one: with flat rows every P of a column moves together.
* column sum: ``[sum P_lo, sum P_hi]`` widened by ``eps_sum = 2^-18`` relative.  The terms are bf16 values summed in fp32;
  most additions are exact and the rest round at 2^-25 of the running sum, about sqrt(n) 2^-26 (2^-21 at n = 1024 per
  accumulator) in total.  This band is statistical (the rigorous n 2^-24 would excuse everything); it is eight times that.
* head mean: replayed exactly (fp32 sum of the G bf16 values in ATen's 4-accumulator order, times fp32(1/G), rounded to bf16,
  which is what ATen's ``mean`` and the head-reduce kernel do); the ends of the ``a_h`` intervals go through it.

A score passes when it lies in its interval; the interval has two or more candidates ("excused") for under 1 % of the scores,
and the same rule accepts torch-CUDA's op sequence on the same inputs, which keeps the rule honest.

One difference from the reference is known and pinned by ``test_subnormal_window_is_the_one_deviation``: the kernels'
``ex2.approx.ftz`` turns a softmax weight below 2^-126 into 0 where torch-CUDA keeps the fp32 subnormal.  The anchor the
kernels are held to applies that flush (the interval reaches 0 where ``z (1 -+ delta_P)`` crosses 2^-126)."""
import math
import time

import pytest
import torch

from helpers import TableRotary, bf16_round
from oracle import pivotkv as op
from oracle import reference_ops as ro
from test_gpu_pivotkv import _cfg, ref_head_scores_cuda

pytestmark = pytest.mark.gpu
BF = torch.bfloat16
LOG2E = 1.4426950408889634
DELTA_P0 = 2.0 ** -19                 # P stage: fixed part of the relative band
DELTA_P1 = 2.0 ** -23                 # P stage: per unit of |s| log2e + |c_q|
EPS_SUM = 2.0 ** -18                  # column-sum stage
MAX_EXCUSED = 0.01
TINY = 2.0 ** -126                    # smallest normal fp32: ex2.approx.ftz returns 0 below it


def _lc():
    from retake import longvideo_cache as lc
    return lc


@pytest.fixture(scope="module", autouse=True)
def _peak_memory():
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    yield
    print(f"\ntest_gpu_score_anchor: peak device memory {torch.cuda.max_memory_allocated() / 1e9:.1f} GB, "
          f"{time.perf_counter() - t0:.0f} s")


# ====================================================================================== the kernel's work partition
# Python replica of score_launch (grid size) and TileRange (pivot_score.cu): a unit is a head's pair of stationary tiles, the
# (unit, streamed tile) space of a layer is cut into geff equal contiguous ranges, a unit is shared by up to three CTAs.
def score_partition(Hl, L, n_keys=None, sms=None):
    """-> dict(nt, nt_a, grid, geff, ctas = set of CTA counts per unit, odd = odd stationary-tile count); n_keys: the compact
    key count of pass 2 with key elision (None: every key is stationary, as in pass 1)"""
    if sms is None:
        sms = torch.cuda.get_device_properties(0).multi_processor_count
    nt = (L + 127) // 128
    half = (nt + 1) // 2
    units = Hl * ((nt + 1) // 2)
    grid = min(max(units * nt // half, 1), sms)
    nt_a = nt if n_keys is None else (n_keys + 127) // 128
    nta = (nt_a + 1) // 2
    Gl = Hl * nta * nt
    geff = min(max(Gl // half, 1), grid)
    per_unit = [0] * (Hl * nta)
    for b in range(geff):
        g0, g1 = Gl * b // geff, Gl * (b + 1) // geff
        for u in range(g0 // nt, (g1 - 1) // nt + 1) if g1 > g0 else ():
            per_unit[u] += 1
    return {"nt": nt, "nt_a": nt_a, "grid": grid, "geff": geff, "ctas": set(per_unit), "odd": nt_a % 2 == 1}


# ================================================================================================== order-free inputs
def _to_dev(x, a):
    """integer-valued [L, heads, D] -> bf16 [1, heads, L, D] view of a token-major tensor, as the attention forward hands
    it over"""
    return (x * a).to(BF).cuda()[None].transpose(1, 2)


def make_qk(pattern, H, KVH, L, D, seed):
    """(q, k, target keys) for one logit pattern; every entry is a power of two times a small integer (module docstring)"""
    g = torch.Generator().manual_seed(seed)
    qi = torch.randint(-2, 3, (L, H, D), generator=g).float()
    ki = torch.randint(-1, 2, (L, KVH, D), generator=g).float()
    a, b, B = 1.0, 1.0, D // 2
    target = None
    if pattern == "noise":
        pass
    elif pattern.startswith("sink"):                      # one key with a logit 30-45 above the rest, for every query
        j = {"sink0": 0, "sink127": min(127, L - 1), "sink_last": L - 1}[pattern]
        a = b = 2.0
        qi[:, :, :B] = 2
        ki[:, :, :B] = 0
        ki[j, :, :B] = 1
        target = [j]
    elif pattern in ("ramp_up", "ramp_down"):             # logits rise / fall with the key index (about 11 in total)
        b = 2.0
        qi[:, :, :B] = 2
        c = (torch.arange(L) * (B + 1)) // L
        if pattern == "ramp_down":
            c = B - c
        ki[:, :, :B] = (torch.arange(B)[None] < c[:, None]).float()[:, None, :]
    elif pattern == "flat":                               # q = 0: every P is bf16(1/L)
        qi.zero_()
    elif pattern == "dup":                                # groups of identical keys: exactly equal scores
        ki = ki[torch.randint(0, max(1, L // 4), (L,), generator=g)]
    elif pattern == "spread":                             # 1 query in 16 is one-hot on a key of its own
        a = 2.0
        hot = torch.arange(0, L, 16)
        tgt = torch.randint(0, L, (hot.numel(),), generator=g)
        for h in range(H):
            qi[hot, h] = 2 * ki[tgt, h // (H // KVH)]
    elif pattern == "underflow":                          # z of a few keys in [2^-134, 2^-126) for every query
        assert D == 128
        a, b = 4.0, 2.0
        width = torch.where(torch.rand(L, generator=g) < 0.5, 31, 32)
        qi.zero_()
        qi[:, :, :32] = 2 * (torch.arange(32)[None] < width[:, None]).float()[:, None, :]
        ki.zero_()
        ki[0, :, :32] = 1                                 # the sink: about +45 for every query
        target = [L // 3, L // 2, L - 1]
        ki[target, :, :32] = -1                           # the keys about 88-91 below every row's log-normaliser
    else:
        raise ValueError(pattern)
    return _to_dev(qi, a), _to_dev(ki, b), target


def _midpoint_gap(x):
    """relative distance of x > 0 to the nearest bf16 rounding midpoint"""
    _, e = torch.frexp(x)
    quantum = torch.ldexp(torch.ones_like(x), (e.clamp_min(-125) - 8).double())
    t = x / quantum
    return (t - torch.floor(t) - 0.5).abs() * quantum / x.clamp_min(1e-300)


def head_mean(a):
    """[KVH, G, L] bf16 values -> bf16(fp32 sum over G in ATen's 4-accumulator order * fp32(1/G)), as float64: the mean of
    the G query heads replayed exactly (monotone in every a_h, so interval ends map to interval ends)"""
    a = a.float()
    G = a.shape[1]
    v = [torch.zeros_like(a[:, 0]) for _ in range(4)]
    for j in range(G):
        v[j & 3] = v[j & 3] + a[:, j]
    s = ((v[0] + v[1]) + v[2]) + v[3]
    return (s * (torch.tensor(1.0, dtype=torch.float32) / torch.tensor(float(G), dtype=torch.float32)).to(s.device)).to(BF).double()


def anchor(q, k):
    """fp64 replay of the reference's chain with a candidate interval per score (module docstring).  Also asserts that the
    bf16 logits of torch.matmul on the GPU equal the exact ones (the inputs are order-free).
    -> {"exact": (lo, hi, pt, gap), "ftz": (...)}: [KVH, L] float64 bf16 values; ``ftz`` flushes softmax weights below
    2^-126 to 0 like the kernels; ``gap`` is the smallest relative distance of an unrounded column sum or head mean of the
    score to a bf16 rounding midpoint (how close the exact chain came to rounding the other way)"""
    _, H, L, D = q.shape
    KVH = k.shape[1]
    G = H // KVH
    inv = torch.tensor(1.0, dtype=torch.float32) / torch.tensor(math.sqrt(D), dtype=torch.float32)
    inv = inv.cuda()
    cols = {v: [torch.empty(H, L, dtype=torch.float64, device="cuda") for _ in range(3)] for v in ("exact", "ftz")}
    for h in range(H):
        qd, kd = q[0, h].double(), k[0, h // G].double()
        s = qd @ kd.t()                                                            # exact: small integers times ab
        logit = (s.float() * inv).to(BF)                                           # bf16(bf16(QK^T) * fp32(1/sqrt D))
        ref_logit = torch.matmul(q[0, h], k[0, h // G].t()) / math.sqrt(D)         # the reference's ops on the GPU
        assert torch.equal(logit, ref_logit), "logits depend on the summation order"
        del s, ref_logit, qd, kd
        x = logit.double()
        del logit
        m = x.amax(1, keepdim=True)
        z = torch.exp(x - m)
        l = z.sum(1, keepdim=True)
        z /= l
        cq = (m + torch.log(l)) * LOG2E
        delta = DELTA_P0 + (x.abs() * LOG2E + cq.abs()) * DELTA_P1
        del x
        zl, zh = z * (1 - delta), z * (1 + delta)
        del delta
        for v in ("exact", "ftz"):
            for i, y in enumerate((zl, zh, z)):
                r = bf16_round(y)
                if v == "ftz":
                    r = torch.where(y < TINY, 0.0, r)
                cols[v][i][h] = r.sum(0)                                           # sum over the queries
                del r
        del z, zl, zh
    out = {}
    for v, (c_lo, c_hi, c_pt) in cols.items():
        a_lo = bf16_round(c_lo * (1 - EPS_SUM)).view(KVH, G, L)
        a_hi = bf16_round(c_hi * (1 + EPS_SUM)).view(KVH, G, L)
        a_pt = bf16_round(c_pt).view(KVH, G, L)
        gap = torch.minimum(_midpoint_gap(c_pt).view(KVH, G, L).amin(1), _midpoint_gap(a_pt.sum(1) / G))
        out[v] = (head_mean(a_lo), head_mean(a_hi), head_mean(a_pt), gap)
    return out


def with_key_patches(anc, mask):
    """the anchor after the reference's key-patch fill: score 1.0, no interval"""
    out = {}
    for v, (lo, hi, pt, gap) in anc.items():
        lo, hi, pt, gap = lo.clone(), hi.clone(), pt.clone(), gap.clone()
        for t in (lo, hi, pt):
            t[:, mask] = 1.0
        gap[:, mask] = math.inf
        out[v] = (lo, hi, pt, gap)
    return out


def check_rule(got, anc, what):
    """every score inside its interval, fewer than 1 % excused; prints how much of the bands was used.  -> excused [KVH, L]"""
    lo, hi, pt, gap = anc
    g = got.double()
    bad = (g < lo) | (g > hi)
    excused = lo != hi
    differ = g != pt
    frac = float(excused.double().mean())
    worst = float(gap[differ].max()) if bool(differ.any()) else 0.0
    print(f"\n{what}: excused {frac:.4%}, differ from the exact chain {float(differ.double().mean()):.4%}, "
          f"largest midpoint gap among those 2^{math.log2(worst) if worst > 0 else -math.inf:.1f}")
    assert not bool(bad.any()), (
        f"{what}: {int(bad.sum())} scores outside their interval, e.g. got {g[bad][:4].tolist()} "
        f"allowed [{lo[bad][:4].tolist()}, {hi[bad][:4].tolist()}]")
    assert frac < MAX_EXCUSED, f"{what}: {frac:.2%} of the scores excused - the case has lost its power"
    return excused


def check_kept(idx, anc_pt, excused, mask, keep, what):
    """kept indices equal topk(anchor score after the mask fill).indices.sort() (KV-head mean and fill by ATen, which the
    select kernel matches bit for bit), except that they may differ among keys with an excused score"""
    s = anc_pt.to(BF).mean(0)
    if mask is not None:
        s = s.masked_fill(mask, 1.0)
    want = s.topk(keep).indices.sort().values
    idx = idx.long()
    if idx.numel() == want.numel() and torch.equal(idx, want):
        return True
    a = torch.zeros(s.numel(), dtype=torch.bool, device=s.device)
    b = a.clone()
    a[idx] = True
    b[want] = True
    diff = a ^ b
    assert idx.numel() == keep and bool(excused.any(0)[diff].all()), (
        f"{what}: kept set differs from the anchor's on {int(diff.sum())} keys, not all of them excused")
    return False


# ======================================================================================================= shape lists
# (H, KVH, L, D, pattern); the coverage test below asserts what these exercise.  A short chunk gets enough heads for about
# a thousand scores, so that the 1 % bound on excused scores is not one or two scores (L = 1 and 129 excepted)
SCORE_CASES = [
    (4, 1, 600, 128, "noise"), (4, 1, 600, 128, "sink_last"), (16, 2, 640, 64, "ramp_up"), (16, 2, 640, 64, "sink127"),
    (7, 1, 2600, 128, "ramp_down"), (7, 1, 2600, 128, "spread"),
    (28, 4, 1000, 128, "noise"), (28, 4, 1000, 128, "flat"), (28, 4, 1000, 128, "sink0"), (28, 4, 1000, 128, "dup"),
    (28, 4, 4096, 128, "ramp_up"), (2, 2, 16384, 128, "noise"), (256, 32, 1024, 128, "noise"),
    (4, 2, 1, 128, "noise"), (8, 8, 127, 64, "sink_last"), (16, 8, 128, 128, "ramp_up"), (14, 2, 129, 128, "sink_last"),
    (14, 2, 129, 64, "flat"),
]
# (H, KVH, L, D, pattern, key count left by the mask (None: no mask), keep)
UPDATE_CASES = [
    (28, 4, 1000, 128, "noise", None, 250), (28, 4, 1000, 128, "ramp_up", 0, 250), (28, 4, 1000, 128, "dup", 1, 250),
    (4, 2, 1000, 128, "noise", 100, 300), (28, 4, 1000, 128, "sink0", 300, 333), (28, 4, 1000, 128, "spread", 700, 500),
    (28, 4, 4096, 128, "noise", 2900, 1024), (28, 4, 4096, 128, "ramp_down", None, 1024),
    (16, 8, 257, 64, "dup", 129, 64),
]


def _free_keys_mask(L, n_free, seed):
    if n_free is None:
        return None
    g = torch.Generator().manual_seed(seed)
    m = torch.ones(L, dtype=torch.bool)
    m[torch.randperm(L, generator=g)[:n_free]] = False
    return m.cuda()


def test_shape_lists_cover_the_partition_edges():
    """units taken by 1, 2 and 3 CTAs, odd and even stationary-tile counts in pass 1 and in the key-elided pass 2, a pass 2
    on fewer CTAs than the grid, one tile, L = 1 / 127 / 128 / 129, D = 64 / 128, G = 1 / 7 / 8, one KV head, 256 heads"""
    p1 = [score_partition(H, L) for H, _, L, _, _ in SCORE_CASES] + [score_partition(H, L) for H, _, L, *_ in UPDATE_CASES]
    p2 = [score_partition(H, L, n) for H, _, L, _, _, n, _ in UPDATE_CASES if n]
    assert {1, 2, 3} <= set().union(*(p["ctas"] for p in p1))
    assert {True, False} == {p["odd"] for p in p1} == {p["odd"] for p in p2}
    assert 3 in set().union(*(p["ctas"] for p in p2))
    assert any(p["geff"] < p["grid"] for p in p2)
    assert any(p["nt"] == 1 for p in p1)
    shapes = [c[:4] for c in SCORE_CASES] + [c[:4] for c in UPDATE_CASES]
    assert {1, 127, 128, 129} <= {L for _, _, L, _ in shapes}
    assert {64, 128} == {D for *_, D in shapes}
    assert {1, 7, 8} <= {H // KVH for H, KVH, _, _ in shapes}
    assert 1 in {KVH for _, KVH, _, _ in shapes} and 256 in {H for H, *_ in shapes}
    # the benchmark shape with its typical compact key count: an odd pass-2 tile count
    assert score_partition(28, 4096, 2900)["odd"]


@pytest.mark.parametrize("H,KVH,L,D,pattern", SCORE_CASES)
def test_scores_meet_the_fp64_anchor(H, KVH, L, D, pattern):
    """rtk_pivot_score (pivot_head_scores) and torch-CUDA's op sequence against the anchor"""
    lc = _lc()
    q, k, _ = make_qk(pattern, H, KVH, L, D, seed=H * 7 + L)
    anc = anchor(q, k)
    got = lc.pivot_head_scores(q, k)
    part = score_partition(H, L)
    check_rule(got, anc["ftz"], f"kernel {H}x{L}x{D} G={H // KVH} {pattern} (CTAs per unit {sorted(part['ctas'])}, "
                                f"{part['nt_a']} tiles)")
    check_rule(ref_head_scores_cuda(q, k), anc["exact"], f"torch-CUDA {H}x{L}x{D} {pattern}")


@pytest.mark.parametrize("pattern", ["noise", "ramp_down"])
def test_scores_in_three_layouts(pattern):
    """the transposed [1, heads, L, D] view, a contiguous copy and a head-major view with a padded token stride read through
    their own tensor maps: all three meet the anchor and agree bit for bit"""
    lc = _lc()
    H, KVH, L, D = 28, 4, 1000, 128
    q, k, _ = make_qk(pattern, H, KVH, L, D, seed=31)

    def padded(x):
        buf = torch.zeros(1, x.shape[1], L, D + 64, dtype=BF, device="cuda")
        buf[..., :D] = x
        return buf[..., :D]
    anc = anchor(q, k)["ftz"]
    res = []
    for name, qq, kk in (("transposed", q, k), ("contiguous", q.contiguous(), k.contiguous()), ("padded", padded(q), padded(k))):
        assert name != "padded" or qq.stride(2) == D + 64
        res.append(lc.pivot_head_scores(qq, kk))
        check_rule(res[-1], anc, f"kernel {pattern} {name}")
    assert torch.equal(res[0], res[1]) and torch.equal(res[0], res[2])


def test_subnormal_window_is_the_one_deviation():
    """Keys whose softmax weight lies in [2^-134, 2^-126) for every query: torch-CUDA keeps the fp32 subnormal weights, so
    their reference score is a tiny positive number; the kernels' ex2.approx.ftz makes it exactly 0.  Pinned as the one
    known difference (DESIGN.md section 2): the kernel gives 0 exactly there and meets the anchor without the flush
    everywhere else; torch-CUDA meets the anchor without the flush everywhere."""
    lc = _lc()
    H, KVH, L, D = 4, 1, 1000, 128
    q, k, target = make_qk("underflow", H, KVH, L, D, seed=5)
    anc = anchor(q, k)
    got = lc.pivot_head_scores(q, k)
    ref = ref_head_scores_cuda(q, k)
    lo, hi, pt, _ = anc["exact"]
    assert bool((lo[:, target] > 0).all()) and float(pt[:, target].max()) < 2.0 ** -110     # inside the window
    assert bool((anc["ftz"][1][:, target] == 0).all())
    print(f"\nsubnormal window: reference scores of the target keys {ref[:, target].float().tolist()}, kernel "
          f"{got[:, target].float().tolist()}")
    check_rule(ref, anc["exact"], "torch-CUDA, underflow window")
    assert bool((ref[:, target] > 0).all())
    assert bool((got[:, target] == 0).all())
    check_rule(got, anc["ftz"], "kernel, underflow window")
    others = torch.ones(L, dtype=torch.bool, device="cuda")
    others[target] = False
    check_rule(got[:, others], tuple(t[:, others] for t in anc["exact"]), "kernel without the target keys, no flush")


def _check_update(lc, q, k, v, keep, mask, anc, what, reforge=False, rot=None, pos=None, mrope=None):
    kk, vv, pp, idx, hs = lc.pivot_update(q, k, v, keep, mask, pos, rot, mrope, reforge)
    if mask is not None:
        anc = with_key_patches(anc, mask)
        assert bool((hs[:, mask] == 1.0).all())
    excused = check_rule(hs, anc["ftz"], what)
    # the select kernel on the kernel's own scores: ATen's mean, fill and top-k exactly
    s = hs.mean(0)
    if mask is not None:
        s = s.masked_fill(mask, 1.0)
    assert torch.equal(idx.long(), s.topk(keep).indices.sort().values)
    same = check_kept(idx, anc["ftz"][2], excused, mask, keep, what)
    _, _, _, idx_ref, _ = ro.pivot_update(q, k, v, keep / q.shape[2] + 1e-9, mask, pos, rot, mrope, reforge)
    same_ref = check_kept(idx_ref, anc["exact"][2], excused, mask, keep, what + " (reference ops)")
    a = torch.zeros(q.shape[2], dtype=torch.bool, device="cuda")
    b = a.clone()
    a[idx.long()] = True
    b[idx_ref] = True
    assert bool(excused.any(0)[a ^ b].all()), f"{what}: kept set differs from the reference's on keys that are not excused"
    print(f"{what}: kept set equal to the anchor's: {same}, to the reference's: {same_ref}")
    i = idx.long()
    assert torch.equal(vv, v[:, :, i])
    return kk, pp, i


@pytest.mark.parametrize("H,KVH,L,D,pattern,n_free,keep", UPDATE_CASES)
def test_update_meets_the_fp64_anchor(H, KVH, L, D, pattern, n_free, keep):
    """rtk_pivot_update without re-forging: head scores by the anchor rule (key patches exactly 1.0), kept indices equal to
    the anchor's and the reference's top-k up to excused scores, K / V rows exact"""
    lc = _lc()
    q, k, _ = make_qk(pattern, H, KVH, L, D, seed=H + L + (n_free or 0))
    v = torch.randn(1, KVH, L, D, generator=torch.Generator().manual_seed(1)).to(BF).cuda()
    mask = _free_keys_mask(L, n_free, seed=L + 1)
    if n_free is not None:
        part = score_partition(H, L, n_free)
        print(f"\npass 2: {part['nt_a']} compact key tiles, {part['geff']} of {part['grid']} CTAs, "
              f"CTAs per unit {sorted(part['ctas'])}")
    kk, _, i = _check_update(lc, q, k, v, keep, mask, anchor(q, k), f"update {H}x{L} {pattern} free={n_free}")
    assert torch.equal(kk, k[:, :, i])


@pytest.mark.parametrize("tables", ["0", "1"])
def test_reforge_update_meets_the_fp64_anchor(tables, monkeypatch):
    """Re-forging with all-zero positions and attention_scaling 1: cos = 1 and sin = 0 exactly, so the un-rotation is the
    identity, but the scoring reads the un-rotated workspace copies through their own tensor maps.  With the rotary
    module's inv_freq (fused un-rotation) and with its cos/sin tables (RTK_ROTARY_TABLES=1, pivot_rope_kernel)."""
    monkeypatch.setenv("RTK_ROTARY_TABLES", tables)
    lc = _lc()
    H, KVH, L, D, keep, mrope = 28, 4, 1000, 128, 250, [16, 24, 24]
    q, k, _ = make_qk("ramp_up", H, KVH, L, D, seed=77)
    v = torch.randn(1, KVH, L, D, generator=torch.Generator().manual_seed(2)).to(BF).cuda()
    rot = TableRotary(D, attention_scaling=1.0)
    rot.inv_freq = rot.inv_freq.cuda()
    pos = torch.zeros(3, 1, L, dtype=torch.int64, device="cuda")
    mask = _free_keys_mask(L, 700, seed=3)
    kk, pp, i = _check_update(lc, q, k, v, keep, mask, anchor(q, k), f"re-forge update, tables={tables}", True, rot, pos,
                              mrope)
    want_pos = pos[..., i].clone()
    want_pos[0] = op.reforge_temporal(want_pos[0], keep, L)
    assert torch.equal(pp, want_pos)
    cos, sin = rot(v, want_pos)
    assert torch.equal(kk, op.rotate(k[:, :, i], op.select_mrope(cos, mrope), op.select_mrope(sin, mrope)))


BATCH_PATTERNS = ["noise", "sink0", "ramp_up", "ramp_down", "flat", "dup", "spread", "sink_last"]


@pytest.mark.parametrize("H,KVH,L,D,layers,reforge", [(16, 8, 300, 64, 35, False), (28, 4, 1000, 128, 6, True)])
def test_batched_update_meets_the_fp64_anchor(H, KVH, L, D, layers, reforge):
    """rtk_pivot_update_batch through PivotKVCache with deferred compression: every layer its own pattern and mask (35
    layers: a group of 32 and one of 3), each layer held to its own anchor"""
    lc = _lc()
    keep = L // 4
    cfg = _cfg(H, KVH, D, layers, keep / L + 1e-9, reforge)
    cfg.longvideo_kwargs["kvcache_compression_kwargs"]["deferred_compression"] = True
    cache = lc.PivotKVCache(cfg)
    rot = TableRotary(D, attention_scaling=1.0, mrope=False)
    rot.inv_freq = rot.inv_freq.cuda()
    free = [None, 0, 1, 100, L // 3, L - 1, L // 2 + 1]
    runs = []
    for layer in range(layers):
        pattern = BATCH_PATTERNS[layer % len(BATCH_PATTERNS)]
        q, k, _ = make_qk(pattern, H, KVH, L, D, seed=layer)
        v = torch.randn(1, KVH, L, D, generator=torch.Generator().manual_seed(layer)).to(BF).cuda()
        n_free = free[layer % len(free)]
        mask = _free_keys_mask(L, n_free, seed=layer)
        cache.keypatches_mask_chunk = mask
        pos = torch.zeros(1, L, dtype=torch.int64, device="cuda")
        cache.update(k, v, layer, {"query_states": q, "position_ids": pos, "rotary_emb": rot, "mrope_section": None})
        runs.append((q, k, v, mask, cache._last_head_scores, cache._last_keep_indices, f"layer {layer} {pattern} free={n_free}"))
    assert len(cache._deferred) == layers
    cache.after_forward()
    for layer, (q, k, v, mask, hs, idx, what) in enumerate(runs):
        anc = anchor(q, k)
        if mask is not None:
            anc = with_key_patches(anc, mask)
        excused = check_rule(hs, anc["ftz"], what)
        check_kept(idx, anc["ftz"][2], excused, mask, keep, what)
        i = idx.long()
        assert torch.equal(cache.layers[layer].keys, k[:, :, i]) and torch.equal(cache.layers[layer].values, v[:, :, i])
        if reforge:
            assert torch.equal(cache.position_cache[layer], torch.zeros(1, keep, dtype=torch.int64, device="cuda"))
