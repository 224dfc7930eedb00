"""GPU parity: DPSelect kernels (through the C ABI) against the oracle and against the reference's own
torch-op sequence executed on the same B200 (the bit-exactness target, SURVEY.md 8a note N4)."""

import pytest
import torch
import torch.nn.functional as F

from helpers import load_golden, scene_video
from oracle import dpselect as od

pytestmark = pytest.mark.gpu


def _mods():
    from retake import visual_compression as vc
    return vc


def ref_dis_cuda(x):
    """reference lines 100-106 verbatim in spirit: stock ATen ops on the GPU."""
    sim = F.cosine_similarity(x[None, :-1], x[None, 1:], dim=-1)[0]
    d = 1 - sim.type(torch.float)
    return torch.cat([torch.ones_like(d[:1]), d], dim=0)


def make_video(kind, T, N, C, seed):
    g = torch.Generator().manual_seed(seed)
    if kind == "rand":
        x = torch.randn(T, N, C, generator=g)
    elif kind == "scene":
        x = scene_video(g, T, N, C)
    else:
        x = scene_video(g, T, N, C, dup_every=4)
    return x.to(torch.bfloat16).cuda()


SHAPES = [("rand", 33, 64, 256, 1), ("scene", 40, 96, 1152, 2), ("dup", 48, 64, 3584, 3), ("rand", 17, 729, 1152, 4),
          ("scene", 128, 256, 3584, 5), ("rand", 9, 16, 512, 6), ("rand", 12, 32, 4096, 7), ("dup", 300, 8, 256, 8)]


@pytest.mark.parametrize("kind,T,N,C,seed", SHAPES)
def test_distance_bit_exact_vs_aten_cuda(kind, T, N, C, seed):
    vc = _mods()
    x = make_video(kind, T, N, C, seed)
    got = vc.dpselect_distance(x)
    want = ref_dis_cuda(x)
    bad = int((got != want).sum())
    assert bad == 0, f"{bad}/{got.numel()} distances differ from ATen-CUDA (max |d| {float((got - want).abs().max())})"


@pytest.mark.parametrize("kind,T,N,C,seed", SHAPES[:4])
def test_distance_bit_exact_vs_oracle_aten_order(kind, T, N, C, seed):
    vc = _mods()
    x = make_video(kind, T, N, C, seed)
    got = vc.dpselect_distance(x).cpu()
    want = od.adjacent_cosine_distance(x.cpu(), reduce="aten_cuda")
    assert torch.equal(got, want)


def test_distance_halo_split_equals_whole():
    vc = _mods()
    x = make_video("scene", 64, 64, 1152, 11)
    whole = vc.dpselect_distance(x)
    parts = [vc.dpselect_distance(x[:16])]
    for a, b in ((16, 40), (40, 41), (41, 64)):
        parts.append(vc.dpselect_distance(x[a - 1:b], halo=True))
    assert torch.equal(torch.cat(parts, 0), whole)


def test_distance_edge_cases():
    vc = _mods()
    x = make_video("rand", 1, 8, 256, 12)
    assert torch.equal(vc.dpselect_distance(x), torch.ones(1, 8, device="cuda"))
    x = make_video("rand", 2, 1, 256, 13)
    assert torch.equal(vc.dpselect_distance(x), ref_dis_cuda(x))
    z = torch.zeros(4, 16, 256, dtype=torch.bfloat16, device="cuda")        # zero rows: eps clamp
    assert torch.equal(vc.dpselect_distance(z), ref_dis_cuda(z))
    from retake._native import RtkError
    with pytest.raises(RtkError):
        vc.dpselect_distance(torch.zeros(4, 4, 100, dtype=torch.bfloat16, device="cuda"))


@pytest.mark.parametrize("sync", [False, True])
@pytest.mark.parametrize("kind,T,N,C,seed", SHAPES)
def test_select_bit_exact_vs_torch_topk_on_cuda(kind, T, N, C, seed, sync):
    vc = _mods()
    x = make_video(kind, T, N, C, seed)
    dis = ref_dis_cuda(x)
    for t in sorted({T, max(1, round(0.5 * T)), max(1, round(0.25 * T)), 1}):
        idx, mask = vc.dpselect_select(dis, t, sync)
        want_idx, peaks = od.dpselect_indices(dis, t, sync, tie="torch")        # torch.topk on this GPU
        want_low, _ = od.dpselect_indices(dis, t, sync, tie="lowest")
        assert torch.equal(idx.long(), want_low), "kernel deviates from the documented lowest-index tie rule"
        assert torch.equal(idx.long(), want_idx), "kernel deviates from torch.topk on CUDA"
        want_mask = peaks[want_idx][:, None].repeat(1, N) if sync else peaks.gather(0, want_idx)
        assert torch.equal(mask, want_mask.flatten())


def test_select_heavy_ties_and_signed_zero():
    vc = _mods()
    g = torch.Generator().manual_seed(5)
    dis = (torch.randint(0, 3, (97, 40), generator=g).float() * 0.5).cuda()
    dis[::7] = -0.0
    dis[0] = 1.0
    for sync in (False, True):
        for t in (1, 13, 48, 97):
            idx, mask = vc.dpselect_select(dis, t, sync)
            want, peaks = od.dpselect_indices(dis, t, sync, tie="torch")
            assert torch.equal(idx.long(), want)


@pytest.mark.parametrize("sync", [False, True])
@pytest.mark.parametrize("kind,T,N,C,seed", SHAPES)
def test_operator_matches_reference_ops_on_cuda(kind, T, N, C, seed, sync):
    """whole operator == oracle restatement fed by ATen-CUDA's own distance and torch.topk on CUDA"""
    vc = _mods()
    x = make_video(kind, T, N, C, seed)
    xc = x.clone()
    for t in sorted({T, max(1, round(0.5 * T)), 1}):
        out, mask, idx = vc.memory_bank_compress_keyframe(x[None], t, 3, sync=sync, return_indices=True)
        assert torch.equal(x, xc), "input was modified"
        dis = ref_dis_cuda(x)
        want_idx, peaks = od.dpselect_indices(dis, t, sync, tie="torch")
        if sync:
            want_out = x[None][:, want_idx]
            want_mask = peaks[want_idx][:, None].repeat(1, N)
        else:
            want_out = x[None].gather(1, want_idx[None, :, :, None].expand(1, -1, -1, C))
            want_mask = peaks.gather(0, want_idx)
        assert out.shape == (1, t, N, C) and out.dtype == torch.bfloat16 and mask.dtype == torch.bool
        assert torch.equal(idx, want_idx)
        assert torch.equal(mask, want_mask.flatten())
        assert torch.equal(out, want_out)
        if t == T:
            assert torch.equal(out[0], x)                      # r = 1.0: identity gather, mask only


def test_golden_fixtures_through_cuda():
    """frozen CPU-reference outputs: equal whenever the CUDA-order distances tie-freely agree"""
    vc = _mods()
    cases = load_golden("dpselect_reference")
    ran = 0
    for c in cases:
        x = c["x"]
        if x.dtype != torch.bfloat16 or x.shape[-1] < 256:
            continue
        out, mask, idx = vc.memory_bank_compress_keyframe(x.cuda(), c["t"], 3, sync=c["sync"], return_indices=True)
        o_out, o_mask, o_idx, _ = od.memory_bank_compress_keyframe(x, c["t"], 3, sync=c["sync"], tie="lowest",
                                                                   reduce="aten_cuda" if not c["sync"] else "torch",
                                                                   return_indices=True)
        if not c["sync"]:
            assert torch.equal(idx.cpu(), o_idx) and torch.equal(mask.cpu(), o_mask) and torch.equal(out.cpu(), o_out)
        if torch.equal(o_mask, c["mask"]) and torch.equal(o_out, c["out"]) and not c["sync"]:
            assert torch.equal(mask.cpu(), c["mask"]) and torch.equal(out.cpu(), c["out"])
            ran += 1
    assert ran >= 6


def test_full_size_config2_properties():
    """BASELINE config 2 (256 frames, 448px, 7B shape): bit-exact vs ATen ops + size-independent properties"""
    vc = _mods()
    T, N, C = 128, 256, 3584
    x = make_video("dup", T, N, C, 21)
    for t, sync in ((128, False), (64, False), (32, False), (64, True)):
        out, mask, idx = vc.memory_bank_compress_keyframe(x[None], t, 3, sync=sync, return_indices=True)
        dis = ref_dis_cuda(x)
        want_idx, peaks = od.dpselect_indices(dis, t, sync, tie="torch")
        assert torch.equal(idx, want_idx)
        idx2 = idx.reshape(t, -1)
        assert bool((idx2[1:] > idx2[:-1]).all())                          # strictly ascending per column
        assert bool((idx2[0] == 0).all())                                  # frame 0 (dis 1 + 2) always survives
        if sync:
            assert torch.equal(out[0], x[idx])
        else:
            assert torch.equal(out[0], x.gather(0, idx[:, :, None].expand(-1, -1, C)))
        assert int(mask.sum()) <= int(peaks.sum()) * (N if sync else 1)


def test_full_size_config4_llava_shape():
    """BASELINE config 4 shape (SigLIP grid N=729, C=1152), 512 frames: bit-exact against the reference's torch op sequence
    executed on the same GPU, both modes, incl. the unaligned row means of sync mode (N % 4 != 0)."""
    from oracle import reference_ops as ro
    vc = _mods()
    T, N, C = 512, 729, 1152
    x = make_video("scene", T, N, C, 31)
    for t, sync in ((512, False), (256, False), (128, True)):
        out, mask, idx = vc.memory_bank_compress_keyframe(x[None], t, 3, sync=sync, return_indices=True)
        want_out, want_mask, want_idx = ro.dpselect(x[None], t, sync)
        assert torch.equal(idx.long(), want_idx) and torch.equal(mask, want_mask) and torch.equal(out, want_out)


def _synthetic_video(T, N, C, seed):
    """scene-structured bf16 video built ON the GPU (scenes of 3..40 grids + 0.3 noise, every 9th grid an exact duplicate)"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.empty(T, N, C, dtype=torch.bfloat16, device="cuda")
    t = 0
    while t < T:
        run = min(T - t, 3 + (seed * 7 + t * 13) % 38)
        scene = torch.randn(N, C, generator=g, device="cuda")
        x[t:t + run] = (scene[None] + 0.3 * torch.randn(run, N, C, generator=g, device="cuda")).to(torch.bfloat16)
        t += run
    x[9::9] = x[8:-1:9][: x[9::9].shape[0]]
    return x


@pytest.mark.parametrize("T,N,C,cases", [
    (1024, 256, 3584, ((1024, False), (512, False), (256, False), (512, True))),      # the 2048-frame headline video
    (2048, 729, 1152, ((2048, False), (1024, False), (512, True))),                   # BASELINE config 4: LLaVA-Video, 2048 frames
])
def test_headline_sizes_bit_exact_vs_reference_ops(T, N, C, cases):
    """VERDICT r1: DPSelect at the benchmark's own sizes (T = 1024 Qwen2-VL grids, T = 2048 LLaVA frames): distances,
    kept indices, masks and compacted embeddings equal the reference's torch-CUDA op sequence bit for bit"""
    from oracle import reference_ops as ro
    vc = _mods()
    x = _synthetic_video(T, N, C, 3)
    assert torch.equal(vc.dpselect_distance(x), ref_dis_cuda(x))
    for t, sync in cases:
        out, mask, idx = vc.memory_bank_compress_keyframe(x[None], t, 3, sync=sync, return_indices=True)
        r_out, r_mask, r_idx = ro.dpselect(x[None], t, sync)
        assert torch.equal(idx.long(), r_idx), (T, t, sync)
        assert torch.equal(mask, r_mask)
        assert torch.equal(out, r_out)
        assert out.shape == (1, t, N, C) and mask.shape == (t * N,)
        del out, r_out
