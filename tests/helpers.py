"""Shared synthetic-input helpers for tests, golden generation and bench (no reference, no oracle)."""
import io
import lzma
import os

import torch


def load_golden(name):
    """the cases frozen by tests/golden/make_golden.py: ``tests/golden/<name>.pt.xz``, an xz-compressed ``torch.save`` file"""
    with lzma.open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name + ".pt.xz")) as f:
        return torch.load(io.BytesIO(f.read()))


def bf16_round(x):
    """round a float64 tensor to the nearest bf16 value (ties to even) in one step, kept as float64; below 2^-126 the
    spacing stays 2^-133, as for bf16 subnormals"""
    _, e = torch.frexp(x)
    quantum = torch.ldexp(torch.ones_like(x), (e.clamp_min(-125) - 8).double())
    return torch.round(x / quantum) * quantum


class TableRotary:
    """Deterministic stand-in for the HF rotary module: callable (x, position_ids) -> (cos, sin)
    with ``attention_scaling`` (``longvideo_cache.py:249,256``).  YaRN-like scaling 1.1386."""

    def __init__(self, head_dim, base=10000.0, attention_scaling=1.1386, mrope=True):
        self.inv_freq = 1.0 / (base ** (torch.arange(0, head_dim, 2, dtype=torch.float32) / head_dim))
        self.attention_scaling = attention_scaling
        self.mrope = mrope

    def __call__(self, x, position_ids):
        pos = position_ids.to(torch.float32)             # [3,1,L] or [1,L]
        freqs = pos[..., None] * self.inv_freq           # [...,L,D/2]
        emb = torch.cat((freqs, freqs), dim=-1)
        cos = emb.cos() * self.attention_scaling
        sin = emb.sin() * self.attention_scaling
        return cos.to(x.dtype), sin.to(x.dtype)


def scene_video(g, T, N, C, sigma=0.3, dup_every=0):
    """scene-structured embeddings (SURVEY.md 8d): x[t] = scene[s(t)] + sigma * eps[t]."""
    x = torch.empty(T, N, C)
    t = 0
    while t < T:
        run = int(torch.randint(2, 7, (1,), generator=g))
        scene = torch.randn(N, C, generator=g)
        for _ in range(run):
            if t >= T:
                break
            x[t] = scene + sigma * torch.randn(N, C, generator=g)
            t += 1
    if dup_every:
        for t in range(dup_every, T, dup_every):
            x[t] = x[t - 1]                               # exact duplicates -> dis == 0 ties
    return x


def index_parity(idx, idx_ref, score_ref, keep):
    """Compare a kept-index set with the reference's ``topk(score, keep).indices.sort()`` (longvideo_cache.py:276-277).

    Returns (identical, justified, n_diff): ``identical`` is exact equality; when the sets differ, ``justified`` says
    whether EVERY index in the symmetric difference carries a reference score within one bf16 ulp of the reference's
    k-th largest score - the only place where cuBLAS' accumulation order (which no other kernel can replay, SURVEY.md
    note N4) may legitimately move a token across the cut.  ``score_ref`` is the reference's bf16 score AFTER the
    key-patch fill."""
    idx, idx_ref = idx.long(), idx_ref.long()
    if idx.numel() == idx_ref.numel() and bool(torch.equal(idx, idx_ref)):
        return True, True, 0
    a = torch.zeros(score_ref.numel(), dtype=torch.bool, device=score_ref.device)
    b = a.clone()
    a[idx] = True
    b[idx_ref] = True
    diff = torch.nonzero(a ^ b)[:, 0]
    bits = score_ref.to(torch.bfloat16).view(torch.int16).int()          # scores are positive: bit patterns are ordered
    kth = torch.sort(bits, descending=True).values[keep - 1]
    ok = bool(((bits[diff] - kth).abs() <= 1).all()) and idx.numel() == idx_ref.numel() == keep
    return False, ok, int(diff.numel())
