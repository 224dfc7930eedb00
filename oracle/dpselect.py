"""Oracle for DPSelect (keyframe / key-patch selection).  TEST INFRASTRUCTURE ONLY.

Restates ``retake/visual_compression.py:86-177`` (``memory_bank_compress_keyframe``)
as explicit arithmetic.  Where the reference delegates to an ATen composite the
individual roundings are written out, so that the CUDA kernels have a spec:

* ``F.cosine_similarity`` on bf16 (``visual_compression.py:100``) is, bit for bit,
  ``n = bf16(sqrt(sum_f32 x^2))``; ``n = max(n, bf16(1e-8))``; ``u = bf16(x / n)``;
  ``p = bf16(u_a * u_b)``; ``sim = bf16(sum_f32 p)``  (SURVEY.md 8a, note N1).
* ``dis = 1 - float(sim)``, row 0 is 1.0 (``:101-106``).
* ``max_pool1d_with_indices(window 3, stride 1, pad 1)`` + ``unique`` + ``nonzero``
  (``:121-123`` / ``:153-156``) selects frame i iff ``d[i] > d[i-1]`` (strict; no left
  neighbour for i = 0) and ``d[i] >= d[i+1]`` (no right neighbour for the last) - the
  pool keeps the FIRST maximum of each window, but the LAST NaN (note N2, ``peak_mask``).
* ``d[peaks] += 2`` in fp32, ``topk(k=t, sorted=False)`` then ascending index sort
  (``:133-135`` / ``:160,167-168``).  ``torch.topk`` leaves the choice among equal keys
  unspecified; the oracle offers the two rules that matter: ``tie="lowest"`` (all keys
  greater than the t-th, then equal keys by ascending index - what ATen's CUDA
  radix-select gather produces, see tests/probes/probe_aten_cuda.py) and
  ``tie="torch"`` (call ``torch.topk`` on the executing device, i.e. whatever the
  reference itself would pick there).

The fp32 accumulation ORDER inside the two reductions is not part of the
reference's text; ``reduce="aten_cuda"`` replays ATen's CUDA reduction tree for a
contiguous row (one warp per row, ``vec`` accumulators per lane, shfl-down tree;
``torch/include/ATen/native/cuda/Reduce.cuh``), ``reduce="torch"`` uses ``Tensor.sum``
of the executing device.
"""
from __future__ import annotations

import torch

BF16 = torch.bfloat16


def _r(x: torch.Tensor) -> torch.Tensor:
    """Round an fp32 tensor to bf16 (round-to-nearest-even) and widen back."""
    return x.to(BF16).to(torch.float32)


def aten_cuda_rowsum(xf: torch.Tensor, vec: int = 8, square: bool = False) -> torch.Tensor:
    """fp32 sum over the last dim of ``xf`` [R, C] in ATen-CUDA order.

    Lane l of a 32-lane warp owns the ``vec``-element vectors l, l+32, l+64, ...; element
    j of every vector goes to accumulator j (``acc = acc + v`` / ``fma(v, v, acc)``);
    accumulators are folded 0+1, +2, ...; lanes are folded with shfl-down offsets
    16, 8, 4, 2, 1.  Requires C % vec == 0 (the kernels have the same contract).
    """
    R, C = xf.shape
    if C % vec:
        raise ValueError("C must be a multiple of the vector width")
    nv = C // vec
    v = xf.reshape(R, nv, vec)
    acc = torch.zeros(R, 32, vec, dtype=torch.float32, device=xf.device)
    k = 0
    while k * 32 < nv:
        chunk = v[:, k * 32:(k + 1) * 32]
        lanes = chunk.shape[1]
        acc[:, :lanes] = acc[:, :lanes] + (chunk * chunk if square else chunk)
        k += 1
    lane = acc[:, :, 0].clone()
    for j in range(1, vec):
        lane = lane + acc[:, :, j]
    off = 16
    while off:
        lane = lane + torch.cat([lane[:, off:], lane[:, 32 - off:]], dim=1)
        off >>= 1
    return lane[:, 0]


def adjacent_cosine_similarity(x: torch.Tensor, reduce: str = "torch", norm_vec: int = 4, sum_vec: int = 8) -> torch.Tensor:
    """``sim[T-1, N]`` (fp32 container; bf16-valued for a bf16 bank) between consecutive frames of ``x[T, N, C]``:
    the rounding chain of ``F.cosine_similarity`` (``visual_compression.py:20,63,100``).

    ``reduce="aten_cuda"``: ``linalg_vector_norm`` on bf16 reduces with 4-element vectors, ``sum`` on bf16
    with 8-element vectors (measured on the B200, tests/probes/probe_aten_cuda2.py Q6/Q7)."""
    T, N, C = x.shape
    xf = x.to(torch.float32)
    lowp = x.dtype == BF16
    rnd = _r if lowp else (lambda t: t)

    def rowsum(a, square=False):
        flat = a.reshape(-1, C)
        if reduce == "aten_cuda":
            return aten_cuda_rowsum(flat, norm_vec if square else sum_vec, square).reshape(a.shape[:-1])
        return (flat * flat if square else flat).sum(-1).reshape(a.shape[:-1])

    n = rnd(torch.sqrt(rowsum(xf, square=True)))
    eps = rnd(torch.tensor(1e-8, dtype=torch.float32, device=x.device))
    n = torch.maximum(n, eps)
    u = rnd(xf / n[..., None])
    p = rnd(u[:-1] * u[1:])
    return rnd(rowsum(p))


def adjacent_cosine_distance(x: torch.Tensor, reduce: str = "torch", norm_vec: int = 4, sum_vec: int = 8) -> torch.Tensor:
    """``dis[T, N]`` fp32 for a memory bank ``x[T, N, C]`` (``visual_compression.py:98-106``): one minus the adjacent
    similarity, row 0 = 1."""
    dis = 1.0 - adjacent_cosine_similarity(x, reduce, norm_vec, sum_vec)
    return torch.cat([torch.ones_like(dis[:1]), dis], dim=0)


def peak_mask(d: torch.Tensor) -> torch.Tensor:
    """Boolean peaks along dim 0 of ``d[T, ...]``: ATen's ``max_pool1d_with_indices(window 3, pad 1)`` loop, literally.
    The window [i-1, i+1] (clipped to [0, T)) starts at its first position with max -inf and takes v when
    ``v > max or isnan(v)``; i is a peak when the loop ends on i.  On finite values: strict rise on the left, no rise on
    the right.  In a run of NaNs the LAST NaN of each window wins (note N2)."""
    T = d.shape[0]
    pos = torch.arange(T, device=d.device).reshape((T,) + (1,) * (d.dim() - 1))
    arg = (pos - 1).clamp_min(0).expand(d.shape)
    mx = torch.full_like(d, float("-inf"))
    for u in (-1, 0, 1):
        j = pos + u
        valid = (j >= 0) & (j < T)
        v = d[(j.clamp(0, T - 1)).flatten()]
        take = valid & ((v > mx) | torch.isnan(v))
        mx = torch.where(take, v, mx)
        arg = torch.where(take, j, arg)
    return arg == pos


def select_top(keys: torch.Tensor, t: int, tie: str = "lowest") -> torch.Tensor:
    """Ascending indices of the ``t`` largest entries along dim 0 of ``keys[T, ...]``."""
    if tie == "torch":
        idx = torch.topk(keys, k=t, dim=0, sorted=False).indices
    elif tie == "lowest":
        idx = torch.sort(keys, dim=0, descending=True, stable=True).indices[:t]
    else:
        raise ValueError(tie)
    return idx.sort(dim=0).values


def dpselect_indices(dis: torch.Tensor, t: int, sync: bool, tie: str = "lowest"):
    """From ``dis[T, N]`` to (kept frame indices, peak mask).

    sync=True : indices [t], peaks [T]        (``visual_compression.py:108-135``)
    sync=False: indices [t, N], peaks [T, N]  (``visual_compression.py:141-169``)
    """
    d = dis.mean(1) if sync else dis
    peaks = peak_mask(d)
    keys = d + 2.0 * peaks.to(d.dtype)
    return select_top(keys, t, tie), peaks


def memory_bank_compress_keyframe(memory_bank: torch.Tensor, tgt_mem_len: int, window_size: int = 3,
                                  sync: bool = True, tie: str = "lowest", reduce: str = "torch",
                                  return_indices: bool = False):
    """Oracle twin of the reference operator (same signature plus oracle knobs)."""
    if window_size != 3:
        raise NotImplementedError("the reference only ever calls this with window_size=3")
    B, T, N, C = memory_bank.shape
    dis = adjacent_cosine_distance(memory_bank[0], reduce=reduce)
    idx, peaks = dpselect_indices(dis, tgt_mem_len, sync, tie)
    if sync:
        out = memory_bank[:, idx]
        mask = peaks[idx][:, None].repeat(1, N)
    else:
        out = memory_bank.gather(1, idx[None, :, :, None].expand(B, -1, -1, C))
        mask = peaks.gather(0, idx)
    if return_indices:
        return out, mask.flatten(), idx, dis
    return out, mask.flatten()
