"""GPU parity of deferred (batched) PivotKV compression - SURVEY.md 8(f2): ``update`` appends, ``after_forward()`` runs the
compression of all layers of the chunk as ONE ``rtk_pivot_update_batch`` call that writes the kept rows in place.  What
every reader of the cache sees must equal compression inside ``update`` (``longvideo_cache.py:217-323``): same kept
indices, same K / V / position caches, same bookkeeping."""
import pytest
import torch

from helpers import TableRotary
from test_gpu_pivotkv import _cfg, _check_keep, qkv, ref_head_scores_cuda, ulp_diff

pytestmark = pytest.mark.gpu
BF = torch.bfloat16


def _lc():
    from retake import longvideo_cache as lc
    return lc


def _positions(L, base, mrope, n_tok=256):
    ar = torch.arange(L, device="cuda")
    if mrope:
        return torch.stack([base + ar // n_tok, (ar % n_tok) // 16, ar % 16])[:, None]
    return (ar + base)[None]


def _run(lc, deferred, H, KVH, L, D, layers, chunks, ratio, reforge, mrope, flush="after_forward", alpha=1.0, hf_rotary=False):
    """drive a cache like the chunk loop does; returns per-chunk observations and the final cache"""
    cfg = _cfg(H, KVH, D, layers, ratio, reforge)
    cfg.longvideo_kwargs["kvcache_compression_kwargs"]["deferred_compression"] = deferred
    cache = lc.PivotKVCache(cfg)
    assert cache.deferred_compression is deferred
    if hf_rotary:
        import bench
        rot = bench.make_rotary(torch.device("cuda"))
    else:
        rot = TableRotary(D, mrope=bool(mrope))
        rot.inv_freq = rot.inv_freq.cuda()
    obs = []
    for c in range(chunks):
        Lc = L if c < chunks - 1 or chunks == 1 else max(1, L // 2 + 3)         # ragged last chunk
        mask = (torch.rand(Lc, generator=torch.Generator().manual_seed(50 + c)) < 0.15).cuda()
        cache.kvcache_compression = True
        cache.keypatches_mask_chunk = mask
        per_layer = []
        for layer in range(layers):
            q, k, v = qkv(H, KVH, Lc, D, alpha, seed=1000 * c + layer)
            base = int(cache.get_prev_temporal_idx(layer)) + 1 if reforge else 100 * c
            pos = _positions(Lc, base, mrope)
            past = cache.get_seq_length(layer)
            ko, vo = cache.update(k, v, layer, {"query_states": q, "position_ids": pos, "rotary_emb": rot,
                                                "mrope_section": mrope})
            # this step's attention sees [past | uncompressed chunk]
            assert ko.shape == (1, KVH, past + Lc, D) and torch.equal(ko[:, :, past:], k) and torch.equal(vo[:, :, past:], v)
            keep = max(1, int(ratio * Lc))
            assert cache.get_seq_length(layer) == past + keep
            per_layer.append((q, k, v, pos, mask, keep, past))
        if flush == "after_forward":
            cache.after_forward()
            if deferred:
                assert not cache._deferred and all(l._deferred_owner is None for l in cache.layers)
        obs.append(per_layer)
    cache.after_forward()
    return cache, obs


SHAPES = [  # H, KVH, L, D, layers, chunks, ratio, reforge, mrope
    (4, 2, 256, 64, 2, 3, 0.5, True, [8, 12, 12]),
    (4, 2, 256, 64, 3, 2, 0.25, False, None),
    (8, 2, 200, 128, 2, 2, 0.3, True, None),
    (28, 4, 1024, 128, 4, 2, 0.122, True, [16, 24, 24]),
    (28, 4, 1024, 128, 3, 2, 0.5, False, [16, 24, 24]),
    (28, 4, 16384, 128, 4, 1, 0.25, True, [16, 24, 24]),       # the length limit, 4 layers in one batched call
]


@pytest.mark.parametrize("H,KVH,L,D,layers,chunks,ratio,reforge,mrope", SHAPES)
def test_deferred_equals_immediate(H, KVH, L, D, layers, chunks, ratio, reforge, mrope):
    lc = _lc()
    a, _ = _run(lc, False, H, KVH, L, D, layers, chunks, ratio, reforge, mrope)
    b, obs = _run(lc, True, H, KVH, L, D, layers, chunks, ratio, reforge, mrope)
    assert a.num_evicted_tokens == b.num_evicted_tokens
    for layer in range(layers):
        assert a.get_seq_length(layer) == b.get_seq_length(layer)
        ka, kb = a.layers[layer].keys, b.layers[layer].keys
        assert ka.shape == kb.shape
        assert torch.equal(a.layers[layer].values, b.layers[layer].values)
        assert torch.equal(ka, kb)
        if reforge:
            assert torch.equal(a.position_cache[layer], b.position_cache[layer])
    # the last chunk's exposed per-layer results
    assert torch.equal(a.last_keep_indices, b.last_keep_indices)
    # a CTA takes the same tile range of every layer as in a single-layer launch: the fp32 partials fold in the same order
    assert torch.equal(a.last_head_scores, b.last_head_scores)


def test_deferred_against_reference_scores():
    """kept rows of every layer against the reference's op sequence on the GPU (no re-forging: K rows are plain gathers)"""
    lc = _lc()
    H, KVH, L, D, layers, ratio = 28, 4, 1024, 128, 5, 0.25
    cfg = _cfg(H, KVH, D, layers, ratio, False)
    cfg.longvideo_kwargs["kvcache_compression_kwargs"]["deferred_compression"] = True
    cache = lc.PivotKVCache(cfg)
    mask = (torch.rand(L, generator=torch.Generator().manual_seed(3)) < 0.2).cuda()
    cache.keypatches_mask_chunk = mask
    pos = _positions(L, 0, None)
    data, entries = [], []
    for layer in range(layers):
        q, k, v = qkv(H, KVH, L, D, 3.0, seed=layer)
        cache.update(k, v, layer, {"query_states": q, "position_ids": pos})
        data.append((q, k, v))
        entries.append(cache._deferred[-1]["outs"])
    assert len(cache._deferred) == layers
    from retake import _native
    n0 = _native.launch_count()
    cache.after_forward()
    # one chain of launches for all layers (no un-rotation here): mask scan, key gather, score pass 1, stats merge, score
    # pass 2, head reduce, select, compact
    assert _native.launch_count() - n0 == 8
    keep = int(ratio * L)
    for layer, ((q, k, v), outs) in enumerate(zip(data, entries)):
        ref = ref_head_scores_cuda(q, k)
        assert bool((outs["head_scores"][:, mask] == 1.0).all())          # key patches are not scored (their score is 1.0)
        d = ulp_diff(outs["head_scores"][:, ~mask], ref[:, ~mask])
        assert int(d.max()) <= 1 and float((d > 0).float().mean()) < 0.02
        _check_keep(outs["keep_idx"], outs["head_scores"].mean(0), ref.mean(0), mask, keep)
        idx = outs["keep_idx"].long()
        assert torch.equal(cache.layers[layer].keys, k[:, :, idx]) and torch.equal(cache.layers[layer].values, v[:, :, idx])


def test_deferred_settles_without_after_forward():
    """a caller that never calls after_forward(): the next update of a layer (or any read) settles the debt first"""
    lc = _lc()
    args = (4, 2, 256, 64, 2, 3, 0.5, True, [8, 12, 12])
    a, _ = _run(lc, False, *args, flush="never")
    b, _ = _run(lc, True, *args, flush="never")
    for layer in range(2):
        assert torch.equal(a.layers[layer].keys, b.layers[layer].keys)
        assert torch.equal(a.layers[layer].values, b.layers[layer].values)
        assert torch.equal(a.position_cache[layer], b.position_cache[layer])
    # reads settle too
    cfg = _cfg(4, 2, 64, 1, 0.5, False)
    cfg.longvideo_kwargs["kvcache_compression_kwargs"]["deferred_compression"] = True
    c = lc.PivotKVCache(cfg)
    q, k, v = qkv(4, 2, 128, 64, 1.0, seed=9)
    c.update(k, v, 0, {"query_states": q, "position_ids": _positions(128, 0, None)})
    assert len(c._deferred) == 1
    keys = c.key_cache[0]
    assert not c._deferred and keys.shape[2] == 64
    assert torch.equal(keys, k[:, :, c.last_keep_indices.long()])


def test_deferred_many_layers_and_hf_rotary():
    """28 layers (the 7B depth) in one batch with the stock HF rotary module, and 35 layers (two groups of <= 32)"""
    lc = _lc()
    a, _ = _run(lc, False, 28, 4, 512, 128, 28, 2, 0.25, True, [16, 24, 24], hf_rotary=True)
    b, _ = _run(lc, True, 28, 4, 512, 128, 28, 2, 0.25, True, [16, 24, 24], hf_rotary=True)
    for layer in range(28):
        assert torch.equal(a.layers[layer].keys, b.layers[layer].keys)
        assert torch.equal(a.layers[layer].values, b.layers[layer].values)
        assert torch.equal(a.position_cache[layer], b.position_cache[layer])
    a, _ = _run(lc, False, 4, 2, 130, 64, 35, 1, 0.5, True, [8, 12, 12])
    b, _ = _run(lc, True, 4, 2, 130, 64, 35, 1, 0.5, True, [8, 12, 12])
    for layer in range(35):
        assert torch.equal(a.layers[layer].keys, b.layers[layer].keys)
        assert torch.equal(a.position_cache[layer], b.position_cache[layer])


def test_deferred_full_size_chunk():
    """7B shape, L = 4096, keep 500 (the benchmark's update), four layers"""
    lc = _lc()
    args = (28, 4, 4096, 128, 4, 2, 500 / 4096, True, [16, 24, 24])
    a, _ = _run(lc, False, *args, hf_rotary=True)
    b, _ = _run(lc, True, *args, hf_rotary=True)
    for layer in range(4):
        assert a.get_seq_length(layer) == b.get_seq_length(layer)
        assert torch.equal(a.layers[layer].values, b.layers[layer].values)
        assert torch.equal(a.layers[layer].keys, b.layers[layer].keys)
        assert torch.equal(a.position_cache[layer], b.position_cache[layer])


def test_deferred_opaque_rotary_falls_back_to_immediate(monkeypatch):
    """an opaque rotary callable (tables must come from calling it) cannot be batched: update compresses right away"""
    lc = _lc()
    monkeypatch.setenv("RTK_ROTARY_TABLES", "1")
    b, _ = _run(lc, True, 4, 2, 256, 64, 2, 2, 0.5, True, [8, 12, 12])
    monkeypatch.setenv("RTK_ROTARY_TABLES", "0")
    a, _ = _run(lc, False, 4, 2, 256, 64, 2, 2, 0.5, True, [8, 12, 12])
    for layer in range(2):
        assert torch.equal(a.layers[layer].keys, b.layers[layer].keys)
        assert torch.equal(a.position_cache[layer], b.position_cache[layer])


def test_deferred_with_positions_rebased_in_place_per_layer():
    """ADVICE r1: the Qwen2-VL attention forward re-bases ONE shared position tensor in place for every layer
    (`pos3d[0, 0, :] += prev + 1 - pos3d[0, 0, 0]`, reference qwen2_vl.py:68-73).  Deferred compression reads the ids at
    after_forward(), so it must have kept its own copy: layers whose `prev` differ would otherwise all be un-rotated and
    re-indexed with the LAST layer's ids."""
    lc = _lc()
    H, KVH, L, D, layers, chunks, ratio, mrope = 4, 2, 256, 64, 4, 3, 0.1, [8, 12, 12]
    rot = TableRotary(D, mrope=True)
    rot.inv_freq = rot.inv_freq.cuda()

    def run(deferred):
        cfg = _cfg(H, KVH, D, layers, ratio, True)
        cfg.longvideo_kwargs["kvcache_compression_kwargs"]["deferred_compression"] = deferred
        cache = lc.PivotKVCache(cfg)
        prevs = []
        for c in range(chunks):
            cache.kvcache_compression = True
            shared = _positions(L, 1000 * c, mrope, n_tok=16).contiguous()       # one tensor for all layers of the chunk
            row = []
            for layer in range(layers):
                q, k, v = qkv(H, KVH, L, D, 3.0, seed=77 * c + layer)
                prev = cache.get_prev_temporal_idx(layer)
                row.append(int(prev))
                shared[0, 0, :] += prev + 1 - shared[0, 0, 0]
                cache.update(k, v, layer, {"query_states": q, "position_ids": shared, "rotary_emb": rot,
                                           "mrope_section": mrope})
            prevs.append(row)
            cache.after_forward()
        return cache, prevs

    a, pa = run(False)
    b, pb = run(True)
    assert pa == pb
    assert any(len(set(row)) > 1 for row in pa[1:]), "the layers must disagree on `prev` for this test to mean anything"
    for layer in range(layers):
        assert torch.equal(a.position_cache[layer], b.position_cache[layer])
        assert torch.equal(a.layers[layer].keys, b.layers[layer].keys)
        assert torch.equal(a.layers[layer].values, b.layers[layer].values)


def test_single_layer_growth_keeps_the_pending_overwrite():
    """ADVICE r1: the same layer updated chunk after chunk with no after_forward() in between (1-layer model / direct cache
    API use): when the buffer grows past its 8192-row capacity the previous chunk's kept rows must already be in place
    before the old buffer is copied"""
    lc = _lc()
    H, KVH, L, D, ratio = 4, 2, 1024, 64, 0.9
    cfg = _cfg(H, KVH, D, 1, ratio, False)
    cache = lc.PivotKVCache(cfg)
    want_k, want_v = [], []
    for c in range(10):                                               # 9 x 921 kept rows + 1024 crosses 8192 at chunk 9
        q, k, v = qkv(H, KVH, L, D, 3.0, seed=300 + c)
        cache.kvcache_compression = True
        ko, vo = cache.update(k, v, 0, {"query_states": q, "position_ids": _positions(L, 0, None)})
        idx = cache.last_keep_indices.long()
        want_k.append(k[:, :, idx])
        want_v.append(v[:, :, idx])
        past = sum(t.shape[2] for t in want_k[:-1])
        assert torch.equal(ko[:, :, :past], torch.cat(want_k[:-1], 2)) if past else True      # what this step's attention sees
    assert cache.layers[0]._kbuf.shape[2] > 8192
    assert torch.equal(cache.layers[0].keys, torch.cat(want_k, 2))
    assert torch.equal(cache.layers[0].values, torch.cat(want_v, 2))
    # and through the bare layer API
    layer = lc.PivotKVLayer()
    ks = []
    for c in range(10):
        _, k, v = qkv(H, KVH, L, D, 1.0, seed=400 + c)
        k_all, _ = layer.update(k, v)
        assert k_all.shape[2] == sum(t.shape[2] for t in ks) + L
        layer.replace_tail(L, k[:, :, :900].contiguous(), v[:, :, :900].contiguous())
        ks.append(k[:, :, :900])
    assert torch.equal(layer.keys, torch.cat(ks, 2))


def test_deferred_unsupported_shape_takes_the_immediate_path():
    """ADVICE r1: a shape outside the batched kernels' envelope (here D = 32) must not touch the cache state before the
    library refuses it"""
    lc = _lc()
    cfg = _cfg(4, 2, 32, 1, 0.5, False)
    cfg.longvideo_kwargs["kvcache_compression_kwargs"]["deferred_compression"] = True
    cache = lc.PivotKVCache(cfg)
    q, k, v = qkv(4, 2, 128, 32, 1.0, seed=1)
    with pytest.raises(Exception):
        cache.update(k, v, 0, {"query_states": q, "position_ids": _positions(128, 0, None)})
    assert not cache._deferred and cache.layers[0]._deferred_owner is None


@pytest.mark.parametrize("deferred", [True, False])
@pytest.mark.parametrize("reforge", [True, False])
def test_chunk_loop_never_synchronises_the_host(deferred, reforge):
    """DPSelect, the re-based ids of a new chunk, every update() and the batched flush only ENQUEUE work: with
    torch's sync debug mode on "error" any blocking call (``.item()``, a pageable host-to-device copy such as
    ``torch.tensor(list, device="cuda")``, ``nonzero`` ...) raises.  Round 2 found one such copy per video in
    ``rebased_position_ids`` - the GPU idled behind it while the host enqueued the first chunk."""
    lc = _lc()
    from retake import visual_compression as vc
    H, KVH, L, D, layers, chunks, ratio, mrope = 8, 2, 256, 64, 3, 3, 0.25, [8, 12, 12]
    rot = TableRotary(D, mrope=True)
    rot.inv_freq = rot.inv_freq.cuda()
    x = torch.randn(12, 64, 256, device="cuda").to(BF)
    data = [[qkv(H, KVH, L, D, 1.0, seed=7 * c + layer) for layer in range(layers)] for c in range(chunks)]
    pos_grid = _positions(L, 0, mrope, n_tok=64)

    def one_video():
        out, mask = vc.memory_bank_compress_keyframe(x[None], 12, 3, sync=False)
        cfg = _cfg(H, KVH, D, layers, ratio, reforge)
        cfg.longvideo_kwargs["kvcache_compression_kwargs"]["deferred_compression"] = deferred
        cache = lc.PivotKVCache(cfg)
        for c in range(chunks):
            cache.kvcache_compression = True
            cache.keypatches_mask_chunk = mask[c * L:(c + 1) * L]
            pos_all = cache.rebased_position_ids(pos_grid, layers)
            for layer in range(layers):
                q, k, v = data[c][layer]
                cache.update(k, v, layer, {"query_states": q, "position_ids": pos_all[layer], "rotary_emb": rot,
                                           "mrope_section": mrope, "position_ids_owned": True})
            cache.after_forward()
        return cache

    ref = one_video()                                   # warm-up: library load, function attributes, allocator blocks
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        cache = one_video()
        with pytest.raises(RuntimeError):               # the detector does see the class of call that was removed
            torch.tensor([1, 2], device="cuda")
    finally:
        torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    for layer in range(layers):
        assert torch.equal(cache.layers[layer].keys, ref.layers[layer].keys)
        assert cache.get_seq_length(layer) == chunks * int(ratio * L)
