"""CPU: the C-ABI library loads and exports every symbol include/rtk_b200.h declares; argument validation
paths that need no GPU; the host wrappers refuse CPU tensors (no fallback)."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "rtk_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(rtk_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from retake import _native
    lib = _native.lib()
    names = _declared()
    assert len(names) >= 10
    for n in names:
        assert hasattr(lib, n), f"{n} declared in rtk_b200.h but not exported"
    assert sorted(_native.EXPORTS) == names
    assert lib.rtk_version() == _native.ABI_VERSION == 3
    assert lib.rtk_error_string(0) == b"ok"
    assert b"aligned" in lib.rtk_error_string(-2)


def test_argument_errors_without_gpu():
    from retake import _native
    lib = _native.lib()
    assert lib.rtk_dpselect_dis(None, 4, 4, 256, 0, None, None) == -1          # RTK_E_BADARG
    buf = ctypes.create_string_buffer(64)
    a = ctypes.addressof(buf)
    a16 = (a + 15) & ~15
    assert lib.rtk_dpselect_dis(a16, 4, 4, 100, 0, a16, None) == -3            # C % 8 / C < 256: RTK_E_UNSUPPORTED
    assert lib.rtk_dpselect_dis(a16 + 2, 4, 4, 256, 0, a16, None) == -2        # RTK_E_ALIGN
    assert lib.rtk_dpselect_select(a16, 4, 4, 9, 0, a16, a16, None) == -1      # t > T
    assert lib.rtk_pivot_score(a16, 4, 128, 512, a16, 3, 128, 384, 16, 128, a16, a16, 1 << 20, None) == -3  # H % KVH
    assert lib.rtk_pivot_score(a16, 4, 128, 512, a16, 2, 128, 256, 16, 96, a16, a16, 1 << 20, None) == -3   # D
    assert lib.rtk_pivot_score(a16, 4, 128, 512, a16, 2, 128, 256, 16, 128, a16, a16, 8, None) == -4        # workspace
    assert lib.rtk_pivot_score_workspace_bytes(28, 4096) == 10 * 28 * 4096 * 4
    assert lib.rtk_pivot_score_workspace_bytes(4, 130) == 10 * 4 * 256 * 4
    assert lib.rtk_pivot_select(a16, 4, 16, None, 17, a16, None, None) == -1   # keep > L
    # one step outside the documented limits: RTK_E_UNSUPPORTED before any CUDA call
    assert lib.rtk_dpselect_select(a16, 8193, 4, 9, 0, a16, a16, None) == -3   # T <= 8192
    assert lib.rtk_dpselect_select(a16, 8193, 4, 9, 1, a16, a16, None) == -3
    for T, N, C in ((8193, 4, 256), (4, 65536, 256), (4, 4, 8200)):            # T <= 8192, N <= 65535, C <= 8192
        assert lib.rtk_mallm_compress(a16, None, T, N, C, 2, 0, 0, a16, a16, a16, 1 << 40, None) == -3, (T, N, C)
    assert lib.rtk_pivot_score(a16, 4, 128, 512, a16, 2, 128, 256, 16385, 128, a16, a16, 1 << 40, None) == -3  # L
    assert lib.rtk_pivot_score(a16, 264, 128, 512, a16, 8, 128, 256, 16, 128, a16, a16, 1 << 40, None) == -3  # H <= 256
    assert lib.rtk_pivot_select(a16, 4, 16385, None, 17, a16, None, None) == -3    # L <= 16384
    # batched update: workspace query, argument errors
    one = lib.rtk_pivot_update_batch_workspace_bytes(28, 4, 4096, 128, 1)
    assert lib.rtk_pivot_update_batch_workspace_bytes(28, 4, 4096, 128, 28) > 27 * (one - 1024) > 0
    assert lib.rtk_pivot_update_batch_workspace_bytes(28, 4, 4096, 128, 64) == lib.rtk_pivot_update_batch_workspace_bytes(28, 4, 4096, 128, 32)
    assert lib.rtk_pivot_update_workspace_bytes(28, 4, 4096, 128) >= one       # rtk_pivot_update runs a one-layer batch
    assert lib.rtk_pivot_update_batch(None, 2, a16, 1 << 20, None) == -1
    from retake.longvideo_cache import _UpdateArgs
    arr = (_UpdateArgs * 2)()
    a256 = (ctypes.addressof(ctypes.create_string_buffer(1024)) + 255) & ~255
    assert lib.rtk_pivot_update_batch(arr, 2, a256, 512, None) == -1           # H == 0
    for x in arr:
        x.H, x.KVH, x.L, x.D, x.keep = 4, 2, 64, 64, 16
    assert lib.rtk_pivot_update_batch(arr, 2, a256, 512, None) == -4           # workspace too small
    arr[0].reforge = 1
    assert lib.rtk_pivot_update_batch(arr, 2, a256, 1 << 30, None) == -3       # reforge without inv_freq: not batchable


def test_host_wrappers_refuse_cpu_tensors():
    from retake import _native
    from retake.visual_compression import memory_bank_compress_keyframe
    x = torch.zeros(1, 4, 4, 256, dtype=torch.bfloat16)
    with pytest.raises(_native.RtkError):
        memory_bank_compress_keyframe(x, 2, 3, sync=False)


def test_build_kvcache_factory():
    import types
    from transformers.cache_utils import DynamicCache
    from retake.longvideo_cache import PivotKVCache, build_kvcache
    cfg = types.SimpleNamespace(hidden_size=256, num_hidden_layers=2, num_attention_heads=4, num_key_value_heads=2)
    assert type(build_kvcache(cfg)) is DynamicCache
    cfg.longvideo_kwargs = {"kvcache_compression": False}
    assert type(build_kvcache(cfg)) is DynamicCache
    cfg.longvideo_kwargs = {"kvcache_compression": True,
                            "kvcache_compression_kwargs": {"compression_ratio": 0.5, "compression_method": "PivotKV",
                                                           "pos_embed_reforge": True}}
    c = build_kvcache(cfg)
    assert isinstance(c, PivotKVCache) and isinstance(c, DynamicCache)
    assert c.head_dim == 64 and c.num_key_value_groups == 2 and c.pos_embed_reforge and c.kvcache_compression
    assert c.get_prev_temporal_idx(0) == -1 and c.num_evicted_tokens == [] and c.position_cache == []
    assert c.deferred_compression is False                 # default: compression inside update(), the reference's call order
    cfg.longvideo_kwargs["kvcache_compression_kwargs"]["deferred_compression"] = True
    d = build_kvcache(cfg)
    assert d.deferred_compression is True and d._deferred == []
    d.after_forward()                                      # nothing pending: no library call, works without a GPU
    del cfg.longvideo_kwargs["kvcache_compression_kwargs"]["deferred_compression"]
    cfg.longvideo_kwargs["kvcache_compression_kwargs"]["compression_method"] = "h2o"
    with pytest.raises(NotImplementedError):
        build_kvcache(cfg)


def test_build_id_matches_sources_and_stale_library_is_refused(monkeypatch):
    """VERDICT r1: nothing used to prove which sources a tested library came from.  The library carries the hash of its
    sources; the binding refuses an in-tree library built from other sources."""
    import importlib.util
    from retake import _native
    lib = _native.lib()
    spec = importlib.util.spec_from_file_location("rtk_build_t", os.path.join(ROOT, "video-retake_b200", "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    sid = mod.source_id()
    assert len(sid) == 16 and lib.rtk_build_id().decode() == sid == _native.build_id()
    assert mod.built_id() == sid                                    # lib/BUILD_ID written next to the .so
    monkeypatch.delenv("RTK_B200_LIB", raising=False)
    monkeypatch.delenv("RTK_ALLOW_STALE_LIB", raising=False)
    monkeypatch.setattr(_native, "_source_id", lambda: "0123456789abcdef")
    with pytest.raises(_native.RtkError, match="built from other sources"):
        _native._check_build_id(lib)
    monkeypatch.setenv("RTK_ALLOW_STALE_LIB", "1")
    _native._check_build_id(lib)                                    # explicit opt-out
    # the SASS summary of the build names the Blackwell opcodes of the scoring object
    import json
    sass = json.load(open(os.path.join(ROOT, "video-retake_b200", "lib", "SASS_SUMMARY.json")))
    assert sass["build_id"] == sid
    ops = sass["opcodes"]["pivot_score.o"]
    assert ops.get("UTCHMMA", 0) > 0 and ops.get("UTMALDG", 0) > 0 and ops.get("LDTM", 0) > 0
    assert sass["opcodes"]["dpselect.o"].get("UBLKCP", 0) > 0


def test_real_reference_loader_agrees_with_the_port():
    """bench.py's CPU arm: the unmodified reference functions (when a reference tree is around) and the op-sequence port
    give the same bits on a small case"""
    from oracle import real_reference, reference_ops as ro
    real = real_reference.load(allow_system_tree=True)       # a CPU test in the build container may use the system tree
    if real is None:
        pytest.skip("no reference tree (RETAKE_REFERENCE, baseline/_ref, /root/reference)")
    vc_ref, cache_cls, base = real
    g = torch.Generator().manual_seed(11)
    x = torch.randn(1, 12, 6, 64, generator=g).to(torch.bfloat16)
    out, mask = vc_ref.memory_bank_compress_keyframe(x.clone(), 5, 3, sync=False)
    pout, pmask, _ = ro.dpselect(x.clone(), 5, False)
    assert torch.equal(out, pout) and torch.equal(mask, pmask)
    H, KVH, D, L = 4, 2, 32, 48
    q = torch.randn(1, H, L, D, generator=g).to(torch.bfloat16)
    k = torch.randn(1, KVH, L, D, generator=g).to(torch.bfloat16)
    v = torch.randn(1, KVH, L, D, generator=g).to(torch.bfloat16)
    cache = cache_cls(real_reference.llm_config(H, KVH, D, 1, 0.5, False))
    cache.kvcache_compression = True
    cache.update(k, v, 0, {"query_states": q, "position_ids": torch.arange(L)[None], "rotary_emb": None, "mrope_section": None})
    kk, vv, _, idx, _ = ro.pivot_update(q, k, v, 0.5)
    assert torch.equal(cache.layers[0].keys, kk) and torch.equal(cache.layers[0].values, vv)


def test_bench_traffic_record_is_tied_to_the_scoring_source(tmp_path, monkeypatch):
    import hashlib
    import json
    import types
    import bench
    sha = hashlib.sha256(open(os.path.join(ROOT, "video-retake_b200", "csrc", "pivot_score.cu"), "rb").read()).hexdigest()[:16]
    prof = tmp_path / "profiles"
    prof.mkdir()
    monkeypatch.setattr(bench, "ROOT", str(tmp_path))
    (tmp_path / "video-retake_b200" / "csrc").mkdir(parents=True)
    (tmp_path / "video-retake_b200" / "csrc" / "pivot_score.cu").write_bytes(
        open(os.path.join(ROOT, "video-retake_b200", "csrc", "pivot_score.cu"), "rb").read())
    s = types.SimpleNamespace(L=4096, deferred=True)
    assert bench.measured_traffic(s) is None                          # no record at all
    (prof / "ncu_score_traffic.json").write_text(json.dumps([{"score_source_sha": "stale", "L": 4096, "deferred": True,
                                                               "bytes_per_layer": 1.0}]))
    assert bench.measured_traffic(s) is None                          # a capture of another kernel is never used
    (prof / "ncu_score_traffic.json").write_text(json.dumps([{"score_source_sha": sha, "L": 4096, "deferred": True,
                                                               "bytes_per_layer": 7.0e7}]))
    assert bench.measured_traffic(s) == 7.0e7
    assert bench.measured_traffic(types.SimpleNamespace(L=6272, deferred=True)) is None
