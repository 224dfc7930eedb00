"""Freeze outputs of the UNMODIFIED reference (SCZwangxiao/video-ReTaKe) into fixtures.

Run in the build container only (it needs ``/root/reference``, which does not travel to
the GPU box):

    python tests/golden/make_golden.py

It imports ``retake.visual_compression.memory_bank_compress_keyframe`` and
``retake.longvideo_cache.PivotKVCache`` from ``/root/reference`` and executes them on CPU
(torch 2.11, transformers 5.5).  ``PivotKVCache.update`` assigns ``self.key_cache[i]``
(transformers 4.48 naming, ``longvideo_cache.py:313``); transformers 5.5 stores
``layers[i].keys`` instead, so the reference class is instantiated through a subclass that
only adds ``key_cache`` / ``value_cache`` list views - the reference code is not edited.

Outputs: ``tests/golden/dpselect_reference.pt.xz``, ``tests/golden/pivotkv_reference.pt.xz`` and
``tests/golden/mallm_reference.pt.xz`` (inputs + outputs, bf16 stored as such; ``torch.save`` files compressed with xz,
which removes the input rows the outputs repeat: 1.5 MB in total, each file under 1 MB; ``helpers.load_golden`` reads them).
"""
import io
import lzma
import os
import sys
import types

import torch

REF = os.environ.get("RETAKE_REFERENCE", "/root/reference")
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from helpers import TableRotary, scene_video  # noqa: E402


def save(cases, name):
    buf = io.BytesIO()
    torch.save(cases, buf)
    with lzma.open(os.path.join(HERE, name + ".pt.xz"), "wb", preset=9 | lzma.PRESET_EXTREME) as f:
        f.write(buf.getvalue())


def load_reference():
    if not os.path.isdir(os.path.join(REF, "retake")):
        raise SystemExit(f"reference tree not found at {REF}")
    sys.path.insert(0, REF)
    import retake.visual_compression as vc   # noqa: E402
    import retake.longvideo_cache as lc      # noqa: E402
    assert vc.__file__.startswith(REF) and lc.__file__.startswith(REF)
    return vc, lc


class _LayerListView:
    """list-like view so that ``cache.key_cache[i] = t`` lands in ``cache.layers[i].keys``."""

    def __init__(self, cache, attr):
        self._c, self._a = cache, attr

    def __getitem__(self, i):
        return getattr(self._c.layers[i], self._a)

    def __setitem__(self, i, v):
        setattr(self._c.layers[i], self._a, v)

    def __len__(self):
        return len(self._c.layers)


def make_shimmed_cache_class(lc):
    class ShimPivotKVCache(lc.PivotKVCache):
        @property
        def key_cache(self):
            return _LayerListView(self, "keys")

        @property
        def value_cache(self):
            return _LayerListView(self, "values")

    return ShimPivotKVCache


def tiny_llm_config(hidden, heads, kv_heads, layers, ratio, reforge):
    cfg = types.SimpleNamespace(hidden_size=hidden, num_hidden_layers=layers, num_attention_heads=heads,
                                num_key_value_heads=kv_heads)
    cfg.longvideo_kwargs = {
        "kvcache_compression": True,
        "kvcache_compression_kwargs": {"compression_ratio": ratio, "compression_method": "pivotkv",
                                       "pos_embed_reforge": reforge},
    }
    return cfg


def gen_dpselect(vc):
    cases = []
    # KAT-D1 (SURVEY.md 8c): unit vectors at given angles, fp32, C=2
    deg0 = [0, 10, 12, 80, 82, 85, 20, 21]
    deg1 = [0, 1, 90, 91, 92, 30, 31, 100]
    ang = torch.deg2rad(torch.tensor([deg0, deg1], dtype=torch.float32)).T  # [8,2]
    X = torch.stack([ang.cos(), ang.sin()], dim=-1)[None]                     # [1,8,2,2]
    for sync in (False, True):
        for t in (8, 5, 3, 2):
            cases.append(("kat_d1", X, t, sync))
    g = torch.Generator().manual_seed(1234)
    for name, T, N, C, dt in [("rand_bf16_a", 24, 16, 256, torch.bfloat16),
                              ("rand_bf16_b", 17, 5, 1152, torch.bfloat16),
                              ("rand_f32", 20, 8, 64, torch.float32)]:
        X = torch.randn(1, T, N, C, generator=g).to(dt)
        for sync in (False, True):
            for t in (T, max(1, round(0.5 * T)), max(1, round(0.25 * T)), 1):
                cases.append((name, X, t, sync))
    for name, T, N, C, dup in [("scene_bf16", 40, 8, 128, 0), ("scene_dup_bf16", 36, 8, 256, 5)]:
        X = scene_video(g, T, N, C, dup_every=dup)[None].to(torch.bfloat16)
        for sync in (False, True):
            for t in (T, T // 2, T // 4):
                cases.append((name, X, t, sync))
    out = []
    for name, X, t, sync in cases:
        Xc = X.clone()
        comp, mask = vc.memory_bank_compress_keyframe(Xc, t, 3, sync=sync)
        assert torch.equal(Xc, X), "reference mutated its input"
        out.append({"name": name, "x": X, "t": t, "sync": sync, "out": comp.clone(), "mask": mask.clone()})
    save(out, "dpselect_reference")
    print("dpselect cases:", len(out))


def gen_pivotkv(lc):
    Cache = make_shimmed_cache_class(lc)
    out = []
    # KAT-P1 (SURVEY.md 8c)
    for dt in (torch.float32, torch.bfloat16):
        for use_mask in (False, True):
            g = torch.Generator().manual_seed(7)
            H, KVH, D, L = 4, 2, 8, 16
            q = torch.randn(1, H, L, D, generator=g).to(dt)
            k = torch.randn(1, KVH, L, D, generator=g).to(dt)
            v = torch.randn(1, KVH, L, D, generator=g).to(dt)
            cache = Cache(tiny_llm_config(H * D, H, KVH, 1, 0.5, False))
            cache.keypatches_mask_chunk = (torch.arange(L) % 5 == 0) if use_mask else None
            pos = torch.arange(L)[None, None].repeat(3, 1, 1)
            ko, vo = cache.update(k, v, 0, {"query_states": q, "position_ids": pos, "rotary_emb": None,
                                            "mrope_section": [1, 1, 2]})
            out.append({"name": "kat_p1", "q": q, "k": k, "v": v, "mask": cache.keypatches_mask_chunk,
                        "ratio": 0.5, "reforge": False, "pos": pos, "mrope": [1, 1, 2],
                        "key_cache": cache.layers[0].keys.clone(), "value_cache": cache.layers[0].values.clone(),
                        "k_out": ko.clone(), "v_out": vo.clone(), "evicted": list(cache.num_evicted_tokens)})
    # multi-chunk, multi-layer replay incl. reforge (call order of qwen2_vl.py:691-718)
    g = torch.Generator().manual_seed(99)
    for name, dt, H, KVH, D, L, chunks, layers, ratio, reforge, mrope, alpha in [
        ("chunks_f32_noreforge", torch.float32, 4, 2, 16, 48, 3, 2, 0.5, False, [2, 3, 3], 1.0),
        ("chunks_f32_reforge", torch.float32, 4, 2, 16, 48, 3, 2, 0.3, True, [2, 3, 3], 1.0),
        ("chunks_bf16_reforge", torch.bfloat16, 4, 2, 64, 64, 2, 2, 0.5, True, [8, 12, 12], 3.0),
        ("chunks_bf16_1d_reforge", torch.bfloat16, 8, 2, 32, 40, 2, 1, 0.25, True, None, 3.0),
        ("chunks_bf16_noreforge", torch.bfloat16, 14, 2, 64, 96, 2, 1, 0.4, False, [8, 12, 12], 3.0),
    ]:
        rot = TableRotary(D, mrope=mrope is not None)
        cache = Cache(tiny_llm_config(H * D, H, KVH, layers, ratio, reforge))
        steps = []
        t0 = 0
        for c in range(chunks):
            cache.kvcache_compression = True
            keymask = torch.rand(L, generator=g) < 0.2
            cache.keypatches_mask_chunk = keymask
            for layer in range(layers):
                q = (torch.randn(1, H, L, D, generator=g) * alpha).to(dt)
                k = (torch.randn(1, KVH, L, D, generator=g) * alpha).to(dt)
                v = torch.randn(1, KVH, L, D, generator=g).to(dt)
                # temporal ids continue after the cached ones when reforging (qwen2_vl.py:256-261)
                base_t = t0
                if reforge:
                    prev = cache.get_prev_temporal_idx(layer)
                    base_t = int(prev) + 1
                tt = base_t + torch.arange(L) // 8
                if mrope is not None:
                    hh = (torch.arange(L) % 8) // 4
                    ww = torch.arange(L) % 4
                    pos = torch.stack([tt, hh, ww])[:, None]
                else:
                    pos = (base_t + torch.arange(L))[None]
                ko, vo = cache.update(k, v, layer, {"query_states": q, "position_ids": pos.clone(),
                                                    "rotary_emb": rot, "mrope_section": mrope})
                steps.append({"chunk": c, "layer": layer, "q": q, "k": k, "v": v, "pos": pos, "mask": keymask,
                              "k_out_shape": tuple(ko.shape),
                              "key_cache": cache.layers[layer].keys.clone(),
                              "value_cache": cache.layers[layer].values.clone(),
                              "position_cache": cache.position_cache[layer].clone() if reforge else None,
                              "evicted": cache.num_evicted_tokens[layer]})
            t0 += L // 8
        out.append({"name": name, "dtype": dt, "H": H, "KVH": KVH, "D": D, "L": L, "ratio": ratio,
                    "reforge": reforge, "mrope": mrope, "rotary": {"head_dim": D, "base": 10000.0,
                                                                    "attention_scaling": 1.1386},
                    "steps": steps})
    save(out, "pivotkv_reference")
    print("pivotkv cases:", len(out))


def gen_mallm(vc):
    """the caller's loop around memory_bank_compress_MALLM / _MALLM_hard (qwen2_vl.py:402-409), every round frozen"""
    g = torch.Generator().manual_seed(4321)
    out = []
    for name, T, N, C, dt, dup, t in [("mallm_f32", 14, 6, 32, torch.float32, 0, 5),
                                      ("mallm_bf16", 16, 9, 64, torch.bfloat16, 0, 6),
                                      ("mallm_dup_bf16", 20, 10, 128, torch.bfloat16, 4, 3),
                                      ("mallm_bf16_wide", 10, 136, 32, torch.bfloat16, 3, 4)]:
        X = scene_video(g, T, N, C, dup_every=dup)[None].to(dt)
        for sync in (False, True):
            bank, size = X.clone(), torch.ones_like(X[:, :, :, 0])
            hard = X.clone()
            rounds = []
            while bank.shape[1] > t:
                bank, size = vc.memory_bank_compress_MALLM(bank, size, sync=sync)
                hard = vc.memory_bank_compress_MALLM_hard(hard, sync=sync)
                rounds.append({"bank": bank.clone(), "size": size.clone(), "hard": hard.clone()})
            keep = [0, len(rounds) // 2, len(rounds) - 1]                # first / middle / last round only (file size)
            out.append({"name": name, "x": X, "t": t, "sync": sync, "n_rounds": len(rounds),
                        "rounds": {i: rounds[i] for i in keep}})
    save(out, "mallm_reference")
    print("mallm cases:", len(out))


if __name__ == "__main__":
    torch.set_num_threads(4)
    vc, lc = load_reference()
    which = sys.argv[1:] or ["dpselect", "pivotkv", "mallm"]
    if "dpselect" in which:
        gen_dpselect(vc)
    if "pivotkv" in which:
        gen_pivotkv(lc)
    if "mallm" in which:
        gen_mallm(vc)
