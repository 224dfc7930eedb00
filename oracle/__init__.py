"""CPU oracle for the DPSelect + PivotKV hot path.  TEST INFRASTRUCTURE ONLY.

This package restates the reference algorithm (SCZwangxiao/video-ReTaKe,
``retake/visual_compression.py:86-177`` and ``retake/longvideo_cache.py:16-334``)
as explicit, op-by-op CPU arithmetic.  It exists so that the CUDA kernels under
``video-retake_b200/csrc`` have something independent to be checked against.

Only ``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` /
``--impl reference`` legs of ``bench.py`` may import it.  The product path
(``video-retake_b200/retake``) never does: it fails loudly when the CUDA
library is missing.

Parity status: PINNED.  The reference has no tests or golden vectors of its
own (SURVEY.md section 4), so the oracle is pinned against outputs of the
*unmodified reference functions executed in the build container* (CPU torch
2.11): ``tests/golden/make_golden.py`` imports ``/root/reference/retake`` and
freezes its outputs into ``tests/golden/*.pt.xz``; ``tests/test_oracle_golden.py``
replays them through this package.  The survey-time known answers KAT-D1 and
KAT-P1 (SURVEY.md section 8c) are part of that set.
"""
