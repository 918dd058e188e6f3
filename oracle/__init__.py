"""CPU oracle for the attention-forward hot path.  TEST INFRASTRUCTURE ONLY.

This package is a CPU restatement (fp32 torch/numpy einsum form) of the
reference's attention forwards.  It exists to CHECK the CUDA path; it is never
the thing shipped or measured.  Only ``tests/``, ``__graft_entry__.smoke()``
and ``bench.py``'s ``cpu_baseline`` / ``--impl reference`` legs may import it.
The product package (``pytorch_attention_b200``) must never import ``oracle``.

Parity pin: the reference repository has no tests, fixtures or golden vectors
(SURVEY.md §4, §8c).  The oracle is therefore pinned against outputs of the
reference itself: ``oracle/make_golden.py`` imports the real modules from
``/root/reference/vision_transformers`` in the build container, checks every
restatement against them (fp32, <= 2e-6 max-abs) and commits seeded
input/output vectors under ``tests/golden/``.  ``tests/test_oracle_golden.py``
re-checks the restatement against those committed vectors on every run, and
``tests/test_oracle_vs_reference.py`` re-checks against further reference
outputs (fresh seeds, configurations without a golden file) that
``oracle/record_reference.py`` recorded into ``tests/golden/reference/fresh_seeds.npz``.
"""
from .attention import (  # noqa: F401
    vit_attention,
    vit_block_attention_half,
    pvt_attention,
    cvt_attention,
    cswin_lepe_attention,
    cswin_block_attention,
    xca_attention,
    class_attention,
    cswin_window_table,
)
