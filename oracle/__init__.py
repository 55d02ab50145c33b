"""CPU restatement ("oracle") of the reference hot path.  TEST INFRASTRUCTURE ONLY.

Only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s CPU-baseline /
`--impl reference` legs may import this package, and only as the checker or the
reported CPU baseline.  Nothing under `buckgnn_b200/` or `Models/` imports it; the
product path raises if the CUDA library is missing instead of falling back here.

PARITY PINNED TO THE REFERENCE'S OWN SOURCE FILE (round 2).  `reference_source.py` executes
the reference's `Models/BuckGNN.py` unmodified (read where it lies, nothing copied) and
`tests/test_reference_source.py` asserts reference == oracle to 1e-6 on the CPU for every
`model_name` x `pooling_layer` x `prediction_type` that works in the reference (forward,
autograd gradients, BatchNorm buffers, the dropout RNG stream), plus the reference's broken
branches.  The golden fixtures of `tests/golden/` are OUTPUTS OF THAT REFERENCE FILE (stamped with
its sha256), so the GPU golden tests compare the CUDA path with the reference, not with this
restatement.

What remains restated: the arithmetic INSIDE two third-party packages the reference imports, which
are neither vendored in the reference project nor dependencies of this one: `torch_geometric`
(`SAGEConv`, `SAGPooling`, `global_mean_pool`) and `torch_scatter` (`scatter_mean`,
`scatter_add`), both unpinned by the reference (`README.md:64-70` names them without versions;
the `lin_l` / `lin_r` parameter names imply PyG >= 1.6 / 2.x).  Their published semantics are
restated at the reference's call sites (`Models/BuckGNN.py:114-176, 203-208, 274, 449, 561`) in
`buckgnn_oracle.py` and anchored by hand-computed known-answer cases and an independent
dense-adjacency formulation (`tests/test_oracle.py`).  The reference ships no tests or vectors of
its own.
"""
