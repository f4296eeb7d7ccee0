"""TEST INFRASTRUCTURE ONLY.

CPU oracle of the MicroDiT training hot path.  Nothing in `micro_diffusion_b200/` may import this
package; only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s CPU-baseline / `--impl reference`
legs use it, and there only as the checker or the timed baseline (plus `tools/stock_torch_gpu.py`, a developer
yardstick that times this same restatement through stock PyTorch on the GPU -- SURVEY.md section 8d's "honest GPU
comparator"; it is not part of the product, the tests or bench.py).

* `oracle.ref_import`  -- loads the UNMODIFIED reference from its source tree (oracle/make_golden.py only).
* `oracle.port`        -- a functional fp32 restatement of the reference algorithm that travels with
                          the repo; pinned against the reference by tests/test_oracle_pinned.py through
                          the fixtures in tests/golden/.
* `oracle.emu_ops`     -- per-kernel CPU restatement of each CUDA op's contract (same buffers, same
                          rounding points); lets the host-side engine be exercised without a GPU.
"""
