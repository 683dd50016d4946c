#!/usr/bin/env python
"""Regenerates the stored outputs of the compiled reference that two tests compare against, on the
seeded inputs those tests generate.  Needs oracle/_ref built by oracle/Makefile (which needs the
reference sources); the tests themselves read only the stored files.

    python tests/golden/make_golden_ref_runs.py cpu [OUT]   # ref_live_cases.npz: reference CPU library
    python tests/golden/make_golden_ref_runs.py gpu [OUT]   # ref_gpu_cases.npz: reference CUDA kernels, on a B200
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "warp-transducer_b200")):
    sys.path.insert(0, p)
from oracle import pyoracle  # noqa: E402


def cpu(out):
    """tests/test_oracle.py::test_live_against_compiled_reference."""
    from test_oracle import live_cases
    assert pyoracle.have_ref_cpu(), "oracle/_ref/libwarprnnt_ref_cpu.so is not built"
    blob = {}
    for k, (acts, labels, tl, ul) in enumerate(live_cases()):
        lp = pyoracle.log_softmax_np(acts)
        c, g = pyoracle.ref_cpu_logprobs(lp, labels, tl, ul, 0, threads=2)
        c_fwd, _ = pyoracle.ref_cpu_logprobs(lp, labels, tl, ul, 0, want_grad=False)
        c64, g64 = pyoracle.ref_cpu_logprobs(pyoracle.log_softmax_np(acts.astype(np.float64)), labels, tl, ul, 0)
        blob.update({"%d.costs_f32" % k: c, "%d.grads_f32" % k: g, "%d.costs_fwd_f32" % k: c_fwd,
                     "%d.costs_f64" % k: c64, "%d.grads_f64" % k: g64})
        print(k, acts.shape, c64)
    np.savez_compressed(out, **blob)


def gpu(out):
    """tests/test_gpu_vs_reference_gpu.py: costs, gradient sample and an input checksum per case."""
    import torch
    from test_gpu_vs_reference_gpu import CASES, call_abi, gather, load_reference_gpu, make_inputs, sample_indices
    assert pyoracle.have_ref_gpu(), "oracle/_ref/libwarprnnt_ref_gpu.so is not built"
    ref = load_reference_gpu()
    blob = {"device": np.array(torch.cuda.get_device_name(0))}
    for name, (N, T, L, V, ragged, seed) in CASES.items():
        acts, labels_np, tl_np, ul_np = make_inputs(N, T, L, V, ragged, seed)
        costs, grads = call_abi(*ref, acts, labels_np, tl_np, ul_np)
        blob.update({name + ".acts_sum": np.float64(acts.sum(dtype=torch.float64).item()),
                     name + ".costs": costs,
                     name + ".grads": gather(grads, sample_indices(acts.shape, labels_np, tl_np, ul_np, seed))})
        print(name, costs[:4], "non-finite in sample:", int((~np.isfinite(blob[name + ".grads"])).sum()), flush=True)
        del acts, grads
        torch.cuda.empty_cache()
    np.savez_compressed(out, **blob)


if __name__ == "__main__":
    mode = sys.argv[1]
    name = {"cpu": "ref_live_cases.npz", "gpu": "ref_gpu_cases.npz"}[mode]
    out = sys.argv[2] if len(sys.argv) > 2 else os.path.join(HERE, name)
    {"cpu": cpu, "gpu": gpu}[mode](out)
    print("wrote", out)
