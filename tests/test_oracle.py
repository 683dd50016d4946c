"""Pins the CPU oracle (oracle/rnnt_oracle.c) before anything is checked against it.

  1. the reference test-suite's own known-answer vectors (tests/golden/known_answers.json)
  2. outputs of the reference itself on seeded random cases (tests/golden/ref_cases.npz,
     produced by the compiled reference CPU library + the reference numpy model)
  3. outputs of the compiled reference CPU library (oracle/_ref/libwarprnnt_ref_cpu.so) on
     seeded inputs, stored in tests/golden/ref_live_cases.npz
"""
import os

import numpy as np

from oracle import pyoracle


def _ka(ka):
    a = np.array(ka["acts"], np.float32).reshape(ka["shape"])
    labels = np.array(ka["labels"], np.int32)
    N, T, U, V = ka["shape"]
    return a, labels, np.full(N, T, np.int32), np.full(N, U - 1, np.int32)


def test_small_known_answer(known_answers):
    ka = known_answers["small"]
    a, y, tl, ul = _ka(ka)
    for dt in (np.float32, np.float64):
        costs, grads, llb = pyoracle.rnnt_logits(a.astype(dt), y, tl, ul, 0)
        assert abs(costs[0] - ka["cost"]) < ka["cost_tol_abs"]       # test_gpu.cu:87-93
        assert np.allclose(costs, ka["cost"], rtol=1e-6)             # test.py:75
        assert np.allclose(grads.reshape(-1), ka["logits_grads"], atol=1e-6)  # test.py:77
        assert abs(llb[0] + costs[0]) < 1e-5
    # CPU convention on host log-softmax (test_cpu.cpp:28-29): forward-only cost
    c, _ = pyoracle.rnnt_logprobs(pyoracle.log_softmax_np(a), y, tl, ul, 0, want_grad=False)
    assert abs(c[0] - ka["cost"]) < 1e-4


def test_options_known_answer(known_answers):
    ka = known_answers["options"]
    a, y, tl, ul = _ka(ka)
    costs, grads, _ = pyoracle.rnnt_logits(a, y, tl, ul, 0)
    assert np.allclose(costs, ka["costs"], atol=ka["tol_abs"])                    # test_gpu.cu:210-222
    assert np.allclose(grads.reshape(-1), ka["logits_grads"], atol=ka["tol_abs"])  # test_gpu.cu:195-207
    # higher-precision copy of the same vectors (test.py:86-149), rtol as the reference uses
    a64 = np.array(ka["acts_f64"]).reshape(ka["shape"])
    c64, g64, _ = pyoracle.rnnt_logits(a64, y, tl, ul, 0)
    assert np.allclose(c64.sum(), sum(ka["costs"]))
    assert np.allclose(g64.reshape(-1), ka["logits_grads_hi"], rtol=1e-3)
    # log-prob-gradient convention (test_cpu.cpp:94-105)
    c, g = pyoracle.rnnt_logprobs(pyoracle.log_softmax_np(a), y, tl, ul, 0)
    assert np.allclose(c, ka["costs"], atol=1e-4)
    assert np.allclose(g.reshape(-1), ka["logprob_grads"], atol=1e-4)


def test_against_committed_reference_outputs(ref_cases):
    for name, cs in ref_cases.items():
        blank = int(cs["blank"])
        c64, g64, llb = pyoracle.rnnt_logits(cs["acts"].astype(np.float64), cs["labels"],
                                             cs["act_lens"], cs["label_lens"], blank)
        assert np.allclose(c64, cs["ref_costs_f64"], rtol=1e-12, atol=1e-10), name
        assert np.allclose(g64, cs["ref_grads_f64"], rtol=1e-9, atol=1e-12), name
        assert np.allclose(-llb, c64, rtol=1e-10), name
        assert np.allclose(c64, cs["np_costs"], rtol=1e-5, atol=1e-5), name
        c32, g32, _ = pyoracle.rnnt_logits(cs["acts"], cs["labels"], cs["act_lens"],
                                           cs["label_lens"], blank)
        assert np.allclose(c32, cs["ref_costs_f32"], rtol=2e-6, atol=1e-5), name
        assert np.allclose(g32, cs["ref_grads_f32"], rtol=1e-4, atol=2e-6), name
        # padded cells carry exactly zero gradient (cpu_rnnt.h:155-158)
        for b in range(cs["acts"].shape[0]):
            T, U = int(cs["act_lens"][b]), int(cs["label_lens"][b]) + 1
            assert not g32[b, T:].any() and not g32[b, :, U:].any(), name


LIVE_SHAPES = [(3, 11, 6, 10), (2, 50, 10, 15), (65, 10, 5, 5), (1, 50, 15, 20)]
REF_LIVE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_live_cases.npz")


def live_cases():
    """Seeded inputs of test_live_against_compiled_reference, one (acts, labels, tl, ul) per shape."""
    rng = np.random.default_rng(7)
    for (N, T, U, V) in LIVE_SHAPES:
        acts = rng.random((N, T, U, V), dtype=np.float32)      # U[0,1) like tests/random.cpp:13-20
        labels = rng.integers(1, V, size=(N, U - 1)).astype(np.int32)
        tl = rng.integers(T // 2 + 1, T + 1, size=N).astype(np.int32)
        ul = rng.integers(0, U, size=N).astype(np.int32)
        tl[0], ul[0] = T, U - 1
        yield acts, labels, tl, ul


def test_live_against_compiled_reference():
    """The compiled reference CPU library's outputs on live_cases() are stored in
    tests/golden/ref_live_cases.npz (tests/golden/make_golden_ref_runs.py cpu)."""
    with np.load(REF_LIVE) as z:
        stored = dict(z)
    for k, (acts, labels, tl, ul) in enumerate(live_cases()):
        ref = {name: stored["%d.%s" % (k, name)] for name in
               ("costs_f32", "grads_f32", "costs_fwd_f32", "costs_f64", "grads_f64")}
        lp = pyoracle.log_softmax_np(acts)
        c_orc, g_orc = pyoracle.rnnt_logprobs(lp, labels, tl, ul, 0, threads=2)
        assert np.allclose(c_orc, ref["costs_f32"], rtol=1e-6, atol=1e-5)
        # fp32 noise floor: exp(lp+alpha+beta-ll) with |ll|~100 has ~4 ulp(100)=3e-5 abs error in
        # BOTH implementations (each is 3e-5 from the fp64 result); the fp64 comparison below is tight
        assert np.allclose(g_orc, ref["grads_f32"], rtol=1e-4, atol=5e-5)
        # forward-only entry (gradients == NULL -> score_forward, rnnt_entrypoint.cpp:70-72)
        c_of, _ = pyoracle.rnnt_logprobs(lp, labels, tl, ul, 0, want_grad=False)
        assert np.allclose(c_of, ref["costs_fwd_f32"], rtol=1e-6, atol=1e-5)
        # logits convention = reference CPU lib composed with log-softmax fwd/bwd
        dx_ref = pyoracle.logits_grad(pyoracle.log_softmax_np(acts.astype(np.float64)), ref["grads_f64"])
        c3, dx_orc, _ = pyoracle.rnnt_logits(acts.astype(np.float64), labels, tl, ul, 0)
        assert np.allclose(c3, ref["costs_f64"], rtol=1e-12)
        assert np.allclose(dx_orc, dx_ref, rtol=1e-9, atol=1e-13)


def test_numeric_gradient_like_reference():
    """Central-difference check as tests/test_cpu.cpp:287-379 (eps 1e-2, rel_diff < 1e-4), fp64."""
    rng = np.random.default_rng(3)
    N, T, U, V = 2, 6, 4, 5
    acts = rng.random((N, T, U, V))
    labels = rng.integers(1, V, size=(N, U - 1)).astype(np.int32)
    tl = np.array([T, T - 2], np.int32)
    ul = np.array([U - 1, U - 2], np.int32)
    _, g, _ = pyoracle.rnnt_logits(acts, labels, tl, ul, 0)
    num = np.zeros_like(acts)
    eps = 1e-4
    flat = acts.reshape(-1)
    for i in range(flat.size):
        old = flat[i]
        flat[i] = old + eps
        cp, _, _ = pyoracle.rnnt_logits(acts, labels, tl, ul, 0, want_grad=False)
        flat[i] = old - eps
        cm, _, _ = pyoracle.rnnt_logits(acts, labels, tl, ul, 0, want_grad=False)
        flat[i] = old
        num.reshape(-1)[i] = (cp.sum() - cm.sum()) / (2 * eps)
    rel = ((g - num) ** 2).sum() / (g ** 2).sum()     # tests/test.h:22-32
    assert rel < 1e-8
