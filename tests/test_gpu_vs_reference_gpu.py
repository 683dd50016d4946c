"""Cross-check against the REFERENCE'S OWN CUDA kernels compiled for sm_100
(oracle/_ref/libwarprnnt_ref_gpu.so, built by oracle/Makefile) on the same inputs, including
BASELINE's headline shape at full size.  The reference's outputs on these seeded inputs, run on a
B200, are stored in tests/golden/ref_gpu_cases.npz (tests/golden/make_golden_ref_runs.py gpu): all
its costs, and its gradient at a fixed seeded sample of elements (uniform over the tensor, plus
blank and label entries of valid cells, where the lattice shows).  The reference GPU path is fp32
throughout, so its own rounding noise (alpha/beta of magnitude ~1e3 carried in fp32) bounds how
tight this can be; the tight parity bound is the fp64 oracle in test_gpu_parity.py."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from oracle import pyoracle

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_gpu_cases.npz")
# name: (N, T, L, V, ragged, seed)
CASES = {"small": (8, 50, 10, 15, True, 5), "readme_small_vocab": (16, 150, 40, 28, True, 5),
         "readme_large_vocab_N4": (4, 150, 20, 5000, True, 5), "headline": (128, 150, 20, 5000, False, 9)}


def make_inputs(N, T, L, V, ragged, seed):
    dev = torch.device("cuda:0")
    U = L + 1
    gen = torch.Generator(device=dev).manual_seed(seed)
    acts = torch.rand((N, T, U, V), generator=gen, device=dev)
    rng = np.random.default_rng(seed)
    labels_np = rng.integers(1, V, size=(N, L)).astype(np.int32)
    tl_np, ul_np = np.full(N, T, np.int32), np.full(N, L, np.int32)
    if ragged:
        tl_np[1::3] = rng.integers(T // 2, T + 1, size=len(tl_np[1::3]))
        ul_np[2::3] = rng.integers(0, L + 1, size=len(ul_np[2::3]))
    return acts, labels_np, tl_np, ul_np


def call_abi(lib, options_type, acts, labels_np, tl_np, ul_np):
    """compute_rnnt_loss of `lib` (this library or the reference's) on device inputs, host costs."""
    N, T, U, V = acts.shape
    dev = acts.device
    labels, tl, ul = (torch.as_tensor(x).to(dev) for x in (labels_np, tl_np, ul_np))
    opt = options_type(loc=1, num_threads=0, stream=torch.cuda.current_stream().cuda_stream,
                       blank_label=0, maxT=T, maxU=U, batch_first=True)
    n = C.c_size_t(0)
    assert lib.get_workspace_size(T, U, N, True, C.byref(n), 4) == 0
    ws = torch.empty(n.value, dtype=torch.uint8, device=dev)
    grads = torch.full_like(acts, float("nan"))
    costs = np.zeros(N, np.float32)
    st = lib.compute_rnnt_loss(acts.data_ptr(), grads.data_ptr(), labels.data_ptr(), ul.data_ptr(),
                               tl.data_ptr(), V, N, costs.ctypes.data, ws.data_ptr(), opt)
    assert st == 0
    torch.cuda.synchronize()
    return costs, grads


def sample_indices(shape, labels_np, tl_np, ul_np, seed, k=2048):
    """k uniform flat indices of the gradient, then k valid cells at the blank or the next label."""
    N, T, U, V = shape
    rng = np.random.default_rng(1000 + seed)
    uniform = rng.integers(0, N * T * U * V, size=k)
    n = rng.integers(0, N, size=k)
    t = (rng.random(k) * tl_np[n]).astype(np.int64)
    u = (rng.random(k) * (ul_np[n] + 1)).astype(np.int64)
    at_label = (np.arange(k) % 2 == 1) & (u < ul_np[n])
    v = np.where(at_label, labels_np[n, np.minimum(u, U - 2)], 0)
    return np.concatenate([uniform, ((n * T + t) * U + u) * V + v])


def load_reference_gpu():
    """The reference's CUDA kernels (oracle/_ref) and the options struct its C-ABI takes."""
    ref = C.CDLL(pyoracle.ref_gpu_path())
    assert ref.get_warprnnt_version() == 1
    ref.compute_rnnt_loss.restype = C.c_int
    ref.compute_rnnt_loss.argtypes = [C.c_void_p] * 5 + [C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                                         pyoracle.RnntOptions]
    ref.get_workspace_size.argtypes = [C.c_int, C.c_int, C.c_int, C.c_bool, C.POINTER(C.c_size_t), C.c_size_t]
    return ref, pyoracle.RnntOptions


def gather(grads, idx):
    return grads.view(-1)[torch.as_tensor(idx, device=grads.device)].cpu().numpy()


@pytest.fixture(scope="module")
def ours():
    import warprnnt_pytorch.warp_rnnt as wr
    with np.load(GOLDEN) as z:
        golden = dict(z)

    def run(name):
        N, T, L, V, ragged, seed = CASES[name]
        acts, labels_np, tl_np, ul_np = make_inputs(N, T, L, V, ragged, seed)
        # the seeded inputs must be the ones the stored reference outputs were computed on
        assert np.isclose(float(acts.sum(dtype=torch.float64)), float(golden[name + ".acts_sum"]), rtol=1e-9)
        costs, grads = call_abi(wr.lib(), wr.rnntOptions, acts, labels_np, tl_np, ul_np)
        assert bool(torch.isfinite(grads).all())
        g = gather(grads, sample_indices(acts.shape, labels_np, tl_np, ul_np, seed)).astype(np.float64)
        return costs, g, golden[name + ".costs"], golden[name + ".grads"].astype(np.float64)
    return run


@pytest.mark.parametrize("name", ["small", "readme_small_vocab", "readme_large_vocab_N4"])
def test_same_answers_as_reference_gpu_kernels(ours, name):
    costs, g, c_ref, gr = ours(name)
    assert np.allclose(costs, c_ref, rtol=1e-5)
    assert ((g - gr) ** 2).sum() / (gr ** 2).sum() < 1e-6      # tests/test.h:22-32 metric
    assert np.allclose(g, gr, rtol=5e-3, atol=2e-6)


def test_headline_shape_full_size_matches_reference_gpu(ours):
    """N=128, T=150, L=20, A=5000: all 2 016 000 000 gradient elements finite, the sample against the reference."""
    costs, g, c_ref, gr = ours("headline")
    assert np.allclose(costs, c_ref, rtol=1e-5)
    assert ((g - gr) ** 2).sum() / (gr ** 2).sum() < 1e-6
    # fp32 reference noise at |ll| ~ 1.4e3 is ~1e-3 relative; ours is far inside it
    worst = float((np.abs(g - gr) / (2e-6 + 1e-2 * np.abs(gr))).max())
    assert worst <= 1.0, worst


@pytest.mark.skipif(not pyoracle.have_ref_gpu(), reason="oracle/_ref/libwarprnnt_ref_gpu.so not built")
@pytest.mark.parametrize("name", list(CASES))
def test_every_element_against_live_reference_gpu(name):
    """Where oracle/_ref is built: the reference's kernels run here reproduce the stored outputs bit
    for bit, and every gradient element of ours is compared with theirs."""
    import warprnnt_pytorch.warp_rnnt as wr
    N, T, L, V, ragged, seed = CASES[name]
    acts, labels_np, tl_np, ul_np = make_inputs(N, T, L, V, ragged, seed)
    c_ref, gr = call_abi(*load_reference_gpu(), acts, labels_np, tl_np, ul_np)
    with np.load(GOLDEN) as z:
        assert np.array_equal(c_ref, z[name + ".costs"])
        assert np.array_equal(gather(gr, sample_indices(acts.shape, labels_np, tl_np, ul_np, seed)), z[name + ".grads"])
    costs, g = call_abi(wr.lib(), wr.rnntOptions, acts, labels_np, tl_np, ul_np)
    assert np.allclose(costs, c_ref, rtol=1e-5)
    rtol = 1e-2 if name == "headline" else 5e-3
    num = den = worst = 0.0
    for b in range(0, N, 16):            # chunked to bound temporaries
        d = (g[b:b + 16] - gr[b:b + 16]).double()
        num += float((d ** 2).sum())
        den += float((gr[b:b + 16].double() ** 2).sum())
        worst = max(worst, float((d.abs() / (2e-6 + rtol * gr[b:b + 16].abs().double())).max()))
    assert num / den < 1e-6, num / den
    assert worst <= 1.0, worst
