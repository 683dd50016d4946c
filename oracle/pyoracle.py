"""ctypes front-end for the CPU checkers.  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs may import this module; the product package never does.

Two checkers live behind it:
  * ``oracle/librnnt_oracle.so``         our C restatement (oracle/rnnt_oracle.c)
  * ``oracle/_ref/libwarprnnt_ref_cpu.so``  the unmodified reference CPU path, compiled
    from /root/reference by oracle/Makefile (prebuilt file travels to the GPU box)
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE_SO = os.path.join(_HERE, "librnnt_oracle.so")
_REF_CPU_SO = os.path.join(_HERE, "_ref", "libwarprnnt_ref_cpu.so")
_REF_GPU_SO = os.path.join(_HERE, "_ref", "libwarprnnt_ref_gpu.so")

_oracle = None
_ref_cpu = None


def build(quiet=True):
    """(Re)build the checker libraries with oracle/Makefile (gcc; reference only if present)."""
    out = subprocess.run(["make", "-C", _HERE, "all"], capture_output=True, text=True)
    if out.returncode != 0:
        raise RuntimeError("oracle build failed:\n" + out.stdout + out.stderr)
    if not quiet:
        print(out.stdout)


def _fp(dt):
    return C.POINTER(C.c_float if dt == np.float32 else C.c_double)


def load_oracle():
    global _oracle
    if _oracle is None:
        if not os.path.exists(_ORACLE_SO):
            build()
        _oracle = C.CDLL(_ORACLE_SO)
    return _oracle


def _ptr(a, ty):
    return a.ctypes.data_as(C.POINTER(ty)) if a is not None else None


def _prep(acts, labels, act_lens, label_lens):
    acts = np.ascontiguousarray(acts)
    assert acts.dtype in (np.float32, np.float64) and acts.ndim == 4
    labels = np.ascontiguousarray(labels, dtype=np.int32)
    act_lens = np.ascontiguousarray(act_lens, dtype=np.int32)
    label_lens = np.ascontiguousarray(label_lens, dtype=np.int32)
    N, T, U, V = acts.shape
    if labels.size == 0:  # U == 1: keep a valid pointer
        labels = np.zeros((N, 1), dtype=np.int32)
    else:
        assert labels.shape == (N, U - 1), (labels.shape, acts.shape)
    return acts, labels, act_lens, label_lens


def rnnt_logits(acts, labels, act_lens, label_lens, blank=0, want_grad=True, threads=0,
                want_lattice=False):
    """GPU convention: logits in -> (costs[N], dense grads wrt logits | None, ll_backward[N]).

    Precision follows acts.dtype (float32 mirrors the reference arithmetic; float64 = truth).
    """
    lib = load_oracle()
    acts, labels, act_lens, label_lens = _prep(acts, labels, act_lens, label_lens)
    N, T, U, V = acts.shape
    dt = acts.dtype
    cty = C.c_float if dt == np.float32 else C.c_double
    fn = lib.oracle_rnnt_logits_f32 if dt == np.float32 else lib.oracle_rnnt_logits_f64
    fn.restype = C.c_int
    costs = np.zeros(N, dtype=dt)
    llb = np.zeros(N, dtype=dt)
    grads = np.empty_like(acts) if want_grad else None
    T0, U0 = int(act_lens[0]), int(label_lens[0]) + 1
    da = np.zeros((T0, U0), dtype=dt) if want_lattice else None
    db = np.zeros((T0, U0), dtype=dt) if want_lattice else None
    rc = fn(_ptr(acts, cty), _ptr(grads, cty), _ptr(labels, C.c_int), _ptr(label_lens, C.c_int),
            _ptr(act_lens, C.c_int), C.c_int(V), C.c_int(N), C.c_int(T), C.c_int(U),
            C.c_int(blank), _ptr(costs, cty), C.c_int(threads), _ptr(da, cty), _ptr(db, cty),
            _ptr(llb, cty))
    if rc != 0:
        raise RuntimeError("oracle_rnnt_logits rc=%d" % rc)
    if want_lattice:
        return costs, grads, llb, da, db
    return costs, grads, llb


def rnnt_logprobs(log_probs, labels, act_lens, label_lens, blank=0, want_grad=True, threads=0):
    """CPU convention: log-probs in -> (costs[N], sparse grads wrt log-probs | None)."""
    lib = load_oracle()
    lp, labels, act_lens, label_lens = _prep(log_probs, labels, act_lens, label_lens)
    N, T, U, V = lp.shape
    dt = lp.dtype
    cty = C.c_float if dt == np.float32 else C.c_double
    fn = lib.oracle_rnnt_logprobs_f32 if dt == np.float32 else lib.oracle_rnnt_logprobs_f64
    fn.restype = C.c_int
    costs = np.zeros(N, dtype=dt)
    grads = np.empty_like(lp) if want_grad else None
    rc = fn(_ptr(lp, cty), _ptr(grads, cty), _ptr(labels, C.c_int), _ptr(label_lens, C.c_int),
            _ptr(act_lens, C.c_int), C.c_int(V), C.c_int(N), C.c_int(T), C.c_int(U),
            C.c_int(blank), _ptr(costs, cty), C.c_int(threads), None, None)
    if rc != 0:
        raise RuntimeError("oracle_rnnt_logprobs rc=%d" % rc)
    return costs, grads


# --------------------------------------------------------------------------------------
# The unmodified reference, through its own C-ABI (include/rnnt.h of the reference).
# --------------------------------------------------------------------------------------
class RnntOptions(C.Structure):
    """rnntOptions, 32 bytes, passed by value (reference include/rnnt.h:43-64)."""
    _fields_ = [("loc", C.c_int), ("num_threads", C.c_uint), ("stream", C.c_void_p),
                ("blank_label", C.c_int), ("maxT", C.c_int), ("maxU", C.c_int),
                ("batch_first", C.c_bool)]


def have_ref_cpu():
    return os.path.exists(_REF_CPU_SO)


def have_ref_gpu():
    return os.path.exists(_REF_GPU_SO)


def ref_gpu_path():
    return _REF_GPU_SO


def load_ref_cpu():
    global _ref_cpu
    if _ref_cpu is None:
        if not have_ref_cpu():
            return None
        _ref_cpu = C.CDLL(_REF_CPU_SO)
        assert _ref_cpu.get_warprnnt_version() == 1
    return _ref_cpu


def ref_cpu_logprobs(log_probs, labels, act_lens, label_lens, blank=0, want_grad=True, threads=0):
    """Reference compute_rnnt_loss(loc=RNNT_CPU, batch_first=true): log-probs in, sparse grads out."""
    lib = load_ref_cpu()
    if lib is None:
        raise RuntimeError("oracle/_ref/libwarprnnt_ref_cpu.so is not built")
    lp, labels, act_lens, label_lens = _prep(log_probs, labels, act_lens, label_lens)
    N, T, U, V = lp.shape
    dt = lp.dtype
    cty = C.c_float if dt == np.float32 else C.c_double
    fn = lib.compute_rnnt_loss if dt == np.float32 else lib.compute_rnnt_loss_fp64
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                   C.c_void_p, C.c_void_p, RnntOptions]
    nbytes = C.c_size_t(0)
    lib.get_workspace_size.argtypes = [C.c_int, C.c_int, C.c_int, C.c_bool,
                                       C.POINTER(C.c_size_t), C.c_size_t]
    rc = lib.get_workspace_size(T, U, N, False, C.byref(nbytes), lp.itemsize)
    assert rc == 0
    ws = np.zeros(nbytes.value, dtype=np.uint8)
    costs = np.zeros(N, dtype=dt)
    grads = np.empty_like(lp) if want_grad else None
    opt = RnntOptions(loc=0, num_threads=threads, stream=None, blank_label=blank, maxT=T, maxU=U,
                      batch_first=True)
    rc = fn(lp.ctypes.data, grads.ctypes.data if want_grad else None, labels.ctypes.data,
            label_lens.ctypes.data, act_lens.ctypes.data, V, N, costs.ctypes.data, ws.ctypes.data,
            opt)
    if rc != 0:
        raise RuntimeError("reference compute_rnnt_loss rc=%d" % rc)
    return costs, grads


def log_softmax_np(x):
    m = x.max(axis=-1, keepdims=True)
    return (x - m) - np.log(np.exp(x - m).sum(axis=-1, keepdims=True))


def logits_grad(lp, g):
    """log_softmax backward: gradient wrt the logits from the gradient g wrt the log-probs lp."""
    return g - np.exp(lp) * g.sum(axis=-1, keepdims=True)


def ref_cpu_logits(acts, labels, act_lens, label_lens, blank=0, threads=0):
    """logits -> log_softmax -> reference CPU lib -> log_softmax backward (what warprnnt_pytorch
    composes on CPU, pytorch_binding/warprnnt_pytorch/__init__.py:95-98 + autograd)."""
    acts = np.ascontiguousarray(acts)
    lp = log_softmax_np(acts)
    costs, g = ref_cpu_logprobs(lp, labels, act_lens, label_lens, blank, True, threads)
    return costs, logits_grad(lp, g).astype(acts.dtype)
