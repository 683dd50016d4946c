#!/usr/bin/env python
"""bench.py — RNN-T loss+grad throughput on B200 (BASELINE.json metric), one JSON line.

    python bench.py --gpus 1 --steps 20 --warmup 3                      # our arm, 1 GPU
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W       # our arm, N GPUs (weak scaling)
    python bench.py --impl reference --gpus 1 --steps K --warmup W      # reference CPU path on host cores
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR    # + the last timed step's outputs as .npy

The inputs are seeded: the same arguments give the same inputs on every run, so the dumped outputs
of two builds can be compared element for element.

A step = one pass of the hot path (log-softmax statistics -> alpha/beta lattice -> dense gradient)
over one batch of synthetic logits; workload = BASELINE config "N=128, T=150, L=20, A=5000 fp32"
per GPU (the configuration the metric is quoted on).  Multi-GPU: every rank owns its own
128-utterance shard (utterances are independent), one NCCL all-reduce of the scalar loss per step.

value         device-resident: inputs already in HBM, compute_rnnt_loss_async + loss all-reduce,
              K steps between CUDA events, max over ranks.
e2e           through the reference-facing C-ABI call compute_rnnt_loss() (host-synchronous, costs to
              the host) with the step's logits coming from pinned host memory inside the timed region.
roofline      the dominant kernel (grad_row_kernel, 8 B/element algorithmic) timed with CUDA events on the
              library's own stream during the timed steps, against MEASURED_PEAKS.json.
parity_check  after the timed region, on EVERY rank: two utterances of the rank's shard (one full-length,
              one ragged) against the fp64 CPU oracle, and all_reduce(loss) == sum(all_gather(local sums)).
c5_strong     BASELINE config 5 as written: 1024 utterances (T=200, L=40, A=5000) split over the G ranks,
              each rank streaming 1024/G/128 micro-batches of 128 utterances through ONE fixed set of
              activation / gradient / workspace buffers per step, one all-reduce per step (strong scaling).
reference_gpu the reference's own CUDA kernels (oracle/_ref/libwarprnnt_ref_gpu.so, built for sm_100 from
              the unmodified reference sources) on the same inputs, tests/test_time.cu's 10-call protocol.
other_workloads  BASELINE configs 2, 4, the config-5 shard, bf16 logits at config 3 and the additive-joint
              training step, each with ms, utt/s and its recomputed roofline fraction (N=1 only).
cpu_baseline  the reference's CPU path (oracle/_ref, else the oracle port) on the host cores.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "warp-transducer_b200"))

WORKLOADS = {   # name: (N per GPU, T, L, V)   BASELINE.json configs
    "c2": (128, 150, 40, 28),
    "c3": (128, 150, 20, 5000),
    "c4": (64, 1500, 300, 50),
    "c5": (128, 200, 40, 5000),     # config 5's micro-batch: 1024 utterances in slabs of 128
}
C5_GLOBAL_BATCH = 1024
METRIC = "RNN-T loss+grad utterances/s at T=150,L=20,A=5000"
UNIT = "utterances/s"


def gen_labels(V, L, N):
    """Labels in [1, V-1] with forced repeats, the same row for every utterance — the recipe of
    the reference harness (tests/random.cpp:22-38, tests/test_time.cu:40-43), numpy generator."""
    rng = np.random.default_rng(1)
    lab = rng.integers(1, V, size=L).astype(np.int32)
    if L >= 3:
        lab[L // 2] = lab[L // 2 + 1]
        lab[L // 2 - 1] = lab[L // 2]
    return np.tile(lab, (N, 1))


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons with NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.maxc, self.stop_flag = index, [], set(), None, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.maxc = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def result(self):
        self.stop_flag = True
        if self.nv is None or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.maxc, "reasons": [], "note": "nvml unavailable"}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.maxc,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def bind_to_gpu_numa_node(index):
    """Pin this process to the CPUs local to GPU `index` (NVML's CPU affinity = the GPU's NUMA node)
    BEFORE any pinned host memory is allocated, so the step's 8 GB staging buffer is first-touched on
    the memory controller next to the GPU's PCIe root.  Round 1: with 8 ranks and no placement the
    pinned-host -> device streams of GPUs 4-7 crossed the socket link and e2e scaled 0.77."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        ncpu = os.cpu_count() or 1
        words = (ncpu + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [w * 64 + b for w in range(words) for b in range(64) if (int(mask[w]) >> b) & 1]
        cpus = [c for c in cpus if c < ncpu]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"cpus": "%d-%d (%d)" % (min(cpus), max(cpus), len(cpus))}
    except Exception as ex:
        return {"error": repr(ex)[:120]}
    return {"error": "empty affinity mask"}


# ----------------------------------------------------------------------------------------------
# CPU arm: the reference's own CPU implementation of the path on the host cores
# ----------------------------------------------------------------------------------------------
def cpu_reference_step_fn(V, T, L, n_utt, threads):
    """Returns (fn, kind): fn() runs logits -> loss + dense logits-gradient for n_utt utterances of
    the workload shape on the CPU.  kind 'reference': torch.log_softmax -> oracle/_ref
    compute_rnnt_loss(loc=CPU, OpenMP) -> log-softmax backward, i.e. exactly what the reference's
    warprnnt_pytorch composes on CPU (__init__.py:95-98 + autograd).  kind 'port': the oracle."""
    import torch
    from oracle import pyoracle
    U = L + 1
    torch.set_num_threads(threads)
    gen = torch.Generator().manual_seed(0)
    acts = torch.rand((n_utt, T, U, V), generator=gen, dtype=torch.float32)
    labels = gen_labels(V, L, n_utt)
    tl = np.full(n_utt, T, np.int32)
    ul = np.full(n_utt, L, np.int32)
    if pyoracle.have_ref_cpu():
        import ctypes as C
        lib = pyoracle.load_ref_cpu()
        fn = lib.compute_rnnt_loss
        fn.restype = C.c_int
        fn.argtypes = [C.c_void_p] * 5 + [C.c_int, C.c_int, C.c_void_p, C.c_void_p, pyoracle.RnntOptions]
        nbytes = C.c_size_t(0)
        lib.get_workspace_size.argtypes = [C.c_int, C.c_int, C.c_int, C.c_bool, C.POINTER(C.c_size_t), C.c_size_t]
        lib.get_workspace_size(T, U, n_utt, False, C.byref(nbytes), 4)
        ws = np.zeros(nbytes.value, np.uint8)
        costs = np.zeros(n_utt, np.float32)
        g = torch.empty_like(acts)
        opt = pyoracle.RnntOptions(loc=0, num_threads=threads, stream=None, blank_label=0, maxT=T,
                                   maxU=U, batch_first=True)

        def step():
            lp = torch.log_softmax(acts, -1)
            rc = fn(lp.data_ptr(), g.data_ptr(), labels.ctypes.data, ul.ctypes.data, tl.ctypes.data,
                    V, n_utt, costs.ctypes.data, ws.ctypes.data, opt)
            assert rc == 0
            dx = g - torch.exp(lp) * g.sum(-1, keepdim=True)
            return float(costs.sum()), dx
        return step, "reference"

    acts_np = acts.numpy()

    def step():
        c, dx, _ = pyoracle.rnnt_logits(acts_np, labels, tl, ul, 0, True, threads)
        return float(c.sum()), dx
    return step, "port"


def cpu_sample_size(V, T, L, N, budget_s):
    """The CPU arm runs the FULL batch (the reference parallelises over utterances with OpenMP,
    cpu_rnnt.h:290, so a partial batch leaves cores idle and understates it) unless the host cannot
    hold it or a pilot says the whole run would exceed budget_s; then the largest multiple of the core
    count that fits."""
    cores = os.cpu_count() or 1
    U = L + 1
    per_utt_bytes = T * U * V * 4 * 5          # acts, log-probs, grads, exp, dx
    try:
        avail = os.sysconf("SC_AVPHYS_PAGES") * os.sysconf("SC_PAGE_SIZE")
    except (ValueError, OSError):
        avail = 64 << 30
    n = min(N, max(1, int(0.6 * avail // per_utt_bytes)))
    pilot = min(n, max(4, min(cores, 16)))
    step, _ = cpu_reference_step_fn(V, T, L, pilot, cores)
    step()
    t0 = time.perf_counter()
    step()
    per_pass_full = (time.perf_counter() - t0) * max(1.0, n / max(pilot, min(cores, n)))
    if per_pass_full > budget_s and n > cores:
        n = max(cores, int(n * budget_s / per_pass_full) // cores * cores)
    return n


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    N, T, L, V = WORKLOADS[args.workload]
    cores = os.cpu_count() or 1
    # full batch per step; the whole --steps/--warmup run is allowed ~12 minutes of CPU time
    n = cpu_sample_size(V, T, L, N, budget_s=720.0 / (args.steps + args.warmup))
    step, kind = cpu_reference_step_fn(V, T, L, n, cores)
    for _ in range(max(args.warmup, 1)):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    value = n / dt
    sample = "%d of %d utterances of the workload per step, shape T=%d U=%d V=%d" % (n, N, T, L + 1, V)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": workload_config(args.workload, 1),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def needs_no_flush(name):
    N, T, L, V = WORKLOADS[name]
    return N * T * (L + 1) * V * 4 > (1 << 30)


def workload_config(name, world):
    N, T, L, V = WORKLOADS[name]
    return {"workload": "%s: N=%d per GPU, T=%d, L=%d (U=%d), A=%d, fp32 logits ~U[0,1), full lengths, blank 0"
                        % (name, N, T, L, L + 1, V),
            "global_batch": N * world, "parallelism": "batch-sharded x%d" % world,
            "l2": ("no flush: per-step inputs (%.2f GB logits) exceed the 126 MB L2" % (N * T * (L + 1) * V * 4 / 1e9))
                  if needs_no_flush(name) else "L2 flushed (256 MB write) before every timed step; steps timed individually"}


# ----------------------------------------------------------------------------------------------
# Our arm: helpers
# ----------------------------------------------------------------------------------------------
class Shard:
    """Device-resident synthetic inputs of one workload on one rank."""

    def __init__(self, torch, wr, dev, name, seed, dtype=None):
        self.N, self.T, self.L, self.V = WORKLOADS[name]
        self.U = self.L + 1
        N, T, U, V, L = self.N, self.T, self.U, self.V, self.L
        gen = torch.Generator(device=dev).manual_seed(seed)
        self.acts = torch.rand((N, T, U, V), generator=gen, device=dev, dtype=torch.float32)
        if dtype is not None:
            self.acts = self.acts.to(dtype)
        self.grads = torch.empty_like(self.acts)
        self.labels_np = gen_labels(V, L, N)
        self.labels = torch.as_tensor(self.labels_np).to(dev)
        self.tl = torch.full((N,), T, dtype=torch.int32, device=dev)
        self.ul = torch.full((N,), L, dtype=torch.int32, device=dev)
        self.costs = torch.empty(N, device=dev)
        self.ws = torch.empty(wr.workspace_size(T, U, N, 4), dtype=torch.uint8, device=dev)
        self.E = N * T * U * V

    def run(self, wr):
        wr.gpu_rnnt_async(self.acts, self.labels, self.tl, self.ul, self.costs, self.grads, 0, 1.0, self.ws)


def time_steps(torch, fn, steps, warmup=3, flush=None):
    """ms per step of fn() on the current stream (CUDA events).  With `flush`, the L2 is overwritten
    before every step and steps are timed one by one."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if flush is None:
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps
    tot = 0.0
    for _ in range(steps):
        flush.zero_()
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        tot += e0.elapsed_time(e1)
    return tot / steps


DUMP_SAMPLE = 1 << 20
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(torch, out_dir, costs, grads, labels_np, loss):
    """Writes what the timed path handed its caller in the last timed step, as float32 .npy files:
    the per-utterance costs, the step's summed loss, and the gradient (8 GB at the flagship shape) at
    fixed seeded positions: DUMP_SAMPLE elements anywhere, DUMP_SAMPLE cells' blank entries and
    DUMP_SAMPLE cells' entries at the cell's next label.  The gradient samples have a fixed size, so
    every workload's dump stays below DUMP_LIMIT_BYTES."""
    N, T, U, V = grads.shape
    rng = np.random.default_rng(0)
    anywhere = rng.integers(0, grads.numel(), size=DUMP_SAMPLE)
    blank = rng.integers(0, N * T * U, size=DUMP_SAMPLE) * V
    cell = rng.integers(0, N * T * (U - 1), size=DUMP_SAMPLE)        # (n, t, u) with u < U - 1
    n, t, u = cell // (T * (U - 1)), cell // (U - 1) % T, cell % (U - 1)
    label = ((n * T + t) * U + u) * V + labels_np[n, u]
    flat = grads.view(-1)
    out = {"costs": costs, "loss": loss}
    for name, idx in (("grads_sample", anywhere), ("grads_blank", blank), ("grads_label", label)):
        out[name] = flat[torch.as_tensor(idx, device=grads.device)]
    out = {name: t.float().cpu().numpy() for name, t in out.items()}
    assert sum(a.nbytes for a in out.values()) <= DUMP_LIMIT_BYTES
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def oracle_check_utterance(torch, acts_b, labels_b, T_b, L_b, cost_b, grads_b):
    """One utterance against the fp64 CPU oracle: (relative cost error, worst element-wise gradient
    excess over rtol 1e-4 + atol 1e-7, aggregate rel_diff).  acts_b/grads_b: [1,T,U,V] CUDA tensors."""
    from oracle import pyoracle
    a = acts_b.float().cpu().numpy().astype(np.float64)
    c_ref, g_ref, _ = pyoracle.rnnt_logits(a, labels_b.reshape(1, -1), np.array([T_b], np.int32),
                                           np.array([L_b], np.int32), 0)
    g = grads_b.float().cpu().numpy().astype(np.float64)
    rel_cost = abs(float(cost_b) - float(c_ref[0])) / max(abs(float(c_ref[0])), 1e-30)
    excess = np.abs(g - g_ref) - (1e-4 * np.abs(g_ref) + 1e-7)
    rd = float(((g - g_ref) ** 2).sum() / max(float((g_ref ** 2).sum()), 1e-300))
    max_rel = float((np.abs(g - g_ref) / (np.abs(g_ref) + 1e-7)).max())
    return rel_cost, float(excess.max()), rd, max_rel


def parity_leg(torch, dist, wr, sh, world, rank, dev):
    """Runs on every rank after the timed region.  (1) utterance 0 of the timed configuration (full
    lengths) and (2) one utterance of a ragged call on the same logits, against the fp64 oracle with the
    north-star tolerance; (3) the collective: all_reduce(sum of local costs) must equal the sum of the
    all_gathered local sums.  Returns this rank's record; rank 0 merges."""
    rec = {"ok": True}
    try:
        sh.run(wr)
        torch.cuda.synchronize()
        local_sum = sh.costs.double().sum()
        rc, ex, rd, mr = oracle_check_utterance(torch, sh.acts[0:1], sh.labels_np[0], sh.T, sh.L,
                                                sh.costs[0].item(), sh.grads[0:1])
        rec["full_utt"] = {"rel_cost": rc, "grad_excess": ex, "rel_diff": rd, "max_rel": mr}
        ok = rc < 1e-4 and ex <= 0.0 and rd < 1e-8
        # ragged: lengths ~U[0.5,1] x max, seed 2 + rank; check the shortest utterance of the shard
        rng = np.random.default_rng(2 + rank)
        tl_r = np.maximum(1, (rng.uniform(0.5, 1.0, sh.N) * sh.T)).astype(np.int32)
        ul_r = (rng.uniform(0.5, 1.0, sh.N) * sh.L).astype(np.int32)
        b = int(np.argmin(tl_r.astype(np.int64) * (ul_r + 1)))
        tl_d, ul_d = torch.as_tensor(tl_r).to(dev), torch.as_tensor(ul_r).to(dev)
        wr.gpu_rnnt_async(sh.acts, sh.labels, tl_d, ul_d, sh.costs, sh.grads, 0, 1.0, sh.ws)
        torch.cuda.synchronize()
        rc, ex, rd, mr = oracle_check_utterance(torch, sh.acts[b:b + 1], sh.labels_np[b], int(tl_r[b]), int(ul_r[b]),
                                                sh.costs[b].item(), sh.grads[b:b + 1])
        rec["ragged_utt"] = {"index": b, "T": int(tl_r[b]), "L": int(ul_r[b]), "rel_cost": rc, "grad_excess": ex,
                             "rel_diff": rd, "max_rel": mr}
        ok = ok and rc < 1e-4 and ex <= 0.0 and rd < 1e-8
        ok = ok and not bool(sh.grads[b, int(tl_r[b]):].any()) and not bool(sh.grads[b, :, int(ul_r[b]) + 1:].any())
        rec["max_rel"] = max(rec["full_utt"]["max_rel"], rec["ragged_utt"]["max_rel"])
        # collective consistency (world == 1: trivially the local sum)
        red = local_sum.clone()
        if world > 1:
            dist.all_reduce(red)
            parts = [torch.zeros_like(local_sum) for _ in range(world)]
            dist.all_gather(parts, local_sum)
            tot = float(torch.stack(parts).sum().item())
        else:
            tot = float(local_sum.item())
        rec["allreduce_rel_err"] = abs(float(red.item()) - tot) / max(abs(tot), 1e-30)
        ok = ok and rec["allreduce_rel_err"] < 1e-12
        rec["ok"] = bool(ok)
    except Exception as ex:
        rec = {"ok": False, "error": repr(ex)[:300]}
    return rec


def c5_strong_leg(torch, dist, wr, world, rank, dev, steps):
    """BASELINE config 5 as written (N=1024, T=200, L=40, A=5000 fp32 over G GPUs): 168 GB of logits and
    as much gradient do not fit one B200, so every rank streams its 1024/G utterances as micro-batches
    of 128 through ONE fixed activation / gradient / workspace set per step (the producer - here a
    device-side refresh of the logits is NOT simulated: the synthetic slab is reused, the kernels read
    and write the full 21 GB + 21 GB per micro-batch from HBM), costs accumulate on the device and one
    scalar all-reduce closes the step.  The reference cannot run this shape at all: 32-bit `mb*T*U*V`
    indexing (cpu_rnnt.h:294-297, gpu_rnnt_kernel.h:7-8)."""
    if C5_GLOBAL_BATCH % (world * 128) != 0:
        return {"skipped": "1024 utterances do not split into 128-utterance micro-batches over %d ranks" % world}
    micro = C5_GLOBAL_BATCH // world // 128
    sh = Shard(torch, wr, dev, "c5", 4321 + rank)
    total = torch.zeros(1, device=dev)

    def step():
        total.zero_()
        for _ in range(micro):
            sh.run(wr)
            total.add_(sh.costs.sum())
        if world > 1:
            dist.all_reduce(total)

    for _ in range(2):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    loss = float(total.item())
    per_gpu_bytes = 12.0 * sh.E * micro
    out = {"workload": "config 5: N=1024 global, T=200, L=40 (U=41), A=5000 fp32, batch-sharded over %d GPU(s)" % world,
           "scaling": "strong", "global_batch": C5_GLOBAL_BATCH, "micro_batches_per_rank": micro,
           "micro_batch": 128, "ms_per_step": ms, "value": C5_GLOBAL_BATCH / (ms * 1e-3), "unit": UNIT,
           "steps": steps, "per_gpu_algorithmic_GBps": per_gpu_bytes / (ms * 1e-3) / 1e9,
           "loss_sum": loss, "buffers": "one fixed 21 GB logits + 21 GB gradient + workspace set per rank",
           "note": "strong-scaling efficiency = ms_per_step(G=1) / (G * ms_per_step(G)), from the driver's per-G runs"}
    del sh
    torch.cuda.empty_cache()
    return out


def reference_gpu_leg(torch, wr, dev, names):
    """tests/test_time.cu's protocol (3 untimed + 10 timed calls, wall clock around the host-synchronous
    compute_rnnt_loss) on the reference's own CUDA kernels compiled for sm_100, and on this library, on the
    same device-resident inputs."""
    import ctypes as C
    from oracle import pyoracle
    path = pyoracle.ref_gpu_path()
    if not os.path.exists(path):
        return {"unavailable": "oracle/_ref/libwarprnnt_ref_gpu.so not built"}
    ref = C.CDLL(path)
    ref.compute_rnnt_loss.restype = C.c_int
    ref.compute_rnnt_loss.argtypes = [C.c_void_p] * 5 + [C.c_int, C.c_int, C.c_void_p, C.c_void_p, wr.rnntOptions]
    ref.get_workspace_size.argtypes = [C.c_int, C.c_int, C.c_int, C.c_bool, C.POINTER(C.c_size_t), C.c_size_t]
    out = {"lib": "oracle/_ref/libwarprnnt_ref_gpu.so (unmodified reference CUDA kernels, -arch sm_100)",
           "protocol": "tests/test_time.cu:89-128: 3 warm-up + 10 timed host-synchronous calls, wall clock"}
    for name in names:
        sh = Shard(torch, wr, dev, name, 99)
        opt = wr.rnntOptions(loc=1, num_threads=0, stream=torch.cuda.current_stream().cuda_stream,
                             blank_label=0, maxT=sh.T, maxU=sh.U, batch_first=True)
        rec = {}
        for label, lib in (("reference_gpu", ref), ("b200", wr.lib())):
            n = C.c_size_t(0)
            lib.get_workspace_size(sh.T, sh.U, sh.N, True, C.byref(n), 4)
            ws = torch.empty(n.value, dtype=torch.uint8, device=dev)
            costs = np.zeros(sh.N, np.float32)
            ts = []
            for _ in range(13):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                st = lib.compute_rnnt_loss(sh.acts.data_ptr(), sh.grads.data_ptr(), sh.labels.data_ptr(),
                                           sh.ul.data_ptr(), sh.tl.data_ptr(), sh.V, sh.N, costs.ctypes.data,
                                           ws.data_ptr(), opt)
                ts.append((time.perf_counter() - t0) * 1e3)
                if st != 0:
                    break
            if st != 0:
                rec[label] = {"error": "status %d" % st}
                continue
            t = float(np.mean(ts[3:]))
            rec[label] = {"ms_per_call": t, "value": sh.N / t * 1e3, "unit": UNIT, "cost0": float(costs[0])}
            del ws
        if "ms_per_call" in rec.get("reference_gpu", {}) and "ms_per_call" in rec.get("b200", {}):
            rec["speedup"] = rec["reference_gpu"]["ms_per_call"] / rec["b200"]["ms_per_call"]
            rec["cost0_rel_diff"] = abs(rec["reference_gpu"]["cost0"] - rec["b200"]["cost0"]) / abs(rec["b200"]["cost0"])
        out[name] = rec
        del sh
        torch.cuda.empty_cache()
    return out


def other_workloads_leg(torch, wr, dev, peaks):
    """Device-resident ms / utt/s / roofline fraction of the configurations the headline does not cover."""
    out = {}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    hbm = peaks["hbm_gbs"]
    for key, name, dtype in (("c2", "c2", None), ("c4", "c4", None), ("c5_shard", "c5", None),
                             ("c3_bf16", "c3", torch.bfloat16)):
        try:
            sh = Shard(torch, wr, dev, name, 7, dtype)
            small = sh.E * sh.acts.element_size() < (1 << 30)
            ms = time_steps(torch, lambda: sh.run(wr), 10, 3, flush if small else None)
            # per-kernel times in a second pass: the event markers between the kernels switch the
            # programmatic-dependent-launch chaining off, so they are not part of the timed pass above
            wr.set_profiling(True)
            wr.profile_collect()
            time_steps(torch, lambda: sh.run(wr), 5, 1, flush if small else None)
            calls, kms = wr.profile_collect()
            wr.set_profiling(False)
            bytes_ = 3.0 * sh.E * sh.acts.element_size()
            out[key] = {"workload": "N=%d T=%d L=%d A=%d %s" % (sh.N, sh.T, sh.L, sh.V, "bf16 logits+grads, fp32 math" if dtype else "fp32"),
                        "ms_per_step": ms, "value": sh.N / (ms * 1e-3), "unit": UNIT,
                        "algorithmic_GBps": bytes_ / (ms * 1e-3) / 1e9, "frac_of_measured_hbm": bytes_ / (ms * 1e-3) / 1e9 / hbm,
                        "frac_of_8TBps": bytes_ / (ms * 1e-3) / 1e9 / 8000.0,
                        "kernel_ms": {"rowstats": kms[0], "lattice": kms[1], "grad": kms[2],
                                      "note": ("this shape runs as 4 overlapped batch groups (a group's wavefront on a side stream beside "
                                               "the streaming passes of the others): rowstats = pass 1 of all groups with the co-running "
                                               "wavefronts, lattice = only the exposed wait before the first pass 2, grad = pass 2 of all "
                                               "groups; the whole kernels alone (RNNT_B200_GROUPS=1) are in profiles/r2_c4_full.md")
                                      if key == "c4" else "separate pass with event markers between the kernels (no launch overlap)"},
                        "l2": "flushed before every step" if small else "inputs exceed L2"}
            del sh
        except Exception as ex:
            out[key] = {"error": repr(ex)[:200]}
        torch.cuda.empty_cache()
    # additive joint network, one training step (forward + backward through autograd)
    try:
        from warprnnt_pytorch.joint import AddJointRNNTLoss
        N, T, L, V = WORKLOADS["c3"]
        U = L + 1
        trans = torch.rand((N, T, V), device=dev, requires_grad=True)
        pred = torch.rand((N, U, V), device=dev, requires_grad=True)
        labels = torch.as_tensor(gen_labels(V, L, N)).to(dev)
        tl = torch.full((N,), T, dtype=torch.int32, device=dev)
        ul = torch.full((N,), L, dtype=torch.int32, device=dev)
        fused = AddJointRNNTLoss()

        def jstep():
            trans.grad = pred.grad = None
            fused(trans, pred, labels, tl, ul).backward()
        ms = time_steps(torch, jstep, 10, 3, flush)
        # traffic floor: read f,g once per pass that needs them (3 passes) + write dF,dG
        floor_bytes = 4.0 * N * (T + U) * V * 4
        out["add_joint_c3"] = {"workload": "additive joint, N=%d T=%d U=%d A=%d fp32, forward+backward" % (N, T, U, V),
                               "ms_per_step": ms, "value": N / (ms * 1e-3), "unit": UNIT,
                               "traffic_floor_GB": floor_bytes / 1e9,
                               "frac_of_measured_hbm_vs_floor": floor_bytes / (ms * 1e-3) / 1e9 / hbm}
    except Exception as ex:
        out["add_joint_c3"] = {"error": repr(ex)[:200]}
    del flush
    torch.cuda.empty_cache()
    return out


# ----------------------------------------------------------------------------------------------
# Our arm
# ----------------------------------------------------------------------------------------------
def run_b200_arm(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    numa = bind_to_gpu_numa_node(local)        # before torch allocates any pinned memory
    import torch
    import torch.distributed as dist
    import warprnnt_pytorch.warp_rnnt as wr

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the B200 arm has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    sh = Shard(torch, wr, dev, args.workload, 1234 + rank)
    N, T, L, V, U, E = sh.N, sh.T, sh.L, sh.V, sh.U, sh.E
    acts, grads, labels, tl, ul, costs, ws = sh.acts, sh.grads, sh.labels, sh.tl, sh.ul, sh.costs, sh.ws
    labels_np = sh.labels_np

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # The scalar-loss all-reduce runs on NCCL's own stream and is consumed one step later, so the
    # compute stream of a rank never stalls on a slower peer inside a step (gradients are local;
    # only the logged loss crosses ranks).  Two alternating buffers keep step k's reduction intact
    # while step k+1 is enqueued.
    loss2 = [torch.zeros(1, device=dev), torch.zeros(1, device=dev)]
    state = {"k": 0, "pending": None}

    def step():
        wr.gpu_rnnt_async(acts, labels, tl, ul, costs, grads, 0, 1.0, ws)
        buf = loss2[state["k"] & 1]
        torch.sum(costs, 0, keepdim=True, out=buf)
        if world > 1 and not os.environ.get("BENCH_NO_ALLREDUCE"):
            if state["pending"] is not None:
                state["pending"].wait()          # step k-1's collective: finished during this step's kernels
            state["pending"] = dist.all_reduce(buf, async_op=True)   # one scalar over NVLink
        state["k"] += 1

    def drain():
        if state["pending"] is not None:
            state["pending"].wait()
            state["pending"] = None

    wr.set_profiling(True)
    # everything with variable host cost (NVML init, thread start, event creation) happens BEFORE the
    # barrier: ranks must leave it aligned, a late starter is waited for by all the others through
    # the loss all-reduce and with K ~ 20 steps of 3.5 ms a 20 ms skew is a 30 % error
    sampler = ClockSampler(local)
    sampler.start()
    kms = np.zeros(3)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(max(args.warmup, 3)):
        step()
    drain()
    wr.profile_collect()                              # drop the warm-up records
    barrier()
    if needs_no_flush(args.workload):
        e0.record()
        for _ in range(args.steps):
            step()                                    # no host synchronisation inside the timed region
        drain()                                       # the last step's all-reduce is inside the timed region
        e1.record()
        barrier()
        total_ms = e0.elapsed_time(e1)
        kms = np.array(wr.profile_collect()[1]) * args.steps
    else:   # working set fits the L2: flush it before every step and time the steps one by one
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        total_ms = 0.0
        for _ in range(args.steps):
            flush.zero_()
            e0.record()
            step()
            drain()
            e1.record()
            kms += np.array(wr.last_kernel_ms())
            e1.synchronize()
            total_ms += e0.elapsed_time(e1)
        barrier()
        del flush
    launches = wr.last_launch_count() * args.steps
    wr.set_profiling(False)
    if args.dump_outputs and rank == 0:
        # before the legs below reuse costs / grads
        dump_outputs(torch, args.dump_outputs, costs, grads, labels_np, loss2[(state["k"] - 1) & 1])

    # ---- secondary, reported separately (SURVEY 8(d)): ragged lengths ~U[0.5,1]*max, seed 2.
    # Padded cells are not read (pass 1 skips them, pass 2 writes zeros), so bytes move less.
    ragged = None
    try:
        rng = np.random.default_rng(2)
        tl_r = torch.as_tensor(np.maximum(1, (rng.uniform(0.5, 1.0, N) * T)).astype(np.int32)).to(dev)
        ul_r = torch.as_tensor((rng.uniform(0.5, 1.0, N) * L).astype(np.int32)).to(dev)
        rms = time_steps(torch, lambda: wr.gpu_rnnt_async(acts, labels, tl_r, ul_r, costs, grads, 0, 1.0, ws),
                         max(3, args.steps // 2), 3)
        valid = float((tl_r.double() * (ul_r.double() + 1)).sum().item())
        ragged = {"ms_per_step": rms, "value": N / (rms * 1e-3), "unit": UNIT + " per GPU",
                  "lengths": "T_b, L_b ~ U[0.5,1] x max (seed 2)", "valid_cell_fraction": valid / (N * T * U),
                  "algorithmic_GBps": (8.0 * valid * V + 4.0 * N * T * U * V) / (rms * 1e-3) / 1e9}
    except Exception as ex:
        ragged = {"error": repr(ex)[:200]}

    # ---- parity on every rank (VERDICT r1: multi-GPU correctness had no driver-side evidence)
    parity_local = parity_leg(torch, dist, wr, sh, world, rank, dev)

    # ---- end to end through compute_rnnt_loss(): pinned host inputs -> device, costs -> host.
    # The batch is fed as CHUNKS of whole utterances: all chunk copies are queued on a copy stream up
    # front, the reference-facing host-synchronous call runs chunk k (after its copy event) while the
    # copies of chunks k+1.. are still in flight.  Every call is the reference's own entry point.
    chunks = 4 if N % 4 == 0 else 1
    nb = N // chunks
    acts_host = torch.empty((N, T, U, V), dtype=torch.float32, pin_memory=True)
    acts_host.copy_(acts)
    labels_host = torch.as_tensor(labels_np).pin_memory()
    tl_host = torch.full((N,), T, dtype=torch.int32).pin_memory()
    ul_host = torch.full((N,), L, dtype=torch.int32).pin_memory()
    costs_host = torch.zeros(N, dtype=torch.float32).pin_memory()
    copy_stream = torch.cuda.Stream(device=dev)
    main_stream = torch.cuda.current_stream()
    ready = [torch.cuda.Event() for _ in range(chunks)]
    opt = wr.rnntOptions(loc=1, num_threads=0, stream=main_stream.cuda_stream,
                         blank_label=0, maxT=T, maxU=U, batch_first=True)
    ws_chunk = wr.workspace_size(T, U, nb, 4)

    def e2e_step():
        copy_stream.wait_stream(main_stream)        # the previous step's kernels are done with the buffers
        with torch.cuda.stream(copy_stream):
            labels.copy_(labels_host, non_blocking=True)
            tl.copy_(tl_host, non_blocking=True)
            ul.copy_(ul_host, non_blocking=True)
            for k in range(chunks):
                acts[k * nb:(k + 1) * nb].copy_(acts_host[k * nb:(k + 1) * nb], non_blocking=True)
                ready[k].record(copy_stream)
        for k in range(chunks):
            main_stream.wait_event(ready[k])
            b0 = k * nb
            st = wr.lib().compute_rnnt_loss(acts[b0:].data_ptr(), grads[b0:].data_ptr(), labels[b0:].data_ptr(),
                                            ul[b0:].data_ptr(), tl[b0:].data_ptr(), V, nb,
                                            costs_host[b0:].data_ptr(), ws.data_ptr(), opt)   # returns with costs on the host
            assert st == 0
        tot = float(costs_host.sum())
        if world > 1:
            t = torch.tensor([tot], device=dev)
            dist.all_reduce(t)
            tot = float(t.item())
        return tot

    assert ws_chunk <= ws.numel()
    e2e_steps = max(3, min(args.steps, 10))
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2e_step()
    barrier()
    f0.record()
    for _ in range(e2e_steps):
        e2e_step()
    f1.record()
    barrier()
    e2e_ms = f0.elapsed_time(f1)
    clocks = sampler.result()
    h2d = acts_host.numel() * 4 + labels_host.numel() * 4 + 2 * N * 4
    d2h = N * 4
    del acts_host

    per_rank = None
    parity = dict(parity_local)
    if world > 1:
        # diagnostics: every rank's own kernel times and loop time (gathered, not used for `value`)
        mine = torch.tensor([total_ms, kms[0] / args.steps, kms[1] / args.steps, kms[2] / args.steps],
                            device=dev, dtype=torch.float64)
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        per_rank = [[round(float(v), 4) for v in r.tolist()] for r in allr]
        t = torch.tensor([total_ms, e2e_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, e2e_ms = t.tolist()
        recs = [None] * world
        dist.all_gather_object(recs, parity_local)
        parity = {"ok": all(r.get("ok") for r in recs),
                  "max_rel": max((r.get("max_rel", float("inf")) for r in recs)),
                  "allreduce_rel_err": max((r.get("allreduce_rel_err", float("inf")) for r in recs)),
                  "per_rank": recs}
    parity["ranks"] = world
    parity["tolerance"] = "|g-g_ref| <= 1e-4 |g_ref| + 1e-7 element-wise, rel_diff < 1e-8, cost rel 1e-4; fp64 CPU oracle"
    ms_per_step = total_ms / args.steps
    value = N * world / (ms_per_step * 1e-3)
    e2e_value = N * world / (e2e_ms / e2e_steps * 1e-3)

    peaks, peak_src = measured_peaks()
    kms /= args.steps
    grad_ms, rows_ms, lat_ms = float(kms[2]), float(kms[0]), float(kms[1])
    achieved = 8.0 * E / (grad_ms * 1e-3) / 1e9 if grad_ms > 0 else None
    roofline = {
        "bound": "hbm", "kernel": "grad_row_kernel (pass 2: read logits 4 B + write gradient 4 B per element)",
        "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
        "frac": achieved / peaks["hbm_gbs"] if achieved else None, "peak_source": peak_src + " (MEASURED_PEAKS.json hbm_gbs)",
        "traffic": None, "traffic_source": "profiles/traffic.json (ncu --set full capture of the same kernel, committed; not re-measured per run)",
        "ms_per_launch": grad_ms,
        "frac_of_8TBps": achieved / 8000.0 if achieved else None,
        "other_kernels": {
            "rowstats_row_kernel": {"ms": rows_ms, "algorithmic_GBps": 4.0 * E / (rows_ms * 1e-3) / 1e9 if rows_ms > 0 else None},
            "lattice_kernel": {"ms": lat_ms, "bound": "latency"},
            "path_12B_per_elt_GBps": 12.0 * E / ((rows_ms + lat_ms + grad_ms) * 1e-3) / 1e9 if grad_ms > 0 else None,
        },
    }
    traffic_file = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(traffic_file):
        try:
            roofline["traffic"] = json.load(open(traffic_file)).get("grad_kernel_c3_bytes")
        except Exception:
            pass

    # ---- BASELINE config 5 as written, on every world size (frees the headline buffers first)
    del acts, grads, ws, sh
    torch.cuda.empty_cache()
    c5 = None
    if not args.no_c5:
        try:
            c5 = c5_strong_leg(torch, dist, wr, world, rank, dev, max(2, min(args.steps, 5)))
        except Exception as ex:
            c5 = {"error": repr(ex)[:300]}

    line = None
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.workload, world),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms / e2e_steps, "steps": e2e_steps,
                    "api": "compute_rnnt_loss (C-ABI, host-synchronous), %d calls of %d utterances per step; the "
                           "logits of every chunk come from pinned host memory each step, chunk k+1 copies while "
                           "chunk k computes" % (chunks, nb),
                    "numa_binding": numa},
            "gpu_launches": launches, "clocks": clocks, "roofline": roofline,
            "parity_check": parity, "c5_strong": c5,
            "lib": os.path.relpath(wr.lib_path(), ROOT),
        }
        line["ragged_lengths"] = ragged
        if per_rank is not None:
            line["per_rank_ms"] = {"columns": ["loop_total", "rowstats", "lattice", "grad"], "rows": per_rank}
    if world > 1:
        dist.barrier()
    if rank == 0 and world == 1 and not args.quick:
        try:
            line["reference_gpu"] = reference_gpu_leg(torch, wr, dev, ["c2", "c3", "c4"])
        except Exception as ex:
            line["reference_gpu"] = {"error": repr(ex)[:300]}
        try:
            line["other_workloads"] = other_workloads_leg(torch, wr, dev, peaks)
        except Exception as ex:
            line["other_workloads"] = {"error": repr(ex)[:300]}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # The CPU baseline runs in a fresh process (`--impl reference`, full batch, 1 warm-up + 1 timed
        # pass): its OpenMP / torch thread pools must not inherit this process's NUMA-local affinity.
        cores = os.cpu_count() or 1
        try:
            import subprocess
            try:
                os.sched_setaffinity(0, range(cores))
            except Exception:
                pass
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload",
                                  args.workload, "--steps", "1", "--warmup", "1"], capture_output=True, text=True,
                                 timeout=900)
            ref_line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
            line["cpu_baseline"] = ref_line["cpu_baseline"]
            line["cpu_baseline"]["sample"] += ", 1 timed pass after 1 warm-up pass, separate process"
        except Exception as ex:   # the baseline is reporting only; never lose the GPU line over it
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": cores, "kind": "unavailable",
                                    "sample": repr(ex)[:200]}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    if not parity.get("ok", False):
        raise SystemExit("bench.py: parity check FAILED: %s" % json.dumps(parity)[:1500])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-c5", action="store_true", help="skip the config-5 strong-scaling leg")
    ap.add_argument("--quick", action="store_true", help="skip the reference-GPU and other-workload legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write rank 0's outputs of the last timed step to DIR/<name>.npy (b200 arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the b200 arm")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        world = int(os.environ.get("WORLD_SIZE", "1"))
        if args.gpus > 1 and world == 1:
            # convenience: relaunch under torchrun when invoked directly with --gpus N
            import subprocess
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                   "--nproc-per-node", str(args.gpus), "--master-addr", "127.0.0.1",
                   "--master-port", os.environ.get("MASTER_PORT", "29517"), os.path.abspath(__file__),
                   "--gpus", str(args.gpus), "--steps", str(args.steps), "--warmup", str(args.warmup),
                   "--workload", args.workload] + (["--no-cpu-baseline"] if args.no_cpu_baseline else []) + \
                  (["--no-c5"] if args.no_c5 else []) + (["--quick"] if args.quick else []) + \
                  (["--dump-outputs", os.path.abspath(args.dump_outputs)] if args.dump_outputs else [])
            raise SystemExit(subprocess.call(cmd))
        run_b200_arm(args)


if __name__ == "__main__":
    main()
