#!/usr/bin/env python
"""bench.py — QPs/sec (fwd+bwd) of the hot path at BASELINE.json's config C2, per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR (b200 arm): after the timed steps, rank 0 writes what the last of them returned to its caller -
z* and the gradients of Q, p, G, h, float64 - as DIR/{z,dQ,dp,dG,dh}.npy (20.8 MB at C2). The inputs are seeded and the
last timed step always runs on the same input copy for the same --steps, so two builds can be compared output for output.

A "step" = QPFunction forward + backward over one batch of 128 random dense QPs
(nz = nineq = 100, neq = 0, fp64; generator of prof-linear.py:64-75).  The path shards
by QP with no data-path collective, so N GPUs run N independent batches ("weak").
Rank 0 prints ONE JSON line (contract in the task statement / DESIGN.md section 6).
`config` is identical in both arms; everything that describes HOW a number was taken is under `detail`.

--impl reference times the reference's own CPU implementation of the path on the box's host cores: the
UNMODIFIED qpth package from oracle/_ref/ (put there by oracle/make_ref.sh; `cpu_baseline.kind` = "reference"),
or, when that directory is absent, the oracle port oracle/pdipm_torch.py (`kind` = "port").

The pipelined legs (`value`, `e2e`) replay CUDA graphs of the user-level step (QPFunction forward + autograd backward, plus
the H2D / D2H copies for `e2e`) on 6 streams in the library's throughput mode (three QPs per SM); `detail.serial_*` is
one stream in latency mode (one QP per SM).

Extra measurements on the b200 line (rank 0): `detail.c4` (BASELINE config 4, cls-layer pattern), `detail.c5`
(config 5: B=8192 scattered from rank 0 over the ranks through NCCL, z* gathered; N > 1 only),
`reference_cuda` (the unmodified reference on CUDA tensors on the same GPU, N = 1 only).
"""
import argparse
import ctypes
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the bench only reads the source tree (it may be read-only)

import numpy as np   # noqa: E402
import torch         # noqa: E402

from qpth_b200.problems import random_qp_batch, algorithmic_bytes_per_qp, algorithmic_flops_per_qp  # noqa: E402

CFG = dict(nBatch=128, nz=100, nineq=100, neq=0)
WORKLOAD = "C2: batch=128 nz=100 nineq=100 neq=0 random dense QP, fp64, fwd+bwd (per GPU)"
METRIC = "QPs/sec (fwd+bwd) batch=128 nz=100 nineq=100"
OPTIONS = "eps=1e-12 maxIter=20 notImprovedLim=3 verbose=-1"
CONFIG = {"workload": WORKLOAD, "per_gpu_batch": CFG["nBatch"], "options": OPTIONS}    # same dict in both arms
DATA = "synthetic (seeded prof-linear.py generator)"
NCOPIES = 8          # rotating input sets: 8 x 20.7 MB = 165 MB > 126 MB of L2
REF_DIR = os.path.join(ROOT, "oracle", "_ref")


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


class ClockSampler:
    """Samples SM clock / throttle reasons of one GPU through NVML (in-process, ~20 us per sample) while the
    timed region runs. (`nvidia-smi -lms` in a subprocess was measurably perturbing launch latency.)"""

    def __init__(self, index, period=0.002):
        self.index, self.period, self.rows, self.ok = index, period, [], False
        self._stop = threading.Event()
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.ok = True
        except Exception:       # noqa: BLE001 - NVML missing: report that instead of failing the bench
            self.ok = False

    def start(self):
        if self.ok:
            self.th = threading.Thread(target=self._run, daemon=True)
            self.th.start()

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(
                    nv, "nvmlDeviceGetCurrentClocksEventReasons") else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((sm, rs))
            except Exception:   # noqa: BLE001
                pass
            self._stop.wait(self.period)

    def stop(self):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["NVML unavailable"]}
        self._stop.set()
        self.th.join(timeout=1.0)
        nv = self.nv
        mx = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
                "hw_power_brake": 0x80}
        reasons = set()
        for _, rs in self.rows:
            for name, bit in bits.items():
                if rs & bit:
                    reasons.add(name)
        sm = [r[0] for r in self.rows]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(mx), "samples": len(sm),
                "reasons": sorted(reasons)}


def bind_to_gpu_numa(index):
    """Pin this process to the CPUs of the NUMA node its GPU hangs off BEFORE any pinned host buffer is allocated
    (first touch puts the pages there): on the 8-GPU boxes GPUs 4-7 sit on node 1, and a rank left on node 0 pays
    the inter-socket hop on every H2D/D2H byte of the e2e leg. Returns a description for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        dom, rest = bus.split(":", 1)
        path = "/sys/bus/pci/devices/%s:%s/numa_node" % (dom[-4:].lower(), rest.lower())
        node = int(open(path).read().strip())
        if node < 0:
            return "numa node unknown (single node)"
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return "numa node %d has no allowed cpus" % node
        os.sched_setaffinity(0, cpus)
        return "bound to numa node %d (%d cpus)" % (node, len(cpus))
    except Exception as exc:    # noqa: BLE001
        return "not bound (%s)" % str(exc)[:80]


def settle(step, min_steps, chunk, max_steps=None):
    """Warm-up: at least `min_steps` steps, then keep going (in chunks) until the CUDA caching allocator has stopped
    growing. On these boxes a fresh cudaMalloc of a 10-20 MB block costs ~10 ms and synchronises, and the pool of a
    loop that allocates ~70 MB per step keeps growing for the first few dozen steps; timing before it has settled
    measures cudaMalloc, not the solver. Returns the number of warm-up steps run."""
    if max_steps is None:
        max_steps = env_int("QPB_BENCH_MAX_SETTLE", 400)      # (lowered only for runs under ncu)
    done = 0
    while done < min_steps:
        step(done); done += 1
    torch.cuda.synchronize()
    stable = 0
    while done < max_steps:
        n0 = torch.cuda.memory_stats().get("num_device_alloc", 0)
        for _ in range(chunk):
            step(done); done += 1
        torch.cuda.synchronize()
        if torch.cuda.memory_stats().get("num_device_alloc", 0) == n0:
            stable += 1
            if stable >= 2:
                break
        else:
            stable = 0
    return done


def make_batches(device, seed0, ncopies, pinned_host=False):
    out = []
    for c in range(ncopies):
        pr = random_qp_batch(seed=seed0 + c, **CFG)
        if pinned_host:
            out.append({k: torch.from_numpy(np.ascontiguousarray(pr[k])).pin_memory() for k in ("Q", "p", "G", "h")})
        else:
            out.append({k: torch.tensor(pr[k], dtype=torch.float64, device=device, requires_grad=True)
                        for k in ("Q", "p", "G", "h")})
    return out


def e2e_leg(f, dev, rank, world, nsteps_req, warmup, dl, graphs=True):
    """The same step through QPFunction with HOST (pinned) buffers, H2D + D2H inside the timed region. NS steps are
    kept in flight on NS CUDA streams (as a serving loop would). Returns (median ms, windows, ksteps, NS, h2d, d2h, how).
    graphs: each stream's step (H2D copies from pinned memory, QPFunction forward, autograd backward, D2H copies) is
    captured once in a CUDA graph and replayed - the eager Python loop needs 0.54 ms of host time per step, as long as
    the step takes on the device (scripts/e2e_host.py); the default-options variant reads a flag back per forward and
    cannot be captured."""
    B, n, m = CFG["nBatch"], CFG["nz"], CFG["nineq"]
    NS = max(1, env_int("QPB_BENCH_E2E_INFLIGHT", 6))
    hb = make_batches(dev, 1000 * rank, NS, pinned_host=True)
    host_out = [{k: torch.empty(s, dtype=torch.float64).pin_memory()
                 for k, s in (("z", (B, n)), ("dQ", (B, n, n)), ("dp", (B, n)), ("dG", (B, m, n)), ("dh", (B, m)))}
                for _ in range(NS)]
    dbuf = [{k: torch.empty(v.shape, dtype=torch.float64, device=dev).requires_grad_(True) for k, v in hb[0].items()}
            for _ in range(NS)]
    streams = [torch.cuda.Stream(device=dev) for _ in range(NS)]
    e = torch.Tensor().to(dev).double()
    from qpth_b200.util import copy_lower_
    lower_band = env_int("QPB_BENCH_DQ_BAND", 0)        # 0: read dQ back in full (measured r2j: strips change nothing,
    q_band = env_int("QPB_BENCH_Q_BAND", 0)             #    the duplex PCIe rate is set by the host -> device direction)
    h2d = sum(v.numel() * 8 for v in hb[0].values())
    d2h = sum(v.numel() * 8 for v in host_out[0].values())
    if lower_band > 0:
        strips = sum(min(n, r0 + lower_band) * (min(n, r0 + lower_band) - r0) for r0 in range(0, n, lower_band))
        d2h += (strips - n * n) * B * 8
    if q_band > 0:
        strips = sum(min(n, r0 + q_band) * (min(n, r0 + q_band) - r0) for r0 in range(0, n, q_band))
        h2d += (strips - n * n) * B * 8

    def e2e_step(i):
        j = i % NS
        with torch.cuda.stream(streams[j]):
            e2e_body(j)

    def e2e_body(j):
        if True:
            src, t, out = hb[j], dbuf[j], host_out[j]
            with torch.no_grad():
                for k, v in src.items():
                    if k == "Q" and q_band > 0:     # Q is symmetric (SPD is a precondition, qp.py:81-85): lower strips only
                        copy_lower_(t[k], v, band=q_band)
                    else:
                        t[k].copy_(v, non_blocking=True)                  # H2D
            for v in t.values():
                v.grad = None
            z = f(t["Q"], t["p"], t["G"], t["h"], e, e)
            z.backward(dl)
            out["z"].copy_(z.detach(), non_blocking=True)                 # D2H
            for k, g in (("dp", "p"), ("dG", "G"), ("dh", "h")):
                out[k].copy_(t[g].grad, non_blocking=True)
            if lower_band > 0:      # dQ = 1/2 (dx z^T + z dx^T) is symmetric (qp.py:157-158): its lower triangle comes back
                copy_lower_(out["dQ"], t["Q"].grad.contiguous(), band=lower_band)
            else:
                out["dQ"].copy_(t["Q"].grad, non_blocking=True)

    for st_ in streams:
        st_.wait_stream(torch.cuda.current_stream())
    ksteps = max(2 * NS, nsteps_req // NS * NS)
    settle(e2e_step, max(4, warmup), 2 * NS)
    how = "eager"
    if graphs and os.environ.get("QPB_BENCH_E2E_GRAPHS", "1") == "1":
        try:
            torch.cuda.synchronize()
            cg = []
            for j in range(NS):
                gph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gph, stream=streams[j]):
                    e2e_body(j)
                cg.append(gph)
            torch.cuda.synchronize()

            def e2e_step(i):                                      # noqa: F811
                j = i % NS
                with torch.cuda.stream(streams[j]):
                    cg[j].replay()
            how = "cuda_graph per stream (H2D + QPFunction forward + autograd backward + D2H captured once, replayed)"
        except Exception as exc:                                  # noqa: BLE001
            sys.stderr.write("bench: e2e graph capture failed (%s); eager loop\n" % str(exc)[:200])
            torch.cuda.synchronize()
    for i in range(ksteps):                # untimed rehearsal: same run-ahead, same allocation pattern
        e2e_step(i)
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    import gc
    gc.collect(); torch.cuda.synchronize()
    windows = []
    for _w in range(5):
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(NS + 1)]
        torch.cuda.synchronize()
        evs[0].record()
        for st_ in streams:
            st_.wait_event(evs[0])
        for i in range(ksteps):
            e2e_step(i)
        for j, st_ in enumerate(streams):
            evs[1 + j].record(st_)
        torch.cuda.synchronize()
        windows.append(max(evs[0].elapsed_time(evs[1 + j]) for j in range(NS)))
    e2e_ms = float(np.median(windows))
    if world > 1:
        tt = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
        torch.distributed.all_reduce(tt, op=torch.distributed.ReduceOp.MAX)
        e2e_ms = float(tt.item())
    return e2e_ms, windows, ksteps, NS, h2d, d2h, how


def run_b200(args, rank, world, local_rank):
    numa = bind_to_gpu_numa(local_rank)
    from qpth_b200 import QPFunction, _lib
    from qpth_b200 import qp as qpmod
    # Every leg of this bench keeps several steps (batches) in flight on several CUDA streams, i.e. more QPs than the
    # GPU has SMs: the library's throughput mode (three QPs per SM at C2; qpth_b200.qp.MODE, a documented user switch whose
    # "auto" default picks it for any batch larger than the SM count). The single-stream figure (detail.serial_*) is
    # taken in latency mode (one QP per SM), the right choice for ONE 128-QP batch at a time.
    bench_mode = os.environ.get("QPB_BENCH_MODE", "throughput")
    qpmod.MODE = bench_mode
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    lib = _lib.load()
    B, n, m = CFG["nBatch"], CFG["nz"], CFG["nineq"]
    f = QPFunction(verbose=-1, check_Q_spd=False)     # fully asynchronous: no host read per step
    e = torch.Tensor().to(dev).double()
    dl = torch.ones(B, n, dtype=torch.float64, device=dev)        # dl_dz = 1 (prof-linear.py:117)
    batches = make_batches(dev, 1000 * rank, NCOPIES)
    eager_z = {}

    def step(i):
        t = batches[i % NCOPIES]
        for v in t.values():
            v.grad = None
        z = f(t["Q"], t["p"], t["G"], t["h"], e, e)
        z.backward(dl)
        eager_z[i % NCOPIES] = z
        return z

    def outputs(j):
        """What the last step on input copy j returned to its caller: z* and the gradients of Q, p, G, h."""
        return dict(z=eager_z[j], **{"d" + k: batches[j][k].grad for k in ("Q", "p", "G", "h")})

    settle_steps = settle(step, args.warmup, NCOPIES)
    # The step is 3 kernels behind ~0.5 ms of Python: capture QPFunction forward + autograd backward of every input
    # copy in a CUDA graph so that the timed loop is not at the mercy of host jitter. Falls back to eager.
    launch_mode = "eager"
    last_iters = None
    serial_step = None

    def capture_graphs(user_level=True):
        """One CUDA graph per input copy of the step. user_level: QPFunction forward + autograd backward (what the e2e leg
        captures, minus the copies); else the two functions QPFunction.forward / .backward call (qpth_b200.qp.solve_forward
        / solve_backward: same kernels, same C-ABI calls, no autograd bookkeeping)."""
        from qpth_b200.qp import solve_forward, solve_backward
        flags, want = [False] * 6, [True, True, True, True, False, False]

        def raw_step(t):
            if user_level:
                for v in t.values():
                    v.grad = None
                z = f(t["Q"], t["p"], t["G"], t["h"], e, e)
                z.backward(dl)
                return f.last_solve(), z
            st_ = solve_forward(t["Q"].detach(), t["p"].detach(), t["G"].detach(), t["h"].detach(), e, e,
                                verbose=-1, check_Q_spd=False)
            return st_, solve_backward(st_, dl, flags, want)

        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream())
        # fresh leaves that only ever see the capture stream (the AccumulateGrad nodes of `batches` belong to the default
        # stream the eager warm-up ran on, which invalidates a capture of backward on another stream)
        leaves = [{k: v.detach().clone().requires_grad_(True) for k, v in t.items()} for t in batches] if user_level else batches
        with torch.cuda.stream(side):
            for t in leaves[:3]:
                raw_step(t)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graphs, keep = [], []
        for t in leaves:
            gph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gph, stream=side):
                keep.append(raw_step(t))
            graphs.append(gph)
        torch.cuda.synchronize()
        keep.append(leaves)

        def graph_outputs(j):
            """outputs(j) of the replayed step: what the last replay of graph j left in its output buffers."""
            if user_level:
                return dict(z=keep[j][1], **{"d" + k: leaves[j][k].grad for k in ("Q", "p", "G", "h")})
            st_, g = keep[j]
            return dict(z=st_.zhat, dQ=g[0], dp=g[1], dG=g[2], dh=g[3])
        return graphs, keep, graph_outputs

    if os.environ.get("QPB_BENCH_GRAPHS", "1") == "1":
        for user_level in (True, False):
            try:
                graphs, keep, outputs = capture_graphs(user_level)

                def step(i):                                      # noqa: F811
                    graphs[i % NCOPIES].replay()
                last_iters = keep[-2][0].iters
                launch_mode = "cuda_graph (QPFunction forward + autograd backward)" if user_level else "cuda_graph (solve_forward + solve_backward)"
                if bench_mode != "latency":                       # the single-stream leg: one QP per SM
                    qpmod.MODE = "latency"
                    lat_graphs, lat_keep, _ = capture_graphs(user_level)
                    qpmod.MODE = bench_mode

                    def serial_step(i):                           # noqa: F811
                        lat_graphs[i % NCOPIES].replay()
                break
            except Exception as exc:                              # noqa: BLE001
                sys.stderr.write("bench: CUDA graph capture (%s) failed (%s)\n" % ("user level" if user_level else "solve_* level", str(exc)[:200]))
                qpmod.MODE = bench_mode
                launch_mode, serial_step = "eager", None
                try:
                    torch.cuda.synchronize()
                except Exception:                                 # noqa: BLE001
                    pass
    # `value`: K steps with the inputs resident in HBM. A step's kernels have 128 CTAs (one QP each); the GPU holds
    # 148 (one QP per SM), 296 or 444 (two / three QPs per SM) at a time and a QP leaves its slot as soon as it has converged
    # (12 Newton iterations on average, 16-18 for the slowest QP of a batch), so a single stream idles most of the
    # machine during the tail of every forward kernel. As in a serving loop (and as in the e2e leg) consecutive steps
    # alternate between INFLIGHT CUDA streams. Every step is still one complete forward + backward over its own
    # batch; the single-stream figure is reported next to it (detail.serial_*).
    inflight = max(1, env_int("QPB_BENCH_INFLIGHT", 6))
    vstreams = [torch.cuda.Stream(device=dev) for _ in range(inflight)]

    def timed_window(nsteps, first, streams):
        """Device time of `nsteps` steps issued round-robin on `streams` (None: the current stream)."""
        torch.cuda.synchronize()
        e0 = torch.cuda.Event(enable_timing=True)
        e0.record()
        if streams is None:
            one = serial_step if serial_step is not None else step
            for i in range(nsteps):
                one(first + i)
            e1 = torch.cuda.Event(enable_timing=True)
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1)
        ends = []
        for st_ in streams:
            st_.wait_event(e0)
        for i in range(nsteps):
            with torch.cuda.stream(streams[i % len(streams)]):
                step(first + i)
        for st_ in streams:
            e1 = torch.cuda.Event(enable_timing=True)
            e1.record(st_)
            ends.append(e1)
        torch.cuda.synchronize()
        return max(e0.elapsed_time(e1) for e1 in ends)

    use_streams = vstreams if inflight > 1 else None
    # the warm-up length depends on the allocator; starting on copy 0 keeps the input copy of every timed step (and so
    # what --dump-outputs writes) a function of --steps alone
    done = -(-settle_steps // NCOPIES) * NCOPIES
    timed_window(args.steps, done, use_streams)       # untimed rehearsal: same run-ahead, same allocation pattern
    done += args.steps
    timed_window(max(4, args.steps // 2), done, None)
    serial_ms = timed_window(args.steps, done, None)  # informational: one stream, steps strictly back to back
    done += args.steps
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    import gc
    gc.collect(); torch.cuda.synchronize()            # (a collection inside the window can cudaFree / cudaFreeHost: tens of ms)
    gc.disable()
    try:
        ms = timed_window(args.steps, done, use_streams)
    finally:
        gc.enable()
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, v in outputs((done + args.steps - 1) % NCOPIES).items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), v.detach().to(torch.float64).cpu().numpy())
    iters_mean = float((last_iters if launch_mode.startswith("cuda_graph") else f.last_solve().iters).float().mean())
    if world > 1:
        tt = torch.tensor([ms], dtype=torch.float64, device=dev)
        torch.distributed.all_reduce(tt, op=torch.distributed.ReduceOp.MAX)
        ms = float(tt.item())
        torch.distributed.barrier()

    # ---- e2e: host buffers, asynchronous options (check_Q_spd=False, verbose=-1) ...
    if os.environ.get("QPB_BENCH_E2E", "1") != "1":               # (development sweeps of the resident number only)
        if rank == 0:
            return {"value": world * B * args.steps / (ms * 1e-3), "ms_per_step": ms / args.steps, "e2e": {"value": 0.0},
                    "detail": {"serial_ms_per_step": serial_ms / args.steps, "steps_in_flight": inflight, "mean_newton_iters": iters_mean}}
        return None
    e2e_ms, windows, ksteps, NS, h2d, d2h, e2e_how = e2e_leg(f, dev, rank, world, args.steps, args.warmup, dl)
    # ... and with the reference's DEFAULT options (check_Q_spd=True, verbose=0): every forward then reads the
    # SPD / inaccurate-solution flags back before it returns (qp.py:81-85, batch.py:205-206), which serialises the host
    e2e_def = None
    if os.environ.get("QPB_BENCH_E2E_DEFAULT", "1") == "1":
        fdef = QPFunction()
        d_ms, d_windows, d_k, _, _, _, _ = e2e_leg(fdef, dev, rank, world, args.steps, args.warmup, dl, graphs=False)
        e2e_def = {"value": world * B * d_k / (d_ms * 1e-3), "windows_ms": d_windows,
                   "options": "QPFunction() defaults: check_Q_spd=True verbose=0 (one blocking flag read per forward)"}
        qpmod.LAZY_CHECKS = True       # the same defaults with the diagnostics deferred (qpth_b200.qp.LAZY_CHECKS)
        try:
            l_ms, l_windows, l_k, _, _, _, _ = e2e_leg(fdef, dev, rank, world, args.steps, args.warmup, dl, graphs=False)
            qpmod.flush_checks()
            e2e_def["lazy_checks"] = {"value": world * B * l_k / (l_ms * 1e-3), "windows_ms": l_windows}
        finally:
            qpmod.LAZY_CHECKS = False
            qpmod._pending.clear()
    c5 = None
    if world > 1 and os.environ.get("QPB_BENCH_C5", "1") == "1":
        c5 = run_c5(rank, world, dev)
    if rank != 0:
        return None

    # ---- the three kernels timed alone through the C ABI, on the stream they are launched on
    plan = _lib.plan_for(n, m, 0, two=(bench_mode == "throughput"))      # the kernels the timed region ran
    t = batches[0]
    f64 = dict(dtype=torch.float64, device=dev)
    L = torch.empty(B * plan.L_elems, **f64); W = torch.empty(B * plan.W_elems, **f64)
    K = torch.empty(B * plan.K_elems, **f64); spd = torch.zeros(B, dtype=torch.int32, device=dev)
    zz = torch.empty(B, n, **f64); ll = torch.empty(B, m, **f64); ss = torch.empty(B, m, **f64)
    iters = torch.empty(B, dtype=torch.int32, device=dev); rr = torch.empty(B, **f64)
    gQ = torch.empty(B, n, n, **f64); gp = torch.empty(B, n, **f64); gG = torch.empty(B, m, n, **f64)
    gh = torch.empty(B, m, **f64); wx = torch.empty(B, n, **f64); wl = torch.empty(B, m, **f64)
    P = lambda x: ctypes.c_void_p(x.data_ptr())
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    Qc, Gc, pc, hc = (t[k].detach().contiguous() for k in ("Q", "G", "p", "h"))
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    kt = []
    for i in range(8):
        ev[0].record()
        _lib.check(lib.qpb200_pre_factor_kkt(ctypes.byref(plan), B, P(Qc), n * n, P(Gc), m * n, None, 0,
                                             P(L), P(W), P(K), P(spd), None, st))
        ev[1].record()
        _lib.check(lib.qpb200_forward(ctypes.byref(plan), B, P(pc), n, P(hc), m, None, 0, P(L), P(W), P(K), 1,
                                      1e-12, 1e-6, 1.5, 3, 20, P(zz), P(ll), P(ss), None, P(iters), P(rr),
                                      None, None, st))
        ev[2].record()
        _lib.check(lib.qpb200_backward(ctypes.byref(plan), B, P(dl), P(zz), P(ll), P(ss), None, P(L), P(W), P(K), 1,
                                       P(gQ), 0, P(gp), 0, P(gG), 0, P(gh), 0, None, 0, None, 0, P(wx), P(wl), None,
                                       None, st))
        ev[3].record()
        torch.cuda.synchronize()
        kt.append([ev[j].elapsed_time(ev[j + 1]) for j in range(3)])
    setup_ms, k_ms, bwd_ms = (float(x) for x in np.mean(np.array(kt[2:]), axis=0))
    # fp64 FMA peak of this box, measured (148 SMs x 8 CTAs x 256 threads x 8 chains)
    probe_out = torch.empty(148 * 8 * 256, **f64)
    pk = []
    for i in range(4):
        ev[0].record()
        _lib.check(lib.qpb200_dfma_probe(148 * 8, 256, 4096, P(probe_out), st))
        ev[1].record(); torch.cuda.synchronize()
        pk.append(ev[0].elapsed_time(ev[1]))
    fp64_peak = 2.0 * 8 * 4096 * 148 * 8 * 256 / (min(pk[1:]) * 1e-3) / 1e12

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except (OSError, ValueError):
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    ab = algorithmic_bytes_per_qp(n, m, 0)
    fwd_bytes = (ab["fwd_in"] + ab["fwd_out"]) * B
    achieved = fwd_bytes / (k_ms * 1e-3) / 1e9
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "latest_traffic.json"))).get("k_forward_dram_bytes")
    except (OSError, ValueError):
        pass
    it_mean = float(iters.float().mean())
    # per-kernel fp64 work (SURVEY 8d, Cholesky form): setup | init + iters x iteration | backward
    nn, mm = float(n), float(m)
    fl_setup = nn ** 3 / 3 + nn * nn * mm + mm * mm * nn
    fl_factor, fl_solve, fl_resid = mm ** 3 / 3, 4 * nn * nn + 2 * mm * mm + 4 * mm * nn, 2 * nn * nn + 4 * mm * nn
    fl_fwd = (fl_factor + fl_solve) + it_mean * (fl_factor + 2 * fl_solve + fl_resid)
    fl_bwd = fl_factor + fl_solve + fl_resid
    tf = lambda fl, ms_: fl * B / (ms_ * 1e-3) / 1e12
    total_qps = world * B * args.steps
    line = {
        "metric": METRIC, "value": total_qps / (ms * 1e-3), "unit": "QPs/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": DATA, "impl": "b200",
        "config": dict(CONFIG),
        "e2e": {"value": world * B * ksteps / (e2e_ms * 1e-3), "unit": "QPs/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "steps": ksteps, "windows_ms": windows, "statistic": "median of 5 windows",
                "best_window_value": world * B * ksteps / (min(windows) * 1e-3),
                "api": "qpth_b200.QPFunction(verbose=-1, check_Q_spd=False); per step: H2D of Q,p,G,h from pinned host memory, fwd, bwd, D2H of z* and all gradients; %d steps in flight on %d CUDA streams" % (NS, NS),
                "steps_in_flight": NS, "launch": e2e_how, "default_options": e2e_def},
        "gpu_launches": 3 * args.steps,
        "clocks": clocks,
        "roofline": {"bound": "hbm", "kernel": "k_forward_fast", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                     "frac": achieved / hbm_peak, "traffic": traffic,
                     "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650",
                     "kernel_ms": k_ms, "algorithmic_bytes_per_launch": fwd_bytes,
                     "note": "latency/fp64-bound path (SURVEY 8d): HBM fraction is small by construction; kernel timed alone (one 128-QP launch)",
                     "fp64": {"peak_tflops_measured": fp64_peak,
                              "forward": {"tflops": tf(fl_fwd, k_ms), "frac": tf(fl_fwd, k_ms) / fp64_peak, "ms": k_ms},
                              "setup": {"tflops": tf(fl_setup, setup_ms), "frac": tf(fl_setup, setup_ms) / fp64_peak, "ms": setup_ms},
                              "backward": {"tflops": tf(fl_bwd, bwd_ms), "frac": tf(fl_bwd, bwd_ms) / fp64_peak, "ms": bwd_ms},
                              "whole_step_pipelined": {"tflops": (fl_setup + fl_fwd + fl_bwd) * B / (ms / args.steps * 1e-3) / 1e12,
                                                       "frac": (fl_setup + fl_fwd + fl_bwd) * B / (ms / args.steps * 1e-3) / 1e12 / fp64_peak}}},
        "cpu_baseline": cpu_baseline() if (world == 1 and os.environ.get("QPB_BENCH_CPU", "1") == "1") else None,   # N=1 only
        "detail": {"l2": "inputs rotate over %d independent batches (%.0f MB > 126 MB L2)" % (NCOPIES, NCOPIES * h2d / 1e6),
                   "mean_newton_iters": iters_mean, "launch": launch_mode, "steps_in_flight": inflight,
                   "serial_ms_per_step": serial_ms / args.steps, "serial_value": total_qps / (serial_ms * 1e-3),
                   "settle_steps": settle_steps, "numa": numa, "mode": bench_mode,
                   "solve_kernels": ("product form" if plan.pf else "round-1") + (", three QPs per SM (192-thread CTAs; W, chol(Q) from L2)" if (plan.pf and plan.pf_three) else ", two QPs per SM (W, chol(Q) from L2)" if (plan.pf and plan.pf_two) else ", one QP per SM"),
                   "serial_kernels": "one QP per SM (latency mode)" if serial_step is not None else "same as value",
                   "kernel_ms_alone": {"setup": setup_ms, "forward": k_ms, "backward": bwd_ms},
                   "parity": "fp64; GPU suite (tests/, -m gpu) vs outputs of the real reference: per-QP relative l2 of z*, nu <= 1e-8; "
                             "lambda, slacks rtol 1e-6 / atol 1e-8 max|ref|; every gradient <= 1e-6 with the denominator floored at "
                             "1e-4 of the batch maximum (tests/parity.py); measured worst case at C2: z 1.5e-11, gradients 1.5e-11"},
    }
    if world == 1 and os.environ.get("QPB_BENCH_C4", "1") == "1":
        try:
            line["detail"]["c4"] = run_c4(dev)
        except Exception as exc:                                  # noqa: BLE001
            line["detail"]["c4"] = {"error": str(exc)[:200]}
    if world == 1 and os.environ.get("QPB_BENCH_REFCUDA", "1") == "1":
        line["reference_cuda"] = reference_cuda(dev)
    if c5 is not None:
        line["detail"]["c5"] = c5
    return line


def run_c4(dev):
    """BASELINE config 4: OptNet cls-layer pattern, nz = nineq = 200, batch 64, shared Q, G, h (example-cls-layer.ipynb).
    Device-resident fwd+bwd through QPFunction, CUDA events, 10 repetitions after warm-up."""
    from qpth_b200 import QPFunction
    from qpth_b200.problems import cls_layer_problem
    pr = cls_layer_problem(64, 200, 200, seed=0)
    t = {k: torch.tensor(pr[k], dtype=torch.float64, device=dev, requires_grad=True) for k in ("Q", "p", "G", "h")}
    e = torch.Tensor().to(dev).double()
    dl = torch.ones(64, 200, dtype=torch.float64, device=dev)
    f = QPFunction(verbose=-1, check_Q_spd=False)

    def one():
        for v in t.values():
            v.grad = None
        z = f(t["Q"], t["p"], t["G"], t["h"], e, e)
        z.backward(dl)
    import gc
    settle(lambda i: one(), 5, 5, max_steps=100)      # until the caching allocator stops calling cudaMalloc (10-20 ms each)
    torch.cuda.synchronize()
    # The legs before this one leave CUDA graphs with private pools and pinned host buffers behind; when Python's
    # collector frees them in the middle of a window (cudaFree / cudaFreeHost block the host for tens of ms) the window
    # measures that, not the solver: collect first, keep the collector off while timing.
    gc.collect(); torch.cuda.synchronize()
    gc.disable()
    reps, times = 10, []
    try:
        for _w in range(5):                           # median of five windows of 10 steps
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                one()
            e1.record(); torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1) / reps)
    finally:
        gc.enable()
    ms = float(np.median(times))
    return {"workload": "C4: cls-layer pattern batch=64 nz=200 nineq=200, shared Q,G,h, batched p, fwd+bwd", "ms_per_step": ms,
            "windows_ms_per_step": times,
            "value": 64 / (ms * 1e-3), "unit": "QPs/s", "mean_newton_iters": float(f.last_solve().iters.float().mean())}


def run_c5(rank, world, dev):
    """BASELINE config 5: ONE job of B = 8192 QPs (nz = nineq = 100) whose inputs live on rank 0; they are scattered to
    the ranks through NCCL (qpth_b200.parallel.sharded_qp), solved (fwd+bwd), z* gathered on rank 0 (the per-sample
    gradients stay sharded, SURVEY 8e). Strong scaling: the total is fixed. Timed on the device, max over ranks, with
    the scatter+gather inside and outside the timed region both stated; rank 0 checks the gathered z* bit-for-bit
    against its own single-GPU solve of sample shards."""
    import torch.distributed as dist
    from qpth_b200 import QPFunction
    from qpth_b200 import parallel
    from qpth_b200.problems import c5_shard
    per = 8192 // 8
    nsh = 8
    glob = None
    if rank == 0:
        parts = [c5_shard(r, per) for r in range(nsh)]
        glob = {k: torch.tensor(np.concatenate([p_[k] for p_ in parts]), dtype=torch.float64, device=dev)
                for k in ("Q", "p", "G", "h")}
    f = QPFunction(verbose=-1, check_Q_spd=False)
    res = {}
    torch.cuda.synchronize()
    torch.cuda.empty_cache()        # (the legs before this one leave CUDA-graph pools behind: keep cudaMalloc out of the timed region)
    for with_comm in (True, False):
        times = []
        zfull = None
        for rep in range(6):
            torch.cuda.synchronize(); dist.barrier()
            out = parallel.sharded_qp_timed(f, glob, 8192, 100, 100, dev, include_comm=with_comm)
            times.append(out["ms"])
            zfull = out["z"]
        key = "ms_with_scatter_gather" if with_comm else "ms_compute_only"
        res[key] = float(np.median(times[2:]))
        res[key + "_all"] = times
    ok = None
    if rank == 0:
        # single-GPU solve of two shards, compared bit-for-bit with the gathered result
        ok = True
        for r in (0, nsh - 1):
            sl = slice(r * per, (r + 1) * per)
            t = {k: glob[k][sl].clone().requires_grad_(False) for k in ("Q", "p", "G", "h")}
            e = torch.Tensor().to(dev).double()
            z1 = f(t["Q"], t["p"], t["G"], t["h"], e, e)
            ok = ok and bool(torch.equal(z1, zfull[sl]))
    return {"workload": "C5: batch=8192 nz=100 nineq=100 scattered from rank 0 over %d GPUs via NCCL, fwd+bwd, z* gathered" % world,
            "scaling": "strong", "n_gpus": world,
            "value_with_scatter_gather": 8192 / (res["ms_with_scatter_gather"] * 1e-3),
            "value_compute_only": 8192 / (res["ms_compute_only"] * 1e-3), "unit": "QPs/s",
            **res, "gathered_z_equals_single_gpu": ok,
            "bytes_scattered": 8192 * (100 * 100 * 2 + 200) * 8 * (world - 1) // world, "bytes_gathered": 8192 * 100 * 8 * (world - 1) // world}


# ---------------------------------------------------------------------------------------------------------
# the reference arm
# ---------------------------------------------------------------------------------------------------------
def load_reference():
    """The UNMODIFIED qpth from oracle/_ref (oracle/make_ref.sh). Returns (QPFunction, kind) or (None, why)."""
    if not os.path.isdir(os.path.join(REF_DIR, "qpth")):
        return None, "oracle/_ref/qpth missing (run oracle/make_ref.sh in the build container)"
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        from qpth.qp import QPFunction as RefQPFunction   # noqa: E402
    return RefQPFunction, "reference"


def ref_fwd_bwd_fn():
    """fwd+bwd callable (dict of CPU/GPU tensors Q,p,G,h; dl) -> None, and its `kind`."""
    RefQP, kind = load_reference()
    if RefQP is not None:
        def run(T, dl):
            t = {k: T[k].detach().clone().requires_grad_(True) for k in ("Q", "p", "G", "h")}
            e = torch.empty(0, dtype=torch.float64, device=T["Q"].device)
            z = RefQP(verbose=-1)(t["Q"], t["p"], t["G"], t["h"], e, e)
            z.backward(dl)
            return z
        return run, "reference", "unmodified qpth (oracle/_ref) QPFunction(verbose=-1) on CPU tensors"
    from oracle import pdipm_torch as pt

    def run(T, dl):                                               # noqa: F811
        e = torch.empty(0, dtype=torch.float64)
        return pt.qp_fwd_bwd(T["Q"], T["p"], T["G"], T["h"], T.get("A", e), T.get("b", e), dl)[0]
    return run, "port", "oracle/pdipm_torch.py (batched torch-CPU restatement of qpth's PDIPM); " + kind


def best_cpu_threads(run, T, dl):
    """Batched 100x100 LAPACK calls do not scale to every core of a big host: use the thread count that maximises the
    reference's own throughput (best of two timings per candidate) so the CPU baseline is not handicapped."""
    ncpu = len(os.sched_getaffinity(0)) or 1
    cands = sorted({c for c in (1, 4, 8, 16, 32) if 1 <= c <= ncpu})     # (64+ threads: 4-100x slower on this workload)
    best, best_t, table = cands[0], float("inf"), {}
    for c in cands:
        torch.set_num_threads(c)
        run(T, dl)
        ts = []
        for _ in range(2):
            t0 = time.perf_counter()
            run(T, dl)
            ts.append(time.perf_counter() - t0)
        table[c] = min(ts)
        if min(ts) < best_t:
            best, best_t = c, min(ts)
    return best, table


def cpu_tensors(seed):
    pr = random_qp_batch(seed=seed, **CFG)
    return {k: torch.from_numpy(np.ascontiguousarray(pr[k])) for k in ("Q", "p", "G", "h", "A", "b")}


def cpu_baseline(sample_reps=5):
    """The reference's CPU implementation on the host cores: fwd+bwd over the C2 batch, bounded sample."""
    run, kind, what = ref_fwd_bwd_fn()
    T = cpu_tensors(0)
    dl = torch.ones(CFG["nBatch"], CFG["nz"], dtype=torch.float64)
    thr, table = best_cpu_threads(run, T, dl)
    torch.set_num_threads(thr)
    run(T, dl)      # warm-up
    ts = []
    for _ in range(sample_reps):
        t0 = time.perf_counter()
        run(T, dl)
        ts.append(time.perf_counter() - t0)
    return {"value": CFG["nBatch"] / min(ts), "unit": "QPs/s", "cores": torch.get_num_threads(), "kind": kind,
            "sample": "%d x the full C2 batch (128 QPs, fwd+bwd), best of %d; %s; thread count calibrated (best of 2 per candidate)" % (sample_reps, sample_reps, what),
            "median_value": CFG["nBatch"] / float(np.median(ts)), "host_cpus": os.cpu_count(),
            "seconds_per_batch_by_threads": {str(k): v for k, v in table.items()}}


def reference_cuda(dev):
    """The unmodified reference on CUDA tensors on this GPU (its un-pivoted LU path, batch.py:9-19), fwd+bwd over the
    C2 batch with torch.cuda.synchronize() on both sides: the "reference on the same box" figure."""
    RefQP, kind = load_reference()
    if RefQP is None:
        return {"unavailable": kind}
    try:
        pr = random_qp_batch(seed=0, **CFG)
        T = {k: torch.tensor(pr[k], dtype=torch.float64, device=dev) for k in ("Q", "p", "G", "h")}
        dl = torch.ones(CFG["nBatch"], CFG["nz"], dtype=torch.float64, device=dev)
        e = torch.empty(0, dtype=torch.float64, device=dev)

        def one():
            t = {k: v.clone().requires_grad_(True) for k, v in T.items()}
            z = RefQP(verbose=-1)(t["Q"], t["p"], t["G"], t["h"], e, e)
            z.backward(dl)
            return z
        one(); torch.cuda.synchronize()
        ts = []
        for _ in range(3):
            torch.cuda.synchronize(); t0 = time.perf_counter()
            z = one()
            torch.cuda.synchronize(); ts.append(time.perf_counter() - t0)
        finite = bool(torch.isfinite(z).all())
        return {"value": CFG["nBatch"] / min(ts), "unit": "QPs/s", "seconds_per_batch": min(ts), "finite": finite,
                "what": "unmodified qpth (oracle/_ref) QPFunction(verbose=-1) on CUDA fp64 tensors, fwd+bwd, best of 3, synchronised"}
    except Exception as exc:                                      # noqa: BLE001
        return {"unavailable": "reference CUDA path failed: %s" % str(exc)[:160]}


def run_reference(args, rank, world):
    """CPU arm: the reference on all the host threads it can use, same workload, metric and unit."""
    if rank != 0:
        return None
    run, kind, what = ref_fwd_bwd_fn()
    batches = [cpu_tensors(c) for c in range(2)]
    dl = torch.ones(CFG["nBatch"], CFG["nz"], dtype=torch.float64)
    thr, table = best_cpu_threads(run, batches[0], dl)
    torch.set_num_threads(thr)
    for i in range(args.warmup):
        run(batches[i % 2], dl)
    t0 = time.perf_counter()
    for i in range(args.steps):
        run(batches[i % 2], dl)
    dt = time.perf_counter() - t0
    val = CFG["nBatch"] * args.steps / dt
    cb = {"value": val, "unit": "QPs/s", "cores": torch.get_num_threads(), "kind": kind,
          "sample": "each step = the full C2 batch (128 QPs, fwd+bwd) on the host CPU; %s; thread count calibrated for best throughput" % what,
          "host_cpus": os.cpu_count(), "seconds_per_batch_by_threads": {str(k): v for k, v in table.items()}}
    return {"metric": METRIC, "value": val, "unit": "QPs/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt * 1e3 / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": DATA,
            "impl": "reference", "config": dict(CONFIG),
            "cpu_baseline": cb,
            "e2e": {"value": val, "unit": "QPs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "detail": {"note": "CPU arm, rank 0 only; " + what}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    args.warmup = max(args.warmup, 3)
    rank, world, local_rank = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    # stdout of this program is ONE JSON line: everything any library prints on fd 1 meanwhile (NCCL prints its version
    # banner there at communicator creation) goes to stderr
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(line) + "\n").encode())

    if args.impl == "reference":
        line = run_reference(args, rank, world)
        if line is not None:
            emit(line)
        return
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    line = run_b200(args, rank, world, local_rank)
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    if line is not None:
        emit(line)


if __name__ == "__main__":
    main()
