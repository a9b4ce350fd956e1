#!/usr/bin/env python
"""bench.py — headline benchmark of the TT core-contraction hot path on B200.

Workload at every N (BASELINE.json configs[4], "cfg5"; SURVEY.md §8(d)-5, §8(e)): 4 096 independent ComplexF64 QTT vectors
(d = 30, n = 2, rank 64), one shared ComplexF64 MPO of rank 4; per vector y = A*x followed by tt_compress!(y, 64)
(truncerr = 0, sweeps = 1).  One "step" = all 4 096 vectors once.  The batch shards over the ranks by vectors with no data-path
collective (strong scaling: the total is fixed).  Metric: tt_rounding sweeps/s — one rounding sweep per vector, so sweeps/s =
vectors/s.  VERDICT r1 asked for this workload as the headline at every N because cfg2 (a single train) does not shard; cfg2,
the cfg4 matvec and the DMRG sweep stay in the line as compact extras (full detail with `--extras-out FILE`; the committed
profiles/bench_extras_N<n>.json were written that way).

  value     device-timed (CUDA events on the library's stream, max over ranks): inputs resident in HBM (10.3 GB at N = 1,
            every chunk of 296 vectors is 0.74 GB, far larger than L2, and is touched once per step);
  e2e       the same step through the public host API on pinned host buffers: per chunk H2D of the input cores,
            `apply_compress`, D2H of the rounded cores into pinned memory, software-pipelined over the chunks of all timed steps
            (the copies of chunk i +- 1 run on the copy stream while chunk i computes) — wall clock, max over ranks;
  roofline  the kernel family that dominates the step (per-family CUDA events over one step, the host threads profiled one after
            the other) against the measured FP64 GEMM peak, plus the whole step against the 13.3 GFLOP/vector model of SURVEY.md
            §8(d)-5; `traffic` = DRAM bytes per launch of the dominant kernel from the committed ncu capture;
  cpu_baseline  the NumPy restatement of the reference algorithm on the host cores (bounded sample, rank 0, N = 1).

`--impl reference` times the reference's own CPU algorithm (oracle/, including the discarded `orthogonalize` of
src/tt_tools.jl:769 that the Julia code executes in every bond step) on a bounded sample of the same workload: every step is
ONE vector of the batch, fully measured (no extrapolation); the run stops after a time budget and reports the steps it measured.

`--dump-outputs DIR` writes what the timed path returned in its last timed step for a fixed, seeded sample of the 4 096 vectors
(the rounded cores, see `write_outputs`), so that two builds can be compared output for output on identical inputs.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the source tree untouched (it may be read-only)

# cfg5
D5, R5, W5, MAXB5, TOTAL5 = 30, 64, 4, 64, 4096
# cfg2
D, NPHYS, RMAX_IN, MAX_BOND = 40, 2, 512, 64
FP64_PEAK_FILE = os.path.join(ROOT, "profiles", "fp64_peak_r01.json")
WORKLOAD = ("cfg5: 4096 independent ComplexF64 QTT vectors (d=30, n=2, rank 64), y = A*x (MPO rank 4) then "
            "tt_compress!(y, 64; truncerr=0, sweeps=1); one rounding sweep per vector")


def cfg5_ranks():
    rks = [min(2 ** k, 2 ** (D5 - k), R5) for k in range(D5 + 1)]
    Rk = [min(4 ** k, 4 ** (D5 - k), W5) for k in range(D5 + 1)]
    return rks, Rk


def cfg5_config(world, chunk):
    return {"workload": WORKLOAD, "d": D5, "n": 2, "rank": R5, "mpo_rank": W5, "max_bond": MAXB5, "total_vectors": TOTAL5,
            "chunk": chunk, "parallelism": f"vectors sharded over {world} rank(s), no data-path collective",
            "cache": "inputs 10.3 GB (0.74 GB per chunk) >> L2, each chunk touched once per step"}


def cfg5_flop_model():
    """algorithmic FLOPs per vector (SURVEY.md §8(d)-5 / Appendix C): Theta GEMMs + projections + R-SVD count, complex = 4 x real"""
    rks, Rk = cfg5_ranks()
    yr = [a * b for a, b in zip(rks, Rk)]
    out = {"gemm": 0.0, "svd": 0.0}
    cur = list(yr)
    for sweep_dir in (range(0, D5 - 1), range(D5 - 2, -1, -1)):
        for k in sweep_dir:
            p, r, q = 2 * cur[k], cur[k + 1], 2 * cur[k + 2]
            kk, m = min(p, q), max(p, q)
            rn = min(kk, MAXB5)
            out["gemm"] += 4.0 * (2.0 * p * r * q + 2.0 * rn * p * q)
            out["svd"] += 4.0 * (6.0 * m * kk * kk + 20.0 * kk ** 3)
            cur[k + 1] = rn
    out["total"] = out["gemm"] + out["svd"]
    return out


def make_mpo(t_or_o):
    rks, Rk = cfg5_ranks()
    rng = np.random.default_rng(7)
    return t_or_o.TToperator(D5, [np.asfortranarray((rng.standard_normal((2, 2, Rk[k], Rk[k + 1])) + 1j * rng.standard_normal((2, 2, Rk[k], Rk[k + 1])))
                                                    / math.sqrt(2.0 * Rk[k + 1])) for k in range(D5)], (2,) * D5, Rk)


def make_vector(seed):
    rks, _ = cfg5_ranks()
    g = np.random.default_rng(seed)
    return [np.asfortranarray((g.standard_normal((2, rks[k], rks[k + 1])) + 1j * g.standard_normal((2, rks[k], rks[k + 1])))
                              / math.sqrt(4.0 * rks[k + 1])) for k in range(D5)]


# 16 rounded vectors of 2.5 MB each: 41 MB of outputs, the whole batch would be 10 GB
DUMP_SAMPLE, DUMP_SEED = 16, 5


def dump_plan(first, nvec, chunk, nw):
    """The vectors `--dump-outputs` writes: a fixed, seeded sample of global ids in [0, TOTAL5), and where this rank finds them,
    {worker: {position of the chunk in that worker's list: [(batch column, global id), ...]}} (chunk c goes to worker c % nw)."""
    ids = np.sort(np.random.default_rng(DUMP_SEED).choice(TOTAL5, DUMP_SAMPLE, replace=False))
    plan = {}
    for g in ids:
        local = int(g) - first
        if 0 <= local < nvec:
            c, b = divmod(local, chunk)
            plan.setdefault(c % nw, {}).setdefault(c // nw, []).append((b, int(g)))
    return ids, plan


def write_outputs(path, ids, kept):
    """DIR/y_core_KK.npy: core KK of the sampled results of apply_compress, float64 of shape (sample, 2, r_KK, r_KK+1, 2) with the
    real and imaginary parts on the last axis; DIR/vector_index.npy: which of the 4 096 vectors they are, in that order."""
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "vector_index.npy"), ids.astype(np.float64))
    for k in range(D5):
        a = np.stack([kept[int(g)][k] for g in ids])
        np.save(os.path.join(path, f"y_core_{k:02d}.npy"), np.stack([a.real, a.imag], axis=-1))


# ---------------------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
            t0 = time.time()                      # nvidia-smi needs ~0.1-0.3 s to print its first row: wait for it (bounded)
            while not self.rows and time.time() - t0 < 1.5:
                time.sleep(0.01)
            self.rows.clear()                     # rows printed before the timed region starts are not under load
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1 for N > 1; the CPU legs are meant to use every host core the BLAS can use."""
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=os.cpu_count() or 1)
    except Exception:
        pass


def host_threads():
    try:
        from threadpoolctl import threadpool_info
        return int(max([p.get("num_threads", 1) for p in threadpool_info()] + [1]))
    except Exception:
        return os.cpu_count() or 1


# ---------------------------------------------------------------------------------------------------------------
# CPU legs (the only place the oracle is executed: as the timed baseline, never as the product)
# ---------------------------------------------------------------------------------------------------------------
def cpu_one_vector(o, A, seed, faithful):
    """one vector of the cfg5 batch through the reference algorithm: A*x (tt_operations.jl:101-111), then the L->R and R->L
    bond truncations of tt_compress! (tt_tools.jl:772-789); faithful=True also runs the orthogonalize of tt_tools.jl:769"""
    rks, _ = cfg5_ranks()
    x = o.TTvector(D5, make_vector(seed), (2,) * D5, rks, [0] * D5)
    t0 = time.perf_counter()
    y = o.apply(A, x)
    for k in list(range(1, D5)) + list(range(D5 - 1, 0, -1)):
        o.tt_bond_truncate(y, k, max_bond=MAXB5, truncerr=0.0, faithful=faithful)
    return time.perf_counter() - t0


def run_reference(args, rank):
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ttn_oracle as o
    use_all_host_threads()
    A = make_mpo(o)
    # one vector takes ~16 s on the GPU box's host cores, so the run is bounded: at most one warm-up vector, and the measured steps
    # stop after `budget` seconds; "steps" is the number actually measured (every one of them in full), never an extrapolation
    budget = float(os.environ.get("TTN_BENCH_REFERENCE_BUDGET_S", "150"))
    nwarm = min(args.warmup, 1)
    times = []
    w0 = time.perf_counter()
    for i in range(nwarm + args.steps):
        el = cpu_one_vector(o, A, 100 + i, faithful=True)
        if i >= nwarm:
            times.append(el)
            if time.perf_counter() - w0 > budget:
                break
    tt = float(np.mean(times)) if times else float("nan")
    val = 1.0 / tt
    cores = host_threads()
    sample = ("each step = ONE of the 4096 vectors through A*x + tt_compress!(y,64) exactly as the reference executes it "
              "(including the orthogonalize of tt_tools.jl:769 whose result is discarded), fully measured; multithreaded "
              f"BLAS/LAPACK inside the vector; NumPy restatement of the reference, not Julia; {len(times)} of the {args.steps} requested "
              f"steps measured within the {budget:.0f} s budget after {nwarm} warm-up vector(s)")
    line = {"impl": "reference", "metric": "tt_rounding sweeps/s", "value": val, "unit": "sweeps/s", "n_gpus": args.gpus,
            "steps": len(times), "steps_requested": args.steps, "warmup": nwarm, "ms_per_step": tt * 1e3, "higher_is_better": True,
            "scaling": "strong",
            "vs_baseline": None, "dtype": "c128", "data": "synthetic", "config": cfg5_config(args.gpus, args.chunk),
            "cpu_baseline": {"value": val, "unit": "sweeps/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "sweeps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------
# ours
# ---------------------------------------------------------------------------------------------------------------
def pinned_chunks(torch, nvec, chunk, rank):
    """this rank's vectors in pinned host memory, one Fortran-ordered (2, r_k, r_{k+1}, chunk) array per site and chunk"""
    rks, _ = cfg5_ranks()
    gen = torch.Generator().manual_seed(1000 + rank)
    chunks, keep = [], []
    for c0 in range(0, nvec, chunk):
        nb = min(chunk, nvec - c0)
        cores = []
        for k in range(D5):
            n_el = 2 * rks[k] * rks[k + 1] * nb
            buf = torch.empty(2 * n_el, dtype=torch.float64).pin_memory()
            buf.normal_(generator=gen)
            buf.mul_(1.0 / math.sqrt(4.0 * rks[k + 1]))
            keep.append(buf)
            cores.append(buf.numpy().view(np.complex128).reshape((2, rks[k], rks[k + 1], nb), order="F"))
        chunks.append(cores)
    return chunks, keep


class ChunkWorker(threading.Thread):
    """One host thread = one library context (compute stream + copy stream + allocation cache, include/ttn_b200.h).  Each worker
    owns every `nw`-th chunk of this rank's vectors; the workers keep one chunk each in flight, so the latency-bound eigensolver
    kernels of one chunk overlap the DMMA GEMMs of the other."""

    def __init__(self, idx, nw, host_chunks, Ad, rks, torch, keep):
        super().__init__(daemon=True)
        import queue
        self.idx, self.nw, self.Ad, self.rks, self.torch, self.keep = idx, nw, Ad, rks, torch, keep
        self.host_chunks = host_chunks[idx::nw]
        self.cmd, self.done = queue.Queue(), queue.Queue()
        self.error = None

    def run(self):
        import ttn_b200 as t
        torch = self.torch
        try:
            t.synchronize()                                   # first library call of this thread: creates its context
            self.stream = torch.cuda.ExternalStream(t.stream_handle())
            self.dev_chunks = [t.DeviceTT.upload_batched(c, (2,) * D5, self.rks) for c in self.host_chunks]
            self.res_bufs = {}
            for c in self.host_chunks:
                nb = c[0].shape[3]
                if nb not in self.res_bufs:
                    self.res_bufs[nb] = [self._result_set(nb), self._result_set(nb)]
            t.synchronize()
            self.done.put("ready")
            while True:
                cmd = self.cmd.get()
                if cmd[0] == "stop":
                    for x in self.dev_chunks:       # handles are released by the thread (context) that created them
                        x.free()
                    self.dev_chunks = []
                    t.synchronize()
                    from ttn_b200 import _lib
                    _lib.load().ttn_shutdown()      # this thread's streams and allocation cache
                    self.done.put("stopped")
                    break
                self.done.put(getattr(self, "_" + cmd[0])(t, *cmd[1:]))
        except Exception as e:   # noqa: BLE001
            self.error = e
            self.done.put(e)

    def _result_set(self, nb):
        res = []
        for k in range(D5):
            rl, rr = min(self.rks[k], MAXB5), min(self.rks[k + 1], MAXB5)
            buf = self.torch.empty(2 * 2 * rl * rr * nb, dtype=self.torch.float64).pin_memory()
            self.keep.append(buf)
            res.append(buf.numpy().view(np.complex128).reshape((2, rl, rr, nb), order="F"))
        return res

    def _device(self, t, nsteps, profile=False, keep=None):
        """nsteps passes over this worker's device-resident chunks; returns the end event (on this worker's stream) + counters.
        `keep` (chunk positions, see dump_plan): the results of those chunks in the last pass stay on the device for `_kept`."""
        if profile:
            t.set_option("reset_flops", 1)
            t.profile(True)
        t.reset_launch_count()
        fb0 = t.get_option("gram_fallbacks")
        last, self.held = None, {}
        for s in range(nsteps):
            for j, xd in enumerate(self.dev_chunks):
                last = t.apply_compress(self.Ad, xd, MAXB5)
                if keep and j in keep and s == nsteps - 1:
                    self.held[j] = last
        ev = self.torch.cuda.Event(enable_timing=True)
        ev.record(self.stream)
        t.synchronize()
        out = {"end": ev, "launches": t.launch_count(), "fallbacks": int(t.get_option("gram_fallbacks") - fb0),
               "out_rks": last.ttv_rks if last is not None else None}
        if profile:
            out["fam"] = t.profile_read()
            t.profile(False)
            out["flops"] = {"gemm": t.get_option("gemm_flops"), "jacobi": t.get_option("heig_flops")}
        return out

    def _kept(self, t, keep):
        """the vectors `keep` ({chunk position: [(batch column, global id), ...]}) names, out of the results `_device` held:
        {global id: list of host cores}; the held results are released"""
        out = {}
        for j, y in self.held.items():
            rks, nb = y.ttv_rks, y.batch
            cores = [np.empty((2, rks[k], rks[k + 1], nb), dtype=np.complex128, order="F") for k in range(D5)]
            y.download_into([a if nb > 1 else a[..., 0] for a in cores])        # a batch of one has no batch axis
            for b, g in keep[j]:
                out[g] = [np.ascontiguousarray(a[..., b]) for a in cores]
            y.free()
        self.held = {}
        return out

    def _e2e(self, t, nsteps):
        """software pipeline over this worker's chunks on pinned host memory, running across the step boundaries: H2D of the next
        chunk and D2H of the previous one run on the copy stream while the current chunk computes; every step moves all of its
        inputs host -> device and all of its results device -> host, and the timed region ends when the last result has landed"""
        hc = self.host_chunks
        seq = [c for _ in range(nsteps) for c in hc]
        if seq:
            mode = os.environ.get("TTN_BENCH_E2E_MODE", "full")      # diagnosis only: "nodown" drops the result copies
            trace = os.environ.get("TTN_BENCH_E2E_TRACE") == "1"
            acc = {"up": 0.0, "compute": 0.0, "down": 0.0, "free": 0.0}
            up = lambda c: t.DeviceTT.upload_batched(c, (2,) * D5, self.rks, asynchronous=True)  # noqa: E731
            nxt = up(seq[0])
            for j, c in enumerate(seq):
                xd = nxt
                t0 = time.perf_counter()
                if j + 1 < len(seq):
                    nxt = up(seq[j + 1])
                t1 = time.perf_counter()
                y = t.apply_compress(self.Ad, xd, MAXB5)
                t2 = time.perf_counter()
                if mode != "nodown":
                    y.download_into(self.res_bufs[c[0].shape[3]][j & 1], asynchronous=True)
                t3 = time.perf_counter()
                xd.free(); y.free()
                t4 = time.perf_counter()
                acc["up"] += t1 - t0; acc["compute"] += t2 - t1; acc["down"] += t3 - t2; acc["free"] += t4 - t3
            if trace:
                print(f"[e2e trace] worker {self.idx}: chunks {len(seq)} host seconds {acc}", file=sys.stderr, flush=True)
            t.copy_synchronize()
        t.synchronize()
        return {"h2d": int(sum(a.nbytes for c in hc for a in c)),
                "d2h": int(sum(sum(a.nbytes for a in self.res_bufs[c[0].shape[3]][0]) for c in hc))}


def bind_to_gpu_numa(local_rank):
    """one process per GPU, bound to the CPUs the GPU hangs off (NVML's ideal CPU set intersected with what the container allows):
    the pinned buffers are then first-touched on that socket and the host <-> device copies of the end-to-end leg do not cross the
    socket interconnect.  Returns the number of CPUs bound, or None when NVML has no answer."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = int(vis.split(",")[local_rank]) if vis else local_rank      # NVML numbers the physical devices
        h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        allowed = os.sched_getaffinity(0)
        nwords = (max(allowed) + 64) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, nwords)
        ideal = {64 * i + b for i, w in enumerate(mask) for b in range(64) if (int(w) >> b) & 1}
        cpus = ideal & allowed
        if not cpus or cpus == allowed:
            return None
        os.sched_setaffinity(0, cpus)
        return len(cpus)
    except Exception:
        return None


def captured_traffic():
    """DRAM bytes per launch (read + write) of the largest kernel of the dominant family, heig_tridiag_kernel<double2> at the cfg5 shape
    (batch 296), from the committed `ncu --set full` capture; None when the summary is not there"""
    try:
        rd = wr = None
        for ln in open(os.path.join(ROOT, "profiles", "ncu_heig_tridiag_c128_r02.txt")):
            f = ln.split()
            if len(f) >= 3 and f[0] == "dram__bytes_read.sum" and rd is None:
                rd = float(f[1]) * {"Mbyte": 1e6, "Kbyte": 1e3, "Gbyte": 1e9, "byte": 1.0}[f[2]]
            if len(f) >= 3 and f[0] == "dram__bytes_write.sum" and wr is None:
                wr = float(f[1]) * {"Mbyte": 1e6, "Kbyte": 1e3, "Gbyte": 1e9, "byte": 1.0}[f[2]]
        return None if rd is None or wr is None else rd + wr
    except Exception:
        return None


def run_ours(args, rank, local_rank, world):
    bound = bind_to_gpu_numa(local_rank) if world > 1 and not args.no_numa_bind else None
    import torch
    import ttn_b200 as t
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        sys.stdout.flush()
        saved = os.dup(1)                 # NCCL may print its banner on stdout: keep stdout clean for the single JSON line
        os.dup2(2, 1)
        try:
            dist_.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            dist_.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
        dist = dist_
    K, W = args.steps, args.warmup
    rks, Rk = cfg5_ranks()
    first, nvec = t.shard_batch(TOTAL5, rank, world)
    chunk = min(args.chunk, nvec)
    Ad = t.DeviceTTO.upload(make_mpo(t))        # read-only, shared by the worker threads
    host_chunks, keep = pinned_chunks(torch, nvec, chunk, rank)
    t.synchronize()
    stream = torch.cuda.ExternalStream(t.stream_handle())
    nw = max(1, min(args.host_threads, len(host_chunks)))
    workers = [ChunkWorker(i, nw, host_chunks, Ad, rks, torch, keep) for i in range(nw)]
    for w in workers:
        w.start()

    def collect():
        res = [w.done.get() for w in workers]
        for r in res:
            if isinstance(r, Exception):
                raise r
        return res

    collect()

    def barrier():
        t.synchronize()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    def allmax(v):
        if dist is None:
            return v
        tm = torch.tensor([v], device="cuda", dtype=torch.float64)
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        return float(tm.item())

    def timed(nsteps, plan=None):
        """all workers idle -> start event -> nsteps passes on every worker -> latest end event of the workers' streams"""
        barrier()
        g0 = torch.cuda.Event(enable_timing=True)
        g0.record()
        for w in workers:
            w.cmd.put(("device", nsteps, False, (plan or {}).get(w.idx)))
        res = collect()
        torch.cuda.synchronize()
        ms = max(g0.elapsed_time(r["end"]) for r in res)
        barrier()
        return ms, res

    # ---- device-resident timing -------------------------------------------------------------------------------
    timed(W)
    dump_ids, plan = dump_plan(first, nvec, chunk, nw) if args.dump_outputs else (None, None)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms, res = timed(K, plan)
    launches = sum(r["launches"] for r in res)
    fallbacks = sum(r["fallbacks"] for r in res)
    clocks = sampler.stop() if rank == 0 else None
    out_rks = res[0]["out_rks"]
    ms_per_step = allmax(ms) / K
    value = TOTAL5 / (ms_per_step * 1e-3)
    if args.dump_outputs:
        for w in workers:
            w.cmd.put(("kept", plan.get(w.idx, {})))
        kept = {g: c for r in collect() for g, c in r.items()}
        if dist is not None:
            parts = [None] * world
            dist.all_gather_object(parts, kept)
            kept = {g: c for p in parts for g, c in p.items()}
        if rank == 0:
            write_outputs(args.dump_outputs, dump_ids, kept)

    # ---- end to end through the host API: pinned host buffers, H2D + apply_compress + D2H per chunk ----------------
    def e2e(nsteps):
        barrier()
        w0 = time.perf_counter()
        for w in workers:
            w.cmd.put(("e2e", nsteps))
        r = collect()
        return (time.perf_counter() - w0) / max(1, nsteps), r

    e2e(min(W, 1))
    e2e_steps = max(1, min(K, args.e2e_steps * world))     # about the same bytes over PCIe per rank at every N
    e2e_s, er = e2e(e2e_steps)
    e2e_s = allmax(e2e_s)
    h2d, d2h = sum(r["h2d"] for r in er), sum(r["d2h"] for r in er)
    if dist is not None:
        tb = torch.tensor([float(h2d), float(d2h)], device="cuda", dtype=torch.float64)
        dist.all_reduce(tb, op=dist.ReduceOp.SUM)
        h2d, d2h = int(tb[0].item()), int(tb[1].item())

    # ---- roofline pass: per-kernel-family CUDA events over one step, with the FLOPs the kernels were asked to execute ------
    # one worker at a time (the others idle), so that a family's event-bracketed time is that of its kernels alone on the GPU and not
    # stretched by the other host thread's kernels sharing the SMs
    ms_prof, pres = 0.0, []
    for w in workers:
        barrier()
        g0 = torch.cuda.Event(enable_timing=True)
        g0.record()
        w.cmd.put(("device", 1, True))
        r = w.done.get()
        if isinstance(r, Exception):
            raise r
        torch.cuda.synchronize()
        ms_prof += g0.elapsed_time(r["end"])
        pres.append(r)
    barrier()
    fam_ms, fam_cnt, executed = {}, {}, {"gemm": 0.0, "jacobi": 0.0}
    for r in pres:
        for k, v in r["fam"].items():
            fam_ms[k] = fam_ms.get(k, 0.0) + v[0]
            fam_cnt[k] = fam_cnt.get(k, 0) + v[1]
        for k in executed:
            executed[k] += r["flops"][k]
    model = cfg5_flop_model()
    peak64 = json.load(open(FP64_PEAK_FILE)) if os.path.exists(FP64_PEAK_FILE) else {"fp64_tflops": 35.45, "c128_tflops": 36.8}
    peak = float(peak64.get("fp64_tflops", 35.45))
    dom = max(fam_ms, key=fam_ms.get)
    names = {"gemm": "gemm_kernel<double2,...> (DMMA: Z = P x, Gram, projection GEMMs of the fused apply + rounding)",
             "jacobi": "heig_* (Gram-path eigensolver: Householder tridiagonalisation, multisection, twisted vectors, back-transformation)"}
    fams = {}
    for k in ("gemm", "jacobi"):
        tfk = executed[k] / (fam_ms[k] * 1e-3) / 1e12 if fam_ms.get(k, 0) > 0 else 0.0
        fams[k] = {"kernel": names[k], "stream_ms_per_step": round(fam_ms.get(k, 0.0), 3), "launches_per_step": fam_cnt.get(k, 0),
                   "executed_gflop_per_vector": executed[k] / nvec / 1e9, "achieved_tflops": tfk, "frac": tfk / peak}
    step_tf = model["total"] * TOTAL5 / (ms_per_step * 1e-3) / 1e12 / world
    exec_tf = (executed["gemm"] + executed["jacobi"]) * (TOTAL5 / nvec) / (ms_per_step * 1e-3) / 1e12 / world
    roofline = {"bound": "tensor", "kernel": names.get(dom, dom), "achieved": fams.get(dom, {}).get("achieved_tflops", 0.0), "peak": peak,
                "unit": "TFLOP/s", "frac": fams.get(dom, {}).get("frac", 0.0), "traffic": captured_traffic(),
                "flop_accounting": "FLOPs the dominant kernel family was asked to execute in the step (GEMM: 8MNK per complex product; "
                                   "eigensolver: LAPACK counts 4/3 n^3 + 2 n^2 nev, x4 complex), counted inside the library, / the summed "
                                   "CUDA-event time of that family in a profiling pass that runs the host threads one after the other (kernels "
                                   "timed without the other thread's kernels sharing the SMs; the timed region itself overlaps the threads, "
                                   "which is why profiled_ms_per_step exceeds ms_per_step)",
                "traffic_note": "dram__bytes_read + dram__bytes_write per launch of heig_tridiag_kernel<double2> (296 matrices of 128 x 128 ComplexF64), "
                                "the largest kernel of the dominant family, from profiles/ncu_heig_tridiag_c128_r02.txt; algorithmic: 39.1 MB "
                                "read (lower triangles) + 39.7 MB of reflectors and tridiagonals written, of which L2 absorbs the writes",
                "peak_source": "measured cuBLAS FP64 GEMM 8192^3 burst on this pool's B200 (profiles/fp64_peak_r01.json; builder-"
                               "measured fallback: MEASURED_PEAKS.json carries no FP64 figure)",
                "families": fams, "family_stream_ms_per_step": {k: round(v, 3) for k, v in fam_ms.items()},
                "profiled_ms_per_step": ms_prof,
                "whole_step": {"survey_model": {"achieved": step_tf, "frac": step_tf / peak,
                                                "gflop_per_vector": model["total"] / 1e9,
                                                "note": "SURVEY.md section 8(d)-5 per-unit figure (Theta GEMMs + projections + R-SVD count 6mk^2+20k^3, "
                                                        "complex = 4 x real) x vectors / step time, per GPU; above 1 because the Gram path and the "
                                                        "fused apply execute fewer FLOPs than that model's algorithm"},
                               "executed": {"achieved": exec_tf, "frac": exec_tf / peak,
                                            "gflop_per_vector": (executed["gemm"] + executed["jacobi"]) / nvec / 1e9}}}
    for w in workers:
        w.cmd.put(("stop",))
    collect()

    # ---- extras: the other components of BASELINE.json's metric (compact in the line, full detail on disk) ----------
    extras, compact = {}, {}
    if not args.no_extras:
        if world > 1:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import shard_bench
            sm = shard_bench.run(torch, dist, rank, world, chi=1024, w=5, reps=10, krylovdim=8)
            extras["matvec_cfg4_sharded"] = sm
            compact["matvec_cfg4_sharded_fused_ms"] = sm.get("fused_ms")
            compact["matvec_cfg4_sharded_tflops"] = sm.get("fused_tflops")
            # cfg4 DMRG sweep over all ranks: replicated sweep, Lanczos matvec of every bond step sharded (csrc/shard.cu)
            def exchange(bts):
                out = [None] * world
                dist.all_gather_object(out, bts)
                return out
            sc = t.ShardContext(np.float64, args.dmrg_chi * args.dmrg_chi * 4, rank, world, exchange)
            ds = bench_dmrg(t, args.dmrg_chi, shard=sc)
            tm = torch.tensor([ds["value"]], device="cuda", dtype=torch.float64)
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            ds["value"] = float(tm.item())
            ds["n_gpus"] = world
            ds["note"] += "; sweep replicated on every rank, Lanczos matvecs sharded over the ranks with the fused all-gather epilogue"
            sc.free()
            extras["dmrg_sweep_sharded"] = ds
            compact["dmrg_sweep_sharded_s"] = ds["value"]
        if rank == 0:
            extras["cfg2"] = bench_cfg2(t, torch, stream)
            compact["cfg2_sweeps_per_s"] = extras["cfg2"]["value"]
            compact["cfg2_e2e_sweeps_per_s"] = extras["cfg2"]["e2e"]["value"]
            extras["matvec_cfg4"] = bench_matvec(t, torch, stream, peak64)
            compact["matvec_cfg4_tflops"] = extras["matvec_cfg4"]["value"]
            compact["matvec_cfg4_frac"] = extras["matvec_cfg4"]["roofline"]["frac"]
            if world == 1 or args.dmrg_all:
                extras["dmrg_sweep"] = bench_dmrg(t, args.dmrg_chi)
                compact["dmrg_sweep_s"] = extras["dmrg_sweep"]["value"]
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import cfg3_bench
            extras["mals_cfg3"] = cfg3_bench.run(bits=20, rmax=128)
            compact["mals_cfg3_s"] = extras["mals_cfg3"].get("value")
            # cfg3 with ranks at the cap: implicit-Euler heat operator, known rank-128 solution (full size), and the same problem at
            # 2 x 10 bits / rmax 32 where the reference's dense-K algorithm is feasible on the CPU (timed below)
            extras["mals_cfg3_heat"] = cfg3_bench.run_heat(bits=20, rmax=128)
            extras["mals_cfg3_heat_small"] = cfg3_bench.run_heat(bits=10, rmax=32, start_rank=16)
            compact["mals_cfg3_heat_s"] = extras["mals_cfg3_heat"]["value"]
            compact["mals_cfg3_heat_max_rank"] = extras["mals_cfg3_heat"]["calls"][0]["max_rank"]
            compact["mals_cfg3_heat_err"] = extras["mals_cfg3_heat"]["calls"][-1]["relative_error"]
    if dist is not None:
        dist.barrier()

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu:
            sys.path.insert(0, os.path.join(ROOT, "oracle"))
            import ttn_oracle as o
            use_all_host_threads()
            Ao = make_mpo(o)
            n_s, tot = 0, 0.0
            while tot < 12.0 and n_s < 8:
                tot += cpu_one_vector(o, Ao, 100 + n_s, faithful=False)
                n_s += 1
            tf = cpu_one_vector(o, Ao, 100, faithful=True)
            cpu = {"value": n_s / tot, "unit": "sweeps/s", "cores": host_threads(), "kind": "port",
                   "sample": f"{n_s} of the 4096 vectors, algorithm-equivalent (the discarded orthogonalize of tt_tools.jl:769 removed), "
                             f"multithreaded BLAS/LAPACK inside each vector",
                   "reference_faithful_value": 1.0 / tf, "reference_faithful_sample": "1 vector including the discarded orthogonalize",
                   "note": "NumPy restatement of the reference, not Julia"}
            if "dmrg_sweep" in extras:
                extras["dmrg_sweep"]["cpu_baseline"] = cpu_dmrg(o, args.dmrg_chi)
                extras["matvec_cfg4"]["cpu_baseline"] = extras["dmrg_sweep"]["cpu_baseline"].get("matvec")
            if "mals_cfg3_heat_small" in extras:
                cb = cpu_cfg3_heat(o, cfg3_bench, 10, 32, 16)
                cb["gpu_first_call_speedup"] = cb["value"] / extras["mals_cfg3_heat_small"]["value"]
                extras["mals_cfg3_heat_small"]["cpu_baseline"] = cb
                compact["mals_cfg3_heat_small_cpu_over_gpu"] = cb["gpu_first_call_speedup"]
        line = {"metric": "tt_rounding sweeps/s", "value": value, "unit": "sweeps/s", "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "c128",
                "data": "synthetic", "config": dict(cfg5_config(world, chunk), out_max_rank=int(max(out_rks)),
                                                    gram_path_fallbacks_in_timed_region=fallbacks, host_threads_per_rank=nw,
                                                    cpus_bound_per_rank=bound),
                "clocks": clocks, "gpu_launches": int(launches),
                "e2e": {"value": TOTAL5 / e2e_s, "unit": "sweeps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": e2e_s * 1e3, "steps": e2e_steps, "mode": os.environ.get("TTN_BENCH_E2E_MODE", "full"),
                        "api": "per chunk: DeviceTT.upload_batched(pinned, asynchronous) -> ttn_b200.apply_compress(A, x, 64) -> "
                               "download_into(pinned, asynchronous); copies on the copy streams overlap the neighbouring chunks' compute; "
                               f"{nw} host thread(s) = library contexts per rank"},
                "roofline": roofline, "cpu_baseline": cpu, "extras": compact}
        if args.extras_out:
            with open(args.extras_out, "w") as f:
                json.dump({"line": line, "extras": extras}, f, indent=1)
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------------
# extras
# ---------------------------------------------------------------------------------------------------------------
def cfg2_ranks(d=D, rmax=RMAX_IN):
    return [min(2 ** k, 2 ** (d - k), rmax) for k in range(d + 1)]


def bench_cfg2(t, torch, stream, reps=5):
    """BASELINE.json configs[1]: tt_compress!(rand_tt d=40 n=2 r=512, 64): a single train, i.e. a 78-step dependency chain"""
    rks = cfg2_ranks()
    rng = np.random.default_rng(1)
    cores, keep = [], []
    for k in range(D):
        c = rng.standard_normal((NPHYS, rks[k], rks[k + 1])) / math.sqrt(NPHYS * rks[k + 1])
        buf = torch.empty(c.size, dtype=torch.float64).pin_memory()
        view = buf.numpy().reshape(c.shape, order="F")
        view[...] = c
        keep.append(buf)
        cores.append(view)
    host_tt = lambda: t.TTvector(D, list(cores), (NPHYS,) * D, list(rks))  # noqa: E731
    base = t.DeviceTT.upload(host_tt())
    for _ in range(3):
        t.tt_compress_(base.copy(), MAX_BOND)
    copies = [base.copy() for _ in range(reps)]
    t.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t.reset_launch_count()
    e0.record(stream)
    for c in copies:
        t.tt_compress_(c, MAX_BOND)
    e1.record(stream)
    t.synchronize()
    ms = e0.elapsed_time(e1) / reps
    launches = t.launch_count() // reps
    t.tt_compress_(host_tt(), MAX_BOND)
    w0 = time.perf_counter()
    for _ in range(reps):
        res = t.tt_compress_(host_tt(), MAX_BOND)
    t.synchronize()
    e2e = (time.perf_counter() - w0) / reps
    return {"metric": "tt_rounding sweeps/s (single train, cfg2)", "value": 1e3 / ms, "unit": "sweeps/s", "ms_per_sweep": ms,
            "launches_per_sweep": int(launches), "out_max_rank": int(max(res.ttv_rks)),
            "e2e": {"value": 1.0 / e2e, "ms": e2e * 1e3, "h2d_bytes": int(sum(c.nbytes for c in cores)),
                    "d2h_bytes": int(sum(c.nbytes for c in res.ttv_vec))},
            "note": "latency bound: 78 dependent bond steps on bond-sized matrices (SURVEY.md section 8(d)-2); fresh 97.9 MB input copy per sweep"}


def bench_matvec(t, torch, stream, peak64, chi=1024, w=5, nn=4, reps=10):
    """local two-site matvec Y = L·W·V·R at cfg4 shapes; F = 4 w n² chi³ + 2 w² n⁴ chi² (SURVEY.md §8(d)-4)"""
    import ctypes as C
    from ttn_b200 import _lib
    lib = _lib.lib()
    rng = np.random.default_rng(4)
    G = np.asfortranarray(rng.standard_normal((w, chi, chi)))
    H = np.asfortranarray(rng.standard_normal((w, chi, chi)))
    Am = np.asfortranarray(rng.standard_normal((w, nn, nn, w)))
    V = np.asfortranarray(rng.standard_normal((chi, nn, chi)))
    mv = C.c_void_p()
    _lib.check(lib.ttn_matvec2_create(0, w, w, chi, chi, nn, G.ctypes.data, Am.ctypes.data, H.ctypes.data, C.byref(mv)))
    dV, dY = C.c_void_p(), C.c_void_p()
    _lib.check(lib.ttn_dev_alloc(V.nbytes, C.byref(dV)))
    _lib.check(lib.ttn_dev_alloc(V.nbytes, C.byref(dY)))
    _lib.check(lib.ttn_h2d(dV, V.ctypes.data, V.nbytes))
    for _ in range(3):
        _lib.check(lib.ttn_matvec2_apply(mv, dV, dY))
    t.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(reps):
        _lib.check(lib.ttn_matvec2_apply(mv, dV, dY))
    e1.record(stream)
    t.synchronize()
    ms = e0.elapsed_time(e1) / reps
    flops = 4.0 * w * nn * chi ** 3 + 2.0 * w * w * nn * nn * chi ** 2
    tf = flops / (ms * 1e-3) / 1e12
    _lib.check(lib.ttn_matvec2_free(mv))
    _lib.check(lib.ttn_dev_free(dV))
    _lib.check(lib.ttn_dev_free(dY))
    pk = float(peak64.get("fp64_tflops_sustained", peak64.get("fp64_tflops", 35.45)))
    return {"metric": "local-matvec FP64 TFLOP/s", "value": tf, "ms": ms, "gflop": flops / 1e9, "chi": chi, "w": w, "n2": nn,
            "symmetrize": False,
            "roofline": {"bound": "tensor", "achieved": tf, "peak": pk, "unit": "TFLOP/s", "frac": tf / pk},
            "note": "one application of K (dmrg.jl:239-244 applies the symmetrised pair: twice this work); working set 0.5 GB > L2"}


def bench_dmrg(t, chi, L=64, kd=8, shard=None):
    """cfg4-style DMRG sweep: Heisenberg XYZ chain L=64 (MPO rank 5), one full two-site sweep from a random TT capped at
    bond `chi`, fixed Lanczos budget (krylovdim 8 x 1 restart) as in SURVEY.md §8(d)-4; symmetrize=True as dmrg.jl:241."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import dmrg_bench
    H = t.DeviceTTO.upload(dmrg_bench.heisenberg(L))
    x0 = t.DeviceTT.upload(dmrg_bench.rand_tt(L, chi))
    t.synchronize()
    t.reset_launch_count()
    t0 = time.perf_counter()
    E, x, rh = t.dmrg_eigsolve(H, x0, N=2, tol=1e-12, sweep_schedule=[2], rmax_schedule=[chi], linsolv_maxiter=1,
                               linsolv_tol=1e-10, krylovdim=kd, symmetrize=True, shard=shard)
    t.synchronize()
    el = time.perf_counter() - t0
    return {"metric": "DMRG sweep s", "value": el, "unit": "s", "L": L, "chi": chi, "krylovdim": kd, "bond_steps": len(E),
            "symmetrize": True, "max_rank": int(max(rh)), "E_last": float(E[-1]), "gpu_launches": int(t.launch_count()),
            "note": "cfg4 (BASELINE.json configs[3]): Heisenberg XYZ L=64, MPO rank 5, one full two-site sweep from a random TT capped "
                    "at chi; the local operator is the symmetrised pair 0.5 (K + K^T) of dmrg.jl:241, as on the CPU leg"}


def cpu_dmrg(o, chi, w=5, nn=4):
    """CPU leg of the DMRG extra: three REAL bulk bond steps of the restated algorithm at full size (symmetrised Lanczos matvecs
    through BLAS GEMMs + gesdd of the 2 chi x 2 chi two-site tensor + environment update), timed; the sweep figure is that mean
    times the ~105 full-rank bond steps of the L = 64 sweep (labelled as such)."""
    import scipy.linalg as sla
    rng = np.random.default_rng(4)
    G = rng.standard_normal((w, chi, chi)); H = rng.standard_normal((w, chi, chi))
    Am = rng.standard_normal((w, nn, nn, w)); V = rng.standard_normal((chi, nn, chi))
    o.dmrg_matvec2_blas(G, Am, V, H)
    t0 = time.perf_counter(); o.dmrg_matvec2_blas(G, Am, V, H); t_mv = time.perf_counter() - t0
    flops = 4.0 * w * nn * chi ** 3 + 2.0 * w * w * nn * nn * chi ** 2
    steps = []
    for _ in range(3):
        t0 = time.perf_counter()
        v = V
        for _ in range(8):                                   # krylovdim 8, symmetrised pair per matvec (dmrg.jl:241)
            v = 0.5 * (o.dmrg_matvec2_blas(G, Am, v, H) + o.dmrg_matvec2_blas(np.transpose(G, (0, 2, 1)), np.transpose(Am, (0, 2, 1, 3)),
                                                                            v, np.transpose(H, (0, 2, 1))))
            v = v / np.linalg.norm(v)
        sla.svd(v.reshape(chi * 2, 2 * chi, order="F"), full_matrices=False, lapack_driver="gesdd")
        steps.append(time.perf_counter() - t0)
    bond = float(np.mean(steps))
    return {"value": 105 * bond, "unit": "s", "cores": host_threads(), "kind": "port", "bulk_bond_step_s": bond, "measured_bond_steps": 3,
            "symmetrize": True,
            "matvec": {"value": flops / t_mv / 1e12, "unit": "TFLOP/s", "seconds": t_mv, "cores": host_threads(), "kind": "port",
                       "sample": "one full-size application (chi=1024) through three BLAS GEMMs"},
            "sample": "three bulk bond steps measured at full size (8 symmetrised Lanczos matvecs + gesdd 2048^2), mean x the ~105 "
                      "full-rank bond steps of the L=64 sweep (environment updates not counted); NumPy restatement, not Julia"}


def cpu_cfg3_heat(o, cfg3_bench, bits, rmax, start_rank, tol=1e-10):
    """CPU leg of the cfg3 (implicit-Euler heat step) extra: one `mals_linsolve` call of the restated algorithm (dense local K,
    mals.jl:148-169, NumPy/LAPACK) on the inputs tools/cfg3_bench.heat_problem builds for the GPU leg at the same (bits, rmax)."""
    A, _, xt, x0 = cfg3_bench.heat_problem(bits, rmax, start_rank)
    d = 2 * bits
    oA = o.TToperator(d, [np.array(c) for c in A.tto_vec], tuple(A.tto_dims), list(A.tto_rks))
    mk = lambda v: o.TTvector(d, [np.array(c) for c in v.ttv_vec], tuple(v.ttv_dims), list(v.ttv_rks), [0] * d)  # noqa: E731
    oxt, ox = mk(xt), mk(x0)
    ob = o.apply(oA, oxt)
    t0 = time.perf_counter()
    ox = o.mals_linsolve(oA, ob, ox, tol=tol, rmax=rmax)
    el = time.perf_counter() - t0
    r = o.add(o.apply(oA, ox), o.scale(-1.0, ob))
    return {"value": el, "unit": "s per call", "kind": "port", "cores": host_threads(), "bits": bits, "rmax": rmax,
            "relative_residual": float(o.norm(r) / o.norm(ob)), "max_rank": int(max(ox.ttv_rks)),
            "sample": "one call on the same inputs as the GPU leg of the same (bits, rmax); dense local K through NumPy/LAPACK, not Julia"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps (each = all 4096 vectors once)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--chunk", type=int, default=296, help="vectors per device batch (cfg5); 296 = two full waves of one matrix per SM")
    ap.add_argument("--host-threads", type=int, default=3, help="library contexts (host threads) per rank: chunks in flight")
    ap.add_argument("--e2e-steps", type=int, default=5, help="upper bound on the end-to-end steps (each moves 2 x 10 GB over PCIe at N=1)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--no-numa-bind", action="store_true", help="N > 1: do not bind each rank to its GPU's CPU set")
    ap.add_argument("--no-extras", action="store_true", help="skip the cfg2 / cfg4 matvec / DMRG sweep / cfg3 extras")
    ap.add_argument("--dmrg-chi", type=int, default=1024, help="bond cap of the DMRG sweep extra (cfg4: 1024)")
    ap.add_argument("--dmrg-all", action="store_true", help="run the DMRG sweep extra at N > 1 as well")
    ap.add_argument("--extras-out", metavar="FILE", help="write the JSON line and the full detail of the extras to FILE")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step for a fixed sample of the "
                                                          "vectors to DIR/<name>.npy (float64, 41 MB)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
