#!/usr/bin/env python
"""bench.py -- traversed edges/sec (mxm TEPS) for FalkorDB's CondTraverse hot path on B200.

A "step" is one pass of the hot path over one batch of synthetic input: a batch of `--sources` source vertices
F (|batch| x n, one entry per row -- cond_traverse.rs:600-601) pushed through a 3-hop GrB_mxm chain F*A*A*A over
GxB_ANY_PAIR_BOOL (cond_traverse.rs:602-605) on a Graph500 RMAT graph, then materialised as sorted CSR (the form
the reference's row iterator walks, cond_traverse.rs:608,644).  TEPS = sum over hops of
flops_h = sum_{(i,k) in F_h} deg_A(k)  divided by the step time  (SURVEY.md 8d).

  value : device-resident -- F already in HBM when the timed region starts; CUDA-event timed on the library's stream
  e2e   : the same batch host to host through ONE C-ABI call per batch, B200_traverse_batch: host source ids in (H2D inside),
          3 hops, the result in host memory as a packed row-major bitmap (128-row slices, D2H on a second stream overlapping
          the next slice's hops) -- the hand-off Matrix.export_auto's rule picks for a result denser than 1/32; the CSR
          hand-off of the same call is timed next to it at N = 1.
  roofline : the dominant kernel family's algorithmic bytes / its event-timed duration against the measured HBM peak, every
          family in `families`, and for the hop what really bounds it (`hop_gather_ceiling`: L1TEX wavefronts per second).
  cpu_baseline : the whole first timed batch on the host (oracle port, all threads) + digest parity of all its rows vs the GPU.

--impl reference times the CPU restatement of the reference algorithm (oracle/, OpenMP on all host cores) on the same
batches.  Multi-GPU: the batch rows are independent, so ranks shard the sources with A replicated and no data-path
collective (weak scaling: fixed sources per rank); ranks bind to their GPU's NUMA node.
Other workloads (--workload): bfs (config 5: partitioned direction-optimising BFS over NCCL), triangles (config 4), delta
(delta-matrix sync kernels at fold sizes), pagerank (FP64 mxv).  The chain line also carries configs 5 and 4 at their stated
sizes as sub-objects `partitioned_bfs` (RMAT-26, rows of A partitioned over the N ranks, NCCL all-gather per level; levels and
min-id parents checked against the oracle) and `masked_triangles` (RMAT-24, strong scaling), each measured by a child process per
rank after the chain's timed regions (--side; a child that fails costs its sub-object only).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scale", type=int, default=24)
    ap.add_argument("--edge-factor", type=int, default=16)
    ap.add_argument("--sources", type=int, default=512,
                    help="frontier rows per batch per GPU (the reference's operator batch is <= 1024 rows, batch.rs:81)")
    ap.add_argument("--hops", type=int, default=3)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--cpu-sources", type=int, default=0, help="sources per CPU sample (0 = auto: ~5 s of CPU work)")
    ap.add_argument("--bits-mode", type=int, default=-1)
    ap.add_argument("--pull-mode", type=int, default=-1)
    ap.add_argument("--pull-kernel", type=int, default=-1, help="-1 library default, 0 = 8-lanes-per-row, 1 = merge-path")
    ap.add_argument("--workload", default="chain", choices=["chain", "bfs", "triangles", "delta", "pagerank"],
                    help="chain = the headline 3-hop mxm chain; bfs = 1-D row-partitioned BFS sweep (BASELINE config 5); "
                         "triangles = masked SpGEMM C<L> = L*L on the symmetrised lower triangle (BASELINE config 4)")
    ap.add_argument("--bfs-sources", type=int, default=16)
    ap.add_argument("--tri-parity", type=int, default=1, help="triangles: check every rank's result block against the oracle (0 = skip)")
    ap.add_argument("--bfs-parity", type=int, default=2, help="sources whose levels / parents are checked against the oracle (0 = none)")
    ap.add_argument("--opt", action="append", default=[], help="library option name=value (B200_set_option), repeatable")
    ap.add_argument("--e2e-format", default="auto", choices=["auto", "csr", "bitmap"],
                    help="result hand-off of the e2e arm: auto = Matrix.export_auto (bitmap when denser than 1/32, else CSR)")
    ap.add_argument("--e2e-subbatches", type=int, default=0,
                    help="row slices of a batch in the bitmap hand-off (falkordb_b200.traverse_to_host): slice k's D2H overlaps "
                         "slice k+1's hops; 0 = 128-row slices (default), 1 = whole batch, blocking export")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--side", default="bfs:26,triangles:24,delta:23,pagerank:22",
                    help="chain workload only: BASELINE configs 5 and 4 measured next to the chain, each as a child process per rank "
                         "(own process group), reported as sub-objects of the chain line; delta / pagerank (single-GPU kernels with "
                         "per-kernel rooflines and parity) at N = 1 only; '' or 'none' = skip")
    ap.add_argument("--side-timeout", type=int, default=300, help="seconds a side workload may take before its children are stopped")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="chain workload, b200 arm: after the timed steps write rank 0's result of the last timed step to DIR as "
                         "float64 .npy files (row_ptr, and a fixed seeded sample of col_idx with its positions) so that two builds "
                         "can be compared output for output")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "b200" or a.workload != "chain"):
        ap.error("--dump-outputs is implemented for the chain workload's b200 arm only")
    return a


DUMP_SAMPLE = 1 << 21          # column indices kept from a larger result: 2 x 16 MB of float64 with their positions


def dump_outputs(out_dir, F):
    """Write the CSR a caller of the chain receives -- row pointers in full, column indices as a sample at positions drawn
    with a fixed seed -- as float64 (exact: every value is below 2^53)."""
    p, j, _ = F.export_csr()
    nnz = len(j)
    if nnz > DUMP_SAMPLE:
        pos = np.sort(np.random.default_rng(12345).choice(nnz, size=DUMP_SAMPLE, replace=False))
    else:
        pos = np.arange(nnz)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "row_ptr.npy"), p.astype(np.float64))
    np.save(os.path.join(out_dir, "col_idx_sample.npy"), j[pos].astype(np.float64))
    np.save(os.path.join(out_dir, "col_idx_sample_pos.npy"), pos.astype(np.float64))


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines = gpu_index, None, []
        self.t0 = self.t1 = None

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        # the sampler is started before the warm-up (its NVML start-up stalls launches for a few ms if it lands inside the
        # timed region); samples stamped inside the timed window are used when there are any, else the ones under warm-up
        lines = self.lines
        if self.t0 is not None and self.t1 is not None:
            inside = [x for x in lines if self.t0 <= x[0] <= self.t1 + 0.1]
            lines = inside or lines
        for _, ln in lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def bind_to_gpu_numa_node(local):
    """Pin this rank's threads (and therefore the first-touch placement of its pinned host buffers) to the NUMA node its GPU
    hangs off: with 8 ranks each streaming ~1 GB per step to the host, buffers on the far socket halve the D2H rate."""
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(local)], text=True).strip()
        bus = out.lower()
        if bus.startswith("00000000:"):
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


def pick_sources(deg, nbatches, nsrc, seed, rank):
    """Seeded batches of distinct source vertices with non-zero out-degree (SURVEY 8d)."""
    rng = np.random.default_rng(seed * 1000003 + rank)
    cand = np.nonzero(deg > 0)[0]
    return [rng.choice(cand, size=nsrc, replace=False).astype(np.uint64) for _ in range(nbatches)]


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_chain(orc, A, src, hops):
    F = orc.build_matrix(len(src), A.nrows, np.arange(len(src)), src)
    flops = 0
    for _ in range(hops):
        F, fl = orc.mxm(F, A, return_flops=True)
        flops += fl
    return F, flops


def host_threads():
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def workload_name(a):
    return f"{a.hops}-hop mxm chain F*A^{a.hops}, RMAT scale-{a.scale} ef{a.edge_factor} seed {a.seed}"


# wall-clock budget of the reference arm's steps + warm-up: the full 512-source batch takes ~12 s on the 128-thread host, so
# the driver's --steps 20 --warmup 5 fits with the SAME batches as the b200 arm (about five minutes, like round 1's arm)
REFERENCE_ARM_BUDGET_S = 360.0


def calibrate_cpu_threads(orc, A, deg, a, all_threads):
    """The CPU arm's team size, measured rather than assumed: all the host threads, half and a quarter of them each run the same
    256-source mini-batch (two rows per thread at the full team), and the fastest wins -- hyper-threads sharing a core's cache, a far
    NUMA node or a CPU quota below the thread count can all make fewer threads faster for this cache-bound kernel.  Returns
    (threads chosen, {threads: seconds})."""
    cand = sorted({t for t in (all_threads, all_threads // 2, all_threads // 4) if t >= 8} | ({all_threads} if all_threads < 8 else set()), reverse=True)
    if len(cand) < 2:
        return all_threads, {}
    probe = pick_sources(deg, 1, min(a.sources, 256), a.seed + 23, 0)[0]
    times = {}
    for t in cand:
        orc.lib().orc_set_num_threads(t)
        orc.chain(A, probe[:t], a.hops, keep=False)                  # workspaces of this team
        t0 = time.perf_counter()
        orc.chain(A, probe, a.hops, keep=False)
        times[t] = time.perf_counter() - t0
    best = min(cand, key=lambda t: times[t])
    if times[all_threads] <= 1.05 * times[best]:                     # within noise: keep every thread
        best = all_threads
    orc.lib().orc_set_num_threads(best)
    return best, {str(k): round(v, 3) for k, v in times.items()}


def workload_config(a, n, nnzA, sources):
    """`config` of the JSON line: what defines the workload, identical for both arms (arm-specific settings go to `options`)"""
    return {"workload": workload_name(a), "n": n, "nnz_A": nnzA, "sources_per_gpu_per_step": sources,
            "l2_policy": ("inputs larger than L2 (A col_idx %.2f GB) and a fresh random source batch every step" % (4 * nnzA / 1e9))
            if 4 * nnzA > 256e6 else "A fits in L2 at this scale (%.3f GB): a smoke configuration, not a bench size" % (4 * nnzA / 1e9)}


def run_reference(a):
    """The reference's CPU implementation of the path.  SuiteSparse:GraphBLAS is not vendored under /root/reference and
    cannot be built here (cmake + generated code), so this arm times the oracle port (kind="port"): row-task Gustavson with
    thread-persistent bitmap workspaces on every host thread (oracle/grb_oracle.c: orc_chain), the whole chain in C.
    Each step = one batch of the b200 arm's workload -- the same --sources per step when steps + warm-up then fit six minutes
    (one untimed full batch decides), else the largest multiple of the thread count that does."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle as orc
    cores = host_threads()
    orc.lib().orc_set_num_threads(cores)       # torchrun pins OMP_NUM_THREADS=1 per rank; this arm owns the host
    t0 = time.time()
    A = orc.rmat_csr(a.scale, a.edge_factor, a.seed)
    gen_s = time.time() - t0
    A = orc.spread(A)                          # pages interleaved over the sockets by first touch (oracle.py: spread)
    deg = np.diff(A.p)
    all_threads = cores
    cores, team_probe = calibrate_cpu_threads(orc, A, deg, a, all_threads)
    S = a.cpu_sources if a.cpu_sources > 0 else a.sources
    probe_s = None
    if a.cpu_sources <= 0:
        # one whole batch of the b200 arm's size decides: the same batches when steps + warm-up then fit the budget, else the
        # largest multiple of the thread count that does (a smaller probe would be pessimistic: few rows per thread, idle threads)
        probe = pick_sources(deg, 1, S, a.seed + 17, 0)[0]
        orc.chain(A, probe[:cores], a.hops, keep=False)                # allocates the per-thread workspaces
        t0 = time.perf_counter()
        orc.chain(A, probe, a.hops, keep=False)
        probe_s = time.perf_counter() - t0
        total = probe_s * max(1, a.steps + a.warmup)
        if total > REFERENCE_ARM_BUDGET_S:
            S = min(S, max(cores, int(S * REFERENCE_ARM_BUDGET_S / total) // cores * cores))
    batches = pick_sources(deg, a.steps + a.warmup, S, a.seed, 0)
    for b in batches[:a.warmup]:
        orc.chain(A, b, a.hops, keep=False)
    flops, t, busy = 0, 0.0, []
    for b in batches[a.warmup:]:
        t0 = time.perf_counter()
        _, fl, _, bz = orc.chain(A, b, a.hops, keep=False)
        t += time.perf_counter() - t0
        flops += fl
        busy.append(bz)
    teps = flops / t
    sample = f"{a.hops}-hop chain, {S} sources/step, RMAT-{a.scale} ef{a.edge_factor}, {a.steps} steps"
    print(json.dumps({
        "impl": "reference", "metric": "traversed edges/sec (mxm TEPS), 3-hop ANY_PAIR mxm chain", "value": teps,
        "unit": "edges/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * t / a.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bool/u32 index", "data": "synthetic",
        "config": workload_config(a, A.nrows, A.nnz, S),
        "options": {"threads": cores, "host_threads": all_threads, "team_size_probe_s": team_probe, "full_batch_probe_s": probe_s,
                    "budget_s": REFERENCE_ARM_BUDGET_S},
        "graph_build_s": round(gen_s, 1), "result_format": "CSR (sorted rows, the form the reference's iterator walks)",
        "cpu_baseline": {"value": teps, "unit": "edges/s", "cores": cores, "kind": "port", "sample": sample,
                         "threads_busy_fraction": float(np.mean(busy)) if busy else None,
                         "algorithm": "Gustavson, one frontier row per task (LPT order), per-thread persistent n-bit accumulators"},
        "e2e": {"value": teps, "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def side_workload(a, workload, scale, extra, port_offset, script=None):
    """Run `bench.py --workload <workload>` as a child process of THIS rank -- under torchrun every rank starts one, and the children
    form their own process group on MASTER_PORT + port_offset -- and return rank 0's JSON line (None on other ranks), or
    {"error": ...}.  A child that crashes, hangs (stopped by PID at the timeout) or prints nothing costs its sub-object, never the
    chain line: the multi-GPU BFS exchange and the N > 1 triangle split had not run on hardware when this was written."""
    env = dict(os.environ)
    env.pop("TORCHELASTIC_USE_AGENT_STORE", None)         # the children's rank 0 hosts its own rendezvous store
    if "MASTER_PORT" in env:
        env["MASTER_PORT"] = str(int(env["MASTER_PORT"]) + port_offset)
    cmd = [sys.executable, script or os.path.abspath(__file__), "--workload", workload, "--gpus", str(a.gpus), "--scale", str(scale),
           "--edge-factor", str(a.edge_factor), "--seed", str(a.seed)] + extra
    t0 = time.time()
    try:
        r = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=a.side_timeout)
    except subprocess.TimeoutExpired:
        return {"error": f"stopped after {a.side_timeout} s"}
    except Exception as ex:
        return {"error": repr(ex)}
    if r.returncode != 0:
        return {"error": f"exit code {r.returncode}", "stderr_tail": r.stderr[-600:]}
    if int(os.environ.get("RANK", "0")) != 0:
        return None
    for ln in reversed(r.stdout.splitlines()):
        if ln.startswith("{"):
            try:
                d = json.loads(ln)
            except ValueError:
                break
            d["child_wall_s"] = round(time.time() - t0, 1)
            for k in ("clocks", "higher_is_better", "vs_baseline", "data"):
                d.pop(k, None)
            return d
    return {"error": "no JSON line from the child", "stderr_tail": r.stderr[-600:]}


def reduce_over_ranks(max_vals, sum_vals, device):
    """Whole-job aggregation for N>1: times are the MAX over ranks, work counters the SUM (one all_reduce each)."""
    import torch
    import torch.distributed as dist
    t = torch.tensor(list(max_vals), device=device, dtype=torch.float64)
    w = torch.tensor(list(sum_vals), device=device, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dist.all_reduce(w, op=dist.ReduceOp.SUM)
    return t.tolist(), w.tolist()


# ------------------------------------------------------------------------------------------------ GPU arm
def run_b200(a):
    import torch
    import torch.distributed as dist
    import falkordb_b200 as fb
    from falkordb_b200._lib import lib
    from falkordb_b200.grb import Matrix

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    all_cpus = set(os.sched_getaffinity(0))
    numa = bind_to_gpu_numa_node(local) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    L = lib()
    fb.init()
    fb.set_option("bits_mode", a.bits_mode)
    fb.set_option("pull_mode", a.pull_mode)
    if a.pull_kernel >= 0:
        fb.set_option("pull_kernel", a.pull_kernel)
    for kv in a.opt:
        k, v = kv.split("=")
        fb.set_option(k, int(v))
    n = 1 << a.scale

    # ---- setup (untimed): graph on device, transpose mirror, source batches ----
    t0 = time.time()
    A = fb.rmat(a.scale, a.edge_factor, a.seed)
    A.prepare(True)
    setup_s = time.time() - t0
    nnzA = A.nvals()
    p, _, _ = (np.empty(n + 1, np.uint64), None, None)
    fb.check(L.B200_Matrix_export_CSR(A.h, p.ctypes.data, None, None, 0))
    deg = np.diff(p.astype(np.int64))
    nb = a.steps + a.warmup
    batches = pick_sources(deg, nb, a.sources, a.seed, rank)
    rows = np.arange(a.sources, dtype=np.uint64)
    stream = torch.cuda.ExternalStream(L.B200_stream())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    pull_flops = [0, 0]               # [flops, hops] that took the pull direction (last_path 3), device-resident arm only

    def chain(F, tally=False):
        fl = 0
        for _ in range(a.hops):
            F.lmxm(A)
            f1 = fb.get_stat("last_flops")
            fl += f1
            if tally and fb.get_stat("last_path") == 3:
                pull_flops[0] += f1
                pull_flops[1] += 1
        F.wait()                      # materialise sorted CSR on the device
        return fl

    # ---- device-resident arm: F0 handles pre-built in HBM, dup'ed inside the step ----
    F0 = []
    for b in batches:
        F = Matrix(a.sources, n, bool)
        F.build(rows, b)
        F.wait()
        F0.append(F)
    clocks = ClockSampler(local)
    clocks.start()
    time.sleep(0.3)                   # let nvidia-smi finish its start-up before anything is timed
    for i in range(a.warmup):
        chain(F0[i].dup())
    fb.set_option("timing", 1)
    fb.reset_stats()
    barrier()
    clocks.mark_begin()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    flops = 0
    nnz_out = 0
    last = None
    for i in range(a.warmup, nb):
        F = F0[i].dup()
        flops += chain(F, tally=True)
        nnz_out += F.nvals()
        if a.dump_outputs and rank == 0 and i == nb - 1:
            last = F                  # outlives the timed window only when it is to be written out
        del F
    e1.record(stream)
    barrier()
    clocks.mark_end()
    clk = clocks.stop()
    ms = e0.elapsed_time(e1)
    launches = fb.get_stat("launches")
    kstats = {}
    for name in ("bits_pull", "bits_pull_long", "bits_push", "heavy_accumulate", "bits_fill", "bits_count", "small_rows"):
        m, nl, by = C.c_double(), C.c_uint64(), C.c_uint64()
        if L.B200_kernel_stats(name.encode(), C.byref(m), C.byref(nl), C.byref(by)) == 0 and nl.value:
            kstats[name] = {"ms": m.value, "launches": nl.value, "bytes": by.value}
    fb.set_option("timing", 0)
    if last is not None:
        dump_outputs(a.dump_outputs, last)
        del last

    # ---- e2e arm: host buffers in, host CSR out, through the public C ABI ----
    # the CSR hand-off needs 4 B per result entry of pinned host memory (6-7 GB at 512 sources): only where it is timed
    max_out = int(max(1, nnz_out // max(1, a.steps)) * 1.5) + 1024 if (world == 1 or a.e2e_format == "csr") else 1024
    out_p = torch.empty(a.sources + 1, dtype=torch.int64).pin_memory().numpy().view(np.uint64)
    out_j = torch.empty(max_out, dtype=torch.int32).pin_memory().numpy().view(np.uint32)
    src_pin = [torch.from_numpy(b.astype(np.int64)).pin_memory().numpy().view(np.uint64) for b in batches]
    rows_pin = torch.from_numpy(rows.astype(np.int64)).pin_memory().numpy().view(np.uint64)

    wpr = (n + 63) // 64
    bm_pin = None
    if a.e2e_format != "csr":
        bm_pin = torch.empty(a.sources * wpr, dtype=torch.int64).pin_memory().numpy().view(np.uint64).reshape(a.sources, wpr)

    def hops_only(F):
        fl = 0
        for _ in range(a.hops):
            F.lmxm(A)
            fl += fb.get_stat("last_flops")
        return fl

    def e2e_step(i, fmt):
        """host sources in -> host result out through the public API; returns (flops, nvals, d2h bytes, format)"""
        nonlocal out_j
        if fmt == "bitmap_sliced":             # dense result known from the warm-up: sliced, overlapped hand-off, ONE C call
            fl, _, _ = fb.traverse_batch(src_pin[i], [A] * a.hops, fb.OUT_BITMAP, out_bitmap=bm_pin)   # H2D of the sources inside
            return fl, 0, bm_pin.nbytes, "bitmap"
        if fmt == "csr_c":                     # B200_traverse_batch with the CSR hand-off
            try:
                fl, nv, _ = fb.traverse_batch(src_pin[i], [A] * a.hops, fb.OUT_CSR, out_p=out_p, out_j=out_j)
            except BufferError:
                out_j = torch.empty(int(len(out_j) * 1.5) + 1024, dtype=torch.int32).pin_memory().numpy().view(np.uint32)
                fl, nv, _ = fb.traverse_batch(src_pin[i], [A] * a.hops, fb.OUT_CSR, out_p=out_p, out_j=out_j)
            return fl, nv, 8 * (a.sources + 1) + 4 * nv, "csr"
        F = Matrix(a.sources, n, bool)
        F.build(rows_pin, src_pin[i])          # H2D of the step's inputs inside GxB_Matrix_build_Scalar
        if fmt != "csr":
            fl = hops_only(F)                  # the result stays a device bit-matrix; no CSR is built for a bitmap hand-off
            nv = F.nvals()
            if fmt == "bitmap" or nv * 32 > a.sources * n:
                F.export_bitmap(bm_pin)        # D2H of the result (row-major packed bitmap)
                return fl, nv, bm_pin.nbytes, "bitmap"
            F.wait()
        else:
            fl = chain(F)
            nv = F.nvals()
        if nv > len(out_j):
            out_j = torch.empty(int(nv * 1.2), dtype=torch.int32).pin_memory().numpy().view(np.uint32)
        fb.check(L.B200_Matrix_export_CSR(F.h, out_p.ctypes.data, out_j.ctypes.data, None, 0))  # D2H of the result
        return fl, nv, 8 * (a.sources + 1) + 4 * nv, "csr"

    def e2e_run(fmt, first, last):
        for i in range(a.warmup):
            e2e_step(i, fmt)
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_wall = time.perf_counter()
        f0.record(stream)
        tot_fl, tot_nv, tot_d2h, kinds = 0, 0, 0, set()
        for i in range(first, last):
            fl, nv, by, kind = e2e_step(i, fmt)
            tot_fl += fl
            tot_nv += nv
            tot_d2h += by
            kinds.add(kind)
        f1.record(stream)
        barrier()
        # device clock on the library stream; spans the host-side gaps between calls too
        return f0.elapsed_time(f1), 1e3 * (time.perf_counter() - t_wall), tot_fl, tot_nv, tot_d2h, "+".join(sorted(kinds))

    e2e_fmt = a.e2e_format
    if e2e_fmt != "csr" and a.e2e_subbatches != 1:
        # Matrix.export_auto's rule decides the format on the first batch; a dense result then goes through the sliced call
        if e2e_fmt == "bitmap" or e2e_step(0, "auto")[3] == "bitmap":
            e2e_fmt = "bitmap_sliced"
    e2e_ms, e2e_wall_ms, e2e_flops, e2e_nnz, e2e_d2h, e2e_kind = e2e_run("csr_c" if e2e_fmt == "csr" else e2e_fmt, a.warmup, nb)
    # secondary: the same arm with a CSR hand-off (3 steps), so both interchange formats are on record
    # (N = 1 only: it pins a multi-GB host buffer per rank and is a side note, not a scaling measurement)
    csr_steps = min(a.steps, 3)
    if a.e2e_format == "csr":
        csr_ms, csr_flops, csr_d2h = e2e_ms, e2e_flops, e2e_d2h
    elif world == 1:
        csr_ms, _, csr_flops, _, csr_d2h, _ = e2e_run("csr_c", a.warmup, a.warmup + csr_steps)
    else:
        csr_ms, csr_flops, csr_d2h, csr_steps = 0.0, 0, 0, 0
    if a.e2e_format == "csr":
        csr_steps = a.steps
    # full-size parity property between the two hand-offs: the bitmap of the last step against the CSR of the same sources
    if e2e_kind == "bitmap":
        Fc = Matrix(a.sources, n, bool)
        Fc.build(rows_pin, src_pin[nb - 1])
        chain(Fc)
        nvc = Fc.nvals()
        if nvc > len(out_j):
            out_j = np.empty(nvc, np.uint32)                 # pageable is fine here: this check is outside every timed region
        fb.check(L.B200_Matrix_export_CSR(Fc.h, out_p.ctypes.data, out_j.ctypes.data, None, 0))
        lp = out_p.astype(np.int64)
        pc = np.bitwise_count(bm_pin).sum(axis=1) if hasattr(np, "bitwise_count") else None
        if pc is not None:
            assert np.array_equal(pc.astype(np.int64), np.diff(lp)), "bitmap row populations differ from the CSR row lengths"
        for r in (0, a.sources - 1):
            cols = out_j[lp[r]:lp[r + 1]].astype(np.int64)
            assert np.all((bm_pin[r, cols >> 6] >> (cols & 63).astype(np.uint64)) & np.uint64(1)), "bitmap misses CSR entries"
        del Fc
    else:
        lp = out_p.astype(np.int64)
    # sortedness + checksum property of the last result (size-independent parity property, cheap)
    lastp = lp
    assert lastp[0] == 0 and np.all(np.diff(lastp) >= 0)
    r0 = out_j[lastp[0]:lastp[1]]
    assert np.all(np.diff(r0.astype(np.int64)) > 0), "row 0 of the result is not strictly ascending"

    # ---- reduce over ranks: time = max, work = sum ----
    if world > 1:
        (ms, e2e_ms, csr_ms), w = reduce_over_ranks([ms, e2e_ms, csr_ms], [flops, e2e_flops, launches, nnz_out, e2e_nnz, csr_flops], "cuda")
        flops, e2e_flops, launches, nnz_out, e2e_nnz, csr_flops = [int(x) for x in w]
    # ---- BASELINE configs 5 and 4 next to the chain, as child processes (every rank takes part; rank 0 keeps the lines) ----
    side = {}
    for spec in [x for x in a.side.split(",") if x and x != "none"]:
        name, _, sc = spec.partition(":")
        if name == "bfs":
            side["partitioned_bfs"] = side_workload(a, "bfs", int(sc or 26), ["--bfs-sources", "8", "--warmup", "2", "--bfs-parity", "1"], 1)
        elif name == "triangles":
            side["masked_triangles"] = side_workload(a, "triangles", int(sc or 24), ["--steps", "3", "--warmup", "1", "--tri-parity", "1"], 2)
        elif name in ("delta", "pagerank") and world == 1:      # single-GPU kernels: delta-matrix sync at fold sizes, FP64 mxv / PageRank
            side["delta_sync" if name == "delta" else "pagerank_fp64"] = side_workload(a, name, int(sc or 22), ["--steps", "3", "--warmup", "1"], 3)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = peaks()
    # dominant kernel = the family with the largest accumulated device time
    roof = None
    if kstats:
        dom = max(kstats, key=lambda k: kstats[k]["ms"])
        ks = kstats[dom]
        per_launch_bytes = ks["bytes"] / ks["launches"]
        per_launch_ms = ks["ms"] / ks["launches"]
        ach = per_launch_bytes / (per_launch_ms * 1e-3) / 1e9 if per_launch_ms > 0 else 0.0
        traffic = None
        try:   # dram__bytes_read+write per launch from the committed ncu --set full captures of this configuration
            tj = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
            fam = {"bits_pull": ("k_pull_seg", "k_pull_small"), "bits_fill": ("k_bits_fill_v3",), "bits_push": ("k_csr_push",),
                   "bits_count": ("k_bits_count_csa",)}
            if (tj["config"]["scale"] == a.scale and tj["config"]["sources"] == a.sources and tj["config"]["edge_factor"] == a.edge_factor
                    and dom in fam and not a.opt):
                traffic = int(sum(tj["dram_bytes_by_kernel"][k] for k in fam[dom]))
        except Exception:
            traffic = None
        roof = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "peak_source": peak_src, "traffic": traffic, "launch_ms": per_launch_ms, "launches": ks["launches"],
                "share_of_step": ks["ms"] / ms,
                "algorithmic_bytes_per_launch": per_launch_bytes,
                "basis": "bytes this kernel family must move per launch (DESIGN.md 4.1), not SURVEY 8(d)'s row-wise figure"}
        try:   # explanatory extras: must never take the bench line down
            # every timed family, same arithmetic (the dominant one above is repeated here)
            roof["families"] = {k: {"ms_per_launch": v["ms"] / v["launches"], "achieved_gbs": v["bytes"] / (v["ms"] * 1e-3) / 1e9 if v["ms"] > 0 else 0.0,
                                    "frac": (v["bytes"] / (v["ms"] * 1e-3) / 1e9 / peak) if v["ms"] > 0 else 0.0,
                                    "share_of_step": v["ms"] / ms} for k, v in kstats.items()}
            if "bits_pull" in kstats and pull_flops[1]:
                kp = kstats["bits_pull"]
                pl_ms = kp["ms"] / kp["launches"]
                # SURVEY 8(d) bytes_mxm for the same launches: 4 B per flop (A's col_idx segment re-read for every frontier row) is
                # the dominant term.  The bit-matrix kernel serves 64*W frontier rows per pass over A, so it never moves these bytes.
                sb = 4.0 * pull_flops[0] / pull_flops[1]
                roof["hop_survey_8d"] = {"bytes_per_launch": sb, "achieved": sb / (pl_ms * 1e-3) / 1e9, "unit": "GB/s",
                                         "frac": sb / (pl_ms * 1e-3) / 1e9 / peak}
                # what actually bounds the hop: one L1TEX wavefront (a 128-byte line through the tag stage) per gathered vertex
                # record -- SPLIT lanes share a record -- against one line per clock per SM at the SM clock sampled during the run
                W = max(1, -(-a.sources // 64))
                Wp = 1
                while Wp < W:
                    Wp <<= 1
                parts = max(1, Wp // 4)                      # 32-byte parts per record
                lanes_per_record = parts                      # lane-split kernels: the parts of a record coalesce into ONE wavefront
                wavefronts = nnzA * 1.0 + nnzA * 4.0 / 128.0  # gathers + the coalesced col_idx stream
                ceiling = 148 * (clk.get("sm_mhz") or 1965.0) * 1e6
                roof["hop_gather_ceiling"] = {"wavefronts_per_launch": wavefronts, "achieved_wavefronts_per_s": wavefronts / (pl_ms * 1e-3),
                                              "ceiling_wavefronts_per_s": ceiling, "frac": wavefronts / (pl_ms * 1e-3) / ceiling,
                                              "lanes_per_record": lanes_per_record,
                                              "note": "L1TEX tag stage: one 128-byte line per clock per SM (scripts/ubench/gather*.cu)"}
        except Exception as ex:
            roof["extras_error"] = repr(ex)
    # SURVEY 8d's row-wise formula (4 B per flop dominant) for the whole step, for reference: a frontier kernel that
    # serves 64*W rows per pass over A reads far fewer bytes than this, so this fraction may exceed 1.
    survey_bytes = 4 * flops + 4 * nnz_out
    survey = {"bytes_mxm_formula": survey_bytes, "achieved": survey_bytes / (ms * 1e-3) / 1e9, "unit": "GB/s",
              "frac_of_peak": survey_bytes / (ms * 1e-3) / 1e9 / peak}

    cpu = None
    if not a.no_cpu_baseline and world == 1:      # the CPU baseline is an N=1 measurement (torchrun also pins OMP to 1 thread)
        try:
            import oracle as orc
            from oracle import CSR
            os.sched_setaffinity(0, all_cpus)
            all_threads = host_threads()
            orc.lib().orc_set_num_threads(all_threads)
            pj = np.empty(nnzA, np.uint32)
            fb.check(L.B200_Matrix_export_CSR(A.h, p.ctypes.data, pj.ctypes.data, None, 0))
            Ao = orc.spread(CSR(n, n, p.astype(np.int64), pj))       # pages interleaved over the sockets by first touch
            del pj
            cores, team_probe = calibrate_cpu_threads(orc, Ao, deg, a, all_threads)
            ncpu = a.cpu_sources if a.cpu_sources > 0 else a.sources
            b = batches[a.warmup][:ncpu]
            orc.chain(Ao, b[: min(len(b), cores)], a.hops, keep=False)          # untimed: allocates the per-thread workspaces
            t0 = time.perf_counter()
            _, cfl, cdg, busy = orc.chain(Ao, b, a.hops, keep=False)
            ct = time.perf_counter() - t0
            # parity at FULL size, every row of the batch: the same sources through the GPU path, compared by digest
            # (nvals, sum mix(row, col), sum mix(row, col, CSR position)) -- B200_Matrix_digest vs orc_digest
            G = Matrix(len(b), n, bool)
            G.build(np.arange(len(b), dtype=np.uint64), b)
            gfl = chain(G)
            parity = bool(np.array_equal(G.digest(), cdg) and gfl == cfl)
            del G
            cpu = {"value": cfl / ct, "unit": "edges/s", "cores": cores, "kind": "port",
                   "sample": f"{a.hops}-hop chain for the {len(b)} sources of the first timed batch ({cfl} flops, {ct:.1f} s)",
                   "threads_busy_fraction": busy, "host_threads": all_threads, "team_size_probe_s": team_probe,
                   "algorithm": "Gustavson, one frontier row per task (LPT order), per-thread persistent n-bit accumulators",
                   "full_size_parity_bit_exact": parity, "parity_rows": len(b), "result_digest": [int(x) for x in cdg]}
        except Exception as ex:  # the baseline must never take the bench line down
            cpu = {"value": None, "error": repr(ex)}

    h2d = 16 * a.sources
    d2h = int(e2e_d2h / a.steps)              # per rank: counted from the buffers export_bitmap / export_CSR copy out
    line = {
        "metric": "traversed edges/sec (mxm TEPS), 3-hop ANY_PAIR mxm chain", "value": flops / (ms * 1e-3), "unit": "edges/s",
        "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms / a.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bool/u32 index", "data": "synthetic",
        "config": workload_config(a, n, nnzA, a.sources),
        "options": {"parallelism": f"replicated A, sources sharded x{world}", "numa_node_bound": numa, "bits_mode": a.bits_mode,
                    "pull_mode": a.pull_mode, "opt": list(a.opt), "setup_s": round(setup_s, 2)},
        "flops_per_step": flops / a.steps, "nnz_out_per_step": nnz_out / a.steps,
        "e2e": {"value": e2e_flops / (e2e_ms * 1e-3), "unit": "edges/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_ms / a.steps, "wall_ms_per_step": e2e_wall_ms / a.steps, "result_format": e2e_kind,
                "api": ("B200_traverse_batch (one C-ABI call per batch: host sources in, host result out; %s)"
                        % ("packed bitmap, 128-row slices, D2H overlapped with the next slice's hops" if e2e_fmt == "bitmap_sliced"
                           else "CSR hand-off" if e2e_kind == "csr" else "bitmap hand-off")),
                "csr_handoff": ({"value": csr_flops / (csr_ms * 1e-3), "unit": "edges/s", "steps": csr_steps,
                                 "ms_per_step": csr_ms / csr_steps, "d2h_bytes_per_step": int(csr_d2h / csr_steps)}
                                if csr_steps and csr_ms > 0 else None)},
        "gpu_launches": int(launches), "kernels": kstats, "roofline": roof, "roofline_survey_formula": survey,
        "cpu_baseline": cpu, "clocks": clk}
    line.update(side)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_bfs(a):
    """BASELINE config 5: BFS frontier sweep, adjacency 1-D row-block partitioned over the ranks; the level loop, the direction
    switch and the NCCL exchange (bitmap or sparse vertex lists) run inside the library (B200_bfs_partitioned, csrc/bfs_do.cu).
    TEPS = edges incident to the reached vertices / time (Graph500 convention, SURVEY 8d), summed over sources; time = device
    events inside the call, max over ranks, plus a wall-clock cross-check.  Parity: the levels and min-id parents of the first
    --bfs-parity sources are compared bit for bit with the oracle on the same graph (outside the timed region)."""
    import torch
    import torch.distributed as dist
    import falkordb_b200 as fb
    from falkordb_b200.dist_bfs import PartitionedBfs, partition
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    fb.init()
    for kv in a.opt:
        k, v = kv.split("=")
        fb.set_option(k, int(v))
    n = 1 << a.scale

    def bcast(b):
        box = [b]
        dist.broadcast_object_list(box, src=0)
        return box[0]

    t0 = time.time()
    pb = PartitionedBfs(a.scale, a.edge_factor, a.seed, rank, world, bcast)
    setup_s = time.time() - t0
    # sources: seeded, restricted to vertices with out-edges; owners publish their degrees through one all-reduce
    rng = np.random.default_rng(a.seed * 7919 + 3)
    cand = rng.choice(n, size=(a.bfs_sources + a.warmup) * 8, replace=False)
    degl = pb.local_degrees()
    mine = (cand >= pb.lo) & (cand < pb.hi)
    vals = np.zeros(len(cand), np.int32)
    vals[mine] = (degl[cand[mine] - pb.lo] > 0).astype(np.int32)
    flag = torch.from_numpy(vals).cuda()
    if world > 1:
        dist.all_reduce(flag, op=dist.ReduceOp.MAX)
    srcs = [int(c) for c, f in zip(cand, flag.cpu().numpy()) if f][: a.bfs_sources + a.warmup]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    clocks = ClockSampler(local)
    clocks.start()
    time.sleep(0.3)
    for s_ in srcs[: a.warmup]:
        pb.run(s_)
    barrier()
    fb.reset_stats()
    clocks.mark_begin()
    t0 = time.perf_counter()
    edges = reached = 0
    dev_ms = exch_ms = 0.0
    agg = {"td_levels": 0, "bu_levels": 0, "sparse_levels": 0, "exchanges": 0, "exchanged_bytes": 0}
    depth = 0
    keep = []
    for s_ in srcs[a.warmup:]:
        host = len(keep) < a.bfs_parity               # parity sources come back to the host; the rest stay in HBM
        lv, par, info = pb.run(s_, on_device=not host)
        edges += info["edges"]                       # identical on every rank (replicated degree table)
        depth = max(depth, info["depth"])
        reached += int((lv >= 0).sum())
        dev_ms += info["device_ms"]
        exch_ms += info["exchange_ms"]
        for k in agg:
            agg[k] += info[k]
        if host:
            keep.append((s_, lv.copy(), par.copy()))
    barrier()
    clocks.mark_end()
    secs = time.perf_counter() - t0
    clk = clocks.stop()
    launches = fb.get_stat("launches")
    if world > 1:
        (secs, dev_ms, exch_ms), (reached, launches) = reduce_over_ranks([secs, dev_ms, exch_ms], [reached, launches], "cuda")
    # ---- parity (untimed): rank 0 regenerates the whole graph on its GPU, exports it, runs the oracle ----
    parity = None
    if a.bfs_parity > 0:
        good = True
        full = []
        for s_, lv, par in keep:
            if world > 1:
                block = partition(n, 0, world)[1]
                pad = torch.full((2, block), -1, dtype=torch.int64, device="cuda")
                pad[0, : len(lv)] = torch.from_numpy(lv).cuda()
                pad[1, : len(par)] = torch.from_numpy(par).cuda()
                out = torch.empty((world, 2, block), dtype=torch.int64, device="cuda")
                dist.all_gather_into_tensor(out.view(-1), pad.view(-1))
                full.append((s_, out[:, 0, :].reshape(-1)[:n].cpu().numpy(), out[:, 1, :].reshape(-1)[:n].cpu().numpy()))
            else:
                full.append((s_, lv, par))
        if rank == 0:
            import oracle as orc
            orc.lib().orc_set_num_threads(len(os.sched_getaffinity(0)))
            pb_A = fb.rmat(a.scale, a.edge_factor, a.seed)
            p_, j_, _ = pb_A.export_csr()
            del pb_A
            Ao = orc.CSR(n, n, p_.astype(np.int64), j_)
            for s_, lv, par in full:
                wl, wp = orc.bfs(Ao, s_)
                good = good and bool(np.array_equal(lv, wl) and np.array_equal(par, wp))
            parity = {"sources_checked": len(full), "levels_and_min_parents_bit_exact": good}
    pb.close()
    if rank == 0:
        k = len(srcs) - a.warmup
        print(json.dumps({
            "metric": "traversed edges/sec (BFS sweep, Graph500 TEPS)", "value": edges / (dev_ms * 1e-3), "unit": "edges/s", "n_gpus": world,
            "steps": k, "warmup": a.warmup, "ms_per_step": dev_ms / max(1, k), "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "bool/u32 index", "data": "synthetic",
            "config": {"workload": f"BFS level+parent sweep, RMAT scale-{a.scale} ef{a.edge_factor}, {k} sources", "n": n,
                       "parallelism": f"1-D row-block partition x{world}; per level one NCCL all-gather on the library stream: n-bit bitmaps "
                                      "(top-down: discovered sets, bottom-up: owned slices) or sentinel-padded vertex lists while the "
                                      "frontier's out-edges number < n/32",
                       "max_depth": depth, "setup_s": round(setup_s, 2)},
            "wall_ms_per_step": 1e3 * secs / max(1, k), "edges_per_bfs": edges / max(1, k), "reached_per_bfs": reached / max(1, k),
            "levels": {kk: agg[kk] / max(1, k) for kk in ("td_levels", "bu_levels", "sparse_levels")},
            "collective": {"name": "ncclAllGather (uint8) on the library stream", "calls_per_bfs": agg["exchanges"] / max(1, k),
                           "us_per_call": (1e3 * exch_ms / agg["exchanges"]) if agg["exchanges"] else None,
                           "share_of_bfs_time": exch_ms / dev_ms if dev_ms else None,
                           "bytes_per_bfs": agg["exchanged_bytes"] / max(1, k)},
            "parity": parity, "gpu_launches": int(launches), "clocks": clk}))
    if world > 1:
        dist.destroy_process_group()


def triangle_row_cuts(lp, lj, world):
    """Row blocks of L with equal WORK for C<L> = L*L, not equal rows (tril(L) of an RMAT graph is heavily skewed: equal-row blocks
    gave 43 % strong-scaling efficiency at N = 4).  What a pair (i, k) of L costs the kernel: the shorter of L(k,:) and L(i,:) drives
    the intersection (ewise.cu: k_masked_pairs), plus a fixed part.  Every rank derives the same cuts from the replicated L.
    Returns (cuts[world + 1], work per block)."""
    n = len(lp) - 1
    degL = np.diff(lp)
    rows_of = np.repeat(np.arange(n, dtype=np.int64), degL)
    work = np.minimum(degL[lj], degL[rows_of]) + 8
    del rows_of
    csum = np.concatenate([[0], np.cumsum(work, dtype=np.int64)])
    rowwork_cum = csum[lp]                                     # work of rows [0, i)
    total_w = int(rowwork_cum[-1])
    cuts = [int(np.searchsorted(rowwork_cum, total_w * g // world, side="left")) for g in range(world + 1)]
    cuts[0], cuts[-1] = 0, n
    per_block = [int(rowwork_cum[cuts[g + 1]] - rowwork_cum[cuts[g]]) for g in range(world)]
    return cuts, per_block


def run_triangles(a):
    """BASELINE config 4: masked ExpandInto SpGEMM, C<L,struct,replace> = L*L over ANY_PAIR with L = tril(A u A') of the
    RMAT graph: which edges close at least one wedge.  Row blocks of the OUTPUT are independent (mask and left operand
    are row-local), so ranks take row blocks of L as the left operand / mask with L replicated as the right operand and
    no exchange.  TEPS = flops / time with flops = sum_{(i,k) in L_block} deg_L(k) (SURVEY 8d)."""
    import torch
    import torch.distributed as dist
    import ctypes as C
    import falkordb_b200 as fb
    from falkordb_b200._lib import lib, check, P
    from falkordb_b200.grb import Matrix, Descriptor
    from falkordb_b200.dist_bfs import partition
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    fb.init()
    fb.set_option("bits_mode", 0)
    n = 1 << a.scale
    L_ = lib()
    h = P()
    check(L_.B200_Matrix_rmat_block(C.byref(h), a.scale, a.edge_factor, a.seed, 0, n, 2))
    Lfull = Matrix(0, 0, bool, _handle=h)
    # row blocks of equal WORK, not equal rows: tril(L) is heavily skewed
    # (equal-row blocks gave 43 % strong-scaling efficiency at N = 4); every rank derives the same split from the replicated L
    lp, lj, _ = Lfull.export_csr()
    lp = lp.astype(np.int64)
    cuts, _ = triangle_row_cuts(lp, lj, world)
    lo, hi = cuts[rank], cuts[rank + 1]
    del lj
    if world > 1:
        hb = P()
        check(L_.B200_Matrix_rmat_block(C.byref(hb), a.scale, a.edge_factor, a.seed, lo, hi, 2))
        Lblk = Matrix(0, 0, bool, _handle=hb)
    else:
        Lblk = Lfull
    stream = torch.cuda.ExternalStream(L_.B200_stream())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    last = {}

    def step():
        Cm = Matrix(hi - lo, n, bool)
        Cm.mxm(Lblk, Lfull, Lblk, Descriptor.RS)
        fl = fb.get_stat("last_flops")
        last["C"] = Cm
        return fl, Cm.nvals()

    for _ in range(a.warmup):
        step()
    barrier()
    fb.set_option("timing", 1)
    fb.reset_stats()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    flops = nnz = 0
    for _ in range(a.steps):
        fl, nv = step()
        flops += fl
        nnz += nv
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    launches = fb.get_stat("launches")
    peak, peak_src = peaks()
    roofs = kernel_rooflines(L_, ("spgemm_masked", "filter"), peak)
    fb.set_option("timing", 0)
    my_ms = ms
    # parity at full size (untimed): this rank's block of the result against the oracle's masked product of the same rows
    parity = None
    if a.tri_parity:
        import oracle as orc
        orc.lib().orc_set_num_threads(max(1, host_threads() // world))
        Lo = orc.CSR(n, n, lp, Lfull.export_csr()[1])
        pb_, jb_ = lp[lo:hi + 1] - lp[lo], Lo.j[lp[lo]:lp[hi]]
        Lb = orc.CSR(hi - lo, n, pb_, jb_)
        want, wfl = orc.mxm(Lb, Lo, Lb, 1, return_flops=True)
        ok = bool(np.array_equal(last["C"].digest(), orc.digest(want)) and wfl * a.steps == flops)
        del want
        flag = torch.tensor([1 if ok else 0], device="cuda")
        if world > 1:
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        parity = {"digest_and_flops_bit_exact_every_rank": bool(flag.item())}
    if world > 1:
        (ms,), (flops, nnz, launches) = reduce_over_ranks([ms], [flops, nnz, launches], "cuda")
    if rank == 0:
        print(json.dumps({
            "parity": parity, "kernels_rank0": roofs, "peak_gbs": peak, "rank0_ms_per_step": my_ms / a.steps,
            "row_cuts": cuts if world <= 8 else None,
            "metric": "traversed edges/sec (masked mxm TEPS, C<L> = L*L)", "value": flops / (ms * 1e-3), "unit": "edges/s",
            "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms / a.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "bool/u32 index", "data": "synthetic",
            "config": {"workload": f"masked SpGEMM C<L,struct> = L*L, L = tril(A u A'), RMAT scale-{a.scale} ef{a.edge_factor}",
                       "n": n, "nnz_L": Lfull.nvals(), "parallelism": f"row blocks of L with equal intersection work x{world}, L replicated, no exchange"},
            "flops_per_step": flops / a.steps, "nnz_out_per_step": nnz / a.steps, "gpu_launches": int(launches)}))
    if world > 1:
        dist.destroy_process_group()


def kernel_rooflines(L, names, peak):
    """per kernel family: event-timed ms / launches / algorithmic bytes (B200_kernel_stats) -> achieved GB/s and fraction of peak"""
    out = {}
    for name in names:
        m, nl, by = C.c_double(), C.c_uint64(), C.c_uint64()
        if L.B200_kernel_stats(name.encode(), C.byref(m), C.byref(nl), C.byref(by)) == 0 and nl.value:
            ach = by.value / (m.value * 1e-3) / 1e9 if m.value > 0 else 0.0
            out[name] = {"ms_per_launch": m.value / nl.value, "launches": nl.value, "algorithmic_bytes_per_launch": by.value / nl.value,
                         "achieved_gbs": ach, "frac_of_hbm_peak": ach / peak}
    return out


def run_delta(a):
    """Delta-matrix sync (SURVEY 8a rows a5-a8; fold formulas versioned_matrix.rs:909-926) at fold sizes: base m = RMAT scale-S
    adjacency (S = --scale, default 23: 1.3e8 entries), dp = 1e6 fresh entries, dm = 1e6 tombstones sampled from m.
      fold      : C<!dm, replace> = m (+) dp           GrB_Matrix_eWiseAdd_BinaryOp with GrB_DESC_RC      (matrix.rs:852-874)
      select    : C<!dm, replace> = m                  GrB_transpose(.., GrB_DESC_RCT0)                  (matrix.rs:824-845)
      tombstone : C = dm (*) m                          GrB_Matrix_eWiseMult_Semiring                     (matrix.rs:876-896)
      transpose : C = m'                                GrB_transpose                                     (matrix.rs:633-662)
    Each is bit-exact against the oracle on a scale-16 instance of the same construction before the timed runs."""
    import torch
    import falkordb_b200 as fb
    import oracle as orc
    from falkordb_b200._lib import lib
    from falkordb_b200.grb import Matrix, Descriptor
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    fb.init()
    L = lib()
    peak, peak_src = peaks()

    def make(scale, ndelta, seed):
        A = fb.rmat(scale, a.edge_factor, seed)
        n = 1 << scale
        p, j, _ = A.export_csr()
        rng = np.random.default_rng(seed + 99)
        pick = np.sort(rng.choice(len(j), size=min(ndelta, len(j)), replace=False))
        rows = (np.searchsorted(p.astype(np.int64), pick, side="right") - 1).astype(np.uint64)
        dm = Matrix(n, n, bool)
        dm.build(rows, j[pick].astype(np.uint64))
        dp = Matrix(n, n, bool)
        dp.build(rng.integers(0, n, ndelta).astype(np.uint64), rng.integers(0, n, ndelta).astype(np.uint64))
        for M_ in (A, dm, dp):
            M_.wait()
        return A, dp, dm, n, (p, j)

    def ops(A, dp, dm, n):
        C1 = Matrix(n, n, bool); C1.element_wise_add(dm, A, dp, Descriptor.RC)
        C2 = Matrix(n, n, bool); C2.select(dm, A)
        C3 = Matrix(n, n, bool); C3.element_wise_multiply(None, dm, A, None)
        C4 = A.transpose()
        return C1, C2, C3, C4

    # parity first (small instance, same construction)
    A, dp, dm, n, (p, j) = make(16, 4000, a.seed)
    Ao = orc.CSR(n, n, p.astype(np.int64), j)
    pd, jd, _ = dp.export_csr(); pm, jm, _ = dm.export_csr()
    dpo, dmo = orc.CSR(n, n, pd.astype(np.int64), jd), orc.CSR(n, n, pm.astype(np.int64), jm)
    got = ops(A, dp, dm, n)
    want = (orc.mask_assign(None, orc.ewise_add(Ao, dpo), dmo, comp=True, structural=False, replace=True),
            orc.mask_assign(None, Ao, dmo, comp=True, structural=False, replace=True), orc.ewise_mult(dmo, Ao), orc.transpose(Ao))
    parity = all(np.array_equal(g.digest(), orc.digest(w)) for g, w in zip(got, want))
    del A, dp, dm, got
    # timed
    scale = a.scale if a.scale != 24 else 23
    A, dp, dm, n, _ = make(scale, 1_000_000, a.seed)
    for _ in range(a.warmup):
        ops(A, dp, dm, n)
    fb.set_option("timing", 1)
    fb.reset_stats()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        ops(A, dp, dm, n)
    fb.sync()
    secs = time.perf_counter() - t0
    roofs = kernel_rooflines(L, ("union", "filter", "transpose"), peak)
    fb.set_option("timing", 0)
    print(json.dumps({"metric": "delta-sync kernels: achieved GB/s on SURVEY 8(d) algorithmic bytes", "value": max((r["achieved_gbs"] for r in roofs.values()), default=0.0),
                      "unit": "GB/s", "n_gpus": 1, "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * secs / a.steps, "higher_is_better": True,
                      "dtype": "bool/u32 index", "data": "synthetic",
                      "config": {"workload": f"fold / select / tombstone / transpose, m = RMAT scale-{scale} ef{a.edge_factor} ({A.nvals()} entries), |dp| = |dm| = 1e6"},
                      "kernels": roofs, "peak_gbs": peak, "peak_source": peak_src, "parity_bit_exact_scale16": parity,
                      "gpu_launches": int(fb.get_stat("launches"))}))


def run_pagerank(a):
    """algo.pageRank's LAGr_PageRank (algo_procedures.rs:744-752: damping 0.85, tol 1e-4, itermax 100) on the RMAT graph; the FP64
    plus_second mxv is the kernel; scores against the oracle (rel 1e-9) at --scale <= 22."""
    import ctypes as CT
    import torch
    import falkordb_b200 as fb
    import oracle as orc
    from falkordb_b200._lib import lib, P
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    fb.init()
    L = lib()
    peak, peak_src = peaks()
    scale = a.scale if a.scale != 24 else 22
    A = fb.rmat(scale, a.edge_factor, a.seed)
    n = 1 << scale
    p, j, _ = A.export_csr()
    G, h = P(), P(A.h.value)
    A.h = P()
    assert L.LAGraph_New(CT.byref(G), CT.byref(h), 1, None) == 0
    L.LAGraph_Cached_AT(G, None)

    def once():
        cen, it = P(), CT.c_int(0)
        assert L.LAGr_PageRank(CT.byref(cen), CT.byref(it), G, 0.85, 1e-4, 100, None) == 0
        return cen, it.value

    for _ in range(a.warmup):
        c, _ = once(); L.GrB_Vector_free(CT.byref(c))
    fb.set_option("timing", 1)
    fb.reset_stats()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        cen, iters = once()
        if _ + 1 < a.steps:
            L.GrB_Vector_free(CT.byref(cen))
    secs = time.perf_counter() - t0
    roofs = kernel_rooflines(L, ("mxv_fp64",), peak)
    fb.set_option("timing", 0)
    nv = CT.c_uint64(n)
    X = np.empty(n, np.float64)
    fb.check(L.GrB_Vector_extractTuples_FP64(None, X.ctypes.data, CT.byref(nv), cen))
    Ao = orc.CSR(n, n, p.astype(np.int64), j)
    orc.lib().orc_set_num_threads(host_threads())
    t0 = time.perf_counter()
    want, wit = orc.pagerank(Ao, float(np.float32(0.85)), float(np.float32(1e-4)), 100)
    cpu_s = time.perf_counter() - t0
    rel = float(np.max(np.abs(X - want) / np.maximum(np.abs(want), 1e-300)))
    nnz = int(p[-1])
    print(json.dumps({"metric": "PageRank edges/sec (nnz * iterations / time)", "value": nnz * iters / (secs / a.steps), "unit": "edges/s", "n_gpus": 1,
                      "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * secs / a.steps, "higher_is_better": True, "dtype": "f64", "data": "synthetic",
                      "config": {"workload": f"LAGr_PageRank(0.85, 1e-4, 100) on RMAT scale-{scale} ef{a.edge_factor}", "n": n, "nnz": nnz, "iterations": iters},
                      "kernels": roofs, "peak_gbs": peak, "peak_source": peak_src,
                      "parity": {"max_rel_err_vs_oracle": rel, "tolerance": 1e-9, "iterations_equal": iters == wit, "ok": bool(rel < 1e-9 and iters == wit)},
                      "cpu_baseline": {"value": nnz * wit / cpu_s, "unit": "edges/s", "cores": host_threads(), "kind": "port"},
                      "gpu_launches": int(fb.get_stat("launches"))}))


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "bfs":
        run_bfs(args)
    elif args.workload == "triangles":
        run_triangles(args)
    elif args.workload == "delta":
        run_delta(args)
    elif args.workload == "pagerank":
        run_pagerank(args)
    else:
        run_b200(args)
