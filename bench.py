#!/usr/bin/env python3
"""bench.py -- the driver's measurement contract for stract_b200.

Headline metric (BASELINE.json): webgraph edges/sec per centrality iteration, on configs[1]
(50M-node / 1B-edge R-MAT host graph, harmonic centrality to convergence on 1xB200; with --gpus N the
same graph is destination-row partitioned over N GPUs = configs[2]).  A "step" is one complete
HarmonicCentrality computation (reset + all HyperBall iterations to convergence) on the graph
resident in HBM; value = kept_edges x iterations / device time.  `e2e` is the same metric through the
C-ABI call sequence a Rust shim makes (sb200_graph_create from HOST buffers -> run -> result to host),
host<->device copies and the on-device CSR staging inside the timed region.

Parity is part of the line: at N = 1 the CPU oracle (oracle/, test infrastructure) computes the SAME
full-size graph on all host threads and its registers / ids / centralities are compared bit for bit
with the GPU's (`parity.c2`); that run is also the `cpu_baseline` (median of 3).  At N > 1 every rank's
register replica and the union of the owned results are compared with the hashes frozen from that
check (tests/golden/path1_c2.json).  BASELINE configs[0] (100k / 1M, the reference's own CPU case)
runs on the GPU as `c1` and is checked against tests/golden/path1_c1.json.  BM25 postings/sec
(configs[3], configs[4]) is reported under "bm25" with its own parity objects (bench_bm25.py).

  python bench.py [--gpus N] [--steps K] [--warmup W]            our CUDA path
  python bench.py --impl reference ...                          the reference's CPU path (oracle port)
  python bench.py --dump-outputs DIR ...                        also write the last timed step's result as DIR/*.npy
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "webgraph_edges_per_sec_per_centrality_iter"
UNIT = "edges/s"
GOLDEN_C2 = os.path.join(ROOT, "tests", "golden", "path1_c2.json")
GOLDEN_C1 = os.path.join(ROOT, "tests", "golden", "path1_c1.json")


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


def workload_config(nodes, edges, kept, n_nodes, iters):
    """The `config` object: identical for every arm and every N (the driver compares the arms on it)."""
    return {"workload": f"webgraph harmonic centrality (HyperBall) to convergence, R-MAT(0.57,0.19,0.19,0.05) {nodes} nodes / "
                        f"{edges} edges, seed 42 (BASELINE configs[1]; with --gpus N the same graph partitioned over N GPUs = configs[2])",
            "kept_edges": kept, "n_nodes": n_nodes, "iterations_per_step": iters,
            "l2_policy": "inputs >> L2: 2 x 1.8 GB register arrays + 3.6 GB CSR per iteration, no flush needed"}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu)], stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, reasons, mx = [], set(), None
        try:
            for line in open(self.path):
                c = [x.strip() for x in line.split(",")]
                if len(c) < 9:
                    continue
                try:
                    sm.append(float(c[1])); mx = float(c[2])
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            sm.sort()
            out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))
        return out


# ------------------------------------------------------------------------------------------------
# result fingerprints (shared by the N = 1 oracle check, the golden file and the N > 1 check)
def sha(a):
    import numpy as np
    return hashlib.sha256(memoryview(np.ascontiguousarray(a)).cast("B")).hexdigest()


def result_checksum(ids_lo, ids_hi, values):
    """Order-independent 64-bit checksum of {(id, centrality)}: a wrapping sum of a mixed word per entry, so the owned
    shares of several ranks add up to the checksum of the whole result."""
    import numpy as np
    with np.errstate(over="ignore"):
        z = (np.asarray(ids_lo, np.uint64) * np.uint64(0x9E3779B97F4A7C15)) ^ (np.asarray(ids_hi, np.uint64) * np.uint64(0xC2B2AE3D27D4EB4F))
        z ^= np.asarray(values, np.float64).view(np.uint64) * np.uint64(0x165667B19E3779F9)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z ^= z >> np.uint64(31)
        return int(z.sum(dtype=np.uint64))


def registers_checksum(regs, owned=None):
    """Wrapping 64-bit sum over (owned) nodes of a mixed word of (position in id order, the node's 64 registers): the owned
    shares of several ranks add up to the checksum of the whole register array."""
    import numpy as np
    a = np.ascontiguousarray(regs).view(np.uint64).reshape(-1, 8)
    with np.errstate(over="ignore"):
        z = np.arange(a.shape[0], dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15)
        for j in range(8):
            z = (z ^ a[:, j]) * np.uint64(0xBF58476D1CE4E5B9)
            z ^= z >> np.uint64(29)
        if owned is not None:
            z = z[np.asarray(owned).astype(bool)]
        return int(z.sum(dtype=np.uint64))


def _i64(x):
    return x - (1 << 64) if x >= (1 << 63) else x


DUMP_MAX_ENTRIES = 1 << 20   # 40 bytes per result entry (f64 centrality + 4 x f64 id words): 40 MB at most
DUMP_SEED = 20240917


def dump_outputs(out_dir, ids_lo, ids_hi, values, stats):
    """--dump-outputs: what one HarmonicCentrality step hands its caller, as .npy files that two builds can be compared on.
    centrality.npy (f64) and node_ids.npy (f64, the u128 id as four exact 32-bit words, low word first) hold the result
    entries, or a fixed seeded sample of DUMP_MAX_ENTRIES of them (same positions for the same result length);
    n_changed.npy (f64) holds the changed-node count of every iteration."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    k = len(values)
    idx = np.arange(k)
    if k > DUMP_MAX_ENTRIES:
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(k, DUMP_MAX_ENTRIES, replace=False))
    words = np.stack([np.asarray(ids_lo)[idx], np.asarray(ids_hi)[idx]], axis=1).astype(np.uint64).view(np.uint32)
    np.save(os.path.join(out_dir, "centrality.npy"), np.asarray(values, np.float64)[idx])
    np.save(os.path.join(out_dir, "node_ids.npy"), words.astype(np.float64))
    np.save(os.path.join(out_dir, "n_changed.npy"), np.array([s["n_changed"] for s in stats], np.float64))


def host_threads():
    """Threads the CPU legs may use: the cores this process is allowed to run on (affinity mask, cgroup CPU quota), not the
    machine's core count -- a GPU lease is often a slice of a bigger host."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]))))
            else:
                q = int(txt[0])
                if q > 0:
                    period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, q // period))
        except (OSError, ValueError, IndexError):
            pass
    return max(1, n)


def _np_u64(t):
    """numpy uint64 view of a host torch tensor / numpy array (no copy)."""
    import numpy as np
    a = t.numpy() if hasattr(t, "numpy") else np.asarray(t)
    return a.view(np.uint64)


# ------------------------------------------------------------------------------------------------
def oracle_c2(cols_host, threads, runs=3, budget_s=150.0):
    """The dense CPU restatement on the full graph: all-threads staging, `runs` timed iteration loops (median),
    final registers / result kept for the comparison.  Returns (oracle handle, info dict)."""
    import numpy as np
    import oracle
    a = [_np_u64(c) for c in cols_host]
    t0 = time.perf_counter()
    o = oracle.DenseHyperBall(*a, threads=threads, mt=True)
    stage_s = time.perf_counter() - t0
    loops, iters = [], 0
    t_all = time.perf_counter()
    for i in range(runs):
        if i:
            o.reset()
        t1 = time.perf_counter()
        iters = o.run()
        loops.append(time.perf_counter() - t1)
        if time.perf_counter() - t_all + loops[-1] > budget_s:
            break
    kept = o.n_edges - o.num_self_loops()
    med = float(np.median(loops))
    return o, {"kept_edges": kept, "n_nodes": o.n_nodes, "iterations": iters, "stage_s": round(stage_s, 2),
               "loop_s": [round(x, 3) for x in loops], "median_loop_s": med, "value": kept * iters / med}


def run_reference(args):
    """--impl reference: the reference's CPU path on this box's host cores.  The reference is Rust (no toolchain in
    this image), so what runs is the oracle port.  Headline = the dense port on ALL host threads over the SAME full
    workload as the GPU arm (a generous stand-in: harmonic.rs:129-154 itself is one sequential iterator over ordered
    maps); `c1` = the structure-faithful single-threaded port on BASELINE configs[0] exactly, which is the case the
    reference's own CPU path is quoted on.  A step = one complete calculate() loop on the staged graph."""
    import numpy as np
    import oracle
    import psutil
    threads = host_threads()
    nodes, edges, scale = args.nodes, args.edges, args.scale
    need = edges * 40 + edges * 36 + 20e9   # edge stream + staging transients + state
    avail = psutil.virtual_memory().available
    note = "full workload"
    if avail < need:
        f = 1
        while (edges // f) * 76 + 20e9 / f > avail and f < 4096:
            f *= 2
        nodes, edges = max(nodes // f, 1000), edges // f
        scale = max(1, int(np.ceil(np.log2(nodes))))
        note = f"host RAM {avail / 2**30:.0f} GiB too small for the 10^9-edge stream: scaled 1/{f}"
    t0 = time.perf_counter()
    d = oracle.synth_edges(1, nodes, edges, seed=42, scale=scale, threads=threads)
    gen_s = time.perf_counter() - t0
    cols = [d["from_lo"], d["from_hi"], d["to_lo"], d["to_hi"], d["rel_flags"]]
    t0 = time.perf_counter()
    o = oracle.DenseHyperBall(*cols, threads=threads, mt=True)
    stage_s = time.perf_counter() - t0
    del d, cols
    kept = o.n_edges - o.num_self_loops()
    budget = args.ref_budget_s
    warm = 0
    t_all = time.perf_counter()
    iters = o.run()
    first = time.perf_counter() - t_all
    if args.warmup > 0:
        warm = 1
    loops = [] if warm else [first]
    while len(loops) < args.steps and (time.perf_counter() - t_all) + first < budget:
        o.reset()
        t1 = time.perf_counter()
        iters = o.run()
        loops.append(time.perf_counter() - t1)
    if not loops:
        loops, warm = [first], 0
    dt = float(np.mean(loops))
    value = kept * iters / dt
    r = o.result()
    fp = {"n_positive": int(len(r["centrality"])), "result_checksum": result_checksum(r["ids_lo"], r["ids_hi"], r["centrality"])}
    n_nodes = o.n_nodes
    o.close()
    # configs[0] exactly: the structure-faithful port, one thread, 20-iteration cap
    u = oracle.synth_edges(0, 100_000, 1_000_000, seed=42, scale=0, threads=threads)
    ua = (u["from_lo"], u["from_hi"], u["to_lo"], u["to_hi"], u["rel_flags"])
    t1 = time.perf_counter()
    fr = oracle.hyperball_faithful(*ua, max_iters=20)
    c1_s = time.perf_counter() - t1
    c1_dense = oracle.DenseHyperBall(*ua)
    c1_kept = c1_dense.n_edges - c1_dense.num_self_loops()
    c1_dense.close()
    c1 = {"workload": "BASELINE configs[0]: uniform 100000 nodes / 1000000 edges, seed 42, <= 20 iterations", "kind": "port",
          "structure": "faithful (ordered maps keyed by u128, heap vector per counter, deep clone per iteration, bloom frontier)",
          "cores": 1, "kept_edges": c1_kept, "iterations": fr["iters"], "ms_per_step": c1_s * 1e3, "value": c1_kept * fr["iters"] / c1_s, "unit": UNIT,
          "centrality_sha256": sha(fr["centrality"])}
    sample = (f"{note}: R-MAT {nodes} nodes / {edges} edges, oracle dense port on {threads} threads, graph staged in RAM "
              f"({stage_s:.1f} s, untimed like the GPU arm's staging), {len(loops)} timed calculate() loops of {iters} iterations "
              f"(requested {args.steps}; bounded by a {budget:.0f} s budget), {warm} warm-up")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": len(loops),
            "warmup": warm, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(args.nodes, args.edges, kept, n_nodes, iters) if note == "full workload" else
                      {"workload": f"webgraph harmonic centrality (HyperBall), R-MAT {nodes} nodes / {edges} edges -- {note}",
                       "kept_edges": kept, "n_nodes": n_nodes, "iterations_per_step": iters},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                             "loop_s": [round(x, 3) for x in loops], "gen_s": round(gen_s, 1), "stage_s": round(stage_s, 1)},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "fingerprint": fp, "c1": c1, "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
def gen_device_graph(torch, L, dev_index, nodes, edges, scale, kind=1):
    from stract_b200._lib import check
    t = [torch.empty(edges, dtype=torch.int64, device=f"cuda:{dev_index}") for _ in range(5)]
    CH = 1 << 27
    for first in range(0, edges, CH):
        cnt = min(CH, edges - first)
        check(L.sb200_synth_edges(kind, nodes, first, cnt, 42, scale, dev_index, *(x.data_ptr() + first * 8 for x in t)))
    return t


def run_c1(torch, device, reps=10):
    """BASELINE configs[0] (100k nodes / 1M edges, <= 20 iterations) on the GPU through the host-buffer C-ABI sequence,
    checked against the frozen oracle output (tests/golden/path1_c1.json)."""
    import numpy as np
    from stract_b200 import synth
    from stract_b200.webgraph import DeviceGraph, HarmonicCentrality, Webgraph
    d = synth.uniform_graph(100_000, 1_000_000, 42)
    g = Webgraph.from_arrays(d["from_lo"], d["from_hi"], d["to_lo"], d["to_hi"], d["rel_flags"])
    for _ in range(2):
        r = HarmonicCentrality.calculate(g, device=device, max_iters=20)
    t0 = time.perf_counter()
    for _ in range(reps):
        r = HarmonicCentrality.calculate(g, device=device, max_iters=20)
    e2e_ms = (time.perf_counter() - t0) / reps * 1e3
    dg = DeviceGraph(g, device=device)
    for _ in range(3):
        dg.reset(); dg.run(20)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(reps):
        dg.reset(); iters, _ = dg.run(20)
    ev1.record(); torch.cuda.synchronize()
    dev_ms = ev0.elapsed_time(ev1) / reps
    regs = dg.registers()
    kept = dg.info()["n_edges_kept"]
    dg.close()
    gold = json.load(open(GOLDEN_C1))
    ok = {"iterations": r.iterations == gold["iterations"], "registers": sha(regs) == gold["registers_sha256"],
          "ids": sha(r.ids_lo) == gold["ids_lo_sha256"] and sha(r.ids_hi) == gold["ids_hi_sha256"],
          "centrality": sha(r.values) == gold["centrality_sha256"]}
    return {"workload": "BASELINE configs[0]: uniform 100000 nodes / 1000000 edges, seed 42, <= 20 iterations",
            "kept_edges": kept, "iterations": r.iterations, "ms_per_step": dev_ms, "value": kept * r.iterations / (dev_ms * 1e-3), "unit": UNIT,
            "e2e_ms_per_step": e2e_ms, "e2e_value": kept * r.iterations / (e2e_ms * 1e-3),
            "parity": {"against": "tests/golden/path1_c1.json (frozen oracle output)", "equal": ok, "green": all(ok.values())},
            "centrality_sha256": sha(r.values)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--nodes", type=int, default=50_000_000)
    ap.add_argument("--edges", type=int, default=1_000_000_000)
    ap.add_argument("--scale", type=int, default=26)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true", help="skip the full-size oracle run (parity + cpu_baseline)")
    ap.add_argument("--no-bm25", action="store_true")
    ap.add_argument("--no-c1", action="store_true")
    ap.add_argument("--no-p2p", action="store_true", help="multi-GPU: NCCL byte-max all-reduce exchange instead of the fused peer-memory stores")
    ap.add_argument("--exchange", default="auto", choices=["auto", "p2p", "symm", "multicast"],
                    help="multi-GPU fused exchange transport: CUDA IPC peer mappings, torch symmetric memory unicast, or NVSwitch "
                         "multicast stores; auto (default) = multicast from 8 GPUs up (measured: 16.9 vs 27.0 ms per step at N = 8, "
                         "profiles/r02_trip10_8gpu_sweep.log), CUDA IPC peer stores + device-side barrier below, and whenever the "
                         "multicast binding is not available")
    ap.add_argument("--sweep", action="store_true", help="N>1: time the exchange variants (side-stream CTAs, subscriber filter, owned item "
                    "list, NVSwitch multicast) on one staged graph in one process and print one JSON line; no bench line")
    ap.add_argument("--ref-budget-s", type=float, default=170.0, help="--impl reference: wall budget of the timed loops")
    ap.add_argument("--write-golden", action="store_true", help="N=1, after a green oracle check: rewrite tests/golden/path1_c2.json")
    ap.add_argument("--dump-outputs", metavar="DIR", help="N=1: write the last timed step's result (sampled to <= 40 MB) as DIR/*.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 0)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and (world > 1 or args.impl != "ours"):
        ap.error("--dump-outputs is supported for the 1-GPU CUDA path only")

    if args.impl == "reference":
        if rank == 0:
            run_reference(args)
        return 0

    import numpy as np
    import torch
    import torch.distributed as dist
    from stract_b200 import kernel_launch_count, lib
    from stract_b200.webgraph import DeviceGraph, HarmonicCentrality, Webgraph

    assert torch.cuda.is_available(), "bench.py needs a GPU (the product path has no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L = lib()
    peaks, peak_src = _peaks()
    full_size = args.nodes == 50_000_000 and args.edges == 1_000_000_000 and args.scale == 26
    if os.environ.get("SB200_BENCH_FINGERPRINT"):   # flow tests: compare N > 1 runs of another graph with this fingerprint file
        global GOLDEN_C2
        GOLDEN_C2 = os.environ["SB200_BENCH_FINGERPRINT"]
        full_size = True

    nodes, edges = args.nodes, args.edges
    tg = time.perf_counter()
    cols = gen_device_graph(torch, L, local_rank, nodes, edges, args.scale)
    torch.cuda.synchronize()
    gen_s = time.perf_counter() - tg
    graph = Webgraph.from_arrays(*cols)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    result = {}
    parity = {}
    W = max(args.warmup, 3)
    if world == 1:
        dg = DeviceGraph(graph, device=local_rank)
        info = dg.info()
        E = info["n_edges_kept"]

        def one_step():
            dg.reset()
            return dg.run()
        for _ in range(W):
            one_step()
        dg.set_profiling(True)
        sampler = ClockSampler(local_rank); sampler.start()
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches_t0 = kernel_launch_count()
        ev0.record()
        tot_iters, stats_last = 0, None
        for _ in range(args.steps):
            iters, stats_last = one_step()
            tot_iters += iters
        ev1.record()
        barrier()
        clocks = sampler.stop()
        launches_timed = kernel_launch_count() - launches_t0
        ms_total = ev0.elapsed_time(ev1)
        prof = dg.profile()
        dg.set_profiling(False)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, *dg.result(), stats_last)
        value = E * tot_iters / (ms_total * 1e-3)
        iters = tot_iters // args.steps
        cap = {}
        try:
            cap = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        except (OSError, ValueError):
            pass
        same_workload = bool(cap) and cap["config"]["nodes"] == args.nodes and cap["config"]["edges"] == args.edges

        def kernel_roofline(p):
            ach = p["alg_bytes"] / (p["ms"] * 1e-3) / 1e9
            r = {"bound": "hbm", "kernel": p["name"], "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                 "frac": ach / peaks["hbm_gbs"], "traffic": None, "dram_frac": None, "peak_source": peak_src,
                 "launches": p["launches"], "avg_launch_ms": p["ms"] / p["launches"],
                 "alg_bytes_per_launch": p["alg_bytes"] / p["launches"], "share_of_step": p["ms"] / ms_total}
            c = cap.get(p["name"]) if same_workload else None
            if c:
                # physical twin of `frac`: DRAM bytes of the committed `ncu --set full` capture of this kernel at this
                # workload over the launch time measured live here
                r["traffic"] = c["dram_bytes_per_launch"]
                r["dram_frac"] = c["dram_bytes_per_launch"] / (r["avg_launch_ms"] * 1e-3) / 1e9 / peaks["hbm_gbs"]
                r["traffic_source"] = c.get("source", cap.get("source"))
            return r
        kern = [kernel_roofline(p) for p in prof if p["launches"]]
        dom = max((k for k in kern if "dense" in k["kernel"]), key=lambda k: k["share_of_step"], default=None)
        result.update(value=value, ms_per_step=ms_total / args.steps, iters=iters, E=E, info=info, clocks=clocks,
                      roofline=dom, launches=launches_timed, kernels=kern,
                      per_iter=[{"t": s["t"], "mode": s["mode"], "n_changed": s["n_changed"], "ms": round(s["ms"], 3)} for s in stats_last])
        exchange_kind = None
    else:
        # configs[2]: the same graph, destination rows partitioned over `world` GPUs
        from stract_b200.webgraph import run_sharded_loop
        # ---- e2e at N > 1: every rank holds ONE contiguous shard of the edge stream in page-locked host memory (as the
        #      reference's workers each hold one webgraph shard); the timed call copies it over the rank's own PCIe link,
        #      all-gathers the stream over NVLink, stages (replicated, DESIGN section 8), exchanges the IPC blobs, runs the
        #      sharded loop and reads back its owned share.  It runs after the kernel-loop measurement, except when that one
        #      binds torch symmetric memory (8 GPUs): then it runs first, the order (CUDA IPC mappings, then symmetric memory)
        #      the 8-GPU sweep exercised.
        e2e_state = {"chk": None}

        def run_e2e_n(free_inputs):
            nonlocal cols, graph
            if args.no_e2e or args.no_p2p:
                return
            import psutil
            from stract_b200.webgraph import ShardedHarmonicCentrality, shard_bounds
            need = edges * 40
            avail = psutil.virtual_memory().available
            ok = torch.tensor([1 if avail > need * 1.3 else 0], device=dev, dtype=torch.int64)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if int(ok.item()) == 0:
                result["e2e_n"] = {"skipped": f"host RAM {avail / 2**30:.0f} GiB < 1.3 x {need / 2**30:.0f} GiB (the page-locked shards of the edge stream)"}
                return
            try:
                s_lo, s_hi = shard_bounds(edges, rank, world)
                hostc = []
                for cc in cols:
                    hh = torch.empty((s_hi - s_lo,), dtype=cc.dtype, pin_memory=True)
                    hh.copy_(cc[s_lo:s_hi])
                    hostc.append(hh)
                hgraph_n = Webgraph.from_arrays(*hostc)
                if free_inputs:
                    cols = graph = None
                torch.cuda.empty_cache()   # the timed call needs room for the gathered stream next to the staging temporaries
                per, d2h_n, its, kept, phases_n = [], 0, 0, 0, []
                n_warm = 2   # device memory pools, NCCL channels and the page-locked result blocks reach steady state
                for step in range(n_warm + max(2, min(args.e2e_steps, 3))):
                    barrier()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    rr = ShardedHarmonicCentrality.calculate(hgraph_n, local_rank, rank, world, exchange="p2p", ingest="shards")
                    chk = float(rr.values[:1024].sum())  # noqa: F841
                    e1.record(); torch.cuda.synchronize()
                    t_ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
                    dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
                    nb = torch.tensor([len(rr.values) * 24, _i64(result_checksum(rr.ids_lo, rr.ids_hi, rr.values))], device=dev, dtype=torch.int64)
                    dist.all_reduce(nb)
                    if step >= n_warm:
                        per.append(float(t_ms.item())); d2h_n = int(nb[0].item()); its = rr.iterations
                        kept = int(rr.info["n_edges_kept"])
                        phases_n.append(rr.info.get("phase_ms"))
                        e2e_state["chk"] = int(nb[1].item()) & ((1 << 64) - 1)
                    del rr
                result["e2e_n"] = {"value": kept * its * len(per) / (sum(per) * 1e-3), "unit": UNIT, "h2d_bytes_per_step": edges * 40,
                                   "d2h_bytes_per_step": d2h_n, "ms_per_step": sum(per) / len(per), "steps": len(per), "pinned_host": True,
                                   "ms_min_median_max": [round(min(per), 1), round(float(np.median(per)), 1), round(max(per), 1)],
                                   "rank0_phase_ms": phases_n,
                                   "note": f"max over ranks per step; each of the {world} ranks copies its 1/{world} shard of the edge stream from page-locked "
                                           "host memory over its own PCIe link, an NCCL all-gather over NVLink assembles the stream on every GPU, "
                                           "then (replicated) staging + CUDA IPC set-up + sharded loop (peer stores + device-side barrier) + owned results to the host",
                                   "exchange": "p2p (CUDA IPC): the end-to-end call always uses this transport"}
                del hostc, hgraph_n
                torch.cuda.empty_cache()
            except Exception as ex:  # noqa: BLE001  (the kernel-loop line must survive a failing end-to-end leg)
                result["e2e_n"] = {"error": repr(ex)[:400]}

        def merge_e2e_parity():
            c2 = parity.get("c2")
            if gold and e2e_state["chk"] is not None and isinstance(c2, dict) and isinstance(c2.get("equal"), dict):
                c2["equal"]["e2e_result_checksum"] = e2e_state["chk"] == gold["result_checksum"]
                c2["green"] = all(c2["equal"].values())

        gold = None
        want = args.exchange
        if want == "auto":
            want = "multicast" if world >= 8 else "p2p"
        if args.no_p2p:
            want = "nccl"
        if args.sweep:
            want = "p2p"   # the sweep walks the CUDA IPC variants on this handle, then binds symmetric memory on a fresh one
        e2e_first = want in ("symm", "multicast") and not args.sweep
        if e2e_first:
            run_e2e_n(False)
        dg = DeviceGraph(graph, device=local_rank, rank=rank, world_size=world)
        exchange_kind = "nccl"
        if want in ("symm", "multicast"):
            kind, ok = None, 0
            try:
                kind = dg.enable_symmetric(multicast=(want == "multicast"))
                ok = 1 if (want == "symm" or kind == "multicast") else 0
            except Exception as ex:  # noqa: BLE001
                print(f"[bench] rank {rank}: symmetric-memory exchange not available: {ex!r}"[:400], file=sys.stderr, flush=True)
            okt = torch.tensor([ok], device=dev, dtype=torch.int64)
            dist.all_reduce(okt, op=dist.ReduceOp.MIN)
            if int(okt.item()) == 1 or args.exchange != "auto":
                if kind is None:
                    raise RuntimeError("--exchange " + args.exchange + ": the symmetric-memory binding failed on this rank")
                exchange_kind = "symmetric-memory " + kind
            else:   # auto: no multicast on this box -- peer stores over CUDA IPC on a fresh handle
                dg.close()
                dg = DeviceGraph(graph, device=local_rank, rank=rank, world_size=world)
                want = "p2p"
        if want == "p2p":
            dg.enable_p2p()
            exchange_kind = "p2p"
        info = dg.info()
        E = info["n_edges_kept"]

        behind_abi = exchange_kind == "p2p"   # sb200_hyperball_run_sharded: round loop + device-side barrier, no NCCL

        if args.sweep:
            # ---- tuning sweep: same staged graph, same process, one variant after the other; each is fingerprinted by the
            #      per-iteration changed counts summed over the ranks (they must equal the first variant's)
            def time_variant(handle, label, run, steps=3, warm=2):
                for _ in range(warm):
                    handle.reset(); run()
                handle.set_profiling(True)
                barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                st = None
                for _ in range(steps):
                    handle.reset(); _t, st = run()
                e1.record()
                barrier()
                prof = handle.profile(); handle.set_profiling(False)
                t_ms = torch.tensor([e0.elapsed_time(e1) / steps], device=dev, dtype=torch.float64)
                dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
                fp = torch.tensor([s["n_changed"] for s in st] + [0] * (32 - len(st)), device=dev, dtype=torch.int64)[:32]
                dist.all_reduce(fp)
                out = {"variant": label, "ms_per_step": round(float(t_ms.item()), 3), "iterations": len(st),
                       "iter_ms_rank0": [round(s["ms"], 3) for s in st],
                       "kernels_rank0": {q["name"]: round(q["ms"] / q["launches"], 3) for q in prof if q["launches"]},
                       "changed_counts": [int(x) for x in fp.tolist()[:len(st)]]}
                if rank == 0:
                    print("[sweep] " + json.dumps(out), file=sys.stderr, flush=True)
                return out
            sweep = []
            variants = [("filter side2", {"publish_all": 0, "quad_side_ctas": 2, "owned_items": 1}),
                        ("filter side0", {"publish_all": 0, "quad_side_ctas": 0, "owned_items": 1}),
                        ("all side0", {"publish_all": 1, "quad_side_ctas": 0, "owned_items": 1}),
                        ("all side2", {"publish_all": 1, "quad_side_ctas": 2, "owned_items": 1}),
                        ("filter side1", {"publish_all": 0, "quad_side_ctas": 1, "owned_items": 1}),
                        ("filter side4", {"publish_all": 0, "quad_side_ctas": 4, "owned_items": 1}),
                        ("filter side8", {"publish_all": 0, "quad_side_ctas": 8, "owned_items": 1})]
            if exchange_kind == "p2p":
                for label, opts in variants:
                    for k_, v_ in opts.items():
                        dg.set_option(k_, v_)
                    sweep.append(time_variant(dg, label, dg.run_sharded))
            dg.close(); dg = None
            try:   # NVSwitch multicast stores over torch symmetric memory (one store per row, the switch replicates), host-side round loop
                dg = DeviceGraph(graph, device=local_rank, rank=rank, world_size=world)
                kind = dg.enable_symmetric(multicast=True)
                for side in (0, 2):
                    dg.set_option("quad_side_ctas", side)
                    sweep.append(time_variant(dg, f"symmetric-memory {kind} side{side}", lambda: run_sharded_loop(dg, world)))
            except Exception as ex:  # noqa: BLE001
                sweep.append({"variant": "symmetric-memory multicast", "error": repr(ex)[:300]})
            finally:
                if dg is not None:
                    dg.close(); dg = None
            if rank == 0:
                ref = sweep[0].get("changed_counts")
                for v in sweep:
                    if "changed_counts" in v:
                        v["same_counts_as_first"] = v["changed_counts"] == ref
                print(json.dumps({"sweep": sweep, "n_gpus": world, "workload": f"R-MAT {args.nodes} nodes / {args.edges} edges (C2), {E} kept edges"}))
            dist.destroy_process_group()
            return 0

        def one_step():
            dg.reset()
            return dg.run_sharded() if behind_abi else run_sharded_loop(dg, world)
        for _ in range(W):
            one_step()
        dg.set_profiling(True)
        sampler = ClockSampler(local_rank); sampler.start()
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches_t0 = kernel_launch_count()
        ev0.record()
        tot_iters, st_last = 0, None
        for _ in range(args.steps):
            t, st_last = one_step()
            tot_iters += t
        ev1.record()
        barrier()
        clocks = sampler.stop()
        roofline_n, kernels_n = None, None
        try:   # rank 0's dominant kernel over its owned share of the rows (algorithmic bytes x owned fraction)
            prof = dg.profile()
            dom = max((p for p in prof if "dense" in p["name"] and p["launches"]), key=lambda p: p["ms"], default=None)
            if dom:
                ach = dom["alg_bytes"] / (dom["ms"] * 1e-3) / 1e9
                roofline_n = {"bound": "hbm", "kernel": dom["name"] + " (rank 0, owned rows)", "achieved": ach, "peak": peaks["hbm_gbs"],
                              "unit": "GB/s", "frac": ach / peaks["hbm_gbs"], "traffic": None, "peak_source": peak_src,
                              "launches": dom["launches"], "avg_launch_ms": dom["ms"] / dom["launches"],
                              "alg_bytes_per_launch": dom["alg_bytes"] / dom["launches"],
                              "note": "includes the stores of the produced rows into the peers' replicas over NVLink"}
            kernels_n = [{"kernel": q["name"], "launches": q["launches"], "avg_launch_ms": q["ms"] / q["launches"]} for q in prof if q["launches"]]
        except Exception:  # noqa: BLE001
            roofline_n = None
        dg.set_profiling(False)
        ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev, dtype=torch.float64)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        ms_total = float(ms.item())
        nl = torch.tensor([kernel_launch_count() - launches_t0], device=dev, dtype=torch.int64)
        dist.all_reduce(nl)
        value = E * tot_iters / (ms_total * 1e-3)
        mine = {"rank": rank, "edges_local": info["n_edges_local"],
                "iter_ms": [round(s["ms"], 3) for s in st_last], "modes": [s["mode"] for s in st_last]}
        allr = [None] * world
        dist.all_gather_object(allr, mine)
        # ---- parity at N > 1: the owned register rows and the owned results of all ranks together against the frozen
        #      N = 1 fingerprint (with the subscriber filter a replica is authoritative only for the rows its rank owns or reads)
        owned, _subs = dg.ownership()
        lo, hi, c = dg.result()
        part = torch.tensor([_i64(registers_checksum(dg.registers(), owned)), _i64(result_checksum(lo, hi, c)), len(c), int(owned.sum())],
                            dtype=torch.int64, device=dev)
        dist.all_reduce(part)   # int64 addition wraps like the uint64 sums
        M = (1 << 64) - 1
        got = {"registers_checksum": int(part[0].item()) & M, "result_checksum": int(part[1].item()) & M, "n_positive": int(part[2].item()),
               "n_nodes": int(part[3].item()), "iterations": tot_iters // args.steps}
        gold = None
        if full_size and os.path.exists(GOLDEN_C2):
            gold = json.load(open(GOLDEN_C2))
        if gold:
            eq = {k: got[k] == gold[k] for k in ("registers_checksum", "result_checksum", "n_positive", "n_nodes", "iterations")}
            parity["c2"] = {"against": "tests/golden/path1_c2.json (fingerprint of the N=1 run that equalled the full-size oracle bit for bit)",
                            "equal": eq, "green": all(eq.values())}
        else:
            parity["c2"] = {"against": None, "green": None, "fingerprint": got}
        result.update(value=value, ms_per_step=ms_total / args.steps, iters=tot_iters // args.steps, E=E, info=info,
                      clocks=clocks, roofline=roofline_n, launches=int(nl.item()), kernels=kernels_n or [], per_iter=allr)
        dg.close()
        dg = None
        if not e2e_first:
            run_e2e_n(True)
        merge_e2e_parity()

    # ---- e2e: the C-ABI call sequence from HOST buffers (N = 1) ----------------------------------
    e2e, host = None, None
    if world == 1 and (not args.no_e2e or not args.no_cpu):
        import psutil
        need = edges * 40
        avail = psutil.virtual_memory().available
        if avail < need * 1.3:
            e2e = {"skipped": f"host RAM {avail / 2**30:.0f} GiB < 1.3x the {need / 2**30:.0f} GiB edge stream"}
        else:
            host = []
            for c in cols:
                try:
                    h = torch.empty(c.shape, dtype=c.dtype, pin_memory=True)
                except Exception:
                    h = torch.empty(c.shape, dtype=c.dtype)
                h.copy_(c)
                host.append(h)
    del cols, graph
    torch.cuda.empty_cache()
    if host is not None and not args.no_e2e:
        pinned = all(h.is_pinned() for h in host)
        hgraph = Webgraph.from_arrays(*host)
        for _ in range(2):  # warm-up: device memory pool and the page-locked result blocks reach steady state
            r = HarmonicCentrality.calculate(hgraph, device=local_rank)
            del r
        barrier()
        per_step, tot, d2h, walls, last_r = [], 0, 0, [], None
        r = None
        for _ in range(args.e2e_steps):
            last_r = r = None   # the caller drops a result before it asks for the next one (its page-locked block is reused)
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            r = HarmonicCentrality.calculate(hgraph, device=local_rank)
            chk = float(r.values[:1024].sum())  # the caller reads the result on the host  # noqa: F841
            ev1.record(); torch.cuda.synchronize()
            per_step.append(ev0.elapsed_time(ev1))
            tot += r.info["n_edges_kept"] * r.iterations
            d2h = len(r.values) * 24
            walls.append({k: round(v, 1) for k, v in (r.info.get("wall_ms") or {}).items()})
            last_r = r
        ms_e = float(sum(per_step))
        e2e = {"value": tot / (ms_e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": edges * 40, "d2h_bytes_per_step": d2h,
               "ms_per_step": ms_e / args.e2e_steps, "steps": args.e2e_steps, "pinned_host": pinned, "workload": "full workload",
               "ms_min_median_max": [round(min(per_step), 1), round(float(np.median(per_step)), 1), round(max(per_step), 1)],
               "stage_ms": last_r.info["stage_ms"], "iterations": last_r.iterations, "step_wall_ms": walls}
        # the e2e result is the one compared with the oracle below (it went through the host-buffer path)
        e2e_result = (last_r.ids_lo, last_r.ids_hi, last_r.values, last_r.iterations)
    else:
        e2e_result = None

    # ---- full-size parity + same-config CPU baseline (N = 1) -------------------------------------
    cpu_baseline = None
    if world == 1 and not args.no_cpu and host is not None:
        threads = host_threads()
        o, oi = oracle_c2(host, threads)
        g_regs = dg.registers()
        lo, hi, c = dg.result()
        ores = o.result()
        eq = {"n_nodes": oi["n_nodes"] == info["n_nodes"], "kept_edges": oi["kept_edges"] == E, "iterations": oi["iterations"] == result["iters"],
              "registers": bool(np.array_equal(g_regs, o.registers_view())),
              "ids": bool(np.array_equal(lo, ores["ids_lo"]) and np.array_equal(hi, ores["ids_hi"])),
              "centrality": bool(np.array_equal(c, ores["centrality"]))}
        if e2e_result is not None:
            eq["e2e_result"] = bool(e2e_result[3] == oi["iterations"] and np.array_equal(e2e_result[0], ores["ids_lo"]) and
                                    np.array_equal(e2e_result[1], ores["ids_hi"]) and np.array_equal(e2e_result[2], ores["centrality"]))
        fp = {"registers_sha256": sha(g_regs), "registers_checksum": registers_checksum(g_regs), "result_checksum": result_checksum(lo, hi, c), "n_positive": int(len(c)),
              "iterations": result["iters"], "centrality_sha256": sha(c), "n_nodes": info["n_nodes"], "kept_edges": E}
        parity["c2"] = {"against": f"oracle dense restatement, full graph, {threads} host threads (bit-exact compare of all "
                                   f"{info['n_nodes']} x 64 registers, ids and f64 centralities)",
                        "equal": eq, "green": all(eq.values()), "fingerprint": fp}
        if args.write_golden and full_size and all(eq.values()):
            with open(GOLDEN_C2, "w") as fh:
                json.dump({"generator": {"fn": "sb200_synth_edges kind 1 (== stract_b200.synth.rmat_graph)", "nodes": nodes, "edges": edges,
                                         "seed": 42, "scale": args.scale}, **fp}, fh, indent=1)
        cpu_baseline = {"value": oi["value"], "unit": UNIT, "cores": threads, "kind": "port",
                        "sample": f"the full workload (same graph as the GPU arm): oracle dense port on {threads} threads, iteration loop "
                                  f"to convergence ({oi['iterations']} iterations), median of {len(oi['loop_s'])} runs; graph staged in RAM "
                                  f"beforehand ({oi['stage_s']} s, all threads)",
                        "loop_s": oi["loop_s"], "stage_s": oi["stage_s"]}
        o.close()
        del o, g_regs
    elif world == 1 and full_size and os.path.exists(GOLDEN_C2):
        gold = json.load(open(GOLDEN_C2))
        lo, hi, c = dg.result()
        eq = {"registers": registers_checksum(dg.registers()) == gold["registers_checksum"], "result_checksum": result_checksum(lo, hi, c) == gold["result_checksum"],
              "n_positive": len(c) == gold["n_positive"], "iterations": result["iters"] == gold["iterations"]}
        parity["c2"] = {"against": "tests/golden/path1_c2.json", "equal": eq, "green": all(eq.values())}
    if dg is not None:
        dg.close()
    del host
    try:
        torch.cuda.empty_cache()
        L.sb200_release_cached_memory(local_rank)
    except Exception:  # noqa: BLE001
        pass

    if rank == 0:
        cfg = workload_config(nodes, edges, result["E"], result["info"]["n_nodes"], result["iters"])
        par = "1 GPU" if world == 1 else (f"destination-row partition x{world}, " + {
            "nccl": "NCCL byte-max all-reduce of the register replicas per iteration",
            "p2p": "fused exchange: pull kernels store produced rows into the subscribing peers' replicas over NVLink (CUDA IPC); round loop "
                   "behind the ABI (sb200_hyperball_run_sharded), device-side barrier + changed-count sum over peer memory, no NCCL in the loop"}.get(
            exchange_kind, "fused exchange over " + str(exchange_kind) + " stores, changed-count all-reduce as barrier"))
        line = {"metric": METRIC, "value": result["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": W, "ms_per_step": result["ms_per_step"], "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": cfg,
                "run": {"parallelism": par, "hbm_bytes": result["info"]["hbm_bytes"], "gen_s": round(gen_s, 2),
                        "stage_ms": result["info"]["stage_ms"]},
                "clocks": result["clocks"], "gpu_launches": result["launches"], "roofline": result["roofline"],
                "kernels": result["kernels"], "per_iter": result["per_iter"], "e2e": e2e if world == 1 else result.get("e2e_n"), "parity": parity}
        if cpu_baseline:
            line["cpu_baseline"] = cpu_baseline
        if world == 1 and not args.no_c1:
            try:
                line["c1"] = run_c1(torch, local_rank)
            except Exception as ex:  # noqa: BLE001
                line["c1"] = {"error": repr(ex)[:300]}
        if not args.no_bm25 and world == 1:
            import bench_bm25
            line["bm25"] = bench_bm25.run(local_rank, peaks, peak_src, cpu=not args.no_cpu)
            for k in ("and_top1000_10M", "or5_signals_100M", "multi_field_10M"):
                if isinstance(line["bm25"].get(k), dict) and "parity" in line["bm25"][k]:
                    parity[k] = line["bm25"][k]["parity"]
                md = (line["bm25"].get(k) or {}).get("max_docs_250k") if isinstance(line["bm25"].get(k), dict) else None
                if md and "parity" in md:
                    parity[k + ".max_docs_250k"] = md["parity"]
        print(json.dumps(line))
        greens = [v.get("green") for v in parity.values() if isinstance(v, dict)]
        if any(g is False for g in greens):
            print("PARITY MISMATCH: " + json.dumps({k: v for k, v in parity.items() if isinstance(v, dict) and v.get("green") is False})[:2000],
                  file=sys.stderr)
            if world > 1:
                dist.destroy_process_group()
            return 3
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
