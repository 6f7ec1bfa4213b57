#!/usr/bin/env python
"""Benchmark of the Fitch/Sankoff construction pass (BASELINE.json metric: node x column updates / s at 1/2/4/8 B200).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config NAME] [--algo fitch|sankoff] [--impl reference] [--dump-outputs DIR]

A "step" is one pass of the hot path (forward + backward + ordered mutation compaction, and for N > 1 the column-range
gather + merge of the per-rank lists on rank 0) over one batch of synthetic columns. The workload is BASELINE.json
configs[3], the configuration the metric's scaling is quoted on: ONE synthetic bacterial-scale alignment, 4k leaves x 5M
columns, whose columns are split into N contiguous ranges (strong scaling; N = 1 runs the same alignment on one GPU:
50 GB of leaf planes + sets fit). Launched by torch.distributed.run for N > 1, one rank per GPU; every rank forms its
part of ONE pmb_group (include/panman_b200.h): the library owns the ranges, the gather into rank 0's mailbox over
NVLink (the packing kernel's stores into peer memory mapped through CUDA IPC), the hand-shakes (stream memory operations)
and the merge; torch.distributed (NCCL) only all-gathers the 128-byte mailbox handles once and reduces the timings.
Prints ONE JSON line (rank 0). At N = 1 the line also carries a `configs` table (every BASELINE.json configuration, both
algorithms where the survey asks for both) measured the same way (CUDA events over --steps pipelined passes). Every timed
loop, the end-to-end figures included, runs --steps steps.  --impl reference times the reference's own CPU
implementation instead.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "fitch_sankoff_node_column_updates_per_sec"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="ecoli4k")
    ap.add_argument("--algo", default=None)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--cols", type=int, default=0, help="override the column count (debug)")
    ap.add_argument("--leaves", type=int, default=0, help="override the leaf count (debug)")
    ap.add_argument("--chunk-nodes", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="N = 1: skip the table of the other configurations")
    ap.add_argument("--no-traffic", action="store_true", help="N = 1: do not measure DRAM traffic with an ncu child run")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the merged lists of the last timed step to DIR/<name>.npy (see dump_outputs); B200 arm only: "
                         "the reference arm sizes its column sample by a timing probe, so its inputs differ from run to run")
    ap.add_argument("--traffic-child", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs the B200 arm: the reference arm sizes its column sample by a timing probe, "
                 "so its inputs, and its lists, differ from run to run")
    return args


def workload(args, name=None, algo=None):
    from panman_b200 import synth

    cfg = dict(synth.CONFIGS[name or args.config])
    if name is None:
        if args.cols:
            cfg["n_cols"] = args.cols
        if args.leaves:
            cfg["n_leaves"] = args.leaves
    algo = algo or (args.algo if name is None else None) or cfg["algos"][0]
    return cfg, algo


# ----------------------------------------------------------------------------- clocks (sampled during the timed region)
class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if not self.nv:
            return
        nv = self.nv
        names = {getattr(nv, k): k for k in dir(nv) if k.startswith("nvmlClocksThrottleReason") and isinstance(getattr(nv, k), int)}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if bit and (r & bit) and name not in ("nvmlClocksThrottleReasonNone", "nvmlClocksThrottleReasonAll"):
                        self.reasons.add(name.replace("nvmlClocksThrottleReason", ""))
            except Exception:
                pass
            time.sleep(0.002)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


# ----------------------------------------------------------------------------- reference / oracle on the host cores
class CpuReference:
    """The reference's own CPU implementation of the path on a column sample: oracle/_ref (the verbatim fitchSankoff.cpp +
    restated string-keyed drivers) when it was built, else the oracle port. Used (a) as the timed CPU baseline and the
    reference arm, (b) as the CHECKER of the GPU lists on the same columns -- never as part of the product path."""

    def __init__(self, tree):
        from oracle.oracle import CHAR_OF, PortOracle, RefOracle, have_ref

        self.tree, self.CHAR_OF = tree, CHAR_OF
        self.port = PortOracle()
        self.kind = "reference" if have_ref() else "port"
        if self.kind == "reference":
            self.ref = RefOracle()

            class T:  # the fields RefOracle.tree needs
                pass

            t = T()
            names = tree.names()
            t.n_nodes, t.names, t.parent, t.child_off, t.child_idx = tree.n_nodes, names, tree.parent, tree.child_off, tree.child_idx
            self.t, self.h = t, self.ref.tree(t)
            self.leaf_names = [names[v] for v in tree.leaves]

    def timed(self, codes, parent_code, algo, n_cols, threads):
        """Seconds for the first n_cols columns of the sample."""
        algo_i = 0 if algo == "fitch" else 1
        if self.kind == "reference":
            rows = self.CHAR_OF[codes[:, :n_cols]]
            cons = self.CHAR_OF[parent_code[:n_cols]]
            seqs = [bytes(r) for r in rows]
            t0 = time.perf_counter()
            self.ref.msa_run(self.h, self.t, algo_i, self.leaf_names, seqs, bytes(cons), "", n_threads=threads)
            return time.perf_counter() - t0
        t0 = time.perf_counter()
        self.port.run(self.tree, algo_i, codes[:, :n_cols], parent_code[:n_cols], n_threads=threads)
        return time.perf_counter() - t0

    def sample(self, codes, parent_code, algo, seconds, threads):
        """Grows the column sample until one run takes about `seconds` (a short probe overweights the fixed costs)."""
        n_all = codes.shape[1]
        nc = min(n_all, max(threads, 16))
        dt = self.timed(codes, parent_code, algo, nc, threads)
        while dt < 0.6 * seconds and nc < n_all:
            nc = int(min(n_all, max(2 * nc, 0.95 * nc * seconds / max(dt, 1e-6))))
            dt = self.timed(codes, parent_code, algo, nc, threads)
        what = "string-keyed reference drivers (verbatim fitchSankoff.cpp)" if self.kind == "reference" else "array port"
        return dict(value=self.tree.n_nodes * nc / dt, unit="node*col/s", cores=threads, kind=self.kind,
                    sample=f"first {nc} columns of the workload ({self.tree.n_nodes} nodes), {dt:.1f} s, {what}, {threads} thread(s)",
                    sample_cols=nc, sample_seconds=dt)

    def lists(self, codes, parent_code, algo, root_override=None):
        """The checker: per-node lists of the sample (array port; pinned to the verbatim build by tests/test_oracle.py)."""
        want, _ = self.port.run(self.tree, 0 if algo == "fitch" else 1, codes, parent_code, root_override, None, None, 0,
                                n_threads=host_threads())
        return want


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def sample_columns(n_leaves, n_cols, seconds=12.0):
    # enough columns for `seconds` of the reference on all host cores (about 4e6 node x columns / s and thread, with a
    # margin), bounded by host memory (about 1 GB of codes); generating them costs CPU time too
    want = int(1.3 * seconds * 4e6 * host_threads() / max(1, 2 * n_leaves - 1))
    return int(min(n_cols, 262144, max(2048, want), max(512, 1_200_000_000 // n_leaves)))


# ----------------------------------------------------------------------------- reference arm
def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from panman_b200 import synth

    cfg, algo = workload(args)
    tree = synth.make_tree(cfg["n_leaves"], cfg["seed"], cfg["kind"])
    n_s = sample_columns(cfg["n_leaves"], cfg["n_cols"])
    codes4, pc = synth.simulate_msa(tree, 0, n_s, synth.MsaSpec(cfg["seed"], cfg["p_sub"], cfg["f_gap"], cfg["p_N"]))
    codes = synth.unpack_nibbles(codes4, n_s).numpy()
    pc = pc.numpy()
    threads = host_threads()
    cpu = CpuReference(tree)
    # every step is one timed run of the reference over a column sample sized for >= 10 s (BASELINE.md section 2)
    probe = cpu.sample(codes, pc, algo, 10.0, threads)
    nc = probe["sample_cols"]
    times = []
    for i in range(args.warmup + args.steps):
        dt = cpu.timed(codes, pc, algo, nc, threads)
        if i >= args.warmup:
            times.append(dt)
    step_s = float(np.mean(times))
    value = tree.n_nodes * nc / step_s
    base = dict(probe, value=value, sample_seconds=step_s,
                sample=f"first {nc} columns of the workload ({tree.n_nodes} nodes), {step_s:.1f} s per step, "
                       f"{'string-keyed reference drivers (verbatim fitchSankoff.cpp)' if cpu.kind == 'reference' else 'array port'}, {threads} thread(s)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "node*col/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * step_s, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "u16 sets / int32 costs (CPU)", "data": "synthetic",
        "config": {"workload": f"{args.config}: {cfg['n_leaves']} leaves x {cfg['n_cols']} columns, {cfg['kind']} tree, {algo}; "
                               f"each step = the first {nc} columns (columns are independent units: the rate is per node x column)"},
        "extrapolated_ms_per_full_pass": 1e3 * tree.n_nodes * cfg["n_cols"] / value,
        "cpu_baseline": base,
        "e2e": {"value": value, "unit": "node*col/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------- B200 arm
def peak_gbs():
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    if "hbm_gbs" in peaks:
        return float(peaks["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth, burst)"
    return 6650.0, "fallback 6650 GB/s (B200_PROFILING.md; MEASURED_PEAKS.json absent)"


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, res):
    """The merged lists a caller of pmb_group_download receives after the last timed step, as out_dir/<name>.npy:
    node_offsets whole, and the records (pos, type_code) whole when they fit in 64 MB in all, else a fixed seeded sample of
    them; record_index.npy says which records were kept. Values are exact in float64 (float32 for the 8-bit type codes).
    The workload is seeded, so the same arguments give the same files on any build that computes the same lists."""
    off = res.node_offsets.astype(np.float64)
    n = len(res.pos)
    k = min(n, (DUMP_BYTES - 4096 - off.nbytes) // 20)  # 4 KB for the .npy headers; record_index, pos f64, type_code f32
    idx = np.arange(n) if k == n else np.sort(np.random.default_rng(0).choice(n, k, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("node_offsets", off), ("record_index", idx.astype(np.float64)), ("pos", res.pos[idx].astype(np.float64)),
                    ("type_code", res.type_code[idx].astype(np.float32))):
        np.save(os.path.join(out_dir, name + ".npy"), a)


def slice_lists(res, n_nodes, a, b):
    node = np.repeat(np.arange(n_nodes), np.diff(res.node_offsets))
    keep = (res.pos >= a) & (res.pos < b)
    off = np.zeros(n_nodes + 1, np.int64)
    off[1:] = np.cumsum(np.bincount(node[keep], minlength=n_nodes))
    return off, res.pos[keep], res.type_code[keep]


def measure_one(pb, synth, torch, name, algo, dev, local, steps, warmup):
    """One configuration on one GPU, device-resident: ms per pass (CUDA events on the library's stream), roofline."""
    cfg = synth.CONFIGS[name]
    algo_i = pb.ALGO_FITCH if algo == "fitch" else pb.ALGO_SANKOFF
    tree = synth.make_tree(cfg["n_leaves"], cfg["seed"], cfg["kind"])
    C = cfg["n_cols"]
    codes4, pc = synth.simulate_msa(tree, 0, C, synth.MsaSpec(cfg["seed"], cfg["p_sub"], cfg["f_gap"], cfg["p_N"]), device=dev)
    ro = synth.unpack_nibbles(codes4[:1], C)[0].to(torch.int8).contiguous() if algo == "sankoff" else None
    ctx = pb.Context(local)
    ctx.set_tree(tree.n_nodes, tree.root, tree.child_off, tree.child_idx, tree.leaf_row)
    ctx.upload(C, tree.n_leaves, codes4, codes4.shape[1], pc, ro)
    del codes4
    lib = torch.cuda.ExternalStream(ctx.stream_handle(), device=dev)
    for _ in range(max(3, warmup)):
        ctx.run_resident_async(algo_i)
    ctx.wait()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(lib)
    for _ in range(steps):
        ctx.run_resident_async(algo_i)
    ctx.join()  # consecutive passes run on several streams (small problems: on two lanes); the main stream now follows them all
    e1.record(lib)
    ctx.wait()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    t = ctx.run_resident(algo_i)
    n_mut = ctx.download(copy=False).n_mut
    alg = ctx.algorithmic_bytes(algo_i)
    peak, _ = peak_gbs()
    out = {"config": name, "algo": algo, "leaves": cfg["n_leaves"], "nodes": tree.n_nodes, "cols": C, "ms": ms,
           "value": tree.n_nodes * C / (ms * 1e-3), "algorithmic_bytes": int(alg), "achieved_gbs": alg / (ms * 1e-3) / 1e9,
           "roofline_frac": alg / (ms * 1e-3) / 1e9 / peak, "n_mut": int(n_mut),
           "phases_ms": {"forward": t.forward_ms, "backward": t.backward_ms, "compact": t.compact_ms}}
    ctx.close()
    torch.cuda.empty_cache()
    return out


def traffic_child(args):
    """Run under ncu by measure_traffic(): the workload once, two passes."""
    import torch

    import panman_b200 as pb
    from panman_b200 import synth

    cfg, algo = workload(args)
    algo_i = pb.ALGO_FITCH if algo == "fitch" else pb.ALGO_SANKOFF
    dev = torch.device("cuda", 0)
    tree = synth.make_tree(cfg["n_leaves"], cfg["seed"], cfg["kind"])
    C = cfg["n_cols"]
    codes4, pc = synth.simulate_msa(tree, 0, C, synth.MsaSpec(cfg["seed"], cfg["p_sub"], cfg["f_gap"], cfg["p_N"]), device=dev)
    ro = synth.unpack_nibbles(codes4[:1], C)[0].to(torch.int8).contiguous() if algo == "sankoff" else None
    ctx = pb.Context(0)
    ctx.set_tree(tree.n_nodes, tree.root, tree.child_off, tree.child_idx, tree.leaf_row)
    ctx.upload(C, tree.n_leaves, codes4, codes4.shape[1], pc, ro)
    for _ in range(2):
        ctx.run_resident(algo_i)
    ctx.close()


def measure_traffic(args):
    """dram__bytes_read.sum + dram__bytes_write.sum of the pass kernels of ONE pass, from an ncu run of a child process on
    the same workload (after the timed region; nothing timed runs under the profiler). None when ncu cannot profile here."""
    import csv
    import shutil

    ncu = shutil.which("ncu") or "/usr/local/cuda/bin/ncu"
    if not os.path.exists(ncu):
        return None, "ncu not found"
    with tempfile.TemporaryDirectory() as td:
        log = os.path.join(td, "traffic.csv")
        cmd = [ncu, "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum", "--clock-control", "none", "--csv", "--log-file", log,
               "--kernel-name", "regex:fitch_|sankoff_|compact_", sys.executable, os.path.abspath(__file__), "--traffic-child",
               "--config", args.config] + (["--algo", args.algo] if args.algo else []) + (["--cols", str(args.cols)] if args.cols else []) \
            + (["--leaves", str(args.leaves)] if args.leaves else [])
        try:
            r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=420, env=dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0]))
        except Exception as e:  # noqa: BLE001
            return None, f"ncu child failed: {e}"
        if r.returncode != 0 or not os.path.exists(log):
            return None, f"ncu child exited {r.returncode}"
        rows = []
        with open(log) as f:
            lines = [ln for ln in f if not ln.startswith("==")]
        for row in csv.DictReader(lines):
            try:
                v = float(row["Metric Value"].replace(",", ""))
            except Exception:
                continue
            unit = row.get("Metric Unit", "byte").lower()
            v *= {"byte": 1, "kbyte": 1e3, "mbyte": 1e6, "gbyte": 1e9}.get(unit, 1)
            rows.append((int(row["ID"]), row["Kernel Name"], v))
        if not rows:
            return None, "ncu produced no metric rows (profiling counters not permitted?)"
        per_launch = {}
        for i, k, v in rows:
            per_launch.setdefault(i, [k, 0.0])[1] += v
        ids = sorted(per_launch)
        half = ids[len(ids) // 2:]  # the second of the two passes
        return int(sum(per_launch[i][1] for i in half)), f"ncu child run, launches {half[0]}..{half[-1]} = one pass ({len(half)} kernels)"


def run_b200_arm(args):
    import torch

    import panman_b200 as pb
    from panman_b200 import synth
    from panman_b200.distributed import connect_group

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; libpanman_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    cfg, algo = workload(args)
    algo_i = pb.ALGO_FITCH if algo == "fitch" else pb.ALGO_SANKOFF
    C = cfg["n_cols"]
    c0, c1 = pb.column_range(world, C, rank)  # strong scaling: ONE alignment, contiguous tile-aligned ranges
    tree = synth.make_tree(cfg["n_leaves"], cfg["seed"], cfg["kind"])
    N = tree.n_nodes
    if args.dump_outputs and 8 * (N + 1) > DUMP_BYTES // 2:  # every rank stops here, none waits for the others in a barrier
        raise SystemExit(f"bench.py: the node offsets of {N} nodes take more than half of the {DUMP_BYTES >> 20} MB of --dump-outputs")
    spec = synth.MsaSpec(cfg["seed"], cfg["p_sub"], cfg["f_gap"], cfg["p_N"])
    codes4, pc = synth.simulate_msa(tree, c0, c1, spec, device=dev)  # this rank's range, generated on its device
    ro = None
    if algo == "sankoff":  # SURVEY 8d: Sankoff runs with --reference = leaf 0
        ro = synth.unpack_nibbles(codes4[:1], c1 - c0)[0].to(torch.int8).contiguous()
    torch.cuda.synchronize()

    g = pb.Group([local], rank_base=rank, world=world)
    ctx = g.ctx(0)
    if args.chunk_nodes:
        ctx.set_option("chunk_nodes", args.chunk_nodes)
    g.set_tree(tree.n_nodes, tree.root, tree.child_off, tree.child_idx, tree.leaf_row)
    g.upload_shard(0, C, tree.n_leaves, codes4, codes4.shape[1], pc, ro)
    g.wait()
    first = ctx.run_resident(algo_i)  # sizes the staging pool; its record count sizes the mailbox
    n_mut_rank = int(ctx.result_device().n_mut)
    if world > 1:
        connect_group(g, dist, n_mut_rank + n_mut_rank // 4 + 4096, device=dev)
    lib_stream = torch.cuda.ExternalStream(ctx.stream_handle(), device=dev)
    lib_end_stream = torch.cuda.ExternalStream(ctx.result_stream_handle(), device=dev)  # compaction (+ packing) stream: a pass ends here

    def barrier():
        g.wait()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    W = max(3, args.warmup)
    for _ in range(W):
        g.run_async(algo_i)
    # everything that takes a rank-dependent time on the host (NVML start-up of the clock sampler, event creation) happens
    # BEFORE the barrier, so that the ranks enter the timed loop together
    sampler = ClockSampler(local)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t0 = time.perf_counter()
    ev0.record(lib_stream)
    for _ in range(args.steps):
        g.run_async(algo_i)  # one C call per step: pass -> pack into rank 0's mailbox -> signal (-> merge on rank 0)
    ev1.record(lib_end_stream)
    if os.environ.get("PMB_BENCH_DEBUG"):
        ta = time.perf_counter()
        g.wait()
        tb = time.perf_counter()
        if world > 1:
            dist.barrier()
        tc = time.perf_counter()
        torch.cuda.synchronize()
        td = time.perf_counter()
        print(f"[rank {rank}] enqueue {1e3 * (ta - t0):.3f} ms, g.wait {1e3 * (tb - ta):.3f}, dist.barrier {1e3 * (tc - tb):.3f}, "
              f"sync {1e3 * (td - tc):.3f}, device {ev0.elapsed_time(ev1):.3f}", file=sys.stderr, flush=True)
    else:
        barrier()  # ends after the last merge on rank 0
    elapsed = time.perf_counter() - t0
    sampler.stop_flag = True
    sampler.join()
    K = args.steps
    dev_ms = ev0.elapsed_time(ev1) / K  # this rank's passes (+ packing) on the stream they were launched on
    launches = ctx.timings().n_launches + (1 if world > 1 else 0) + (4 if world > 1 and rank == 0 else 0)
    alg_bytes = ctx.algorithmic_bytes(algo_i)
    el = torch.tensor([elapsed, dev_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(el, op=dist.ReduceOp.MAX)
    elapsed, dev_ms_max = float(el[0]), float(el[1])
    value = N * C * K / elapsed

    # ---- the result of the last step (outside the timed region): merged lists on rank 0, and the parity check
    res = g.download(copy=True) if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, res)
    run_merge_ms = None
    if rank == 0:  # the <= 6 run-merge into NucMut fields follows the gather (outside the timed region; for information)
        nm = g.merge_runs()
        n_nucmut = int(nm[0][-1])
        del nm
        torch.cuda.synchronize()
        t_rm = time.perf_counter()
        g.merge_runs(to_host=False)  # device side only: seven small launches over the node-major list
        torch.cuda.synchronize()
        run_merge_ms = 1e3 * (time.perf_counter() - t_rm)
    parity = None
    if rank == 0:
        parity = parity_check(args, tree, cfg, algo, spec, res, world, synth, torch)
    # phase split of one pass: a few synchronous passes after the timed region (same kernels, same inputs)
    fwd = bwd = cmp_ = 0.0
    for _ in range(3):
        t = ctx.run_resident(algo_i)
        fwd += t.forward_ms / 3
        bwd += t.backward_ms / 3
        cmp_ += t.compact_ms / 3
    if world > 1:
        dist.barrier()

    # ---- end to end through the reference-facing C-ABI call with HOST buffers (H2D and D2H inside the timed region)
    e2e = None
    if not args.no_e2e:
        h_codes = torch.empty(codes4.shape, dtype=torch.uint8, pin_memory=True).copy_(codes4)
        h_pc = torch.empty(pc.shape, dtype=torch.uint8, pin_memory=True).copy_(pc)
        h_ro = None if ro is None else torch.empty(ro.shape, dtype=torch.int8, pin_memory=True).copy_(ro)
        torch.cuda.synchronize()

        def e2e_step():
            g.upload_shard(0, C, tree.n_leaves, h_codes, h_codes.shape[1], h_pc, h_ro)  # host -> device, this rank's range
            g.run_async(algo_i)
            return g.download(copy=False)  # waits; on rank 0: merged lists device -> host

        e2e_step()
        barrier()
        e2e_steps = K
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            r2 = e2e_step()
        barrier()
        e2e_t = time.perf_counter() - t0
        e2 = torch.tensor([e2e_t], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(e2, op=dist.ReduceOp.MAX)
        h2d = int(h_codes.numel() + h_pc.numel() + (0 if h_ro is None else h_ro.numel()))
        e2e = {"value": N * C * e2e_steps / float(e2[0]), "unit": "node*col/s", "h2d_bytes_per_step": h2d * world if world > 1 else h2d,
               "d2h_bytes_per_step": int((N + 1) * 8 + (r2.n_mut if rank == 0 else 0) * 5), "steps": e2e_steps,
               "ms_per_step": 1e3 * float(e2[0]) / e2e_steps,
               "api": "pmb_group_upload_shard (pinned host buffers) + pmb_group_run_async + pmb_group_download on every rank"}
        # ---- the same through the denser boundary format: this rank's range clade-run encoded (pmb_runs_encode, once, on the
        # host, outside the timed region -- as the nibble packing of h_codes is), then per step: events host -> device,
        # expansion into the same bit-planes on the device, the pass, lists device -> host
        runs, enc_s, setup_error = None, 0.0, None
        try:  # a rank that cannot encode (host memory) must not leave the others waiting in a barrier
            t_enc = time.perf_counter()
            runs = pb.Runs.of_tree(tree, c1 - c0, h_codes.numpy(), h_pc.numpy())
            enc_s = time.perf_counter() - t_enc
        except Exception as e:  # noqa: BLE001
            setup_error = str(e)
        ok = torch.tensor([0.0 if setup_error else 1.0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        try:
            if float(ok[0]) < 1.0:
                raise RuntimeError(setup_error or "pmb_runs_encode failed on another rank")

            def runs_step():
                g.upload_shard_runs(0, C, runs, h_pc, h_ro)
                g.run_async(algo_i)
                return g.download(copy=False)

            r3 = runs_step()
            same = None
            if rank == 0:
                same = bool(np.array_equal(r3.node_offsets, res.node_offsets) and np.array_equal(r3.pos, res.pos)
                            and np.array_equal(r3.type_code, res.type_code))
            barrier()
            runs_steps = K
            t0 = time.perf_counter()
            for _ in range(runs_steps):
                r3 = runs_step()
            barrier()
            e3 = torch.tensor([time.perf_counter() - t0, enc_s, float(runs.nbytes + h_pc.numel() + (0 if h_ro is None else h_ro.numel()))],
                              dtype=torch.float64, device=dev)
            e3max = e3.clone()
            if world > 1:
                dist.all_reduce(e3max, op=dist.ReduceOp.MAX)
                dist.all_reduce(e3, op=dist.ReduceOp.SUM)
            e2e["clade_runs"] = {
                "value": N * C * runs_steps / float(e3max[0]), "unit": "node*col/s", "ms_per_step": 1e3 * float(e3max[0]) / runs_steps,
                "steps": runs_steps, "h2d_bytes_per_step": int(e3[2]), "d2h_bytes_per_step": e2e["d2h_bytes_per_step"],
                "host_encode_seconds_once": float(e3max[1]), "events_per_column": runs.n_events / max(1, c1 - c0),
                "ms_per_step_if_encoded_every_step": 1e3 * float(e3max[1]) + 1e3 * float(e3max[0]) / runs_steps,
                "lists_identical_to_the_matrix_entry": same,
                "api": "pmb_runs_encode once (host, outside the timed region); per step pmb_group_upload_shard_runs (page-locked events) "
                       "+ pmb_group_run_async + pmb_group_download on every rank",
                "note": "same pass, same results; only the form in which the leaf codes cross PCIe differs. `e2e.value` above stays the "
                        "nibble-matrix entry (the conservative figure)"}
        except Exception as e:  # noqa: BLE001
            e2e["clade_runs"] = {"error": str(e)}
        if runs is not None:
            runs.close()
        del h_codes, h_pc

    if rank != 0:
        g.close()
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = peak_gbs()
    achieved = alg_bytes / (dev_ms_max * 1e-3) / 1e9  # this rank's algorithmic bytes / the slowest rank's pass time
    set_mb = (tree.n_leaves * 0.5 + (N - tree.n_leaves) * (2 if algo == "fitch" else 4)) * (c1 - c0) / 1e6
    line = {
        "metric": METRIC, "value": value, "unit": "node*col/s", "n_gpus": world,
        "steps": K, "warmup": W, "ms_per_step": 1e3 * elapsed / K, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None,
        "dtype": "u16 Fitch sets as 16 bit-planes" if algo == "fitch" else "2-bit Sankoff excess as 32 bit-planes", "data": "synthetic",
        "config": {"workload": f"{args.config}: {cfg['n_leaves']} leaves ({N} nodes) x {C} columns, {cfg['kind']} tree, {algo}, seed {cfg['seed']}; "
                               f"the columns are split into {world} contiguous 1024-aligned range(s), rank 0 owns [{c0},{c1})",
                   "l2": f"inputs larger than L2: leaf planes + set matrix = {set_mb:.0f} MB per rank and pass",
                   "parallelism": (f"column ranges x{world} (pmb_group), tree replicated; per-rank lists packed into rank 0's mailbox over NVLink "
                                   "(peer stores of the packing kernel, CUDA IPC mapping), stream-memory-op hand-shake, merge on rank 0 "
                                   "overlapping the next pass") if world > 1 else "single GPU",
                   "n_mut": int(res.n_mut), "n_nucmut_after_run_merge": n_nucmut,
                   "run_merge_device_ms": run_merge_ms},
        "device_ms_per_step": dev_ms_max,
        "phases_ms": {"forward": fwd, "backward": bwd, "compact": cmp_, "note": "rank 0, 3 synchronous passes after the timed region"},
        "gpu_launches": int(launches * K),
        "clocks": sampler.summary(),
        "parity_check": parity,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": None, "peak_source": peak_src,
                     "kernel": "one pass on one rank = persistent forward kernel + persistent backward kernel + compaction"
                               + (" + packing into the mailbox" if world > 1 else "")
                               + "; duration = CUDA events around the timed passes on the library's stream / steps, max over ranks",
                     "algorithmic_bytes_per_pass": int(alg_bytes)},
    }
    if e2e:
        line["e2e"] = e2e
    g.close()
    del g, codes4
    torch.cuda.empty_cache()
    if world == 1:
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args, tree, cfg, algo, spec, synth)
        if not args.no_configs:
            table = []
            for name, a in (("sars20k", "fitch"), ("indel10k", "fitch"), ("indel10k", "sankoff"), ("caterpillar100k", "fitch"),
                            ("caterpillar100k", "sankoff")):
                try:
                    table.append(measure_one(pb, synth, torch, name, a, dev, local, K, args.warmup))
                except Exception as e:  # noqa: BLE001
                    table.append({"config": name, "algo": a, "error": str(e)})
            table.append({"config": args.config, "algo": algo, "leaves": cfg["n_leaves"], "nodes": N, "cols": C, "ms": dev_ms_max,
                          "value": N * C / (dev_ms_max * 1e-3), "algorithmic_bytes": int(alg_bytes), "achieved_gbs": achieved,
                          "roofline_frac": achieved / peak, "n_mut": int(res.n_mut), "phases_ms": line["phases_ms"]})
            line["configs"] = table
        if not args.no_traffic:
            traffic, how = measure_traffic(args)
            if traffic is None:
                try:
                    traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(f"{args.config}:{algo}")
                    how += "; value from profiles/traffic.json (earlier ncu capture)"
                except Exception:
                    pass
            line["roofline"]["traffic"] = traffic
            line["roofline"]["traffic_source"] = how
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def parity_check(args, tree, cfg, algo, spec, res, world, synth, torch):
    """Outside the timed region, rank 0: the merged lists of the last timed step against the oracle on column slices --
    one around every range boundary (shards meet there) and one in the middle -- plus the whole-result invariants."""
    try:
        cpu = CpuReference(tree)
        C, N = cfg["n_cols"], tree.n_nodes
        assert res.n_mut == int(res.node_offsets[-1]) == len(res.pos)
        if len(res.pos):
            assert int(res.pos.min()) >= 0 and int(res.pos.max()) < C
            d = np.diff(res.pos.astype(np.int64))
            starts = res.node_offsets[1:-1]
            starts = starts[(starts > 0) & (starts < len(res.pos))]
            d[starts - 1] = 1
            assert bool((d > 0).all()), "positions not ascending inside a node's list"
        width = int(max(256, min(2048, 40_000_000 // max(1, N))))
        centres = sorted({pb_range(world, C, r)[0] for r in range(1, world)} | {C // 2})
        checked = 0
        for c in centres:
            a, b = max(0, c - width // 2), min(C, c + width // 2)
            if b <= a:
                continue
            s4, spc = synth.simulate_msa(tree, a, b, spec, device="cuda")
            codes = synth.unpack_nibbles(s4, b - a).cpu().numpy()
            ro = codes[0].astype(np.int8) if algo == "sankoff" else None
            want = cpu.lists(codes, spc.cpu().numpy(), algo, ro)
            off, pos, tc = slice_lists(res, N, a, b)
            if not (np.array_equal(off, want.node_offsets) and np.array_equal(pos, want.pos + a) and np.array_equal(tc, want.type_code)):
                return f"MISMATCH in columns [{a},{b})"
            checked += b - a
        return f"ok ({checked} columns in {len(centres)} slice(s) bit-exact vs the oracle incl. every range boundary; whole result sorted and consistent)"
    except AssertionError as e:
        return f"FAILED invariant: {e}"


def pb_range(world, n_cols, rank):
    import panman_b200 as pb

    return pb.column_range(world, n_cols, rank)


def cpu_baseline(args, tree, cfg, algo, spec, synth):
    """N = 1, rank 0: the reference's CPU implementation on a bounded column sample, all host cores and -- the way the
    reference ships its -M Fitch loop (src/panman.cpp:1381, serial) -- one thread."""
    n_s = sample_columns(cfg["n_leaves"], cfg["n_cols"])
    codes4, pc = synth.simulate_msa(tree, 0, n_s, spec)
    codes = synth.unpack_nibbles(codes4, n_s).numpy()
    cpu = CpuReference(tree)
    out = cpu.sample(codes, pc.numpy(), algo, args.cpu_seconds, host_threads())
    one = cpu.sample(codes, pc.numpy(), algo, max(3.0, args.cpu_seconds / 2), 1)
    out["as_shipped_1_thread"] = {"value": one["value"], "unit": "node*col/s", "cores": 1, "sample": one["sample"]}
    return out


def main():
    args = parse()
    if args.traffic_child:
        traffic_child(args)
    elif args.impl == "reference":
        run_reference_arm(args)
    else:
        run_b200_arm(args)


if __name__ == "__main__":
    main()
