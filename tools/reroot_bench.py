#!/usr/bin/env python
"""Reroot of an MSA-built PanMAT on one GPU: the device replay of the mutation lists (pmb_upload_replay) against the uploads it
replaces, at BASELINE.json configs 2, 4 and 5 (synth.CONFIGS sars20k, ecoli4k, caterpillar100k).

Per config, alternating within the call (median of --reps rounds of replay / dense / runs):
  * pmb_upload_replay, the whole call (host clock) and its device span (CUDA events on pmb_stream);
  * the replay's kernels alone (torch.profiler, one profiled call of its own) and their write rate over the leaf planes
    (0.5 byte per leaf x column);
  * expand_runs_kernel rebuilding the same planes from a host encoding (pmb_upload_runs, whole call);
  * the dense pmb_upload_nuc of the same matrix from page-locked memory;
  * the rerooted pass (pmb_run_resident, device time).
Writes one JSON file with the card's name and power limit, read in the same call."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import panman_b200 as pb  # noqa: E402
from panman_b200 import synth  # noqa: E402
from panman_b200.host import reroot_newick  # noqa: E402

REPLAY_KERNELS = ("replay_", "cub::", "DeviceRadixSort", "DeviceScan", "pack_colparams")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def new_tree_of(st, tip):
    names = st.names()
    old_nw = _newick(st, names)
    t = reroot_newick(old_nw, names[tip])
    row_of = {names[v]: int(st.leaf_row[v]) for v in range(st.n_nodes) if st.leaf_row[v] >= 0}
    lr = np.asarray([row_of[n] if t.leaf_row[v] >= 0 else -1 for v, n in enumerate(t.names)], np.int32)
    return t, lr


def _newick(st, names):
    out, stack = [], [(int(st.root), 0)]
    while stack:
        v, k = stack.pop()
        b, e = int(st.child_off[v]), int(st.child_off[v + 1])
        if b == e:
            out.append(names[v])
            continue
        out.append("(" if k == 0 else ("," if k < e - b else ""))
        if k < e - b:
            stack.append((v, k + 1))
            stack.append((int(st.child_idx[b + k]), 0))
        else:
            out.append(")")
    return "".join(out) + ";"


def timed(fn, stream):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    a.record(stream)
    fn()
    b.record(stream)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, a.elapsed_time(b)


def kernel_ms(fn):
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        us = getattr(e, "device_time_total", None)
        if us is None:
            us = e.cuda_time_total
        if us:
            out[e.key] = out.get(e.key, 0.0) + us / 1e3
    return out


def bench_config(name, reps):
    cfg = synth.CONFIGS[name]
    st = synth.make_tree(cfg["n_leaves"], cfg["seed"], cfg["kind"])
    C, L = cfg["n_cols"], st.n_leaves
    codes4, pc = synth.simulate_msa(st, 0, C, synth.MsaSpec(cfg["seed"], cfg["p_sub"], cfg["f_gap"], cfg["p_N"]), device="cuda")
    h_codes = torch.empty(codes4.shape, dtype=torch.uint8, pin_memory=True).copy_(codes4)
    del codes4
    torch.cuda.empty_cache()
    h_pc = pc.cpu().numpy()
    ctx = pb.Context(0)
    ctx.set_tree(st.n_nodes, st.root, st.child_off, st.child_idx, st.leaf_row)
    ctx.upload(C, L, h_codes, h_codes.shape[1], h_pc)
    ctx.run_resident(pb.ALGO_FITCH)
    po, pos, info, nucs, _ = ctx.merge_runs()
    tip = int(np.nonzero(st.leaf_row >= 0)[0][L // 3])
    tip_row = int(st.leaf_row[tip])
    nt, nlr = new_tree_of(st, tip)

    class Old:
        n_nodes, root, child_off, child_idx, leaf_row = st.n_nodes, st.root, st.child_off, st.child_idx, st.leaf_row

    ctx.set_tree(nt.n_nodes, nt.root, nt.child_off, nt.child_idx, nlr)
    stream = torch.cuda.ExternalStream(ctx.stream_handle())
    runs = pb.Runs(nt.n_nodes, nt.root, nt.child_off, nt.child_idx, nlr, C, h_codes.numpy(), h_codes.shape[1], h_pc)
    # the dense and runs uploads carry the same root override as the replay: the tip's codes
    ro = synth.unpack_nibbles(h_codes[tip_row:tip_row + 1].cuda(), C)[0].cpu().numpy().astype(np.int8)
    replay = lambda: ctx.upload_replay(Old, po, pos, info, nucs, C, h_pc, tip_row)  # noqa: E731
    dense = lambda: ctx.upload(C, L, h_codes, h_codes.shape[1], h_pc, ro)  # noqa: E731
    enc = lambda: ctx.upload_runs(runs, h_pc, ro)  # noqa: E731
    for f in (replay, dense, enc):  # warm-up of every path and of its buffers
        f()
    rows = {"replay": [], "replay_device": [], "dense": [], "runs": [], "pass": []}
    for _ in range(reps):
        h, d = timed(replay, stream)
        rows["replay"].append(h)
        rows["replay_device"].append(d)
        rows["pass"].append(ctx.run_resident(pb.ALGO_FITCH).total_ms)
        rows["dense"].append(timed(dense, stream)[0])
        rows["runs"].append(timed(enc, stream)[0])
    k_rep = kernel_ms(replay)
    k_runs = kernel_ms(enc)
    plane_bytes = L * ((C + 1023) // 1024) * 1024 / 2
    rep_k = sum(v for k, v in k_rep.items() if any(s in k for s in REPLAY_KERNELS))
    exp_k = sum(v for k, v in k_rep.items() if "expand_runs" in k)
    med = {k: statistics.median(v) for k, v in rows.items()}
    out = dict(config=name, n_leaves=L, n_cols=C, n_pieces=int(len(pos)), n_records=int((info >> 4).astype(np.int64).sum()),
               plane_bytes=plane_bytes, reps=reps,
               replay_call_ms=med["replay"], replay_device_span_ms=med["replay_device"],
               replay_kernels_ms=rep_k + exp_k, replay_records_and_events_kernels_ms=rep_k, replay_expand_kernel_ms=exp_k,
               replay_kernels_plane_write_GBps=plane_bytes / ((rep_k + exp_k) * 1e-3) / 1e9,
               runs_upload_call_ms=med["runs"],
               runs_expand_kernel_ms=sum(v for k, v in k_runs.items() if "expand_runs" in k),
               dense_pinned_upload_call_ms=med["dense"], rerooted_pass_ms=med["pass"],
               replay_faster_than_dense=med["replay"] < med["dense"],
               kernels_of_replay_ms=k_rep, all_rounds=rows)
    runs.close()
    ctx.close()
    del h_codes
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="sars20k,ecoli4k,caterpillar100k")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "reroot_bench.json"))
    args = ap.parse_args()
    res = dict(card=card(), results=[])
    for name in args.configs.split(","):
        r = bench_config(name, args.reps)
        print(json.dumps({k: v for k, v in r.items() if k not in ("kernels_of_replay_ms", "all_rounds")}), flush=True)
        res["results"].append(r)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
