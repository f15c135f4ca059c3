"""Cost of collating across ranks (msg_config.collate = MSG_COLLATE_RANKS) against grouped input on the same ranks.

Run one process per GPU:
  python -m torch.distributed.run --nproc-per-node N profiles/collate_ranks_probe.py --records 10000000 --out DIR

Workload: the config-5 shape of profiles/collate_probe.py (1M-gene catalogue, filter -l 80 -p 95 -z 80 --besthit,
--multi proportional; its generator and device coordinate sort), `--records` records PER RANK as device-resident 10 M
record chunks.  Every chunk has its own QNAME range.
  grouped : the generator's QNAME-grouped chunks, collate = 0 (the multi-GPU path without an exchange)
  coord   : the same chunks sorted by (tid, pos), collate = MSG_COLLATE_RANKS: (N-1)/N of the heads leave each GPU
The arms alternate (warm-up + `--reps` timed runs).  Per rank: push time (device events), the exchange phases and bytes
and the local collation from the MSG_TRACE_FINISH lines, the finish time, device memory held after the finish, and
whether both arms give the same integers (abundances within 1e-9 relative).  Rank 0 writes DIR/collate_ranks_N<N>.json
with every rank's numbers, and the card's name and power limit read in the same run.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "profiles")]
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import msamtools_b200 as m  # noqa: E402
from msamtools_b200 import synth  # noqa: E402
import collate_probe as CP  # noqa: E402

EXCH = re.compile(r"exchange: partition \+ send gather ([\d.]+) ms, agree ([\d.]+) ms, send/recv ([\d.]+) ms, receive scan ([\d.]+) ms; "
                  r"sent (\d+) records, (\d+) head bytes \((\d+) to peers\); received (\d+) records, (\d+) head bytes \((\d+) from peers\)")
LOCAL = re.compile(r"\[msg collate\] (\d+) records, (\d+) head bytes: partition ([\d.]+) ms, sort ([\d.]+) ms, grouped gather ([\d.]+) ms, pipeline ([\d.]+) ms")
INTS = ("mapped_inserts", "uniq", "multi", "purged", "iterations", "n_lists")


def run_arm(chunks, collate, tlen, rank, world, uid, trace_file):
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info()
    ctx = m.Context(collate=collate, n_targets=len(tlen), device=rank, n_ranks=world, rank=rank, nccl_unique_id=uid, **CP.FILT)
    try:
        ctx.mark(0)
        for raw_d, off_d in chunks:
            ctx.push_device(raw_d.data_ptr(), int(off_d[-1]), off_d.data_ptr(), off_d.numel() - 1)
        ctx.mark(1)
        push_ms = ctx.elapsed_ms(0, 1)
        sys.stderr.flush()
        saved = os.dup(2)
        with open(trace_file, "w") as fh:
            os.dup2(fh.fileno(), 2)
            try:
                t0 = time.perf_counter()
                ctx.mark(2)
                ab, st = ctx.finish_profile()
                ctx.mark(3)
                wall = (time.perf_counter() - t0) * 1e3
            finally:
                os.dup2(saved, 2); os.close(saved)
        finish_ms = ctx.elapsed_ms(2, 3)
        free1, _ = torch.cuda.mem_get_info()
        trace = open(trace_file).read()
        res = dict(push_ms=push_ms, finish_ms=finish_ms, finish_wall_ms=wall, context_bytes_after_finish=int(free0 - free1))
        e = EXCH.search(trace)
        if e:
            g = e.groups()
            res.update(partition_send_gather_ms=float(g[0]), agree_ms=float(g[1]), send_recv_ms=float(g[2]), receive_scan_ms=float(g[3]),
                       sent_records=int(g[4]), sent_bytes=int(g[5]), sent_to_peers_bytes=int(g[6]),
                       recv_records=int(g[7]), recv_bytes=int(g[8]), recv_from_peers_bytes=int(g[9]))
        lc = LOCAL.search(trace)
        if lc:
            res.update(local_partition_ms=float(lc.group(3)), local_sort_ms=float(lc.group(4)), local_grouped_gather_ms=float(lc.group(5)),
                       local_pipeline_ms=float(lc.group(6)))
        return res, ab, st
    finally:
        ctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, nargs="+", default=[10_000_000, 100_000_000], help="records per rank")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", default=None, help="directory for collate_ranks_N<N>.json (rank 0)")
    a = ap.parse_args()
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    os.environ["MSG_TRACE_FINISH"] = "1"
    torch.cuda.set_device(rank)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        uid = [m.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        uid = uid[0]
        smi = subprocess.run(["nvidia-smi", "-i", str(rank), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True).stdout.strip()
        tlen = synth.target_lengths(synth.make_params("genes1m", n_records=1, seed=CP.SEED))
        tmp = tempfile.mkdtemp(prefix=f"collate_ranks_probe_{rank}_")
        trace_file = os.path.join(tmp, "trace.txt")
        out = dict(gpu=smi, world=world, workload="config-5 shape per rank: 1M genes, filter -l 80 -p 95 -z 80 --besthit, proportional; "
                   "device-resident 10 M-record chunks", sizes=[])
        for total in a.records:
            grouped, coord = [], []
            nch = (total + CP.CHUNK - 1) // CP.CHUNK
            for k in range(nch):
                n = min(CP.CHUNK, total - k * CP.CHUNK)
                raw, off = CP.gen_chunk(rank * nch + k, n)          # every rank's chunks have their own QNAME ranges
                raw_d = torch.empty(len(raw) + 64, dtype=torch.uint8, device="cuda")
                raw_d[:len(raw)] = torch.from_numpy(np.ascontiguousarray(raw)).to("cuda")
                raw_d[len(raw):] = 0
                off_d = torch.from_numpy(off.astype(np.int64)).to("cuda")
                grouped.append((raw_d, off_d)); coord.append(CP.coord_permute_device(raw_d, off_d))
                del raw, off
            torch.cuda.synchronize()
            runs = {"grouped": [], "coord": []}
            outs = {}
            for rep in range(a.reps + 1):
                for arm in ("grouped", "coord"):
                    res, ab, st = run_arm(grouped if arm == "grouped" else coord, m._lib.MSG_COLLATE_RANKS if arm == "coord" else 0,
                                          tlen, rank, world, uid, trace_file)
                    if rep:
                        runs[arm].append(res)
                    outs[arm] = (ab, st)
            (ab0, s0), (ab1, s1) = outs["grouped"], outs["coord"]
            den = np.maximum(np.abs(ab0), np.abs(ab1))
            rel = float(np.max(np.where(den > 0, np.abs(ab0 - ab1) / np.where(den > 0, den, 1), 0)))
            row = dict(rank=rank, records_per_rank=total, runs=runs, integers_equal=all(s0[k] == s1[k] for k in INTS),
                       max_rel_abundance_diff=rel, stats={k: s1[k] for k in INTS})
            rows = [None] * world
            dist.all_gather_object(rows, row)
            if rank == 0:
                out["sizes"].append(rows)
                print(json.dumps(dict(world=world, records_per_rank=total, ranks=[
                    dict(rank=r["rank"], integers_equal=r["integers_equal"], rel=r["max_rel_abundance_diff"], stats=r["stats"],
                         coord=r["runs"]["coord"][-1], grouped=r["runs"]["grouped"][-1]) for r in rows])), flush=True)
            del grouped, coord
            torch.cuda.empty_cache()
        if rank == 0 and a.out:
            os.makedirs(a.out, exist_ok=True)
            with open(os.path.join(a.out, f"collate_ranks_N{world}.json"), "w") as fh:
                json.dump(out, fh, indent=1)
    finally:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
