"""Cost of profiling input that is not grouped by QNAME (msg_config.collate) against grouped input, on one GPU.

Workload: the config-5 shape of bench.py (alignments to a 1M-gene catalogue, filter -l 80 -p 95 -z 80 --besthit,
--multi proportional), records resident in HBM, pushed as device chunks of 10 M records each.
  grouped : the generator's QNAME-grouped chunks, collate = 0
  coord   : the same chunks, each sorted by (tid, pos) with unmapped records last, collate = 1
Each chunk comes from its own QNAME range, so sorting every chunk by coordinate puts as many reads out of order as
sorting the whole input would; the collation itself does not depend on the input order (hash partition, per-bucket
sort, then a gather from the arena in grouped order).

Per size the two arms alternate (warm-up + `--reps` timed runs each).  Reported: device-event time of the pushes (for
collate: validation + head gather into the arena), the finish (collate: partition, bucket sort, grouped gather and the
pipeline, from the library's MSG_TRACE_FINISH line; grouped: PropSharing only), device memory the context holds after
the finish, and whether both arms give the same integers and abundances (1e-9 relative).

  python profiles/collate_probe.py --records 10000000 100000000 --out collate_probe.json
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
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402

import msamtools_b200 as m  # noqa: E402
from msamtools_b200 import synth  # noqa: E402

CHUNK = 10_000_000
SEED = 20240611
FILT = dict(l=80, p=95, z=80, besthit=True, kept=False, profile=True, multi="proportional")


def gen_chunk(k, n):
    p = synth.make_params("genes1m", n_records=n, seed=SEED + k, qname_base=k * 4 * CHUNK)
    raw, off, _ = synth.generate(p)
    return raw[:int(off[-1])], off


def coord_permute_device(raw_d, off_d):
    """the chunk's records sorted by (tid, pos), unmapped / tid -1 last, on the device with torch"""
    n = off_d.numel() - 1
    starts = off_d[:-1]
    def i32(at):
        b = torch.stack([raw_d[starts + at + j].to(torch.int64) for j in range(4)], 1)
        v = b[:, 0] | (b[:, 1] << 8) | (b[:, 2] << 16) | (b[:, 3] << 24)
        return torch.where(v >= 2 ** 31, v - 2 ** 32, v)
    tid, pos = i32(4), i32(8)
    flag = raw_d[starts + 18].to(torch.int64) | (raw_d[starts + 19].to(torch.int64) << 8)
    unm = ((tid < 0) | ((flag & 4) != 0)).to(torch.int64)
    key = (unm << 62) | ((tid + 1) << 32) | (pos + 1)
    perm = torch.argsort(key, stable=True)
    lens = (off_d[1:] - off_d[:-1])[perm]
    new_off = torch.zeros(n + 1, dtype=torch.int64, device=raw_d.device)
    new_off[1:] = torch.cumsum(lens, 0)
    out = torch.empty_like(raw_d)
    B = 1_000_000
    for lo in range(0, n, B):
        hi = min(n, lo + B)
        p = perm[lo:hi]
        L = lens[lo:hi]
        src0 = off_d[:-1][p]
        base = torch.repeat_interleave(src0 - new_off[lo:hi], L)
        dst = torch.arange(int(new_off[lo]), int(new_off[hi]), device=raw_d.device, dtype=torch.int64)
        out[dst] = raw_d[dst + base]
    out[int(new_off[-1]):] = 0
    return out, new_off


def run_arm(chunks, collate, tlen, trace_file):
    free0, total = torch.cuda.mem_get_info()
    ctx = m.Context(collate=collate, n_targets=len(tlen), **FILT)
    try:
        ctx.mark(0)
        for raw_d, off_d in chunks:
            ctx.push_device(raw_d.data_ptr(), int(off_d[-1]), off_d.data_ptr(), off_d.numel() - 1)
        ctx.mark(1)
        push_ms = ctx.elapsed_ms(0, 1)
        # the library prints the collation phases to fd 2 with MSG_TRACE_FINISH
        sys.stderr.flush()
        saved = os.dup(2)
        with open(trace_file, "w") as fh:
            os.dup2(fh.fileno(), 2)
            try:
                t0 = time.perf_counter()
                ctx.mark(2)
                ab, st = ctx.finish_profile()
                ctx.mark(3)
                finish_wall = (time.perf_counter() - t0) * 1e3
            finally:
                os.dup2(saved, 2); os.close(saved)
        finish_ms = ctx.elapsed_ms(2, 3)
        free1, _ = torch.cuda.mem_get_info()
        trace = open(trace_file).read()
        ph = {}
        mt = re.search(r"\[msg collate\] (\d+) records, (\d+) head bytes: partition ([\d.]+) ms, sort ([\d.]+) ms, grouped gather ([\d.]+) ms, pipeline ([\d.]+) ms", trace)
        if mt:
            ph = dict(head_bytes=int(mt.group(2)), partition_ms=float(mt.group(3)), bucket_sort_ms=float(mt.group(4)),
                      grouped_gather_ms=float(mt.group(5)), pipeline_ms=float(mt.group(6)))
        res = dict(push_ms=push_ms, finish_ms=finish_ms, finish_wall_ms=finish_wall, context_bytes_after_finish=int(free0 - free1), **ph)
        return res, ab, st
    finally:
        ctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, nargs="+", default=[10_000_000, 100_000_000])
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    os.environ["MSG_TRACE_FINISH"] = "1"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    tlen = synth.target_lengths(synth.make_params("genes1m", n_records=1, seed=SEED))
    out = dict(gpu=smi, workload="config-5 shape: 1M genes, filter -l 80 -p 95 -z 80 --besthit, proportional; device-resident 10 M-record chunks",
               sizes=[])
    tmp = tempfile.mkdtemp(prefix="collate_probe_")
    trace_file = os.path.join(tmp, "trace.txt")
    for total in a.records:
        grouped, coord = [], []
        for k in range(0, (total + CHUNK - 1) // CHUNK):
            n = min(CHUNK, total - k * CHUNK)
            raw, off = gen_chunk(k, n)
            raw_d = torch.empty(len(raw) + 64, dtype=torch.uint8, device="cuda")
            raw_d[:len(raw)] = torch.from_numpy(np.ascontiguousarray(raw)).to("cuda")
            raw_d[len(raw):] = 0
            off_d = torch.from_numpy(off.astype(np.int64)).to("cuda")
            c_raw, c_off = coord_permute_device(raw_d, off_d)
            grouped.append((raw_d, off_d)); coord.append((c_raw, c_off))
            del raw, off
        torch.cuda.synchronize()
        runs = {"grouped": [], "coord": []}
        outs = {}
        for rep in range(a.reps + 1):
            for arm in ("grouped", "coord"):
                res, ab, st = run_arm(grouped if arm == "grouped" else coord, arm == "coord", tlen, trace_file)
                if rep:
                    runs[arm].append(res)
                outs[arm] = (ab, st)
        (ab0, s0), (ab1, s1) = outs["grouped"], outs["coord"]
        ints = all(s0[k] == s1[k] for k in ("mapped_inserts", "uniq", "multi", "purged", "iterations", "n_lists", "n_entries"))
        den = np.maximum(np.abs(ab0), np.abs(ab1))
        rel = float(np.max(np.where(den > 0, np.abs(ab0 - ab1) / np.where(den > 0, den, 1), 0)))
        out["sizes"].append(dict(records=total, runs=runs, integers_equal=ints, max_rel_abundance_diff=rel,
                                 stats_grouped={k: v for k, v in s0.items() if k != "delta"}))
        print(json.dumps(out["sizes"][-1]), flush=True)
        del grouped, coord
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(out, fh, indent=1)
    print(json.dumps(dict(gpu=smi)))


if __name__ == "__main__":
    main()
