"""Cost of exact mode (msg_config.exact) against the default f64-atomic path, on one GPU.

Shapes (bench.py CONFIGS):
  config3 : catalog10k (F = 10^4), plain `profile`
  config5 : genes1m (F = 10^6), filter -l 80 -p 95 -z 80 --besthit fused with the profile
each with --multi=proportional and --multi=equal.  Records are generated once, held in HBM and pushed as device
chunks of 10 M records.  Per shape and mode the two arms (default, exact) alternate: one warm-up and `--reps` timed
runs each.  Reported per run, from device events (the context's marks and the library's MSG_TRACE_FINISH lines):
  finish_ms        msg_finish_profile of the first finish after the pushes (exact: includes the transposition)
  refinish_ms      a second finish on the same state (exact: the incidence is reused)
  transpose_ms     exact only: the one-off transposition (and, equal mode, the in-order sum of the shares)
  loop_ms, per_iteration_ms   PropSharing loop, and per iteration
  longest_incidence           exact only: the most lists holding one feature (the longest serial chain of adds)
The pushes (identical in both arms but for the list keys) are timed too.  A separate check runs exact mode against the
CPU oracle on a QNAME-grouped subsample (>= 1 M records) of each shape and asserts bit-equal abundances.

  python profiles/exact_probe.py --records 20000000 --out exact_probe.json
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
SHAPES = {"config3": dict(preset="catalog10k", opts={}),
          "config5": dict(preset="genes1m", opts=dict(l=80, p=95, z=80, besthit=True, kept=False))}
FINISH_RE = re.compile(r"\[msg finish rank 0\].*init ([\d.]+) ms, loop ([\d.]+) ms, tail ([\d.]+) ms")
EXACT_RE = re.compile(r"\[msg exact\] (\d+) lists, (\d+) entries, longest incidence (\d+): transposition(?: \+ equal shares)? ([\d.]+) ms")


def gen(preset, total):
    chunks = []
    for k in range(0, (total + CHUNK - 1) // CHUNK):
        n = min(CHUNK, total - k * CHUNK)
        p = synth.make_params(preset, n_records=n, seed=SEED + k, qname_base=k * 4 * CHUNK)
        raw, off, _ = synth.generate(p)
        raw = raw[:int(off[-1])]
        raw_d = torch.zeros(len(raw) + 64, dtype=torch.uint8, device="cuda")
        raw_d[:len(raw)] = torch.from_numpy(np.ascontiguousarray(raw)).to("cuda")
        off_d = torch.from_numpy(off.astype(np.int64)).to("cuda")
        chunks.append((raw_d, off_d))
    torch.cuda.synchronize()
    return chunks


def traced_finish(ctx, trace_file):
    sys.stderr.flush()
    saved = os.dup(2)
    with open(trace_file, "w") as fh:
        os.dup2(fh.fileno(), 2)
        try:
            ctx.mark(2)
            ab, st = ctx.finish_profile()
            ctx.mark(3)
        finally:
            os.dup2(saved, 2); os.close(saved)
    return ab, st, ctx.elapsed_ms(2, 3), open(trace_file).read()


def run_arm(chunks, T, mode, opts, exact, trace_file):
    ctx = m.Context(profile=True, multi=mode, n_targets=T, exact=exact, **opts)
    try:
        ctx.mark(0)
        for raw_d, off_d in chunks:
            ctx.push_device(raw_d.data_ptr(), int(off_d[-1]), off_d.data_ptr(), off_d.numel() - 1)
        ctx.mark(1)
        res = dict(push_ms=ctx.elapsed_ms(0, 1))
        ab, st, res["finish_ms"], tr = traced_finish(ctx, trace_file)
        _, _, res["refinish_ms"], tr2 = traced_finish(ctx, trace_file)
        mf = FINISH_RE.search(tr)
        if mf and mode == "proportional":
            res["loop_ms"] = float(mf.group(2))
            res["per_iteration_ms"] = res["loop_ms"] / max(st["iterations"], 1)
        mx = EXACT_RE.search(tr)
        if mx:
            res.update(lists=int(mx.group(1)), entries=int(mx.group(2)), longest_incidence=int(mx.group(3)), transpose_ms=float(mx.group(4)))
        return res, ab, st
    finally:
        ctx.close()


def oracle_check(shape, records):
    """exact mode against the CPU oracle on a QNAME-grouped subsample: bit-equal abundances and equal counters"""
    from oracle import oracle as orc
    orc.load()
    cfg = SHAPES[shape]
    p = synth.make_params(cfg["preset"], n_records=records, seed=SEED + 999)
    raw, off, _ = synth.generate(p)
    T = len(synth.target_lengths(p))
    opts = cfg["opts"]
    idx = None
    if opts:
        idx = orc.filter_stream(raw, off, orc.filter_cfg(**{k: v for k, v in opts.items() if k != "kept"}))
    out = {}
    for mode, share in (("proportional", 3), ("equal", 2)):
        eab, est, eui, ed = orc.profile(raw, off, idx, T, share)
        with m.Context(profile=True, multi=mode, n_targets=T, exact=True, **opts) as ctx:
            ctx.push(raw, off)
            ui, d = ctx.pull_counts()
            ab, st = ctx.finish_profile()
        same = bool(np.array_equal(ab.view(np.uint64), eab.view(np.uint64)) and np.array_equal(d.view(np.uint64), ed.view(np.uint64))
                    and np.array_equal(ui, eui) and all(st[k] == est[k] for k in ("mapped_inserts", "uniq", "multi", "purged", "iterations", "converged")))
        out[mode] = dict(records=records, bit_equal=same, iterations=st["iterations"])
        assert same, (shape, mode)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=20_000_000)
    ap.add_argument("--check-records", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--shapes", nargs="+", default=list(SHAPES))
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    os.environ["MSG_TRACE_FINISH"] = "1"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    out = dict(gpu=smi, records=a.records, shapes={})
    trace_file = os.path.join(tempfile.mkdtemp(prefix="exact_probe_"), "trace.txt")
    for shape in a.shapes:
        cfg = SHAPES[shape]
        t0 = time.time()
        chunks = gen(cfg["preset"], a.records)
        T = len(synth.target_lengths(synth.make_params(cfg["preset"], n_records=1, seed=SEED)))
        res = dict(gen_s=time.time() - t0, oracle=oracle_check(shape, a.check_records), modes={})
        for mode in ("proportional", "equal"):
            runs = {"default": [], "exact": []}
            stats = {}
            for rep in range(a.reps + 1):
                for arm in ("default", "exact"):
                    r, ab, st = run_arm(chunks, T, mode, cfg["opts"], arm == "exact", trace_file)
                    if rep:
                        runs[arm].append(r)
                    stats[arm] = (ab, st)
            (ab0, s0), (ab1, s1) = stats["default"], stats["exact"]
            den = np.maximum(np.abs(ab0), np.abs(ab1))
            rel = float(np.max(np.where(den > 0, np.abs(ab0 - ab1) / np.where(den > 0, den, 1), 0)))
            res["modes"][mode] = dict(runs=runs, iterations=(s0["iterations"], s1["iterations"]), max_rel_default_vs_exact=rel,
                                      features_differing=int(np.count_nonzero(ab0.view(np.uint64) != ab1.view(np.uint64))))
            print(json.dumps({shape: {mode: res["modes"][mode]}}), flush=True)
        out["shapes"][shape] = res
        del chunks
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(out, fh, indent=1)
    print(json.dumps(dict(gpu=smi)))


if __name__ == "__main__":
    main()
