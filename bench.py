#!/usr/bin/env python
"""bench.py -- `M alignments/s filter+besthit+profile` on B200 (BASELINE.json metric).

Default workload = BASELINE.json configs[4], the configuration the metric is quoted on: alignments to a
1 M-gene catalogue, sharded on QNAME-group boundaries over the ranks (weak scaling: --records per GPU per step,
default 100 M = 10 chunks of 10 M name-sorted PE150 records, 29.5 GB resident per GPU), through
`filter -l 80 -p 95 -z 80 --besthit | profile --multi=proportional`.  A step = msg_reset, one push per chunk
(decode + filter statistics, best-hit, insert counting), msg_finish_profile (PropSharing loop; at N > 1 the
cross-GPU exchange is inside it).

  value      whole-job throughput, chunks resident in HBM when the timed region starts (CUDA events, max over ranks)
  e2e        same metric through the public host API: pinned HOST chunks pushed with msg_push_async (two in flight),
             the abundance vector read back, all inside the timed region
  roofline   dominant kernel (decode + fused filter statistics): algorithmic bytes per launch / its CUDA-event
             launch time vs the measured HBM peak; `step` = the same arithmetic for the whole step
  cpu_baseline  the reference's own object code (oracle/_ref) on a bounded sample, on the box's host cores
  parity     every run checks its own results before printing: a >= 1 M-record subsample of this very workload goes
             through the same (multi-GPU) path and is compared with the CPU oracle; abundance vectors must be
             bit-identical on all ranks

`--config 1|3|4` select the other BASELINE.json configs (single GPU); `--impl reference` times the reference's CPU
implementation of the selected config on the box's host cores.
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from (which may be read-only)

METRIC = "M alignments/s filter+besthit+profile"
FILTER = dict(l=80, p=95, z=80)
SEED = 13579
QNAME_ORIGIN = 100_000_000          # every QNAME is "sim" + 9 digits on every rank and chunk (same bytes per record everywhere)

CONFIGS = {
    5: dict(preset="genes1m", records=100_000_000, chunk=10_000_000,
            workload="configs[4]: alignments to a 1M-gene catalogue, QNAME-group sharded over the GPUs: "
                     "filter -l 80 -p 95 -z 80 --besthit | profile --multi=proportional",
            ctx=dict(besthit=True, profile=True, multi="proportional", kept=False, **FILTER),
            ref_filter=["filter", "-b", "-u", "-l", "80", "-p", "95", "-z", "80", "--besthit"],
            ref_second=["profile", "--label", "S", "--multi=proportional"]),
    12: dict(preset="community", records=10_000_000, chunk=10_000_000,       # the round-1 bench line: F = 100, flagged-word exchange
             workload="configs[1] data shape (synthetic community PE150, 100 genomes) through filter -l 80 -p 95 -z 80 --besthit | "
                      "profile --multi=proportional",
             ctx=dict(besthit=True, profile=True, multi="proportional", kept=False, **FILTER),
             ref_filter=["filter", "-b", "-u", "-l", "80", "-p", "95", "-z", "80", "--besthit"],
             ref_second=["profile", "--label", "S", "--multi=proportional"]),
    1: dict(preset="community", records=20_000_000, chunk=20_000_000,
            workload="configs[1]: synthetic community PE150, 100 genomes: filter -l 80 -p 95 -z 80 with record output",
            ctx=dict(records=True, kept=False, **FILTER),
            ref_filter=["filter", "-b", "-u", "-l", "80", "-p", "95", "-z", "80"], ref_second=None),
    3: dict(preset="catalog10k", records=20_000_000, chunk=20_000_000,
            workload="configs[2]: name-sorted alignments, 10k references, 30% multi-mappers: profile --multi=proportional",
            ctx=dict(profile=True, multi="proportional", do_filter=False),
            ref_filter=["profile", "--label", "S", "--multi=proportional"], ref_second=None),
    4: dict(preset="community", records=20_000_000, chunk=20_000_000,
            workload="configs[3]: filter -l 80 -p 95 -z 80 fused with coverage --summary, 100 genomes, 1 GPU",
            ctx=dict(coverage=True, coverage_summary=True, kept=False, **FILTER),
            ref_filter=["filter", "-b", "-u", "-l", "80", "-p", "95", "-z", "80"], ref_second=["coverage", "--summary"]),
}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def source_stamp(files):
    h = hashlib.sha1()
    for f in files:
        with open(os.path.join(ROOT, f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,"
         "clocks.mem,temperature.gpu")

    def __init__(self, device, interval_ms=20):
        self.device, self.rows, self.proc, self.interval_ms = device, [], None, interval_ms

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", str(self.interval_ms),
                                          "-i", str(self.device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, pw, mem, temp, reasons = [], [], [], [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
            except (ValueError, IndexError):
                continue
            try:
                mem.append(float(r[9])); temp.append(float(r[10]))
            except (ValueError, IndexError):
                pass
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        # median over the samples taken under load (power above the idle floor), else over all of them
        hot = [s for s, p in zip(sm, pw) if p > 300.0]
        return {"sm_mhz": statistics.median(hot or sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "samples_under_load": len(hot), "power_w_max": max(pw) if pw else None,
                "mem_mhz_min": min(mem) if mem else None, "temp_c_max": max(temp) if temp else None}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", str(rank)))
    return rank, world, local


# ------------------------------------------------------------------------------------------------ synthetic workload
def chunk_plan(cfg, records, chunk_records, world):
    nchunks = max(1, (records + chunk_records - 1) // chunk_records)
    per = records // nchunks
    stride = (int(per / 2.4) // 100_000 + 1) * 100_000            # > inserts per chunk (>= 2.9 records per insert in every preset)
    if QNAME_ORIGIN + world * nchunks * stride >= 1_000_000_000:
        sys.exit("bench.py: records x ranks too large for 9-digit QNAMEs")
    return nchunks, per, stride


def chunk_params(cfg, rank, k, nchunks, per, stride, n_records=None):
    from msamtools_b200 import synth
    return synth.make_params(cfg["preset"], n_records=per if n_records is None else n_records, seed=SEED,
                             qname_base=QNAME_ORIGIN + (rank * nchunks + k) * stride)


def gen_chunk(cfg, rank, k, plan, raw=None, off=None, n_records=None):
    from msamtools_b200 import synth
    p = chunk_params(cfg, rank, k, *plan, n_records=n_records)
    n = p.n_records
    if raw is None:
        raw = np.empty((n + 64) * 330, dtype=np.uint8)
    if off is None:
        off = np.empty(n + 66, dtype=np.uint64)
    raw, off, _ = synth.generate(p, raw, off)
    return raw, off


def target_lengths(cfg):
    from msamtools_b200 import synth
    return synth.target_lengths(synth.make_params(cfg["preset"], n_records=1, seed=SEED))


def gen_threads(world, nchunks):
    cores = os.cpu_count() or 1
    t = max(1, min(nchunks, cores // max(world, 1)))
    try:
        import psutil
        avail = psutil.virtual_memory().available
        t = max(1, min(t, int(avail * 0.45 / (3.6e9 * world))))      # every in-flight chunk holds ~3.3 GB of host memory
    except Exception:
        pass
    return t


# ------------------------------------------------------------------------------------------------ reference arm (CPU)
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "msamtools")


def have_ref_binary():
    return os.path.exists(REF_BIN) and os.access(REF_BIN, os.X_OK)


def scratch_dir(prefix, need_bytes):
    """tmpfs if it has room for the shards (so that the CPU arm does not wait for a disk), else the default temp dir"""
    import shutil
    import tempfile
    for base in ("/dev/shm", tempfile.gettempdir()):
        try:
            if os.path.isdir(base) and shutil.disk_usage(base).free > need_bytes * 1.25 + (1 << 28):
                return tempfile.mkdtemp(prefix=prefix, dir=base)
        except OSError:
            pass
    return tempfile.mkdtemp(prefix=prefix)


def bam_header_blob(names, tlen):
    import struct
    text = ("@HD\tVN:1.6\tSO:queryname\n" + "".join("@SQ\tSN:%s\tLN:%d\n" % (n, int(l)) for n, l in zip(names, tlen))).encode()
    parts = [b"BAM\1", struct.pack("<i", len(text)), text, struct.pack("<i", len(names))]
    for n, l in zip(names, tlen):
        nb = n.encode() + b"\0"
        parts.append(struct.pack("<i", len(nb)) + nb + struct.pack("<i", int(l)))
    return b"".join(parts)


def write_bgzf0(path, blobs):
    """level-0 ("stored") BGZF, so that the reference arm pays (almost) nothing for inflate"""
    import struct
    import zlib
    data = b"".join(bytes(b) for b in blobs)
    with open(path, "wb") as fh:
        for o in range(0, len(data), 0xff00):
            blk = data[o:o + 0xff00]
            co = zlib.compressobj(0, zlib.DEFLATED, -15)
            comp = co.compress(blk) + co.flush()
            fh.write(b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0" + struct.pack("<H", len(comp) + 25))
            fh.write(comp + struct.pack("<II", zlib.crc32(blk) & 0xffffffff, len(blk)))
        fh.write(bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000"))


class RefPipelines:
    """The reference's own object code (oracle/_ref/msamtools: msamtools v1.1.3 sources compiled against the I/O shim)
    run as its documented pipe, one pipe per QNAME-boundary shard (the reference is single-threaded), shards on
    tmpfs as level-0 BGZF BAM so that inflate cost is negligible."""

    def __init__(self, cfg, raw, off, tlen, n_pipes, per_pipe):
        import msamtools_b200 as m
        self.cfg = cfg
        hdr = bam_header_blob([f"g{i:07d}" for i in range(len(tlen))], tlen)
        n = len(off) - 1
        self.dir = scratch_dir("msb200_ref_", int(off[min(n, n_pipes * per_pipe)]) + n_pipes * (len(hdr) + (64 << 20)))
        self.paths, self.n = [], 0
        a = 0
        for k in range(n_pipes):
            want = min(n, a + per_pipe)
            b = m.split_point(raw, off, want) if want < n else n
            if b <= a:
                break
            path = os.path.join(self.dir, f"shard{k}.bam")
            write_bgzf0(path, [hdr, raw[int(off[a]):int(off[b])]])
            self.paths.append(path)
            self.n += b - a
            a = b

    def run(self):
        t0 = time.perf_counter()
        procs = []
        for i, path in enumerate(self.paths):
            out = os.path.join(self.dir, f"out{i}.gz")
            first = [REF_BIN] + self.cfg["ref_filter"]
            if self.cfg["ref_second"] is None:
                if first[1] == "profile":
                    first += ["-o", out]
                f = subprocess.Popen(first + [path], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
                procs.append((f,))
            else:
                f = subprocess.Popen(first + [path], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL)
                g = subprocess.Popen([REF_BIN] + self.cfg["ref_second"] + ["-o", out, "-"], stdin=f.stdout, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
                f.stdout.close()
                procs.append((g, f))
        for ps in procs:
            for p in ps:
                if p.wait() != 0:
                    raise RuntimeError("reference pipeline failed")
        return time.perf_counter() - t0

    def procs_per_pipe(self):
        return 1 if self.cfg["ref_second"] is None else 2

    def describe(self):
        cmd = "msamtools " + " ".join(self.cfg["ref_filter"])
        if self.cfg["ref_second"] is not None:
            cmd += " | msamtools " + " ".join(self.cfg["ref_second"])
        return (f"{self.n} alignments per step as {len(self.paths)} QNAME-boundary shards (level-0 BGZF BAM on tmpfs), one `{cmd}` pipe "
                f"per shard ({self.procs_per_pipe()} process(es) each; the reference is single-threaded); reference arithmetic "
                f"(oracle/_ref = the reference's unmodified C sources), shim I/O (not htslib 1.24)")

    def close(self):
        import shutil
        shutil.rmtree(self.dir, ignore_errors=True)


def oracle_port_run(cfg, raw, off, tlen, sample_records, threads):
    """Fallback when oracle/_ref is absent: the oracle port, one in-memory pipeline per thread (config 5 only)."""
    from concurrent.futures import ThreadPoolExecutor
    import msamtools_b200 as m
    from oracle import oracle as orc
    orc.load()
    n = min(sample_records, len(off) - 1)
    cuts = [0]
    for t in range(1, threads):
        cuts.append(max(m.split_point(raw, off, n * t // threads), cuts[-1]))
    cuts.append(m.split_point(raw, off, n) or n)
    ocfg = orc.filter_cfg(besthit=True, **FILTER)
    shards = [(raw[int(off[a]):int(off[b])], (off[a:b + 1] - off[a]).copy()) for a, b in zip(cuts[:-1], cuts[1:]) if b > a]
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=threads) as ex:      # ctypes releases the GIL inside the C call
        list(ex.map(lambda sh: orc.pipeline(sh[0], sh[1], ocfg, len(tlen), 3)[1]["n_kept"], shards))
    return cuts[-1], time.perf_counter() - t0, len(shards)


def ref_sample(cfg, args, plan, cores):
    """host-side sample of the workload for the CPU arm: chunk 0 of rank 0, `pipes x per` records"""
    procs = 2 if cfg["ref_second"] is not None else 1
    pipes = args.cpu_threads // procs if args.cpu_threads else max(1, min(cores // procs, 16))
    # per pipe: enough records that the reference's per-process fixed cost (parsing a 1 M-line header, writing a 1 M-row table:
    # about a second at config 5) does not dominate its rate
    per = args.cpu_sample // pipes if args.cpu_sample else 2_000_000
    raw, off = gen_chunk(cfg, 0, 0, plan, n_records=pipes * per + 1000)      # the same generator stream as rank 0's chunk 0, continued
    return raw, off, pipes, per


def cuda_library_mapped():
    """whether THIS process has the product's CUDA library mapped (the reference arm must not need it)"""
    try:
        with open("/proc/self/maps") as f:
            return "libmsamtools_b200" in f.read()
    except OSError:
        return None


def config_json(cfg, key, plan, records, n_refs):
    """identical in both arms (the driver compares them): only what defines the workload, nothing measured"""
    return {"workload": cfg["workload"], "config_index": key, "preset": cfg["preset"], "records_per_gpu_per_step": int(records),
            "chunks_per_step": int(plan[0]), "n_references": int(n_refs), "seed": SEED,
            "l2": "inputs larger than L2 (every chunk is ~%.1f GB of records vs 126 MB)" % (plan[1] * 295 / 1e9)}


def run_reference(args):
    rank, world, local = dist_env()
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    cores = os.cpu_count() or 1
    records = args.records or cfg["records"]
    plan = chunk_plan(cfg, records, args.chunk_records or cfg["chunk"], world)
    tlen = target_lengths(cfg)
    raw, off, pipes, per = ref_sample(cfg, args, plan, cores)
    if have_ref_binary() and not args.cpu_port:
        rp = RefPipelines(cfg, raw, off, tlen, pipes, per)
        try:
            for _ in range(max(1, min(args.warmup, 2))):
                rp.run()
            tot_t = sum(rp.run() for _ in range(args.steps))
        finally:
            rp.close()
        n, used, kind, sample = rp.n, rp.procs_per_pipe() * len(rp.paths), "reference", rp.describe()
    else:
        threads = args.cpu_threads or min(cores, 32)
        tot_t = 0.0
        for _ in range(args.steps):
            n, dt, nsh = oracle_port_run(cfg, raw, off, tlen, pipes * per, threads)
            tot_t += dt
        used, kind = threads, "port"
        sample = f"{n} alignments per step in {nsh} QNAME-boundary shards, one in-memory oracle pipeline per thread (oracle/msam_oracle.c)"
    v = n * args.steps / tot_t / 1e6
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "M alignments/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int32+f64", "data": "synthetic",
            "config": config_json(cfg, args.config, plan, records, len(tlen)),
            "cpu_baseline": {"value": v, "unit": "M alignments/s", "cores": used, "kind": kind, "host_cores_available": cores, "sample": sample},
            "e2e": {"value": v, "unit": "M alignments/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "cuda_library_mapped": cuda_library_mapped()}
    print(json.dumps(line))


def cpu_baseline_entry(cfg, args, plan, tlen):
    cores = os.cpu_count() or 1
    raw, off, pipes, per = ref_sample(cfg, args, plan, cores)
    if have_ref_binary() and not args.cpu_port:
        rp = RefPipelines(cfg, raw, off, tlen, pipes, per)
        try:
            rp.run()                                   # page-cache / exec warm-up
            dt = min(rp.run() for _ in range(2))
        finally:
            rp.close()
        out = {"value": rp.n / dt / 1e6, "unit": "M alignments/s", "cores": rp.procs_per_pipe() * len(rp.paths), "kind": "reference",
               "host_cores_available": cores, "sample": rp.describe() + "; best of 2"}
    else:
        threads = args.cpu_threads or min(cores, 32)
        nn, dt, nsh = oracle_port_run(cfg, raw, off, tlen, pipes * per, threads)
        out = {"value": nn / dt / 1e6, "unit": "M alignments/s", "cores": threads, "kind": "port", "host_cores_available": cores,
               "sample": f"first {nn} alignments of chunk 0 in {nsh} QNAME-boundary shards, one in-memory oracle pipeline per thread"}
    if args.config == 5:
        one_n, one_dt, _ = oracle_port_run(cfg, raw, off, tlen, min(1_000_000, len(off) - 1), 1)
        out["oracle_port_single_thread_value"] = one_n / one_dt / 1e6
    return out


# ------------------------------------------------------------------------------------------------ host ingest (R3: file to result)
def write_bgzf_threads(path, blobs, level=1, threads=8):
    """BGZF at `level` with the blocks deflated on worker threads (zlib releases the GIL)"""
    import struct
    import zlib
    from concurrent.futures import ThreadPoolExecutor
    data = b"".join(bytes(b) for b in blobs)
    starts = list(range(0, len(data), 0xff00))

    def pack(group):
        out = []
        for o in group:
            blk = data[o:o + 0xff00]
            co = zlib.compressobj(level, zlib.DEFLATED, -15)
            comp = co.compress(blk) + co.flush()
            out.append(b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0" + struct.pack("<H", len(comp) + 25) + comp +
                       struct.pack("<II", zlib.crc32(blk) & 0xffffffff, len(blk)))
        return b"".join(out)

    groups = [starts[i:i + 64] for i in range(0, len(starts), 64)]
    with ThreadPoolExecutor(max_workers=threads) as ex, open(path, "wb") as fh:
        for part in ex.map(pack, groups):
            fh.write(part)
        fh.write(bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000"))
    return len(data)


def ingest_entry(cfg, plan, tlen, raw, off, cli=None, env_extra=None, thread_counts=(1, 4, 16), with_reference=True):
    """R3 of SURVEY 8d, reported separately from the kernels (north_star): a level-1 BGZF BAM of the workload on tmpfs through the
    drop-in CLI (`filter ... | profile ...`, file to result) with 1 / 4 / 16 host threads -- host read+inflate GB/s and the
    per-phase wall times from the CLI's own timers, alignments/s by wall clock -- and the reference's object code on the same file.
    (`cli` / `env_extra`: the CPU tests run this leg against a build of the CLI on the null device of tests/hostprof.)"""
    import re
    import tempfile
    cli = cli or os.path.join(ROOT, "msamtools_b200", "bin", "msamtools")
    if not os.path.exists(cli):
        return {"unavailable": "msamtools_b200/bin/msamtools not built"}
    n = len(off) - 1
    d = scratch_dir("msb200_ingest_", int(raw.nbytes))
    path = os.path.join(d, "in.bam")
    cores = os.cpu_count() or 1
    payload = write_bgzf_threads(path, [bam_header_blob([f"g{i:07d}" for i in range(len(tlen))], tlen), raw], level=1, threads=min(cores, 16))
    out = {"file": f"{n} alignments of chunk 0, BGZF level 1 on tmpfs", "payload_bytes": int(payload), "file_bytes": os.path.getsize(path), "threads": {}}
    f_args = cfg["ref_filter"][:1] + [a for a in cfg["ref_filter"][1:]]

    def pipe(binary, env):
        t0 = time.perf_counter()
        if cfg["ref_second"] is None:
            a = [binary] + f_args + (["-o", os.path.join(d, "o.gz")] if f_args[0] == "profile" else []) + [path]
            p1 = subprocess.run(a, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, env=env)
            err, rc = p1.stderr, p1.returncode
        else:
            with open(os.path.join(d, "second.err"), "wb") as e2:
                p1 = subprocess.Popen([binary] + f_args + [path], stdout=subprocess.PIPE, stderr=subprocess.PIPE, env=env)
                p2 = subprocess.Popen([binary] + cfg["ref_second"] + ["-o", os.path.join(d, "o.gz"), "-"], stdin=p1.stdout, stdout=subprocess.DEVNULL,
                                      stderr=e2, env=env)
                p1.stdout.close()
                err = p1.stderr.read()
                rc = p2.wait() | p1.wait()
            with open(os.path.join(d, "second.err"), "rb") as e2:
                err += e2.read()
        return time.perf_counter() - t0, err.decode(errors="replace"), rc

    def phases(err):
        """"# phase <command> <name>: <seconds> s" lines of both processes (MSAMTOOLS_TIMING=1)"""
        out = {}
        for c, nm, sec in re.findall(r"^# phase (\S+) (.+?): ([0-9.]+) s\b", err, flags=re.M):
            out[f"{c}: {nm}"] = float(sec)
        return out

    try:
        for thr in thread_counts:
            if thr > cores and thr != 1:
                continue
            env = dict(os.environ, MSAMTOOLS_TIMING="1", MSAMTOOLS_THREADS=str(thr), **(env_extra or {}))
            pipe(cli, env)                                  # warm-up (CUDA context creation is part of every CLI run; page cache)
            dt, err, rc = pipe(cli, env)
            m = re.search(r"host ingest ([0-9.]+) GB in ([0-9.]+) s", err)
            out["threads"][str(thr)] = {"file_to_result_M_aln_per_s": n / dt / 1e6, "wall_s": dt, "rc": rc,
                                        "inflate_gbs": (float(m.group(1)) / float(m.group(2))) if m and float(m.group(2)) > 0 else None,
                                        "phases_s": phases(err)}
        if have_ref_binary() and with_reference:
            dt, _, rc = pipe(REF_BIN, dict(os.environ))
            out["reference_single_pipe"] = {"file_to_result_M_aln_per_s": n / dt / 1e6, "wall_s": dt, "rc": rc,
                                            "note": "the reference's object code on the same file: one process per command, single-threaded inflate (shim I/O)"}
    finally:
        import shutil
        shutil.rmtree(d, ignore_errors=True)
    return out


# ------------------------------------------------------------------------------------------------ parity inside the bench
def close_rel(a, b, rel=1e-9):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return bool(np.all(np.abs(a - b) <= rel * np.maximum(np.abs(a), np.abs(b))))


def parity_check(m, cfg, plan, tlen, rank, world, local, dist, bcast):
    """A subsample of this workload (the first `v` records of every rank's chunk 0, >= 1 M records in total) through the
    same contexts' code path (same options, same n_ranks: fused pass + the in-kernel cross-GPU exchange) vs the CPU
    oracle run over the concatenation of all ranks' subsamples.  Integers / bytes exact, abundances within 1e-9 relative."""
    from oracle import oracle as orc
    opts = cfg["ctx"]
    v = 1_000_000 if world == 1 else 500_000
    raw, off = gen_chunk(cfg, rank, 0, plan, n_records=v)
    uid = bcast(m.nccl_unique_id() if (world > 1 and rank == 0) else None)
    kw = dict(n_targets=len(tlen), device=local, n_ranks=world, rank=rank, nccl_unique_id=uid)
    if opts.get("coverage"):
        kw["target_len"] = tlen
    ab = st = cov = rec = None
    with m.Context(**kw, **opts) as ctx:
        ctx.push(raw, off)
        kept = ctx.kept_count()
        if opts.get("profile"):
            ab, st = ctx.finish_profile()
        if opts.get("coverage"):
            cov = ctx.finish_coverage()
        if opts.get("records"):
            rec = ctx.pull_records()[0]
    res = {"subsample_records_per_rank": int(len(off) - 1)}
    digest = hashlib.sha1(ab.tobytes()).hexdigest() if ab is not None else ""
    if dist is not None:
        box = [None] * world
        dist.all_gather_object(box, (digest, int(kept)))
        digests, kepts = [b[0] for b in box], [b[1] for b in box]
    else:
        digests, kepts = [digest], [int(kept)]
    res["ranks_bit_identical"] = len(set(digests)) == 1
    ok = res["ranks_bit_identical"]
    if rank == 0:
        orc.load()
        raws, offs, base = [raw], [off], int(off[-1])
        for r in range(1, world):
            rr, ro = gen_chunk(cfg, r, 0, plan, n_records=v)
            raws.append(rr); offs.append(ro[1:] + np.uint64(base)); base += int(ro[-1])
        raw_all, off_all = (np.concatenate(raws), np.concatenate(offs)) if world > 1 else (raw, off)
        res["records"] = int(len(off_all) - 1)
        do_filter = opts.get("do_filter", True)
        ocfg = orc.filter_cfg(besthit=bool(opts.get("besthit")), **FILTER) if do_filter else None
        idx = orc.filter_stream(raw_all, off_all, ocfg) if do_filter else None
        ints = {"kept_records": (int(sum(kepts)), int(len(idx)) if idx is not None else int(len(off_all) - 1))}
        if opts.get("profile"):
            eab, est, _, _ = orc.profile(raw_all, off_all, idx, len(tlen), 3)
            ints.update({k: (int(st[k]), int(est[k])) for k in ("mapped_inserts", "uniq", "multi", "purged", "iterations", "converged", "n_lists")})
            res.update(abundance_within_1e9=close_rel(ab, eab), em_iterations=int(est["iterations"]), multi_lists=int(est["n_lists"]),
                       max_rel_err=float(np.max(np.abs(ab - eab) / np.maximum(np.maximum(np.abs(ab), np.abs(eab)), 1e-300))))
            ok = ok and res["abundance_within_1e9"]
        if opts.get("coverage"):
            ecov = orc.coverage(raw_all, off_all, idx, tlen)
            res["coverage_exact"] = bool(all(np.array_equal(a_, b_) for a_, b_ in zip(cov, ecov[:3])))
            ok = ok and res["coverage_exact"]
        if opts.get("records"):
            res["record_bytes_exact"] = bool(bytes(rec) == bytes(orc.emit_records(raw_all, off_all, idx, ocfg)))
            ok = ok and res["record_bytes_exact"]
        res["integers_exact"] = all(a_ == b_ for a_, b_ in ints.values())
        if not res["integers_exact"]:
            res["integer_mismatches"] = {k: v2 for k, v2 in ints.items() if v2[0] != v2[1]}
        ok = ok and res["integers_exact"]
    ok = bool(bcast(ok if rank == 0 else None))
    return ok, res


# ------------------------------------------------------------------------------------------------ output dump
DUMP_LIMIT = 64_000_000             # bytes of .npy files in all


def step_outputs(ctx, cfg, out, kept):
    """What a caller of the timed step receives, by name: the profile (abundance vector and statistics) or the coverage
    summary of the whole step, whichever the config asks for, and the kept-record count and (when the config outputs
    records) the filtered record bytes of the step's last chunk, the only chunk they are kept for."""
    res = {"kept_records_last_chunk": kept}
    if cfg["ctx"].get("profile"):
        ab, st = out
        res["abundance"] = ab
        res.update({"profile_" + k: v for k, v in st.items()})
    elif cfg["ctx"].get("coverage"):
        res.update(zip(("coverage_covered", "coverage_touched", "coverage_total"), out))
    if cfg["ctx"].get("records"):
        res["records_last_chunk"] = ctx.pull_records()[0]
    return res


def dump_outputs(path, arrays):
    """Every array as <path>/<name>.npy in float64 (byte data in float32; both hold the values exactly).  An array that does
    not fit in what is left of DUMP_LIMIT is replaced by a sample of its elements at positions drawn with the workload's seed,
    and the positions go to <name>_sample_index.npy, so that two builds run with the same arguments dump the same elements."""
    os.makedirs(path, exist_ok=True)
    left = DUMP_LIMIT - 256 * (len(arrays) + 1)            # room for the .npy headers
    for name, a in sorted(arrays.items(), key=lambda kv: np.size(kv[1])):
        a = np.asarray(a)
        dt = np.dtype(np.float32 if a.dtype == np.uint8 else np.float64)
        if a.size * dt.itemsize > left:
            idx = np.unique(np.random.default_rng(SEED).integers(0, a.size, left // (dt.itemsize + 8)))
            np.save(os.path.join(path, name + "_sample_index.npy"), idx.astype(np.float64))
            left -= idx.size * 8
            a = a.reshape(-1)[idx]
        np.save(os.path.join(path, name + ".npy"), a.astype(dt))
        left -= a.size * dt.itemsize


# ------------------------------------------------------------------------------------------------ our arm
def run_ours(args):
    import msamtools_b200 as m
    from concurrent.futures import ThreadPoolExecutor, as_completed
    rank, world, local = dist_env()
    if args.gpus != world and world == 1 and args.gpus > 1:
        sys.exit("bench.py --gpus N>1 must be launched with torch.distributed.run (one rank per GPU)")
    key = args.config
    cfg = CONFIGS[key]
    if key not in (5, 12) and world > 1:
        sys.exit("bench.py: --config 1|3|4 are single-GPU lines")
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def bcast(x):
        if dist is None:
            return x
        box = [x]
        dist.broadcast_object_list(box, src=0)
        return box[0]

    def max_over_ranks(x):
        if dist is None:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if dist is None:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.int64, device="cuda")
        dist.all_reduce(t)
        return int(t.item())

    records = args.records or cfg["records"]
    plan = chunk_plan(cfg, records, args.chunk_records or cfg["chunk"], world)
    nchunks = plan[0]
    tlen = target_lengths(cfg)
    has_profile = bool(cfg["ctx"].get("profile"))
    has_cov = bool(cfg["ctx"].get("coverage"))
    has_rec = bool(cfg["ctx"].get("records"))

    # ---- parity first (also warms every code path up)
    parity_ok, parity = (None, {"skipped": "--no-parity"})
    if not args.no_parity:
        parity_ok, parity = parity_check(m, cfg, plan, tlen, rank, world, local, dist, bcast)
        if not parity_ok:
            if rank == 0:
                print(json.dumps({"metric": METRIC, "parity_checked": False, "parity": parity}))
            sys.exit("bench.py: parity check against the oracle FAILED")

    uid = bcast(m.nccl_unique_id() if (world > 1 and rank == 0) else None)
    kw = dict(n_targets=len(tlen), device=local, n_ranks=world, rank=rank, nccl_unique_id=uid)
    if has_cov:
        kw["target_len"] = tlen
    ctx = m.Context(**kw, **cfg["ctx"])

    def barrier():
        ctx.sync()
        if dist is not None:
            import torch
            dist.barrier()
            torch.cuda.synchronize()

    # ---- the rank's shard: nchunks chunks, generated on the host cores, uploaded to HBM; the first e2e_chunks stay in pinned memory
    n_e2e = max(1, min(nchunks, args.e2e_chunks))
    per = plan[1]
    pinned, host_chunks, dev_chunks = [], {}, {}
    for k in range(n_e2e):
        pinned.append((m.PinnedBuffer((per + 64) * 330, device=local), m.PinnedBuffer((per + 66) * 8, device=local)))

    def job(k):
        if k < n_e2e:
            return k, gen_chunk(cfg, rank, k, plan, pinned[k][0].array, pinned[k][1].array.view(np.uint64))
        return k, gen_chunk(cfg, rank, k, plan)

    t_gen = time.perf_counter()
    n_local = raw_bytes = 0
    with ThreadPoolExecutor(max_workers=gen_threads(world, nchunks)) as ex:
        for fut in as_completed([ex.submit(job, k) for k in range(nchunks)]):
            k, (raw, off) = fut.result()
            d_raw, d_off = ctx.device_alloc(raw.nbytes), ctx.device_alloc(off.nbytes)
            ctx.device_upload(d_raw, raw); ctx.device_upload(d_off, off)
            dev_chunks[k] = (d_raw, raw.nbytes, d_off, len(off) - 1)
            n_local += len(off) - 1; raw_bytes += raw.nbytes
            if k < n_e2e:
                host_chunks[k] = (raw, off)
            del raw, off
    t_gen = time.perf_counter() - t_gen
    order = sorted(dev_chunks)

    def finish():
        if has_profile:
            return ctx.finish_profile()
        if has_cov:
            return ctx.finish_coverage()
        ctx.sync()
        return None

    host_t = [0.0, 0.0, 0.0]                       # wall clock spent inside reset / pushes / finish (diagnostics: where a step's time goes on the host)

    def step_resident():
        t_a = time.perf_counter()
        ctx.reset()
        t_b = time.perf_counter()
        for k in order:
            ctx.push_device_async(*dev_chunks[k])
        ctx.wait()
        t_c = time.perf_counter()
        out_ = finish()
        t_d = time.perf_counter()
        host_t[0] += t_b - t_a; host_t[1] += t_c - t_b; host_t[2] += t_d - t_c
        return out_

    for _ in range(args.warmup):
        out = step_resident()
    ctx.timing(reset=True)
    host_t[:] = [0.0, 0.0, 0.0]
    # every rank samples its own GPU; the samplers start BEFORE the barrier: round 1 started rank 0's nvidia-smi between the
    # barrier and the first timed step, and the other ranks' timed regions then contained their wait for rank 0 (tens of ms of
    # process start-up on an 8-GPU node, i.e. +1 ms per step of a 20 x 1 ms region: the "N = 2 anomaly" of round 1)
    sampler = ClockSampler(local, 20 if rank == 0 else 100)
    sampler.start()
    time.sleep(0.05)
    barrier()
    ctx.mark(0)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = step_resident()
    ctx.mark(1)
    dev_ms = ctx.elapsed_ms(0, 1)
    barrier()
    wall_ms = 1e3 * (time.perf_counter() - t0)
    tim = ctx.timing(reset=True)
    kept_last = int(ctx.kept_count())
    step_ms = max_over_ranks(max(dev_ms, 0.0) / args.steps)
    wall_step_ms = max_over_ranks(wall_ms / args.steps)
    n_total = sum_over_ranks(n_local)
    value = n_total / (step_ms * 1e-3) / 1e6
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, step_outputs(ctx, cfg, out, kept_last))

    # the job's own result must be the same bits on every rank, and obey the conservation laws of the profile
    job_check = {}
    if has_profile:
        ab, st = out
        digest = hashlib.sha1(ab.tobytes()).hexdigest()
        if dist is not None:
            box = [None] * world
            dist.all_gather_object(box, digest)
        else:
            box = [digest]
        job_check = {"ranks_bit_identical": len(set(box)) == 1,
                     "uniq_plus_multi_eq_inserts": int(st["uniq"]) + int(st["multi"]) == int(st["mapped_inserts"]),
                     "abundance_sum_eq_inserts_minus_purged": bool(abs(ab.sum() - (st["mapped_inserts"] - st["purged"])) <= 1e-6 * max(st["mapped_inserts"], 1)),
                     "inserts": int(st["mapped_inserts"]), "multi_lists": int(st["n_lists"]), "purged": int(st["purged"]),
                     "em_iterations": int(st["iterations"]), "em_converged": int(st["converged"])}
        parity_ok = bool(parity_ok is not False and all(v for k2, v in job_check.items() if isinstance(v, bool))) if parity_ok is not None else None

    # ---- end to end: pinned HOST chunks through the public push API, H2D + D2H inside the timed region
    e2e_order = sorted(host_chunks)
    rec_out = m.PinnedBuffer(max(host_chunks[k][0].nbytes for k in e2e_order) + 4096, device=local) if has_rec else None

    def step_e2e():
        ctx.reset()
        for k in e2e_order:
            ctx.push_async(*host_chunks[k])
        ctx.wait()
        res = finish()
        if has_rec:
            ctx.pull_records(rec_out.array)          # the filtered records come back into pinned host memory
        return res

    n_e2e_local = sum(len(host_chunks[k][1]) - 1 for k in e2e_order)
    e2e = None
    if args.e2e_steps > 0:
        for _ in range(max(1, min(args.warmup, 2))):
            step_e2e()
        ctx.timing(reset=True)
        barrier()
        t0 = time.perf_counter()
        e2e_steps = max(1, min(args.steps, args.e2e_steps))
        for _ in range(e2e_steps):
            step_e2e()
        barrier()
        e2e_ms = max_over_ranks(1e3 * (time.perf_counter() - t0) / e2e_steps)
        tim2 = ctx.timing(reset=True)
        n_e2e_total = sum_over_ranks(n_e2e_local)
        e2e_bytes = sum(host_chunks[k][0].nbytes for k in e2e_order)
        e2e = {"value": n_e2e_total / (e2e_ms * 1e-3) / 1e6, "unit": "M alignments/s", "ms_per_step": e2e_ms,
               "records_per_gpu_per_step": int(n_e2e_local), "chunks_per_step": len(e2e_order),
               "h2d_bytes_per_step": int(tim2["h2d_bytes"] // e2e_steps), "d2h_bytes_per_step": int(tim2["d2h_bytes"] // e2e_steps),
               "h2d_gbs": (tim2["h2d_bytes"] / e2e_steps) / (e2e_ms * 1e-3) / 1e9,
               "bam_gbs_per_gpu": e2e_bytes / (e2e_ms * 1e-3) / 1e9,
               "api": "msg_push_async x chunks (pinned host buffers, two chunks in flight) + msg_wait + msg_finish_*",
               "h2d_mode": ("zero-copy: decode windows pulled from the pinned host chunks over PCIe (h2d bytes = window chunks requested + offset "
                            "index DMA; SEQ/QUAL never leave the host)") if tim2.get("zero_copy_chunks", 0) else "staged: whole chunks DMA'd into two device slots"}
    clocks = sampler.stop()                             # sampled across both timed regions (resident + e2e)
    per_rank = {"rank": rank, "decode_launch_ms": tim["decode_ms"] / max(tim["decode_launches"], 1), "step_ms": max(dev_ms, 0.0) / args.steps,
                "host_ms_per_step": {"reset": 1e3 * host_t[0] / args.steps, "push": 1e3 * host_t[1] / args.steps, "finish": 1e3 * host_t[2] / args.steps},
                "sm_mhz": clocks["sm_mhz"], "mem_mhz_min": clocks.get("mem_mhz_min"), "temp_c_max": clocks.get("temp_c_max"), "reasons": clocks["reasons"]}
    if dist is not None:
        ranks_info = [None] * world
        dist.all_gather_object(ranks_info, per_rank)
    else:
        ranks_info = [per_rank]

    for k in order:
        ctx.device_free(dev_chunks[k][0]); ctx.device_free(dev_chunks[k][2])

    if rank == 0:
        peak, peak_src = peaks()
        launches = max(tim["decode_launches"], 1)
        dec_ms = tim["decode_ms"] / launches
        alg_per_launch = tim["alg_bytes"] / launches
        achieved = alg_per_launch / (dec_ms * 1e-3) / 1e9
        alg_step = tim["alg_bytes"] / args.steps
        if has_rec:       # A_out(rec) = 8 + B_rec + keep * B_rec (SURVEY 8d): the records are read once and the survivors written once
            alg_step = raw_bytes + 8 * n_local + raw_bytes * kept_last / max(n_local, 1)
        traffic = traffic_stale = None
        tpath = os.path.join(ROOT, "profiles", "decode_traffic.json")
        if os.path.exists(tpath):
            with open(tpath) as fh:
                tj = json.load(fh)
            if tj.get("config_index") == key and abs(tj.get("records_per_launch", 0) - n_local / nchunks) < 1000:
                if tj.get("source_stamp") == source_stamp(["msamtools_b200/csrc/decode.cuh", "msamtools_b200/csrc/common.cuh"]):
                    traffic = tj.get("dram_bytes_per_launch")
                else:       # the kernel source changed after the ncu capture: `traffic` stays null, the last capture is shown as what it is
                    traffic_stale = {"dram_bytes_per_launch": tj.get("dram_bytes_per_launch"), "measured_on_source_stamp": tj.get("source_stamp"),
                                     "note": "ncu capture of an EARLIER build of this kernel (decode.cuh changed since); not this run's traffic"}
        line = {
            "metric": METRIC, "value": value, "unit": "M alignments/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int32+f64", "data": "synthetic",
            "config": config_json(cfg, key, plan, records, len(tlen)),
            "run": {"records_per_gpu": int(n_local), "raw_bytes_per_gpu": int(raw_bytes), "kept_records_last_chunk": kept_last,
                    "wall_ms_per_step": wall_step_ms, "generation_s": round(t_gen, 1),
                    "host_ms_per_step": {"reset": 1e3 * host_t[0] / args.steps, "push": 1e3 * host_t[1] / args.steps, "finish": 1e3 * host_t[2] / args.steps},
                    "job": job_check},
            "parity_checked": bool(parity_ok) if parity_ok is not None else False, "parity": parity,
            "roofline": {"bound": "hbm", "kernel": "decode_kernel (record decode + fused filter statistics)",
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
                         "traffic": traffic, "traffic_last_capture": traffic_stale, "alg_bytes_per_launch": alg_per_launch, "launch_ms": dec_ms, "launches_per_step": launches / args.steps,
                         "full_scan_gbs": (raw_bytes + 8 * n_local) / nchunks / (dec_ms * 1e-3) / 1e9, "kernel_share_of_step": dec_ms * launches / args.steps / step_ms,
                         "step": {"alg_bytes": alg_step, "achieved": alg_step / (step_ms * 1e-3) / 1e9, "frac": alg_step / (step_ms * 1e-3) / 1e9 / peak}},
            "e2e": e2e,
            "gpu_launches": int(tim["kernel_launches"]),
            "clocks": clocks,
            "ranks": ranks_info,
        }
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_entry(cfg, args, plan, tlen)
        if world == 1 and not args.no_ingest:
            line["ingest"] = ingest_entry(cfg, plan, tlen, *host_chunks[0])
        print(json.dumps(line))
    ctx.close()
    if rec_out is not None:
        rec_out.close()
    for a, b in pinned:
        a.close(); b.close()
    if dist is not None:
        dist.destroy_process_group()
    if parity_ok is False:
        sys.exit("bench.py: result checks FAILED")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=5, choices=sorted(CONFIGS), help="BASELINE.json config (1-based: 5 = the 1M-gene catalogue job the metric is quoted on)")
    ap.add_argument("--records", type=int, default=0, help="alignments per GPU per step (default: the config's)")
    ap.add_argument("--chunk-records", type=int, default=0, help="alignments per pushed chunk")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--e2e-chunks", type=int, default=3, help="chunks kept in pinned host memory for the end-to-end leg")
    ap.add_argument("--cpu-sample", type=int, default=0)
    ap.add_argument("--cpu-threads", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-ingest", action="store_true", help="skip the BGZF file-to-result (host ingest) leg")
    ap.add_argument("--cpu-port", action="store_true", help="time the in-memory oracle port even when oracle/_ref exists")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one returned as DIR/<name>.npy "
                                                          "(float32/float64, at most 64 MB in all; a larger output is sampled): the "
                                                          "step's profile or coverage summary, and the kept count and records of its "
                                                          "last chunk")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
