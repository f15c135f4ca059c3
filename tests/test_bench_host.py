"""CPU: host-side logic of bench.py -- the workload plan (chunking, 9-digit QNAME ranges that never overlap between ranks and
chunks), the `config` object both arms print (the driver compares them), and the reference arm end to end on a small sample."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

sys.path.insert(0, ROOT)
import bench  # noqa: E402


@pytest.mark.parametrize("world", [1, 2, 8])
def test_chunk_plan_and_qname_ranges(world):
    cfg = bench.CONFIGS[5]
    plan = bench.chunk_plan(cfg, cfg["records"], cfg["chunk"], world)
    nchunks, per, stride = plan
    assert nchunks * per == cfg["records"] and nchunks == 10
    bases = sorted(bench.chunk_params(cfg, r, k, *plan).qname_base for r in range(world) for k in range(nchunks))
    assert len(set(bases)) == world * nchunks
    assert min(np.diff(bases)) >= stride if len(bases) > 1 else True
    assert stride > per / 2.7                                   # more QNAME numbers than inserts in a chunk (>= 2.7 records per insert)
    assert bases[0] >= 100_000_000 and bases[-1] + stride < 1_000_000_000      # "sim" + 9 digits everywhere


def test_both_arms_print_the_same_config():
    cfg = bench.CONFIGS[5]
    plan = bench.chunk_plan(cfg, cfg["records"], cfg["chunk"], 1)
    a = bench.config_json(cfg, 5, plan, cfg["records"], 1_000_000)
    plan8 = bench.chunk_plan(cfg, cfg["records"], cfg["chunk"], 8)
    b = bench.config_json(cfg, 5, plan8, cfg["records"], 1_000_000)
    assert a == b and "configs[4]" in a["workload"] and a["records_per_gpu_per_step"] == 100_000_000


def test_small_chunk_is_a_prefix_of_the_full_chunk():
    """the in-run parity check regenerates `v` records of every rank's chunk 0: that must be a prefix of the chunk the rank pushes"""
    cfg = bench.CONFIGS[12]
    plan = bench.chunk_plan(cfg, 40_000, 20_000, 2)
    full, foff = bench.gen_chunk(cfg, 1, 0, plan)
    part, poff = bench.gen_chunk(cfg, 1, 0, plan, n_records=5_000)
    n = len(poff) - 1
    assert 5_000 <= n < 5_100 and np.array_equal(poff, foff[:n + 1]) and np.array_equal(part, full[:int(poff[-1])])


def test_dump_outputs_exact_bounded_and_repeatable(tmp_path, monkeypatch):
    """--dump-outputs: values exact in float64 (bytes in float32); an output past the size limit is replaced by a sample
    taken at the same positions on every run"""
    monkeypatch.setattr(bench, "DUMP_LIMIT", 200_000)
    rng = np.random.default_rng(3)
    arrays = {"abundance": rng.random(5_000), "kept_records_last_chunk": 123_456, "profile_delta": [0.5, 0.25], "profile_converged": 1,
              "records_last_chunk": rng.integers(0, 256, 1_000_000, dtype=np.uint8)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b")) == sorted([k + ".npy" for k in arrays] + ["records_last_chunk_sample_index.npy"])
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in names) <= 200_000
    for f in names:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == (np.float32 if f == "records_last_chunk.npy" else np.float64) and np.array_equal(a, b)
    got = {f[:-4]: np.load(tmp_path / "a" / f) for f in names}
    assert np.array_equal(got["abundance"], arrays["abundance"]) and got["kept_records_last_chunk"] == 123_456
    assert got["profile_delta"].tolist() == [0.5, 0.25] and got["profile_converged"] == 1
    idx = got["records_last_chunk_sample_index"].astype(np.int64)
    assert len(idx) > 1000 and np.all(np.diff(idx) > 0)
    assert np.array_equal(got["records_last_chunk"], arrays["records_last_chunk"][idx])


def test_reference_arm_runs_on_the_host(tmp_path):
    if not bench.have_ref_binary():
        pytest.skip("oracle/_ref not built")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "12", "--cpu-sample", "40000",
                        "--cpu-threads", "4", "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["value"] > 0 and line["cpu_baseline"]["kind"] == "reference"
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["config"]["config_index"] == 12
    assert line["cuda_library_mapped"] is False                                      # the arm's own process never mapped the CUDA library


def test_ingest_leg_against_the_null_device(tmp_path):
    """bench.py's file-to-result leg (BGZF file -> `filter | profile` through the CLI, per-phase timers of both processes parsed
    from stderr) run end to end on a build of the CLI over the null device of tests/hostprof (no GPU here): host logic only"""
    import shutil
    if not shutil.which("gcc"):
        pytest.skip("no gcc")
    sys.path.insert(0, os.path.join(ROOT, "tests", "hostprof"))
    import run as hostprof
    cli = hostprof.build()
    cfg = bench.CONFIGS[12]
    plan = bench.chunk_plan(cfg, 60_000, 60_000, 1)
    raw, off = bench.gen_chunk(cfg, 0, 0, plan)
    tlen = bench.target_lengths(cfg)
    out = bench.ingest_entry(cfg, plan, tlen, raw[:int(off[-1])], off, cli=cli, thread_counts=(1, 4))
    assert set(out["threads"]) == {"1", "4"}
    for t in out["threads"].values():
        assert t["rc"] == 0 and t["file_to_result_M_aln_per_s"] > 0 and t["inflate_gbs"] > 0
        assert {"filter: open + header", "filter: stream", "profile: stream", "profile: table"} <= set(t["phases_s"])
