"""CPU: the C-ABI library loads, exports every symbol include/msamtools_b200.h declares, and the
product path fails loudly (never falls back) when there is no GPU.  No compute calls here."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import msamtools_b200 as m
from conftest import ROOT


def declared_symbols():
    with open(os.path.join(ROOT, "include", "msamtools_b200.h")) as fh:
        text = re.sub(r"/\*.*?\*/", "", fh.read(), flags=re.S)
    return sorted(set(re.findall(r"\b(msg_[a-z_0-9]+)\s*\(", text)))


def test_exports_match_header():
    lib = m._lib.load()
    decl = declared_symbols()
    assert decl == sorted(m._lib.EXPORTS)
    for name in decl:
        assert getattr(lib, name) is not None
    assert lib.msg_abi_version() == m._lib.MSG_ABI_VERSION


def test_struct_layout_matches_header(tmp_path):
    assert C.sizeof(m._lib.MsgConfig) == 80
    assert C.sizeof(m._lib.MsgProfileStats) == 4 * 6 + 8 * 20 + 16
    assert C.sizeof(m._lib.MsgTiming) == 88
    # field by field against the compiler's view of include/msamtools_b200.h (same names, offsets and sizes)
    import shutil
    import subprocess
    if not shutil.which("gcc"):
        pytest.skip("no gcc")
    structs = {"msg_config": m._lib.MsgConfig, "msg_profile_stats": m._lib.MsgProfileStats, "msg_timing": m._lib.MsgTiming}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "msamtools_b200.h"', 'int main(void) {']
    for cname, ct in structs.items():
        lines.append(f'  printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, _ in ct._fields_:
            lines.append(f'  printf("{cname}.{fname} %zu %zu\\n", offsetof({cname}, {fname}), sizeof((({cname} *)0)->{fname}));')
    lines += ['  return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines) + "\n")
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    got = dict((l.split()[0], [int(x) for x in l.split()[1:]]) for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    for cname, ct in structs.items():
        assert got[cname] == [C.sizeof(ct)]
        for fname, _ in ct._fields_:
            f = getattr(ct, fname)
            assert got[f"{cname}.{fname}"] == [f.offset, f.size], f"{cname}.{fname}"


def test_no_cpu_fallback():
    # in a child process that sees no CUDA device (none installed, or all of them hidden from it)
    import subprocess
    import sys
    code = ("import msamtools_b200 as m\n"
            "try:\n"
            "    m.Context(l=80, n_targets=1)\n"
            "    print('created')\n"
            "except m.MsgError as e:\n"
            "    print(e.code, e.text)\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, check=True)
    out = r.stdout.strip()
    assert out != "created", "a context was created without a CUDA device"
    rc, text = out.split(" ", 1)
    assert int(rc) == m._lib.MSG_ENODEV
    assert "no CPU fallback" in text


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "msamtools_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".c", ".h")):
                with open(os.path.join(dp, f)) as fh:
                    src = fh.read()
                code = "\n".join(l for l in src.splitlines() if "import" in l or "dlopen" in l or "CDLL" in l or "#include" in l)
                assert "oracle" not in code, f"{f} reaches into oracle/"


def test_host_index_helpers():
    from msamtools_b200 import synth
    p = synth.make_params("mixed", n_records=5000, seed=1)
    raw, off, _ = synth.generate(p)
    off2 = m.index_records(raw)
    assert np.array_equal(off, off2)
    n = len(off) - 1
    k = m.split_point(raw, off, n // 2)
    assert 0 < k <= n // 2
    # names differ across the cut, and the record before it is mapped with tid >= 0
    def name(i):
        o = int(off[i]); lq = int(raw[o + 12]); return bytes(raw[o + 36:o + 36 + lq])
    assert name(k - 1) != name(k)
    o = int(off[k - 1])
    assert not (int(raw[o + 18]) & 4) and int(np.frombuffer(raw[o + 4:o + 8].tobytes(), dtype="<i4")[0]) >= 0
    with pytest.raises(m.MsgError):
        m.index_records(raw[:-3])
