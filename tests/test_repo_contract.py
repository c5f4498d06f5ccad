"""Repository-level contracts checked on the CPU: the product never touches the oracle, the bench's
reference arm prints a well-formed line, the build hook works."""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "fuzzysearch_b200")
    offenders = []
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f), errors="replace").read()
                if re.search(r"^\s*(import|from)\s+oracle\b|fzoracle|libfzoracle|oracle/_ref", text, re.M):
                    offenders.append(os.path.join(dirpath, f))
    assert not offenders, offenders
    header = open(os.path.join(ROOT, "include", "fuzzb200.h")).read()
    assert "oracle" not in header


def test_emulator_never_reaches_the_product_build():
    """tests/emu compiles the product sources with -DFZB_EMU for the CPU suite.  The shipped library must never be
    built that way, and nothing in the package may load the emulated one."""
    mk = open(os.path.join(ROOT, "fuzzysearch_b200", "csrc", "Makefile")).read()
    assert "FZB_EMU" not in mk
    for dirpath, _, files in os.walk(os.path.join(ROOT, "fuzzysearch_b200")):
        for f in files:
            if f.endswith(".py"):
                text = open(os.path.join(dirpath, f)).read()
                assert "emu" not in text.lower().replace("enumerate", ""), os.path.join(dirpath, f)
    for f in ("bench.py", "__graft_entry__.py"):
        assert "libfuzzb200_emu" not in open(os.path.join(ROOT, f)).read() and \
            "FZB_TEST_BACKEND" not in open(os.path.join(ROOT, f)).read(), f
    so = os.path.join(ROOT, "fuzzysearch_b200", "libfuzzb200.so")
    if os.path.exists(so):
        blob = open(so, "rb").read()
        assert b"cuda-emu" not in blob and b"fzb_emu_switch" not in blob


def test_reference_arm_prints_the_contract_line():
    if not os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "fuzzysearch")):
        import pytest
        pytest.skip("oracle/_ref not built (needs /root/reference)")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload",
                          "ascii64m_lev_m20_k2", "--steps", "1", "--warmup", "0", "--cpu-sample-mib", "16",
                          "--ref-cores", "2"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "GB/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["cpu_baseline"]["kind"] == "reference" and line["cpu_baseline"]["cores"] == 2
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"]
    assert line["config"]["workload"] == "ascii64m_lev_m20_k2" and line["metric"] == "haystack_GB_per_s_scanned"
    assert line["steps"] == 1 and len(line["cpu_baseline"]["step_values"]) == 1
    assert line["cpu_baseline"]["single_core_value"] > 0


def test_reference_arm_never_loads_the_product_library(tmp_path):
    """`bench.py --impl reference` must time the reference alone: no fuzzysearch_b200 import, no
    libfuzzb200.so mapped (the driver lists the shared objects each arm loaded)."""
    if not os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "fuzzysearch")):
        import pytest
        pytest.skip("oracle/_ref not built (needs /root/reference)")
    probe = tmp_path / "probe.py"
    probe.write_text(
        "import runpy, sys, atexit\n"
        "def report():\n"
        "    maps = open('/proc/self/maps').read()\n"
        "    sys.stderr.write('PRODUCT_LIB_MAPPED=%d\\n' % ('libfuzzb200' in maps))\n"
        "    sys.stderr.write('PRODUCT_PKG_IMPORTED=%d\\n' % any(m.startswith('fuzzysearch_b200') for m in sys.modules))\n"
        "atexit.register(report)\n"
        "sys.argv = ['bench.py', '--impl', 'reference', '--workload', 'ascii64m_lev_m20_k2', '--steps', '1',\n"
        "            '--warmup', '0', '--cpu-sample-mib', '4', '--ref-cores', '1']\n"
        "runpy.run_path(BENCH, run_name='__main__')\n".replace("BENCH", repr(os.path.join(ROOT, "bench.py"))))
    out = subprocess.run([sys.executable, str(probe)], capture_output=True, text=True, timeout=600)
    assert "PRODUCT_LIB_MAPPED=0" in out.stderr and "PRODUCT_PKG_IMPORTED=0" in out.stderr, out.stderr[-2000:]


def test_graft_entry_exposes_build_and_smoke():
    sys.path.insert(0, ROOT)
    import __graft_entry__ as g
    assert callable(g.build) and callable(g.smoke)


@pytest.mark.gpu
def test_bench_dumps_what_the_last_timed_step_returned(tmp_path, cuda_device):
    """`--steps K` times exactly K searches and `--dump-outputs DIR` writes the final list of the last one; the
    inputs are seeded, so two runs write the same arrays."""
    def run(name, steps):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "ascii64m_lev_m20_k2",
                              "--steps", str(steps), "--warmup", "0", "--e2e-steps", "0", "--no-cpu-baseline",
                              "--dump-outputs", str(tmp_path / name)], capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr[-2000:]
        line = json.loads(out.stdout.strip().splitlines()[-1])
        assert sorted(os.listdir(tmp_path / name)) == ["dist.npy", "end.npy", "start.npy"]
        return line, {n: np.load(tmp_path / name / (n + ".npy")) for n in ("start", "end", "dist")}

    line1, one = run("one", 1)
    line3, three = run("three", 3)
    assert line1["steps"] == 1 and line3["steps"] == 3
    assert line1["parity"]["ok"] and line1["matches_per_step"] == line1["parity"]["final"] == len(one["start"]) > 0
    for n in one:
        assert one[n].dtype == np.float64 and np.array_equal(one[n], three[n]), n
    assert np.all(one["start"] < one["end"]) and np.all(np.diff(one["start"]) > 0)
    assert set(np.unique(one["dist"])) <= {0.0, 1.0, 2.0}
