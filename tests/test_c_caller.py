"""The C-ABI library compiled into and LINKED against a plain C host (tests/c_caller/caller.c), as the
reference driver would be: `gcc caller.c -I include -L sagecal_b200 -ldirac_b200`.  On a CPU box the
host only calls the index helpers and takes the address of every entry point; on the GPU box it also
runs precalculate_coherencies + sagefit_visibilities."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_LAYOUT = os.path.join(ROOT, "tests", "golden", "ref_layout.txt")


def build(tmp_path):
    exe = os.path.join(str(tmp_path), "caller")
    libdir = os.path.join(ROOT, "sagecal_b200")
    cmd = ["gcc", "-O1", "-Wall", "-Werror", "-o", exe, os.path.join(ROOT, "tests", "c_caller", "caller.c"),
           "-I", os.path.join(ROOT, "include"), "-L", libdir, "-ldirac_b200", "-lm",
           "-Wl,-rpath," + libdir]
    subprocess.check_call(cmd)
    return exe


def test_c_host_links_and_calls_host_helpers(tmp_path):
    exe = build(tmp_path)
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and "C_CALLER OK" in out.stdout, (out.returncode, out.stdout, out.stderr)


@pytest.mark.gpu
def test_c_host_runs_the_solver(tmp_path):
    exe = build(tmp_path)
    out = subprocess.run([exe, "gpu"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "C_CALLER OK" in out.stdout, (out.returncode, out.stdout, out.stderr)


def test_link_order_puts_the_hot_path_on_this_library(tmp_path):
    """INTEGRATION.md section 2 on a CPU box: `-ldirac_b200` in front of the reference's library
    (oracle/_ref, the reference CPU path compiled from its own sources) takes over the hot-path
    symbols and leaves the rest with the reference."""
    refdir = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.exists(os.path.join(refdir, "libdirac_ref.so")):
        pytest.skip("oracle/_ref not built (needs /root/reference)")
    exe = os.path.join(str(tmp_path), "link_order")
    libdir = os.path.join(ROOT, "sagecal_b200")
    cmd = ["gcc", "-O1", "-Wall", "-o", exe, os.path.join(ROOT, "tests", "c_caller", "link_order.c"),
           "-I", os.path.join(ROOT, "include"), "-L", libdir, "-ldirac_b200", "-L", refdir,
           "-ldirac_ref", "-ldl", "-lm", "-Wl,-rpath," + libdir, "-Wl,-rpath," + refdir,
           "-Wl,--allow-shlib-undefined"]
    subprocess.check_call(cmd)
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, (out.stdout, out.stderr)
    got = dict(line.split() for line in out.stdout.strip().splitlines())
    ours = [s for s, lib in got.items() if lib == "libdirac_b200.so"]
    theirs = [s for s, lib in got.items() if lib == "libdirac_ref.so"]
    assert sorted(theirs) == ["my_dnrm2", "my_dscal", "update_w_and_nu"], got
    assert len(ours) == len(got) - 3 and "sagefit_visibilities" in ours and "whiten_data" in ours, got


def test_struct_layouts_equal_the_reference_headers(tmp_path):
    """baseline_t, clus_source_t, exinfo_*, elementcoeff, the prefix of persistent_data_t and the
    STYPE_ / DOBEAM_ / STAT_ / SM_ constants: same sizes, offsets and values as a caller compiled
    against the reference's Dirac.h / Dirac_radio.h sees (74 lines compared).  That caller is built
    where the reference sources are (DIRAC_REFERENCE); elsewhere what it printed is read back from
    tests/golden/ref_layout.txt (stored by a run with DIRAC_REF_GOLDEN=record)."""
    src = os.path.join(ROOT, "tests", "c_caller", "layout.c")

    def layout(name, flags):
        exe = os.path.join(str(tmp_path), name)
        subprocess.check_call(["gcc", "-w", "-o", exe, src] + flags)
        return subprocess.run([exe], capture_output=True, text=True, timeout=60).stdout

    ours = layout("ours", ["-I", os.path.join(ROOT, "include")])
    if os.environ.get("DIRAC_REFERENCE"):
        refinc = os.path.join(os.environ["DIRAC_REFERENCE"], "src", "lib")
        want = layout("ref", ["-DUSE_REF", "-I", refinc + "/Dirac", "-I", refinc + "/Radio"])
        if os.environ.get("DIRAC_REF_GOLDEN") == "record":
            with open(REF_LAYOUT, "w") as f:
                f.write(want)
    else:
        with open(REF_LAYOUT) as f:
            want = f.read()
    assert ours == want and len(want.splitlines()) > 70
