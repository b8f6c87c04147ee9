"""The shared-memory ring of the temporally blocked kernel (csrc/lbm_tb.cuh), on the CPU.

Each stage keeps a population only as long as the next stage pulls it: 2 slots for the populations pulled from x+1,
3 for those that stay in their column, 4 for those pulled from x-1.  tests/cpp/tb_ring_schedule.cpp replays both
marches with the kernel's own ring functions and checks that every pull gets the cell it asks for, that no slot is
read and written between the same two barriers, and that the ghost rows' one-off fill reaches every slot.  The ring
size is what lets four blocks of 128 rows share an SM at depth 3; the build log pins that the kernel keeps its
registers to the 128 that four blocks allow, without a spill."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "highperformancecomputing-latticeboltzmannmethod_b200", "csrc")
CUDA_INC = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
PTXAS_LOG = os.path.join(CSRC, "build", "lbm_tb.o.ptxas.log")


@pytest.fixture(scope="module")
def schedule_exe(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("cpp") / "tb_ring_schedule")
    subprocess.run(["g++", "-std=c++17", "-O1", "-I" + CSRC, "-I" + CUDA_INC,
                    os.path.join(ROOT, "tests", "cpp", "tb_ring_schedule.cpp"), "-o", exe], check=True)
    return exe


def test_every_pull_gets_its_cell_and_no_slot_is_read_and_written_between_two_barriers(schedule_exe):
    """Both marches, depths 2 and 3, chunks of 1 .. 64 columns: every step, ramp-up and ramp-down included; before
    them, tb_ring_fill into a ring of NaN."""
    out = subprocess.run([schedule_exe], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    assert re.fullmatch(r"ok \d+\n", out.stdout) and int(out.stdout.split()[1]) > 10000, out.stdout


def test_four_depth_three_rings_fit_an_sm(schedule_exe):
    ring = int(subprocess.run([schedule_exe, "bytes"], capture_output=True, text=True, check=True).stdout)
    assert ring <= 2 * 27 * 128 * 8  # 55 296 B per block
    assert 4 * (ring + 1024) <= 228 * 1024  # + the 1 KB the runtime reserves per block


def kernel_properties(log, template_args):
    """{registers, spill_stores, spill_loads} of the k_tb instantiation whose mangled template arguments are given."""
    text = open(log).read()
    m = re.search(r"Function properties for (\S*k_tbI%sEEvNS_6TbArgsEi)\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, "
                  r"(\d+) bytes spill loads\n.*?Used (\d+) registers" % re.escape(template_args), text, re.S)
    assert m, "k_tb<%s> not in %s" % (template_args, log)
    return {"registers": int(m.group(5)), "spill_stores": int(m.group(3)), "spill_loads": int(m.group(4))}


def test_the_default_depth_three_kernel_fits_128_registers_without_a_spill():
    """k_tb<3, 128, FORCED = false, SKEW = true, FUSED = false>: what the 4096 x 8192 slab runs."""
    if not os.path.exists(PTXAS_LOG):
        pytest.skip("no ptxas log: the library was not built in this tree (make -C csrc writes it)")
    p = kernel_properties(PTXAS_LOG, "Li3ELi128ELb0ELb1ELb0E")
    assert p["registers"] <= 128 and p["spill_stores"] == 0 and p["spill_loads"] == 0, p
