"""CPU: the update-schedule field of wdpm_config - the ctypes mirror and the C header agree on where it lives, and
it takes a reserved slot: the struct keeps its size and the ABI its version."""
import ctypes as C
import shutil
import subprocess
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


def test_config_mirror_matches_the_header(tmp_path):
    from wdpm_b200 import solver
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    src = tmp_path / "offsets.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "wdpm_b200.h"\n'
                   "int main(void) { printf(\"%zu %zu %zu %d %d %d\\n\", sizeof(wdpm_config), offsetof(wdpm_config, schedule),\n"
                   "    offsetof(wdpm_config, reserved), WDPM_ABI_VERSION, WDPM_SCHEDULE_OPENCL, WDPM_SCHEDULE_SERIAL); return 0; }\n")
    exe = tmp_path / "offsets"
    subprocess.run([cc, "-I", str(ROOT / "include"), str(src), "-o", str(exe)], check=True)
    size, off_sched, off_res, abi, opencl, serial = (int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True,
                                                                                      check=True).stdout.split())
    assert size == C.sizeof(solver._Config) == 88
    assert off_sched == solver._Config.schedule.offset
    assert off_res == solver._Config.reserved.offset
    assert abi == 1
    assert (opencl, serial) == (solver.SCHED_OPENCL, solver.SCHED_SERIAL) == (0, 1)


def test_zeroed_config_keeps_the_opencl_schedule():
    from wdpm_b200 import solver
    assert solver._Config().schedule == solver.SCHED_OPENCL
