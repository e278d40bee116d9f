"""Checkpoints without a GPU: the command-line host refuses a resume file it cannot use, and checkpoints under
`chain`, before any solver is created; the ctypes mirror declares the new entry points."""
import os
import subprocess

import pytest

from conftest import gunzip_to


@pytest.fixture(scope="module")
def host_bin():
    from wdpm_b200 import build
    build.build_library()
    return build.build_host()


def _add(host_bin, tmp_path, env):
    dem = gunzip_to("basin5.asc.gz", tmp_path / "basin5.asc")
    argv = ["add", str(dem), "NULL", str(tmp_path / "o.asc"), "NULL", "10", "1.0", "1.0", "1", "1", "0.005", "0"]
    return subprocess.run([str(host_bin)] + argv, capture_output=True, text=True, env=dict(os.environ, **env), timeout=120)


@pytest.mark.parametrize("content,why", [(None, "No such file"), (b"not a checkpoint" * 20, "wrong magic"),
                                         (b"WDPMCKPT\x01\x00\x00\x00" + bytes(40), "truncated")])
def test_resume_refuses_an_unusable_file(host_bin, tmp_path, content, why):
    ck = tmp_path / "ck.bin"
    if content is not None:
        ck.write_bytes(content)
    res = _add(host_bin, tmp_path, {"WDPM_B200_RESUME": str(ck)})
    assert res.returncode == 1 and why in res.stderr, res.stdout[-300:] + res.stderr
    assert "solver" not in res.stdout + res.stderr  # refused before any solver exists
    assert not (tmp_path / "o.asc").exists()


@pytest.mark.parametrize("var", ["WDPM_B200_CHECKPOINT", "WDPM_B200_RESUME"])
def test_chain_refuses_checkpoints(host_bin, tmp_path, var):
    dem = gunzip_to("basin5.asc.gz", tmp_path / "basin5.asc")
    pf = tmp_path / "add.txt"
    pf.write_text(f"add {dem} NULL {tmp_path / 'o.asc'} NULL 10 1.0 1.0 1 1 0.005 0\n")
    res = subprocess.run([str(host_bin), "chain", str(pf)], capture_output=True, text=True, timeout=120,
                         env=dict(os.environ, **{var: str(tmp_path / "ck.bin")}))
    assert res.returncode == 1 and var in res.stderr and "chain" in res.stderr
    assert "solver" not in res.stdout + res.stderr
    assert not (tmp_path / "o.asc").exists()


def test_mirror_declares_the_checkpoint_entry_points():
    from wdpm_b200 import Solver
    from wdpm_b200.stripes import DistributedSolver, StripeSolver
    for cls in (Solver, StripeSolver, DistributedSolver):
        for name in ("checkpoint_arm", "checkpoint_wait", "set_outlet_drains"):
            assert callable(getattr(cls, name, None)), (cls, name)
