"""CPU: row stripes at the partition's limits.

* The striped-oracle emulation of tests/test_stripes_cpu.py at world 8 on 70 rows: every stripe holds exactly 9
  padded rows, the fewest the library accepts (kHaloBelow + kHaloAbove), so every owned row of a middle stripe is
  exported (rows 0-5 up, rows 6-8 down). The assembled grid must equal the single-domain oracle for every module.
* plan_stripes (the Python partition) against set_create of the command-line host (wdpm_b200/host/wdpm_host.c),
  compiled here with stub library calls: for 16..200 rows and 2..8 requested stripes both must cut the same bands,
  and where plan_stripes refuses a count, set_create must fall back to the largest count plan_stripes accepts. A
  difference would give a Python host and the command line different partitions of the same DEM.
"""
import shutil
import subprocess
from pathlib import Path

import pytest
import torch.multiprocessing as mp

from test_stripes_cpu import _free_port, _worker
from wdpm_b200 import stripes

ROOT = Path(__file__).resolve().parent.parent


def test_nine_row_plan_shapes():
    """The shapes the GPU tests rely on: 9N - 2 rows give N stripes of 9 padded rows; 9N - 1, 9N and 9N + 1 rows give
    a last stripe of 10, 11 and 12 rows and 9 rows elsewhere. 9N - 3 and 9N - 4 rows still make 3N row triples, but
    the last is partial: N stripes would leave 8 or 7 rows to the last one, which the library refuses, so N is
    refused."""
    for n in (2, 3, 4, 8):
        assert [p.rows for p in stripes.plan_stripes(9 * n - 2, n)] == [9] * n
        for extra, last in ((1, 10), (2, 11), (3, 12)):
            assert [p.rows for p in stripes.plan_stripes(9 * n - 2 + extra, n)] == [9] * (n - 1) + [last]
        for rows in (9 * n - 3, 9 * n - 4, 9 * n - 5):
            with pytest.raises(ValueError):
                stripes.plan_stripes(rows, n)


def test_every_stripe_gets_nine_rows():
    for rows in range(16, 201):
        for n in range(1, 9):
            try:
                plan = stripes.plan_stripes(rows, n)
            except ValueError:
                assert rows + 2 < 9 * n
                continue
            assert min(p.rows for p in plan) >= 9 and sum(p.rows for p in plan) == rows + 2, (rows, n)


@pytest.mark.parametrize("module", [0, 1, 2, 3], ids=["add", "subtract", "drain", "drain-set"])
def test_striped_oracle_on_eight_nine_row_stripes(module):
    world, rows, cols = 8, 70, 40
    assert {p.rows for p in stripes.plan_stripes(rows, world)} == {9}
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, rows, cols, module, 7, 4321 + module, q)) for r in range(world)]
    for p in procs:
        p.start()
    ok, ndiff = q.get(timeout=300)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    assert ok, f"{ndiff} cells differ"


# set_create of the host, with the library calls it makes replaced by stubs that record each stripe's config
_HARNESS = r"""
#define main wdpm_host_main
#include "wdpm_host.c"
#undef main

static int n_created, rec_row0[MAX_GPUS], rec_rows[MAX_GPUS];

const char *wdpm_last_error(void) { return "stub"; }
int wdpm_device_count(void) { return MAX_GPUS; }
int wdpm_create(const wdpm_config *cfg, wdpm_solver **out)
{
    rec_row0[n_created] = cfg->stripe_row0;
    rec_rows[n_created] = cfg->stripe_rows;
    *out = (wdpm_solver *)(intptr_t)(++n_created);
    return WDPM_OK;
}
int wdpm_stripe_band(wdpm_solver *s, int32_t *band_row0, int32_t *band_rows, int32_t *owned_row0, int32_t *owned_rows)
{
    (void)s;
    *band_row0 = *band_rows = *owned_row0 = *owned_rows = 0;
    return WDPM_OK;
}
int wdpm_stripe_export(wdpm_solver *s, wdpm_stripe_endpoint *self) { (void)s; memset(self, 0, sizeof *self); return WDPM_OK; }
int wdpm_stripe_connect(wdpm_solver *s, const wdpm_stripe_endpoint *above, const wdpm_stripe_endpoint *below)
{
    (void)s; (void)above; (void)below;
    return WDPM_OK;
}

int main(int argc, char **argv)
{
    const int r0 = atoi(argv[1]), r1 = atoi(argv[2]), n0 = atoi(argv[3]), n1 = atoi(argv[4]);
    for (int rows = r0; rows <= r1; rows++)
        for (int want = n0; want <= n1; want++) {
            wdpm_config cfg;
            memset(&cfg, 0, sizeof cfg);
            cfg.rows = rows;
            cfg.cols = 5;
            solver_set ss;
            n_created = 0;
            set_create(&ss, cfg, want);
            printf("%d %d %d", rows, want, ss.n);
            for (int g = 0; g < n_created; g++) printf(" %d %d", rec_row0[g], rec_rows[g]);
            printf("\n");
        }
    (void)argc;
    return 0;
}
"""


@pytest.fixture(scope="module")
def set_create_bin(tmp_path_factory):
    gcc = shutil.which("gcc") or "/usr/bin/gcc"
    d = tmp_path_factory.mktemp("set_create")
    src = d / "harness.c"
    src.write_text(_HARNESS)
    exe = d / "harness"
    # only set_create and what it calls are kept (--gc-sections), so the library's other entry points need no stubs
    cmd = [gcc, "-O1", "-std=c11", "-ffunction-sections", "-fdata-sections", "-Wl,--gc-sections",
           "-I", str(ROOT / "include"), "-I", str(ROOT / "wdpm_b200" / "host"), str(src), "-o", str(exe), "-lm", "-lpthread"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    return exe


def test_plan_stripes_equals_the_hosts_set_create(set_create_bin):
    res = subprocess.run([str(set_create_bin), "16", "200", "2", "8"], capture_output=True, text=True, timeout=60)
    assert res.returncode == 0, res.stderr
    lines = res.stdout.split("\n")[:-1]
    assert len(lines) == 185 * 7
    lowered = 0
    for ln in lines:
        v = [int(x) for x in ln.split()]
        rows, want, n, bands = v[0], v[1], v[2], list(zip(v[3::2], v[4::2]))
        assert len(bands) == n, ln
        # set_create lowers the count to the largest one plan_stripes accepts
        expect_n = want
        while expect_n > 1:
            try:
                stripes.plan_stripes(rows, expect_n)
                break
            except ValueError:
                expect_n -= 1
        lowered += expect_n < want
        assert n == expect_n, ln
        if n == 1:
            assert bands == [(0, 0)], ln   # a plain solver: no stripe fields
            continue
        plan = stripes.plan_stripes(rows, n)
        assert bands == [(p.row0, p.rows) for p in plan], (ln, plan)
        assert min(r for _, r in bands) >= 9, ln   # wdpm_create refuses a stripe of fewer rows
    assert lowered > 0
