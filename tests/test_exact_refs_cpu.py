"""The host-side references of tests/test_gpu_production_path.py on hand-computed 2 x 3 grids (no GPU needed)."""
import numpy as np

from test_gpu_production_path import NODATA, exact_checksum, oracle_block_outlets, ordered_sum, reduction_chain
from wdpm_b200 import ascgrid

M64 = 1 << 64


def test_exact_checksum_by_hand():
    w = np.array([[1.0, 0.0, -0.0], [0.5, 2.0, 0.0]])
    # bits(1.0) = 0x3FF0..., bits(-0.0) = 2^63, bits(0.5) = 0x3FE0..., bits(2.0) = 0x4000...; weights 2 * idx + 1
    want = (0x3FF0000000000000 * 1 + (1 << 63) * 5 + 0x3FE0000000000000 * 7 + 0x4000000000000000 * 9) % M64
    assert exact_checksum(w) == want
    # the same rows as the owned part of a larger DEM: first owned row 4, 10 columns per DEM row
    want = sum(b * (2 * ((4 + i) * 10 + j) + 1) for (i, j), b in
               {(0, 0): 0x3FF0000000000000, (0, 2): 1 << 63, (1, 0): 0x3FE0000000000000, (1, 1): 0x4000000000000000}.items()) % M64
    assert exact_checksum(w, global_row0=4, dem_cols=10) == want
    # fp32: the 32-bit patterns, zero-extended
    w32 = w.astype(np.float32)
    want = (0x3F800000 * 1 + 0x80000000 * 5 + 0x3F000000 * 7 + 0x40000000 * 9) % M64
    assert exact_checksum(w32) == want
    # row chunking does not change the value, and the sum wraps modulo 2^64
    big = np.full((2, 3), -np.inf)   # 0xFFF0... times weights 1..11: far above 2^64
    want = sum(0xFFF0000000000000 * (2 * k + 1) for k in range(6)) % M64
    assert exact_checksum(big) == exact_checksum(big, rows_per_chunk=1) == want


def test_reduction_chain_by_hand():
    # 2 x 3 interior: 4 x 5 padded cells; one SM -> 8 reduce blocks: 1 * 1 + 5 + 8 + 8
    assert reduction_chain(4, 5, 1) == 22
    # 1022^2 on 148 SMs: 1184 blocks, ceil(1024/1184) = 1 row and ceil(1024/256) = 4 columns per thread
    assert reduction_chain(1024, 1024, 148) == 4 + 13 + 1184
    # 8000 x 530 on 148 SMs: ceil(8002/1184) = 7 rows of ceil(532/256) = 3 columns
    assert reduction_chain(8002, 532, 148) == 21 + 13 + 1184


def test_oracle_block_outlets_by_hand(oracle):
    """One Drain iteration with the outlet at padded (1, 3), traced by hand through runoff.cl's arithmetic: every value
    is a short dyadic fraction, so the fp64 and fp32 results are exact and equal."""
    for dt in (np.float64, np.float32):
        d = np.array([[10, 10, 10], [10, 10, NODATA]], dtype=dt)
        w = np.array([[0.5, 0.25, 0.125], [0.002, 0.0, 7.0]], dtype=dt)
        D, W = ascgrid.pad_grid(d, dt(NODATA)), ascgrid.pad_grid(w, dt(0))
        md, ms, wet, totals = oracle_block_outlets(oracle, W, D, 0.004, 1, [(1, 3)], np.array([0.125], dtype=dt))
        # 0.002 < 0.004 is cleared; the water on the NODATA cell stays and is not counted
        want = np.array([[0.35888671875, 0.0128173828125, 0.0], [0.05126953125, 0.0, 7.0]], dtype=dt)
        assert np.array_equal(W[1:-1, 1:-1], want)
        assert md == 0.2371826171875      # cell (1, 2): 0.25 -> 0.0128173828125
        assert ms == 0.4229736328125 and wet == 3
        # (0.125 + 0.125) + 0.28125 at sub-pass (1, 2), then + 0 + 0.0457763671875 at (2, 2)
        assert totals.dtype == dt and totals.tolist() == [0.5770263671875]
        assert ordered_sum(np.array([0.5, 0.25, 2.0 ** -30], dtype=dt), dt) == dt(dt(0.75) + dt(2.0 ** -30))
