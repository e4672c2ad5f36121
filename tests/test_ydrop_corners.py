"""The y-drop extension kernel source (ydrop_warp.cuh) on the CPU warp emulator, against the oracle's ydrop_extend at the
corners of the penalty range the gapped stage accepts: y-drop 1000..20000, gap open 0..2000, gap extend 10..60. The 16-bit
score frames of the kernel are argued for y-drop up to 20000; mimeo's own runs only ever use 9400 / 400 / 30. Each corner
runs a few random extensions of a single homologous core in both directions (the host's wide-band rerun included) and one
identical-sequence case. These stay well inside the wide kernel's 2048 diagonals; the bands that outgrow it come from
anchors inside repeat pairs and are covered by tests/test_ydrop_band.py."""
import numpy as np
import pytest

from oracle import lastz_oracle as lo
from tests.test_ydrop_emu import check, emu_lib, make_case


@pytest.mark.parametrize('gap_extend', [10, 30, 60])
@pytest.mark.parametrize('gap_open', [0, 400, 2000])
@pytest.mark.parametrize('ydrop', [1000, 9400, 20000])
def test_ydrop_kernel_source_at_penalty_corners(ydrop, gap_open, gap_extend):
    l = emu_lib()
    p = lo.default_params(3000, ydrop=ydrop, gap_open=gap_open, gap_extend=gap_extend)
    rng = np.random.default_rng(ydrop + 7 * gap_open + 131 * gap_extend)
    for _ in range(5):
        core = int(rng.integers(200, 1200))
        flank = [int(rng.integers(0, 400)) for _ in range(4)]
        t, q = make_case(rng, flank, core, float(rng.uniform(0.02, 0.2)), float(rng.uniform(0.0, 0.02)), int(rng.choice([1, 3, 40])),
                         n_frac=float(rng.choice([0.0, 0.01])))
        check(l, t, q, flank[0] + core // 2, min(len(q) - 1, flank[2] + core // 2), p)
    t = rng.integers(0, 4, 1500).astype(np.uint8)
    check(l, t, t.copy(), 750, 750, p)
