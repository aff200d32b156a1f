"""CPU premise of test_gpu_param_range.py at every point of the parameter grid (param_range.py): with a lattice-valued BSK and LUTs
(DESIGN section 4), the oracle's f64 PBS rounded to 2^s equals the exact integer PBS (orc.pbs_exact_batch) on every word, and its
residual stays within 2^(s-4).  At B * l = 52 the lattice unit is only 2^12; the residual of each point is printed."""
import time

import numpy as np
import pytest

from helpers import assert_on_lattice, lattice_bsk, lattice_inputs, lattice_luts, lattice_shift, pbs_steps
from param_range import ROTATION_POINTS


@pytest.mark.parametrize("pt", ROTATION_POINTS, ids=[pt.id for pt in ROTATION_POINTS])
def test_lattice_premise_grid(orc, pt):
    p = pt.params(orc)
    s = lattice_shift(p)
    bsk = lattice_bsk(orc, p, seed=0x5100 + pt.n, nnz=pt.nnz, cmax=pt.cmax)
    luts = lattice_luts(p, 3, seed=0x5101 + pt.B)
    rows = 6 if p.poly_size <= 4096 else 3
    small = lattice_inputs(p, rows, seed=0x5102 + pt.l)
    idx = (np.arange(rows) % 3).astype(np.uint32)
    fk = orc.FourierKey(p, bsk)
    t0 = time.time()
    exact = orc.pbs_exact_batch(p, bsk, small, luts, idx)
    assert not (exact & np.uint64((1 << s) - 1)).any(), "the exact PBS left the lattice"
    got = orc.pbs_f64_batch(p, fk, small, luts, idx)
    assert_on_lattice(got, exact, s, f"oracle f64 {pt.id} ({time.time() - t0:.1f} s)",
                      run_rows=lambda k, r: orc.pbs_f64_batch(p, fk, small[r], luts, idx[r], max_steps=k),
                      ref_rows=lambda k, r: orc.pbs_exact_batch(p, bsk, small[r], luts, idx[r], max_steps=k),
                      n_steps=pbs_steps(p))
