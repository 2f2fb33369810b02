# -*- coding: utf-8 -*-
"""`bench.py --dump-outputs`: the stored sample must be the same on every run (two builds are
compared element for element) and fit its byte budget."""
import numpy as np
import torch

import bench


def test_dump_index_fixed_sorted_in_range():
    total, n = 3_072_000_000, 3_750_000            # C4's Tx, float32 budget
    i = bench.dump_index(total, n)
    assert len(i) == n and i.dtype == np.int64
    assert np.all(np.diff(i) > 0) and i[0] >= 0 and i[-1] < total
    assert np.array_equal(i, bench.dump_index(total, n))
    assert bench.dump_index(10, 10) is None


def test_output_arrays_whole_or_sampled():
    t = torch.randn(2, 3, 50, dtype=torch.complex64)
    a = bench.output_arrays({'Tx': t, 'Wx': 2 * t})
    assert a['Tx'].dtype == np.float32 and a['Tx'].shape == (2, 3, 50, 2)
    assert np.array_equal(a['Wx'][..., 1], (2 * t).imag.numpy())
    t64 = t.to(torch.complex128)
    b = bench.output_arrays({'Tx': t64, 'Wx': t64}, budget=2 * 16 * 40)
    idx = bench.dump_index(t64.numel(), 40)
    assert b['Tx'].dtype == np.float64 and b['Tx'].shape == (40, 2)
    assert np.array_equal(b['Tx'][:, 0], t64.reshape(-1).real.numpy()[idx])
    assert sum(v.nbytes for v in b.values()) <= 2 * 16 * 40
