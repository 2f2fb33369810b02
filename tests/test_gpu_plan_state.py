# -*- coding: utf-8 -*-
"""State a CWT plan must not pick up from outside itself.

* Experiment switches that once chose between kernel variants (tile sizes, butterflies per
  thread, the pass-1 kernel, outputs per thread of the interpolation kernel, the float64
  interpolation window) are gone: setting them before a plan is created changes nothing.
* Kernel launch state (dynamic shared-memory limits, SM counts) belongs to a device: the same
  transform on a second GPU of the process gives the same result as on the first."""
import os
import numpy as np
import pytest

from conftest import relerr
from oracle import ssq_oracle as O

pytestmark = pytest.mark.gpu

# values that selected a non-default variant before the switches were removed
REMOVED = [('SSQB_BPT', '2'), ('SSQB_LOGE', '13'), ('SSQB_P1V', '0'), ('SSQB_INTERP_PPK', '8'),
           ('SSQB_F64_REGWIN', '0')]


@pytest.fixture(scope='module')
def S():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import ssqueezepy_b200 as S_
    return S_


def _np(t):
    return t.detach().cpu().numpy()


def _run(S, dtype, N, env=None, device=0):
    """ssq_cwt of a chirp through a plan created for this call (with `env` set)"""
    import torch
    wav = S.Wavelet(('gmw', {'beta': 12, 'gamma': 3, 'dtype': dtype}))
    scales = 2 ** (np.arange(-10, 70) / 8.)         # 0.42 .. 370
    x = O.chirp(N, 0, dtype)[None]
    old = {k: os.environ.get(k) for k in (env or {})}
    S.CwtPlan._cache.clear()
    try:
        os.environ.update(env or {})
        with torch.cuda.device(device):
            Tx, Wx, _, _, dWx = S.ssq_cwt(x, wav, scales=scales, get_dWx=True)
            torch.cuda.synchronize()
            return _np(Tx), _np(Wx), _np(dWx)
    finally:
        S.CwtPlan._cache.clear()
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _assert_same(ref, out, dtype, what):
    T0, W0, dW0 = ref
    T1, W1, dW1 = out
    assert np.array_equal(W0, W1) and np.array_equal(dW0, dW1), what
    assert np.array_equal(T0 != 0, T1 != 0), what
    assert relerr(T1, T0) < (2e-6 if dtype == 'float32' else 1e-13), what


# The default routes give these scales to the Nyquist-cut, short-block and gridded rows; without
# the gridded and short-block routes they fall to the block, direct and two-pass rows.  n_up = 2^16
# and 2^18: pass 1 of the two-pass rows at 128 and 512 points.
@pytest.mark.parametrize('routes', [{}, {'SSQB_NO_GRID': '1', 'SSQB_NO_SBLK': '1'}],
                         ids=['default', 'block-direct-twopass'])
@pytest.mark.parametrize('dtype,N', [('float32', 40100), ('float32', 150100),
                                     ('float64', 40100), ('float64', 150100)])
def test_removed_switches_have_no_effect(S, dtype, N, routes):
    ref = _run(S, dtype, N, routes)
    for name, value in REMOVED:
        _assert_same(ref, _run(S, dtype, N, dict(routes, **{name: value})), dtype, name)


def test_second_device_same_result(S):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 CUDA devices")
    dtype, N = 'float32', 40200
    _assert_same(_run(S, dtype, N, device=0), _run(S, dtype, N, device=1), dtype, 'cuda:1')
