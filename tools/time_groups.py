"""Step time of one ssq_cwt configuration for several group sizes (SSQB_GROUP, read per call).
Usage: python tools/time_groups.py N na dtype wavelet B g1,g2,...   (0 = one group)"""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import ssqueezepy_b200 as S
from ssqueezepy_b200 import _lib
from ssqueezepy_b200._ssq_cwt import ssq_cwt_host_params
from ssqueezepy_b200.algos import make_reassign_desc
from ssqueezepy_b200.utils.common import p2up, EPS32, EPS64
from oracle import ssq_oracle as O

N, na, dtype, name, B = int(sys.argv[1]), int(sys.argv[2]), sys.argv[3], sys.argv[4], int(sys.argv[5])
groups = [int(g) for g in sys.argv[6].split(',')]
opts = {'dtype': dtype}
if name == 'gmw':
    opts.update(beta=12, gamma=3)
wav = S.Wavelet((name, opts))
ow = O.OracleWavelet(name, dtype, **{k: v for k, v in opts.items() if k != 'dtype'})
scales = O.bench_scales(ow, N, na)
lib = _lib.load(require_device=True)
n_up, n1, _ = p2up(N)
hp = ssq_cwt_host_params(N, wav, scales, 'log', 'peak', True, 1.)
plan = S.CwtPlan.get(wav, hp['scales'], N, n_up, n1, 'reflect', 1.)
desc = make_reassign_desc(hp['ssq_freqs'], hp['const'], plan.na, hp['logscale'], True,
                          10 * (EPS64 if dtype == 'float64' else EPS32), dtype)
plan.set_reassign(desc, 'prof')
x = torch.as_tensor(np.stack([O.chirp(N, b, dtype) for b in range(B)]), device='cuda')
cdt = torch.complex128 if dtype == 'float64' else torch.complex64
Wx = torch.empty((B, na, N), dtype=cdt, device='cuda'); Tx = torch.empty_like(Wx)
st = torch.cuda.current_stream().cuda_stream
run = lambda: _lib.check(lib.ssqb_ssq_cwt_exec(plan.handle, x.data_ptr(), B, Wx.data_ptr(), Tx.data_ptr(), None, st))
bytes_step = (4 if dtype == 'float32' else 8) * (1 + 4 * na) * N * B
for g in groups:
    os.environ['SSQB_GROUP'] = str(g)
    for _ in range(3):
        run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    it = 5
    e0.record()
    for _ in range(it):
        run()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / it
    print("B=%d group=%d: %.3f ms/step  %.1f Msamples/s  hbm_frac %.3f"
          % (B, g, ms, B * N / ms / 1e3, bytes_step / ms / 1e6 / 6572.2), flush=True)
