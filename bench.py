#!/usr/bin/env python
# -*- coding: utf-8 -*-
"""Benchmark of the ssq_cwt hot path (BASELINE.json metric: Msamples/s, 300 scales, N=160k, fp32).

    python bench.py --gpus N --steps K --warmup W            # this repo (B200)
    python bench.py --impl reference --steps K --warmup W    # the reference's own CPU path

Workload (`config.workload`), the one the north-star target is quoted on: BASELINE configs[3] --
batched ssq_cwt, GMW(beta=12, gamma=3), 300 log scales, float32, 64 synthetic linear chirps of
N = 160 000 samples (SURVEY 8d).  The 64 signals are sharded over the N GPUs of the job
(64/N per GPU per step, no data-path collective): STRONG scaling.  One "step" = one full pass of
the hot path (pad -> FFT -> 300 x (wavelet multiply, inverse transform, derivative) -> phase
transform -> reassignment) over the 64 signals.  `--config C2` times BASELINE configs[1] instead
(one Morlet signal per GPU per step, weak scaling; also reported as the `c2` extra key of the
default run), `--config C5` configs[4] (float64, N = 2^20, 512 scales, one signal per GPU).

Numbers on the JSON line:
  value      Msamples/s, inputs resident in HBM, CUDA events around the K steps, barrier +
             synchronize on both sides, max over ranks
  e2e        same metric through the C ABI with HOST buffers (pinned): H2D of x and D2H of
             Tx, Wx inside the timed region (ssqb_ssq_cwt_exec_host: chunks of two signals
             ping-pong between two staging slots, copies overlap the transform)
  roofline   dominant kernel class: algorithmic bytes per launch / mean launch duration (CUDA
             events on the launch stream, separate profiling pass) against MEASURED_PEAKS.json;
             whole-step fraction; fp32 flop fraction (SURVEY 8d "report both")
  cpu_baseline / --impl reference
             the UNMODIFIED reference (ssqueezepy 0.6.6 installed into baseline/_ref, numba +
             scipy.fft, SSQ_PARALLEL=1 on all host cores, reused Wavelet, warm JIT) on a bounded
             sample of the same workload: one signal per step.  Falls back to the oracle port
             (kind "port") only if the package cannot be imported.

`--dump-outputs DIR` writes what the last timed step computed, Tx.npy and Wx.npy (rank 0's
shard on several GPUs), so that two builds can be compared output for output: the inputs are
the same seeded chirps on every run.  A complex array is stored as its real view (float32 or
float64, trailing axis of 2: real, imaginary); one larger than DUMP_BYTES / 2 is stored as a
fixed sample of its flattened elements (one per stride, seeded offset within each stride:
`dump_index`), so the files stay below 64 MB in all.  Wx repeats bit for bit from run to run;
the fused reassignment adds into Tx with atomics, so Tx's last bits follow the summation order
and two runs agree only to rounding (DESIGN section 2: bins exact, Tx <= 2e-6 norm-wise).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "ssq_cwt Msamples/s (300 scales, N=160k, fp32)"
CONFIGS = {
    # name: (wavelet spec, dtype, N, na, global batch (None: one signal per GPU), scaling)
    'C4': (('gmw', {'beta': 12, 'gamma': 3}), 'float32', 160_000, 300, 64, 'strong'),
    'C2': (('morlet', {}), 'float32', 160_000, 300, None, 'weak'),
    'C5': (('gmw', {'beta': 12, 'gamma': 3, 'dtype': 'float64'}), 'float64', 1 << 20, 512, None, 'weak'),
}
FP32_PEAK_TFLOPS = 75.0          # 148 SMs x 128 FMA lanes x 2 x 1.965 GHz (CUDA cores, nominal)
DUMP_BYTES = 60_000_000          # --dump-outputs: all files together (Tx and Wx, headers aside)


def config_dict(name):
    spec, dtype, N, na, gb, scaling = CONFIGS[name]
    wl = {'C4': "batched ssq_cwt gmw(beta=12,gamma=3) 300 log scales float32, 64 chirps x N=160000 "
                "(BASELINE configs[3]) sharded over the GPUs",
          'C2': "ssq_cwt morlet(mu=13.4) 300 log scales float32 N=160000 (BASELINE configs[1]), "
                "one signal per GPU per step",
          'C5': "ssq_cwt gmw(beta=12,gamma=3) 512 log scales float64 N=1048576 (BASELINE configs[4]), "
                "one signal per GPU per step"}[name]
    return {"workload": wl, "global_batch": gb, "n_samples": N, "n_scales": na,
            "compute_dtype": dtype, "padtype": "reflect", "scaling": scaling}


def bytes_per_sample(dtype, na):
    return (4 if dtype == 'float32' else 8) * (1 + 4 * na)      # SURVEY 8(d): read x, write Tx, Wx


def flops_per_signal(N, na):
    n_up = 1 << (1 + int(round(np.log2(N))))
    return (2 * na + 1) * 5 * n_up * np.log2(n_up) + 20 * na * N            # SURVEY 8(d)


def _peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.isfile(path):
        with open(path) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
         'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index=0):
        self.lines, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + self.Q,
                 '--format=csv,noheader,nounits', '-lms', '100'],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for ln in self.lines:
            f = [c.strip() for c in ln.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def chirp(N, b=0, dtype='float32'):
    """Unit-amplitude linear chirp, fs=1, seeded per signal index (SURVEY 8d)."""
    u, v = np.random.default_rng(1234 + b).random(2)
    f0, f1 = 0.02 + 0.03 * u, 0.20 + 0.20 * v
    t = np.arange(N) / N
    return np.cos(2 * np.pi * (f0 * N * t + 0.5 * (f1 - f0) * N * t**2)).astype(dtype)


def log_scales(cwt_scalebounds, wavelet, N, na):
    """SURVEY 8d scale recipe (explicit log array inside the wavelet's valid range)."""
    mn, mx = cwt_scalebounds(wavelet, N, preset='maximal')
    nv = int(np.ceil(na / np.log2(mx / mn)))
    p0 = int(np.floor(nv * np.log2(mn)))
    return 2 ** (np.arange(p0, p0 + na) / nv)


def dump_index(total, n, seed=0):
    """Sorted flat indices of a fixed sample of n out of `total` elements: one in each of n equal
    strides, at a seeded offset.  None when n covers them all."""
    if total <= n:
        return None
    stride = total // n
    return np.arange(n, dtype=np.int64) * stride + np.random.default_rng(seed).integers(0, stride, n)


def output_arrays(outs, budget=DUMP_BYTES):
    """{name: float array on the host} of complex device tensors, sampled by `dump_index` to share
    `budget` bytes evenly."""
    import torch
    res = {}
    for name, t in outs.items():
        idx = dump_index(t.numel(), budget // len(outs) // t.element_size())
        if idx is not None:
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        res[name] = torch.view_as_real(t).cpu().numpy()
    return res


def bind_to_gpu_numa(local_rank):
    """Pin this process (and so its pinned host buffers, first touch) to the CPUs local to
    its GPU: the 8 GPUs of the box hang off two sockets."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id
        dom = torch.cuda.get_device_properties(local_rank).pci_domain_id
        dev = torch.cuda.get_device_properties(local_rank).pci_device_id
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/local_cpulist" % (dom, bus, dev)
        with open(path) as f:
            txt = f.read().strip()
        cpus = set()
        for part in txt.split(','):
            a, _, b = part.partition('-')
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return txt
    except Exception as e:                     # not fatal: only the e2e line cares
        return "unbound (%s)" % e
    return "unbound"


# ---------------------------------------------------------------------------
# reference arm / cpu_baseline
# ---------------------------------------------------------------------------
def _import_reference():
    os.environ['SSQ_GPU'] = '0'
    os.environ['SSQ_PARALLEL'] = '1'
    os.environ.setdefault('NUMBA_CACHE_DIR', '/tmp/numba_cache_ssq_ref')
    cores = os.cpu_count() or 1
    # torchrun exports OMP_NUM_THREADS=1; the reference's prange kernels use numba's pool
    os.environ['NUMBA_NUM_THREADS'] = str(cores)
    os.environ['OMP_NUM_THREADS'] = str(cores)
    ref = os.path.join(ROOT, 'baseline', '_ref')
    if not os.path.isdir(os.path.join(ref, 'ssqueezepy')):
        raise ImportError("baseline/_ref/ssqueezepy missing (run __graft_entry__.build())")
    sys.path.insert(0, ref)
    import ssqueezepy                                   # noqa: the unmodified reference
    assert os.path.realpath(ssqueezepy.__file__).startswith(os.path.realpath(ref))
    return ssqueezepy


def cpu_reference_run(cfg_name, steps, warmup):
    """Time the reference's SSQ_PARALLEL CPU path, one signal of the workload per step."""
    spec, dtype, N, na, gb, _ = CONFIGS[cfg_name]
    cores = os.cpu_count() or 1
    try:
        sp = _import_reference()
        from ssqueezepy.utils import cwt_scalebounds
        wav = sp.Wavelet(spec if spec[1] else spec[0])
        scales = log_scales(cwt_scalebounds, wav, N, na)
        kind = "reference"
        how = ("ssqueezepy %s from baseline/_ref (numba %s threads, scipy.fft workers=%d), "
               "reused Wavelet object (Psih cache)" % (sp.__version__, os.environ['NUMBA_NUM_THREADS'], cores))

        def run(b):
            return sp.ssq_cwt(chirp(N, b, dtype), wav, scales=scales)
    except Exception as e:                                       # labelled fallback
        from oracle import ssq_oracle as O
        okw = {k: v for k, v in spec[1].items() if k != 'dtype'}
        wav = O.OracleWavelet(spec[0], dtype, **okw)
        scales = O.bench_scales(wav, N, na)
        use_c = O.c_reassign_available()
        kind = "port"
        how = "oracle port (reference not importable: %s); scipy.fft workers=%d" % (e, cores)

        def run(b):
            return O.ssq_cwt(chirp(N, b, dtype), wav, scales, workers=cores, use_c=use_c)
    nsig = gb or 1
    for i in range(max(warmup, 1)):
        run(i % nsig)
    ts = []
    for i in range(steps):
        t0 = time.perf_counter()
        run((warmup + i) % nsig)
        ts.append(time.perf_counter() - t0)
    mean = float(np.mean(ts))
    return {"value": N / mean / 1e6, "unit": "Msamples/s", "cores": cores, "kind": kind,
            "sample": "%d steps of ONE %d-sample signal of the workload each (the reference "
                      "materialises [B,na,n_up] arrays, so a batch is looped per signal, SURVEY 8d); "
                      "%d warm-up calls; %s" % (steps, N, max(warmup, 1), how),
            "ms_per_step": mean * 1e3, "min_ms": float(np.min(ts)) * 1e3}


def run_reference(args):
    if int(os.environ.get('RANK', '0')) != 0:
        return
    base = cpu_reference_run(args.config, args.steps, args.warmup)
    _, dtype, N, na, gb, scaling = CONFIGS[args.config]
    line = {"metric": METRIC, "value": base["value"], "unit": "Msamples/s", "impl": "reference",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": base["ms_per_step"], "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None, "dtype": "f32" if dtype == 'float32' else "f64",
            "data": "synthetic", "config": config_dict(args.config),
            "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": base["value"], "unit": "Msamples/s",
                    "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit_line(line)


# ---------------------------------------------------------------------------
# this repo
# ---------------------------------------------------------------------------
class Workload:
    """Plan + device buffers of one configuration on the current GPU."""

    def __init__(self, cfg_name, B, first_signal):
        import torch
        import ssqueezepy_b200 as S
        from ssqueezepy_b200 import _lib
        from ssqueezepy_b200._ssq_cwt import ssq_cwt_host_params
        from ssqueezepy_b200.algos import make_reassign_desc
        from ssqueezepy_b200.utils import cwt_scalebounds
        from ssqueezepy_b200.utils.common import EPS32, EPS64, p2up
        spec, dtype, N, na, gb, _ = CONFIGS[cfg_name]
        self.name, self.B, self.N, self.na, self.dtype = cfg_name, B, N, na, dtype
        self.lib = _lib.load(require_device=True)
        self._lib = _lib
        wav = S.Wavelet(spec if spec[1] else spec[0])
        scales = log_scales(cwt_scalebounds, wav, N, na)
        n_up, n1, _ = p2up(N)
        hp = ssq_cwt_host_params(N, wav, scales, 'log', 'peak', True, 1.)
        self.plan = S.CwtPlan.get(wav, hp['scales'], N, n_up, n1, 'reflect', 1.)
        desc = make_reassign_desc(hp['ssq_freqs'], hp['const'], self.plan.na, hp['logscale'], True,
                                  10 * (EPS64 if dtype == 'float64' else EPS32), dtype)
        self.plan.set_reassign(desc, 'bench')
        self.ssq_freqs = np.asarray(hp['ssq_freqs'])[::-1].copy()      # as ssq_cwt returns them
        x = np.stack([chirp(N, first_signal + b, dtype) for b in range(B)])
        self.x_host = torch.from_numpy(x).pin_memory()
        self.x_dev = self.x_host.cuda()
        cdt = torch.complex128 if dtype == 'float64' else torch.complex64
        self.cdt = cdt
        self.Wx = torch.empty((B, na, N), dtype=cdt, device='cuda')
        self.Tx = torch.empty_like(self.Wx)
        self.stream = torch.cuda.current_stream().cuda_stream
        self.bytes_per_step = bytes_per_sample(dtype, na) * N * B

    def step(self):
        self._lib.check(self.lib.ssqb_ssq_cwt_exec(self.plan.handle, self.x_dev.data_ptr(), self.B,
                                                   self.Wx.data_ptr(), self.Tx.data_ptr(), None,
                                                   self.stream))

    def alloc_host_out(self):
        import torch
        self.Wx_h = torch.empty((self.B, self.na, self.N), dtype=self.cdt).pin_memory()
        self.Tx_h = torch.empty((self.B, self.na, self.N), dtype=self.cdt).pin_memory()

    def step_host(self):
        self._lib.check(self.lib.ssqb_ssq_cwt_exec_host(self.plan.handle, self.x_host.data_ptr(),
                                                        self.B, self.Wx_h.data_ptr(),
                                                        self.Tx_h.data_ptr(), None, self.stream))

    def profile(self, reps=2):
        import ctypes as C
        import torch
        lib, _lib = self.lib, self._lib
        _lib.check(lib.ssqb_cwt_plan_set_profiling(self.plan.handle, 1))
        for _ in range(reps):
            self.step()
        torch.cuda.synchronize()
        n = len(_lib.PROFILE_KINDS)
        pms = (C.c_double * n)(); pl = (C.c_longlong * n)(); pr = (C.c_longlong * n)()
        _lib.check(lib.ssqb_cwt_plan_get_profile(self.plan.handle, pms, pl, pr))
        _lib.check(lib.ssqb_cwt_plan_set_profiling(self.plan.handle, 0))
        return {k: {"ms_total": pms[i] / reps, "launches": int(pl[i]) // reps, "rows": int(pr[i]) // reps}
                for i, k in enumerate(_lib.PROFILE_KINDS) if pl[i]}


def timed_steps(w, steps, warmup, world, dist, sampler=None):
    import torch

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()
    for _ in range(warmup):
        w.step()
    sync_all()
    if sampler is not None:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = w._lib.launch_count()
    e0.record()
    for _ in range(steps):
        w.step()
    e1.record()
    sync_all()
    ms = torch.tensor([e0.elapsed_time(e1)], device='cuda', dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item()) / steps, (w._lib.launch_count() - l0)


def run_b200(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    spec, dtype, N, na, gb, scaling = CONFIGS[args.config]
    if gb is not None:
        if gb % world:
            raise SystemExit("global batch %d does not divide over %d GPUs" % (gb, world))
        B = gb // world
        first = rank * B
        total_signals = gb
    else:
        B, first, total_signals = 1, rank, world
    w = Workload(args.config, B, first)

    sampler = ClockSampler(local) if rank == 0 else None
    ms_per_step, launches = timed_steps(w, args.steps, args.warmup, world, dist, sampler)
    dumped = output_arrays({'Tx': w.Tx, 'Wx': w.Wx}) if args.dump_outputs and rank == 0 else None
    if rank == 0:
        # the timed region can be shorter than nvidia-smi's sampling period: keep the same step
        # loop running for another 0.5 s so the clocks line has enough samples
        t_probe = time.perf_counter() + 0.5
        while time.perf_counter() < t_probe:
            w.step()
            torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    if clocks is not None:
        clocks["window"] = "timed region + 0.5 s of the same step loop"
    value = total_signals * N / (ms_per_step * 1e-3) / 1e6

    # ---- e2e: host buffers through the C ABI (H2D + transform + D2H) -------------------------
    w.alloc_host_out()
    e2e_steps = max(1, min(args.steps, 3))
    w.step_host()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        w.step_host()
    torch.cuda.synchronize()
    t_e2e = torch.tensor([(time.perf_counter() - t0) / e2e_steps], device='cuda', dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    e2e_val = total_signals * N / float(t_e2e.item()) / 1e6
    esz = 8 if dtype == 'float32' else 16
    h2d = int(total_signals * N * (esz // 2))
    d2h = int(2 * total_signals * na * N * esz)
    del w.Wx_h, w.Tx_h

    # ---- e2e with the consumer on the device: x in, ridge indices out ------------------------------
    # (extract_ridges is the main consumer of Tx; returning N x n_ridges indices instead of two
    # planes takes PCIe out of the picture: SURVEY 8f row 4)
    e2e_ridges = None
    if args.ridges and args.config != 'C5':
        import ssqueezepy_b200 as S
        idx_h = torch.empty((B, N, 1), dtype=torch.int64).pin_memory()

        def step_ridges():
            w.x_dev.copy_(w.x_host, non_blocking=True)
            w.step()
            idx = S.extract_ridges(w.Tx, w.ssq_freqs, penalty=2., n_ridges=1, bw=4, transform='cwt')
            idx_h.copy_(idx, non_blocking=True)
            torch.cuda.synchronize()
        step_ridges()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(2):
            step_ridges()
        tr = torch.tensor([(time.perf_counter() - t0) / 2], device='cuda', dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tr, op=dist.ReduceOp.MAX)
        e2e_ridges = {"value": total_signals * N / float(tr.item()) / 1e6, "unit": "Msamples/s",
                      "ms_per_step": float(tr.item()) * 1e3, "h2d_bytes_per_step": h2d,
                      "d2h_bytes_per_step": int(total_signals * N * 8),
                      "note": "pinned x in -> ssq_cwt -> extract_ridges(Tx, penalty=2, n_ridges=1, bw=4) "
                              "on the device -> ridge indices back to pinned host memory"}

    # ---- optional NCCL gather of the outputs (timed separately; SURVEY 8e) ------------------------
    gather_ms = None
    if world > 1 and args.gather:
        from ssqueezepy_b200.distributed import gather_batch
        torch.cuda.synchronize(); dist.barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        out = gather_batch(w.Tx, total_signals)
        g1.record(); torch.cuda.synchronize()
        gm = torch.tensor([g0.elapsed_time(g1)], device='cuda', dtype=torch.float64)
        dist.all_reduce(gm, op=dist.ReduceOp.MAX)
        gather_ms = float(gm.item())
        del out

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- roofline (separate profiling pass, rank 0) ---------------------------------------------
    peak, peak_src = _peaks()
    prof = w.profile()
    bps = bytes_per_sample(dtype, na)
    row_kinds = {k: v for k, v in prof.items() if k in ('row_kernels_with_epilogue',
                                                        'grid_interp_with_epilogue')}
    dom = max(row_kinds, key=lambda k: row_kinds[k]["ms_total"]) if row_kinds else max(prof, key=lambda k: prof[k]["ms_total"])
    d = prof[dom]
    alg_bytes_launch = bps * N * (d["rows"] / max(d["launches"], 1)) / na
    dur = d["ms_total"] / max(d["launches"], 1) * 1e-3
    achieved = alg_bytes_launch / dur / 1e9
    step_gbs = w.bytes_per_step / (ms_per_step * 1e-3) / 1e9
    flops = flops_per_signal(N, na) * B / (ms_per_step * 1e-3) / 1e12
    traffic, traffic_note = None, "no whole-step ncu capture committed yet"
    tpath = os.path.join(ROOT, 'profiles', 'r2_traffic.json')
    if os.path.isfile(tpath):
        with open(tpath) as f:
            tr = json.load(f)
        traffic = (tr.get('dram_bytes_per_launch') or {}).get(dom)
        traffic_note = ("%s; figure = mean DRAM bytes per launch of the dominant class in that capture "
                        "(8 signals per launch, as in the timed run); whole step: %.2fx the algorithmic bytes"
                        % (tr.get('note'), tr.get('traffic_over_algorithmic', float('nan'))))
    tot = sum(v["ms_total"] for v in prof.values())
    roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "traffic_note": traffic_note,
                "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes_launch,
                "mean_launch_ms": dur * 1e3,
                "whole_step": {"achieved": step_gbs, "frac": step_gbs / peak},
                "flop_frac": {"achieved_tflops": flops, "peak_tflops": FP32_PEAK_TFLOPS,
                              "frac": flops / FP32_PEAK_TFLOPS,
                              "note": "nominal FFT flop count of SURVEY 8d over the step time, against "
                                      "the fp32 CUDA-core peak; the gridded rows do far fewer flops "
                                      "than that count" } if dtype == 'float32' else None,
                "kernel_share_of_step": {k: v["ms_total"] / max(tot, 1e-12) for k, v in prof.items()},
                "profile": prof}

    # ---- extra: BASELINE configs[1] (one Morlet signal) on this GPU -------------------------------
    c2 = None
    if args.config == 'C4' and not args.no_c2:
        del w
        torch.cuda.empty_cache()
        w2 = Workload('C2', 1, 0)
        ms2, _ = timed_steps(w2, 20, 3, 1, None)
        c2 = {"value": 160_000 / (ms2 * 1e-3) / 1e6, "unit": "Msamples/s", "ms_per_step": ms2,
              "hbm_frac": w2.bytes_per_step / (ms2 * 1e-3) / 1e9 / peak,
              "config": config_dict('C2')["workload"]}
        del w2
        torch.cuda.empty_cache()

    cpu = None
    if world == 1:
        cpu = cpu_reference_run(args.config, 2, 1)
    line = {"metric": METRIC, "value": value, "unit": "Msamples/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None, "dtype": "f32" if dtype == 'float32' else "f64", "data": "synthetic",
            "config": config_dict(args.config),
            "run": {"batch_per_gpu_per_step": B,
                    "outputs": "Tx, Wx complex [B,%d,%d] left on the producing GPU" % (na, N),
                    "l2": "each step streams %.0f MB of outputs per GPU (> 126 MB L2) between re-uses "
                          "of any line" % (bps * N * B / 1e6),
                    "parallelism": "batch-sharded x%d, no data-path collective" % world,
                    "groups": "each rank's batch runs in zero-ahead groups of signals (8 of >= 32, else half "
                              "the batch): the row kernels of a group store the zeros of the next group's Tx",
                    "numa_binding": numa},
            "clocks": clocks, "gpu_launches": int(launches),
            "e2e": {"value": e2e_val, "unit": "Msamples/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                    "note": "ssqb_ssq_cwt_exec_host: pinned host x in, Tx and Wx copied back to pinned "
                            "host buffers; PCIe-bound (%.1f GB back per step per GPU)" % (d2h / world / 1e9)},
            "e2e_ridges": e2e_ridges, "gather_ms": gather_ms, "roofline": roofline, "c2": c2}
    if cpu is not None:
        line["cpu_baseline"] = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}
    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + '.npy'), a)
    emit_line(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


_REAL_STDOUT = None


def guard_stdout():
    """stdout carries exactly ONE JSON line: libraries that print there (NCCL's version
    banner does, at communicator creation) are pointed at stderr for the rest of the run."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit_line(line):
    data = (json.dumps(line) + '\n').encode()
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        os.write(1, data)
    else:
        os.write(_REAL_STDOUT, data)


def main():
    guard_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--config', default='C4', choices=list(CONFIGS))
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--no-c2', action='store_true', help='skip the extra configs[1] measurement')
    ap.add_argument('--gather', action='store_true', help='also time an NCCL all_gather of Tx')
    ap.add_argument('--no-ridges', dest='ridges', action='store_false',
                    help='skip the e2e variant that returns ridges instead of planes')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write Tx, Wx of the last timed step to DIR/<name>.npy (b200 only)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs needs --impl b200')
    if args.warmup < 3 and args.impl == 'b200':
        args.warmup = 3
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
