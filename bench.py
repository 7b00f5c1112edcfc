#!/usr/bin/env python
"""Benchmark of the hot path on BASELINE.json's metric: trajectory-steps/s (batch x t_steps / s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg2] [--no-secondary]
                    [--dump-outputs DIR]

A "step" is one full solve of the workload (one pass of the hot path over one batch).
Workload cfg2 (BASELINE.json configs[1], the configuration the metric is quoted on):
    Milstein Ito/diagonal, batch=65536, state=64, t=1000 steps (dt=2^-10), fp32, full output series
    ts = arange(1001)*dt, SDE = per-channel GBM (f = mu*y, g = sigma*y) as ordinary torch callables,
    Brownian motion = torchsde_b200.BrownianInterval (counter-based, regenerated in registers).

Output: ONE JSON line (rank 0).  Besides the contract's keys:
  parity_check   rows of the TIMED output buffers compared with the numpy oracle on the same Philox path
  roofline       the dominant solver-owned kernel (fused Milstein tableau), CUDA-event probe + ncu traffic
  kernels        the same probe for every solver-owned kernel of the step
  cpu_baseline   the REFERENCE itself (google-research/torchsde, staged unmodified in oracle/_ref by build()) on the
                 host cores, bounded sample; the numpy oracle port is reported beside it
  secondary      the other BASELINE.json configs (cfg3 / cfg4 / cfg5), measured in the same process on every rank
`--impl reference` times the unmodified reference on the host cores for the same config / metric / unit.
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from (which may be read-only)

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOADS = {
    # BASELINE.json configs[1] — the configuration the metric is quoted on (the headline)
    'cfg2': dict(method='milstein', sde_type='ito', kind='gbm', B=65536, D=64, M=64, T=1000, dt=2.0 ** -10,
                 E_bytes_per_traj_step=13 * 64 * 4, S_tableau_bytes_per_traj_step=5 * 64 * 4),
    'cfg2_small': dict(method='milstein', sde_type='ito', kind='gbm', B=4096, D=64, M=64, T=100, dt=2.0 ** -10,
                       E_bytes_per_traj_step=13 * 64 * 4, S_tableau_bytes_per_traj_step=5 * 64 * 4),
    # honest HBM-bound point of SURVEY §8(d): working set 320 MiB >> L2
    'cfg2_b262144': dict(method='milstein', sde_type='ito', kind='gbm', B=262144, D=64, M=64, T=100, dt=2.0 ** -10,
                         E_bytes_per_traj_step=13 * 64 * 4, S_tableau_bytes_per_traj_step=5 * 64 * 4),
    # BASELINE.json configs[2], substituted (reference SRK rejects general noise, srk.py:35): parity/measurement cases
    'cfg3_srk_additive': dict(method='srk', sde_type='ito', kind='additive', B=8192, D=32, M=16, T=500,
                              dt=2.0 ** -10, levy='space-time', E_bytes_per_traj_step=(11 * 32 + 5 * 32 * 16) * 4),
    # same SDE, g returned as a stride-0 (batch-broadcast) view: nothing of size (B, d, m) ever exists
    'cfg3_srk_additive_expand': dict(method='srk', sde_type='ito', kind='additive_expand', B=8192, D=32, M=16, T=500,
                                     dt=2.0 ** -10, levy='space-time',
                                     E_bytes_per_traj_step=(11 * 32 + 5 * 32 * 16) * 4),
    'cfg3_euler_general': dict(method='euler', sde_type='ito', kind='general', B=8192, D=32, M=16, T=500,
                               dt=2.0 ** -10, E_bytes_per_traj_step=(6 * 32 + 2 * 32 * 16) * 4),
    'cfg3_heun_general': dict(method='heun', sde_type='stratonovich', kind='general', B=8192, D=32, M=16, T=500,
                              dt=2.0 ** -10, E_bytes_per_traj_step=2 * (6 * 32 + 2 * 32 * 16) * 4),
    # cfg2 with per-trajectory parameters (mu, sigma of shape (B, D)): f/g/vjp are contiguous element-wise
    # products, i.e. PyTorch's vectorised kernels instead of its broadcasting ones.  E = 7 (solver) + 3*3 = 16 D s.
    'cfg2_pertraj': dict(method='milstein', sde_type='ito', kind='gbm_pertraj', B=65536, D=64, M=64, T=1000,
                         dt=2.0 ** -10, E_bytes_per_traj_step=16 * 64 * 4, S_tableau_bytes_per_traj_step=5 * 64 * 4),
    # general noise in the HBM-bound regime (g = 256 MiB per evaluation)
    'cfg3_euler_general_large': dict(method='euler', sde_type='ito', kind='general', B=65536, D=64, M=16, T=100,
                                     dt=2.0 ** -10, E_bytes_per_traj_step=(6 * 64 + 2 * 64 * 16) * 4),
    # other diagonal tableaus at the cfg2 size
    'cfg2_euler': dict(method='euler', sde_type='ito', kind='gbm', B=65536, D=64, M=64, T=200, dt=2.0 ** -10,
                       E_bytes_per_traj_step=8 * 64 * 4),
    'cfg2_srk': dict(method='srk', sde_type='ito', kind='gbm', B=65536, D=64, M=64, T=200, dt=2.0 ** -10,
                     levy='space-time', E_bytes_per_traj_step=41 * 64 * 4),
    'cfg2_milstein_gf': dict(method='milstein', sde_type='ito', kind='gbm', B=65536, D=64, M=64, T=200,
                             dt=2.0 ** -10, options={'grad_free': True}, E_bytes_per_traj_step=15 * 64 * 4),
}
METRIC = "trajectory-steps/s (batch x t_steps / s)"
REF_DIR = os.path.join(ROOT, 'oracle', '_ref', 'pkg')  # oracle/stage_reference.py


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        return float(json.load(open(path))['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (profiling recipe)."""
    Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.proc = None
        self.index = index
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.Q}',
                                          '--format=csv,noheader,nounits', '-lms',
                                          os.environ.get('TSDE_BENCH_SAMPLER_MS', '200')],  # (the recipe's period)
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.monotonic(), line.strip()))

    def mark(self):
        """The timed region starts here: the process was started (and NVML initialised) before the warm-up, so that
        its start-up does not run against the first timed steps; only samples taken from now on are reported."""
        self.t_mark = time.monotonic()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        t_mark = getattr(self, 't_mark', 0.0)
        timed = [ln for t, ln in self.lines if t >= t_mark] or [ln for _, ln in self.lines[-1:]]
        for ln in timed:
            p = [x.strip() for x in ln.split(',')]
            if len(p) < 6:
                continue
            try:
                sm.append(float(p[0]))
                mx.append(float(p[1]))
            except ValueError:
                continue
            for n, v in zip(names, p[2:6]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def build_sde(w, device, dtype=torch.float32):
    from tests import problems
    torch.manual_seed(1147481649)
    kind = w.get('kind', 'gbm')
    if kind == 'gbm':
        sde = problems.GBMDiagonal(w['D'], w['sde_type'], seed=1147481649 % 1000, dtype=dtype)
    elif kind == 'gbm_pertraj':
        sde = problems.GBMPerTrajectory(w['B'], w['D'], w['sde_type'], seed=649, dtype=dtype)
    else:
        sde = problems.make(kind, w['D'], w['M'], w['sde_type'], dtype=dtype, seed=649)
    return sde.to(device)


def common_config(args, w, world):
    """The `config` object — identical for the `ours` and the `reference` arm (same workload, same sizes)."""
    return {"workload": args.workload, "method": w['method'], "sde_type": w['sde_type'],
            "noise": "diagonal" if w.get('kind', 'gbm').startswith('gbm') else w['kind'],
            "batch_per_gpu": w['B'], "state": w['D'], "brownian": w['D'] if w.get('kind', 'gbm').startswith('gbm') else w['M'],
            "t_steps": w['T'], "dt": w['dt'], "output": "full series (T+1,B,D)",
            "parallelism": f"batch-sharded x{world}"}


# -------------------------------------------------------------------------------------------------
# CPU arms: (1) the reference itself, staged unmodified under oracle/_ref; (2) the numpy oracle port
# -------------------------------------------------------------------------------------------------
def import_reference():
    """`torchsde` v0.2.6 as staged by build() (oracle/stage_reference.py) plus the stand-in for its one missing
    pure-Python dependency.  Returns the module or None."""
    if not os.path.isdir(os.path.join(REF_DIR, 'torchsde')):
        return None
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    import torchsde  # noqa: the reference, NOT this repository's package (which is `torchsde_b200`)
    assert os.path.realpath(torchsde.__file__).startswith(os.path.realpath(REF_DIR))
    return torchsde


def cpu_reference_run(ref, w, n_steps):
    """One solve of the first `n_steps` steps of the workload by the reference's own stock code path
    (torchsde.sdeint + torchsde.BrownianInterval, CPU tensors, all host threads); BASELINE.md §3.
    Returns (traj-steps/s, seconds)."""
    B, D, dt = w['B'], w['D'], w['dt']
    M = D if w.get('kind', 'gbm').startswith('gbm') else w['M']
    sde = build_sde(w, 'cpu')
    y0 = torch.full((B, D), 0.1)
    ts = torch.arange(n_steps + 1, dtype=torch.float32) * dt
    bm = ref.BrownianInterval(t0=0.0, t1=n_steps * dt, size=(B, M), dtype=torch.float32, entropy=1147481649, dt=dt,
                              levy_area_approximation=w.get('levy', 'none'))
    t0 = time.perf_counter()
    with torch.no_grad():
        ys = ref.sdeint(sde, y0, ts, bm=bm, method=w['method'], dt=dt, options=dict(w.get('options', {})))
    el = time.perf_counter() - t0
    assert ys.shape == (n_steps + 1, B, D)
    return B * n_steps / el, el


def cpu_port_run(w, n_steps, threads, B=None):
    """Oracle Milstein (oracle/solvers.py) + oracle counter-based Brownian cells on `threads` host
    threads (rows are independent; numpy releases the GIL inside ufuncs).  Returns traj-steps/s."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import brownian as obm
    from oracle import solvers
    B = B or w['B']
    D = w['D']
    dt = w['dt']
    sde_t = build_sde(w, 'cpu')
    mu = sde_t.mu.detach().numpy()
    sigma = sde_t.sigma.detach().numpy()

    class NpGBM:  # numpy callables of the same synthetic SDE (f = mu*y, g = sigma*y; gdg = vjp)
        noise_type, sde_type = 'diagonal', w['sde_type']
        f = staticmethod(lambda t, y: mu * y)
        g = staticmethod(lambda t, y: sigma * y)
        gdg = staticmethod(lambda t, y, v2: (sigma * y) * v2 * sigma)

    ts = np.array([0.0, n_steps * dt], dtype=np.float32)
    chunks = np.array_split(np.arange(B), threads)

    def work(rows):
        r0, n = int(rows[0]), len(rows)

        def bm(ta, tb, return_U=False):
            k = int(round(float(ta) / dt))
            W, _ = obm.cell(1234567, 1000 + k, float(tb) - float(ta), n, D, np.float32, False, row_offset=r0)
            return W
        y0 = np.full((n, D), 0.1, dtype=np.float32)
        solvers.make('milstein', NpGBM, bm, dt).integrate(y0, ts)

    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=threads) as ex:
        list(ex.map(work, chunks))
    el = time.perf_counter() - t0
    return B * n_steps / el, el


_REF_THREADS = {}


def best_reference_threads(ref, w):
    """The reference is a Python loop over small ATen ops: beyond a few dozen threads the OpenMP fork/join cost of
    every op exceeds its work (measured on the 128-core GPU host: 47 k traj-steps/s at 128 threads against > 10x that
    at 16-32).  'All the host threads it can use' therefore means the thread count at which it is fastest: try a
    ladder on 2 steps each and keep the best.  Returns (threads, {threads: traj-steps/s})."""
    key = (w['B'], w['D'], w['method'])
    if key not in _REF_THREADS:
        n = os.cpu_count() or 1
        tried = {}
        for c in sorted({min(c, n) for c in (8, 16, 32, 64, n)}):
            torch.set_num_threads(c)
            cpu_reference_run(ref, w, 1)
            tried[c] = cpu_reference_run(ref, w, 2)[0]
        _REF_THREADS[key] = (max(tried, key=tried.get), tried)
    torch.set_num_threads(_REF_THREADS[key][0])
    return _REF_THREADS[key]


def cpu_baseline_sample(w, budget_s=20.0):
    """Bounded sample for the `ours` arm's `cpu_baseline`: the reference on the host cores (1 warm-up of 2 steps,
    then best of 3 solves of n steps, n sized for ~budget_s seconds in total), and the numpy port beside it."""
    out = {}
    ref = import_reference()
    if ref is not None:
        threads, tried = best_reference_threads(ref, w)
        _, el = cpu_reference_run(ref, w, 2)
        n = int(max(2, min(64, (budget_s / 3.5) / max(el / 2, 1e-3))))
        vals = [cpu_reference_run(ref, w, n)[0] for _ in range(3)]
        out = {"value": max(vals), "unit": "traj-steps/s", "cores": torch.get_num_threads(), "kind": "reference",
               "sample": f"torchsde v0.2.6 sdeint (CPU, fp32) B={w['B']} D={w['D']}, first {n} of {w['T']} steps, "
                         f"best of 3 after a warm-up", "host_cores": os.cpu_count(),
               "threads_tried": {str(k): round(v) for k, v in tried.items()}}
    if w['method'] == 'milstein' and w.get('kind', 'gbm') == 'gbm' and not w.get('options'):
        threads, tried = best_cpu_threads(w)
        port, _ = cpu_port_run(w, 4, threads)
        port_info = {"value": port, "unit": "traj-steps/s", "cores": threads, "kind": "port",
                     "sample": f"numpy oracle port, first 4 of {w['T']} steps",
                     "threads_tried": {str(k): round(v) for k, v in tried.items()}}
        if not out:
            out = dict(port_info, host_cores=os.cpu_count())
        else:
            out["port"] = port_info
    return out or None


def run_reference(args, w, rank, world):
    if rank != 0:
        return
    ref = import_reference()
    line = {"impl": "reference", "metric": METRIC, "unit": "traj-steps/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": common_config(args, w, world), "gpu_launches": 0}
    if ref is not None:
        # size the per-step sample so that warmup + steps solves end within a few minutes (~100 s)
        threads, tried = best_reference_threads(ref, w)
        _, el = cpu_reference_run(ref, w, 2)
        per_step = max(el / 2, 1e-3)
        budget = float(os.environ.get('TSDE_BENCH_REF_BUDGET_S', 100.0))
        n_steps = int(max(2, min(w['T'], budget / (args.warmup + args.steps) / per_step)))
        vals = []
        for i in range(args.warmup + args.steps):
            v, el = cpu_reference_run(ref, w, n_steps)
            if i >= args.warmup:
                vals.append((v, el))
        kind, cores = "reference", torch.get_num_threads()
        sample = (f"torchsde v0.2.6 (unmodified, oracle/_ref) sdeint on CPU tensors, torch threads={cores} of "
                  f"{os.cpu_count()} host cores (fastest of {sorted(tried)}); each bench step = first {n_steps} of {w['T']} steps of the workload "
                  f"(B={w['B']} D={w['D']}; per-step cost is constant for sequential access)")
    else:
        threads, tried = best_cpu_threads(w)
        n_steps = 8
        vals = []
        for i in range(args.warmup + args.steps):
            v, el = cpu_port_run(w, n_steps, threads)
            if i >= args.warmup:
                vals.append((v, el))
        kind, cores = "port", threads
        sample = f"numpy oracle port (oracle/_ref absent), first {n_steps} of {w['T']} steps per bench step"
    value = float(np.mean([v for v, _ in vals]))
    ms = float(np.mean([el for _, el in vals]) * 1e3)
    line.update({"value": value, "ms_per_step": ms,
                 "cpu_baseline": {"value": value, "unit": "traj-steps/s", "cores": cores, "kind": kind,
                                  "sample": sample, "host_cores": os.cpu_count()},
                 "e2e": {"value": value, "unit": "traj-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
    print(json.dumps(line), flush=True)


_CPU_THREADS = {}


def best_cpu_threads(w):
    """The numpy port stops scaling once its per-thread slices get small (interpreter overhead under the GIL), so
    'all the host threads' is not its fastest setting: try a ladder of thread counts on one step each and keep the
    fastest, so that the CPU arm is reported at its best.  Returns (threads, {threads: traj-steps/s})."""
    key = (w['B'], w['D'])
    if key not in _CPU_THREADS:
        n = os.cpu_count() or 1
        tried = {}
        for c in sorted({min(c, n) for c in (4, 8, 16, 32, n)}):
            cpu_port_run(w, 1, c)                      # warm-up (thread start, allocations)
            tried[c] = max(cpu_port_run(w, 1, c)[0], cpu_port_run(w, 1, c)[0])
        _CPU_THREADS[key] = (max(tried, key=tried.get), tried)
    return _CPU_THREADS[key]


# -------------------------------------------------------------------------------------------------
# GPU arm
# -------------------------------------------------------------------------------------------------
DUMP_SERIES_ROWS = 128      # trajectories whose whole series is written by --dump-outputs
DUMP_FINAL_ROWS = 1 << 16   # terminal states written by --dump-outputs (all of them up to this batch)
DUMP_SEED = 20261017


def dump_outputs(out_dir, ys):
    """Write what the solve returned, as float32 .npy files under `out_dir`:
      ys_final.npy          terminal states ys[-1], (B, D); above DUMP_FINAL_ROWS trajectories a fixed sample of rows
      ys_series_rows.npy    the whole series (T+1, rows, D) of a fixed sample of DUMP_SERIES_ROWS trajectories
    Rows are tests.helpers.sample_rows(B, n, DUMP_SEED): the same for every run of a workload, so two builds can be
    compared output for output.  At most 64 MiB in all for every workload of WORKLOADS.  Several ranks: rank 0's
    batch."""
    from tests import helpers
    os.makedirs(out_dir, exist_ok=True)
    B = ys.shape[1]
    arrays = {}
    for name, n, series in (('ys_final', DUMP_FINAL_ROWS, False), ('ys_series_rows', DUMP_SERIES_ROWS, True)):
        idx = torch.arange(B, device=ys.device) if n >= B else \
            torch.from_numpy(helpers.sample_rows(B, n, DUMP_SEED)).to(ys.device)
        arrays[name] = (ys[:, idx] if series else ys[-1, idx]).float().cpu().numpy()
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20, {k: a.shape for k, a in arrays.items()}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), a)


def parity_check(w, sde, bm, ys, row_offset, n_rows=256):
    """Compare `n_rows` random trajectories of the timed output buffers with the numpy oracle integrating the same
    Philox-defined Brownian path (oracle/: test infrastructure used here as the checker of the measured run)."""
    from oracle import solvers
    from tests import helpers, problems
    B, D, dt = w['B'], w['D'], w['dt']
    M = D if w.get('kind', 'gbm').startswith('gbm') else w['M']
    rows = helpers.sample_rows(B, n_rows, seed=20260923)
    got = ys[:, torch.from_numpy(rows).to(ys.device)].cpu().numpy()
    sde_cpu = build_sde(w, 'cpu')
    kind = w.get('kind', 'gbm')
    if kind == 'gbm_pertraj':
        return None
    want_u = w.get('levy', 'none') != 'none'
    oracle_bm = helpers.oracle_grid_bm(bm, rows, M, np.float32, want_u)
    ts = (np.arange(w['T'] + 1, dtype=np.float32) * np.float32(dt))
    t0 = time.perf_counter()
    ref, _ = solvers.make(w['method'], problems.NumpySDE(sde_cpu), oracle_bm, dt, dict(w.get('options', {}))).integrate(
        np.full((len(rows), D), 0.1, dtype=np.float32), ts)
    scale = float(np.abs(ref).max())
    # relative to |ref| where the process stays away from zero (GBM: positive), floored at 5 % of the sample's scale
    # for processes that cross zero (additive / general noise), where a pure relative error is meaningless
    floor = 1e-3 * scale if kind.startswith('gbm') else 5e-2 * scale
    rel = np.abs(got.astype(np.float64) - ref) / np.maximum(np.abs(ref), floor)
    return {"rows": int(len(rows)), "t_points": int(ref.shape[0]), "max_rel_err": float(rel.max()),
            "rel_err_floor": floor, "max_abs_err": float(np.abs(got - ref).max()), "ref_scale": scale,
            "against": "numpy oracle (oracle/solvers.py + oracle/philox.py) on the same global rows of the same path",
            "source": "output series of the last timed solve", "oracle_seconds": round(time.perf_counter() - t0, 2)}


def run_ours(args, w, rank, world, local_rank):
    import torch.distributed as dist
    import torchsde_b200 as tsde
    from torchsde_b200 import _cabi
    from torchsde_b200._core import graph as graph_mod
    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    _cabi.lib()  # fail loudly if the CUDA library is missing: there is no fallback
    B, D, T, dt = w['B'], w['D'], w['T'], w['dt']
    sde = build_sde(w, dev)
    ts = (torch.arange(T + 1, dtype=torch.float32) * dt).to(dev)
    y0_host = torch.full((B, D), 0.1, dtype=torch.float32).pin_memory()
    y0_dev = y0_host.to(dev)
    out_host = torch.empty((B, D), dtype=torch.float32).pin_memory()
    # static_output: the solve returns the plan-owned series instead of a copy of it (16.8 GB at cfg2); every timed
    # region below consumes the result before the next solve overwrites it
    opts = {'cuda_graph': not args.no_graph, 'static_output': True}
    if args.row_split > 1:
        opts['row_split'] = args.row_split
    row_offset = rank * B  # weak scaling: every rank integrates its own B trajectories of one global batch

    M = D if w.get('kind', 'gbm').startswith('gbm') else w['M']
    opts.update(w.get('options', {}))
    last = {}

    def solve(y0, entropy):
        bm = tsde.BrownianInterval(0.0, T * dt, size=(B, M), dtype=torch.float32, device=dev, entropy=entropy,
                                   levy_area_approximation=w.get('levy', 'none'))
        bm.shard_rows(row_offset)
        last['bm'] = bm
        with torch.no_grad():
            return tsde.sdeint(sde, y0, ts, bm=bm, method=w['method'], dt=dt, options=dict(opts))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- device-resident throughput (`value`) ----
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for i in range(args.warmup):
        solve(y0_dev, 1000 + i)
    barrier()
    launches0 = _cabi.LAUNCHES
    sampler.mark()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(args.steps):
        ys = solve(y0_dev, 2000 + i)
    ev1.record()
    barrier()
    elapsed = ev0.elapsed_time(ev1) * 1e-3
    clocks = sampler.stop() if rank == 0 else None
    eager_launches = _cabi.LAUNCHES - launches0
    plan = graph_mod.LAST_PLAN if opts['cuda_graph'] else None
    launches_per_solve = plan.abi_launches if plan is not None else eager_launches // max(args.steps, 1)
    finite = bool(torch.isfinite(ys[-1]).all().item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ys)   # before the next solve overwrites the plan-owned series
    parity = parity_check(w, sde, last['bm'], ys, row_offset) if rank == 0 else None

    # ---- end to end through the public API with HOST buffers (`e2e`) ----
    gathered = torch.empty((world * B, D), dtype=torch.float32, device=dev) if world > 1 else None

    def e2e_step(i):
        y0 = y0_host.to(dev, non_blocking=True)           # H2D of the step's inputs
        ys = solve(y0, 3000 + i)
        if world > 1:
            # the one collective of the path (SURVEY §8e): gather the row shards' terminal states over NVLink
            dist.all_gather_into_tensor(gathered, ys[-1].contiguous())
        out_host.copy_(ys[-1], non_blocking=True)          # D2H of the step's result (terminal states)
        return ys

    # warm-up of THIS path as well (the first all_gather sets up NCCL's channels for the collective: ~100 ms that
    # an N = 2 run without it showed as +6 ms per step)
    for i in range(args.warmup):
        ys = e2e_step(-1 - i)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        ys = e2e_step(i)
    e1.record()
    barrier()
    e2e_elapsed = e0.elapsed_time(e1) * 1e-3

    per_rank_ms = [elapsed / args.steps * 1e3]
    if world > 1:
        mine = torch.tensor([elapsed], device=dev, dtype=torch.float64)
        every = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(every, mine)
        per_rank_ms = [float(x.item()) / args.steps * 1e3 for x in every]
        t = torch.tensor([elapsed, e2e_elapsed], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed, e2e_elapsed = t.tolist()
    total_traj_steps = world * B * T * args.steps
    value = total_traj_steps / elapsed
    e2e_value = total_traj_steps / e2e_elapsed

    # ---- rooflines of the solver-owned kernels, timed in situ (rank 0) ----
    headline = args.workload.startswith('cfg2') and w['method'] == 'milstein' and not w.get('options') \
        and w.get('kind', 'gbm') == 'gbm'
    del ys
    last.clear()
    roof = kernel_rooflines(w, dev) if (rank == 0 and headline) else None
    cpu = cpu_baseline_sample(w) if (rank == 0 and not args.no_cpu) else None
    secondary = None
    if not args.no_secondary and args.workload == 'cfg2':
        graph_mod.drop_plans(sde)       # the cfg2 plan pins 16.8 GB: release it before the other workloads
        del sde
        torch.cuda.empty_cache()
        try:
            secondary = run_secondary(rank, world, dev)
        except Exception as exc:  # the headline line must survive a failure in the extra workloads (reported, loudly)
            import traceback
            traceback.print_exc()
            secondary = {"error": f"{type(exc).__name__}: {exc}"}
    if rank != 0:
        return
    peak, peak_src = peaks()
    E = w['E_bytes_per_traj_step']
    traffic = ncu_traffic()
    line = {
        "metric": METRIC, "value": value, "unit": "traj-steps/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": elapsed / args.steps * 1e3, "higher_is_better": True,
        "scaling": "strong" if args.strong else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": common_config(args, w, world),
        "impl_details": {"cuda_graph": opts['cuda_graph'], "row_split": args.row_split,
                         "result": "plan-owned static series (options static_output=True): valid until the next solve",
                         "l2_policy": "inputs larger than L2: per-step working set 80 MiB + 16 MiB ys row streamed "
                                      "into a 16.8 GB series", "finite": finite},
        "parity_check": parity,
        "clocks": clocks,
        "per_rank_ms_per_step": [round(x, 3) for x in per_rank_ms],
        "e2e": {"value": e2e_value, "unit": "traj-steps/s", "h2d_bytes_per_step": int(y0_host.numel() * 4),
                "d2h_bytes_per_step": int(out_host.numel() * 4), "ms_per_step": e2e_elapsed / args.steps * 1e3,
                "result_copied": "ys[-1] (terminal states)", "warmup": args.warmup,
                "collective": None if world == 1 else "one NCCL all_gather of the terminal states per solve"},
        "gpu_launches": int(launches_per_solve * args.steps),
        "gpu_launches_note": "C-ABI kernel launches of this library captured in the replayed CUDA graph "
                             "(counted during capture) x timed solves; PyTorch's kernels for the user's f/g/vjp are "
                             "not counted",
        "host_launch_calls_in_timed_region": int(eager_launches),
        "roofline": None if roof is None else dict(
            roof['step_milstein'], bound="hbm", peak=peak, unit="GB/s", peak_source=peak_src,
            traffic=traffic.get('step_milstein'), traffic_source=traffic.get('source'),
            kernel="ew_fast_kernel<float, MilsteinOp, COUNTER> (tsde_step_milstein)",
            timing="CUDA events around a graph replay of back-to-back launches of the kernel (how the solver "
                   "issues them), cfg2 tensor sizes, rotating buffer sets larger than L2; median of 7"),
        "kernels": None if roof is None else {k: dict(v, traffic=traffic.get(k)) for k, v in roof.items()},
        "roofline_whole_step": {"E_bytes_per_traj_step": E, "achieved": value / world * E / 1e9, "peak": peak,
                                "unit": "GB/s", "frac": value / world * E / 1e9 / peak,
                                "note": "SURVEY §8(d) E-bytes: solver kernels + the synthetic SDE's own f/g/vjp"},
        "cpu_baseline": cpu,
        "secondary": secondary,
    }
    print(json.dumps(line), flush=True)


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the solver kernels at the cfg2 shape, from the
    committed `ncu --set full` capture (profiles/ncu_traffic.json is written by profiles/ncu_extract.py from the
    .ncu-rep; nothing is profiled inside the timed run)."""
    path = os.path.join(ROOT, 'profiles', 'ncu_traffic.json')
    if os.path.exists(path):
        return json.load(open(path))
    return {}


def kernel_rooflines(w, dev):
    """Average duration of each solver-owned kernel of the step at the workload's tensor sizes: CUDA events on the
    launching stream around back-to-back launches through the C ABI captured in a CUDA graph, each launch on a
    different buffer set (12 sets, > 126 MB L2)."""
    import ctypes
    from torchsde_b200 import _cabi
    B, D, dt = w['B'], w['D'], w['dt']
    lib = _cabi.lib()
    key = torch.tensor([987654321], dtype=torch.int64, device=dev)
    L = _cabi.make_launch(torch.float32, _cabi.NOISE_DIAGONAL, B, D, D)
    nz = _cabi.Noise()
    nz.source, nz.key, nz.cell_id, nz.n_cells, nz.h, nz.h_total = _cabi.SRC_COUNTER, key.data_ptr(), 7, 1, dt, dt
    peak, _ = peaks()

    def milstein(s):
        _cabi.check(lib.tsde_step_milstein(ctypes.byref(L), ctypes.byref(nz), s[0].data_ptr(), s[1].data_ptr(),
                                           s[2].data_ptr(), s[3].data_ptr(), dt, s[4].data_ptr()), "tsde_step_milstein")

    def seed(s):
        _cabi.check(lib.tsde_milstein_vjp_seed(ctypes.byref(L), ctypes.byref(nz), s[0].data_ptr(), dt, 1,
                                               s[1].data_ptr()), "tsde_milstein_vjp_seed")

    out = {}
    for name, nt, launch in (('step_milstein', 5, milstein), ('milstein_vjp_seed', 2, seed)):
        nset = max(2, min(12, int(2e9 // (nt * B * D * 4))))
        sets = [[torch.rand(B, D, device=dev) for _ in range(nt)] for _ in range(nset)]
        for s_ in sets:
            launch(s_)
        torch.cuda.synchronize(dev)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            L.stream = torch.cuda.current_stream(dev).cuda_stream  # launch on the capturing stream
            for s_ in sets:
                launch(s_)
        L.stream = torch.cuda.current_stream(dev).cuda_stream
        graph.replay()
        torch.cuda.synchronize(dev)
        times = []
        for _ in range(7):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            graph.replay()
            e1.record()
            torch.cuda.synchronize(dev)
            times.append(e0.elapsed_time(e1) * 1e3 / nset)
        us = float(np.median(times))
        nbytes = nt * D * 4 * B
        out[name] = {"achieved": nbytes / (us * 1e-6) / 1e9, "frac": nbytes / (us * 1e-6) / 1e9 / peak,
                     "algorithmic_bytes_per_launch": nbytes, "avg_launch_us": us}
        del sets, graph
    return out


# -------------------------------------------------------------------------------------------------
# the other BASELINE.json configs, in the same process (every rank; weak scaling like the headline)
# -------------------------------------------------------------------------------------------------
def _timed(fn, warmup, steps, dev, world):
    import torch.distributed as dist
    for i in range(warmup):
        fn(i)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    gc_was_on = gc.isenabled()
    gc.disable()   # as `timeit` does: a full collection (tens of ms with this process's object count) inside a 1-2 ms
    try:           # host-paced sweep is not the code under test
        e0.record()
        for i in range(steps):
            out = fn(100 + i)
        e1.record()
    finally:
        if gc_was_on:
            gc.enable()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    el = e0.elapsed_time(e1) * 1e-3 / steps
    if world > 1:
        t = torch.tensor([el], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        el = float(t.item())
    return el, out


def run_secondary(rank, world, dev):
    """cfg3 (three solver/noise combinations), cfg4 (sdeint_adjoint forward + backward, batch-sharded with the one
    all-reduce of the parameter gradients) and cfg5 (Brownian query sweeps).  Device-resident, CUDA events, max over
    ranks; every rank owns the config's batch (weak scaling), rows keyed by their global index."""
    import torchsde_b200 as tsde
    from torchsde_b200 import parallel
    from torchsde_b200._core import graph as graph_mod
    from tests import problems
    peak, _ = peaks()
    res = {"note": "per-GPU batch = the config's batch (weak scaling); value = all ranks' trajectory-steps / max-over-"
                   "ranks device time; roofline_frac = E-bytes (SURVEY §8d) x value / n_gpus / measured HBM peak"}
    # ---- cfg3 ----
    for name in ('cfg3_srk_additive', 'cfg3_srk_additive_expand', 'cfg3_euler_general', 'cfg3_heun_general'):
        w = WORKLOADS[name]
        B, D, M, T, dt = w['B'], w['D'], w['M'], w['T'], w['dt']
        sde = build_sde(w, dev)
        ts = (torch.arange(T + 1, dtype=torch.float32) * dt).to(dev)
        y0 = torch.full((B, D), 0.1, device=dev)
        keep = {}

        def solve(i, w=w, sde=sde, ts=ts, y0=y0, keep=keep):
            bm = tsde.BrownianInterval(0.0, w['T'] * w['dt'], size=(w['B'], w['M']), dtype=torch.float32, device=dev,
                                       entropy=500 + i, levy_area_approximation=w.get('levy', 'none'))
            bm.shard_rows(rank * w['B'])
            keep['bm'] = bm
            with torch.no_grad():
                return tsde.sdeint(sde, y0, ts, bm=bm, method=w['method'], dt=w['dt'],
                                   options={'cuda_graph': True, 'static_output': True})
        el, ys = _timed(solve, 3, 5, dev, world)
        parity = parity_check(w, sde, keep['bm'], ys, rank * B) if rank == 0 else None
        v = world * B * T / el
        res[name] = {"value": v, "unit": "traj-steps/s", "ms_per_solve": el * 1e3,
                     "config": {"method": w['method'], "noise": w['kind'], "batch_per_gpu": B, "state": D,
                                "brownian": M, "t_steps": T},
                     "roofline_frac": v / world * w['E_bytes_per_traj_step'] / 1e9 / peak,
                     "parity_check": None if parity is None else {k: parity[k] for k in ('rows', 'max_rel_err')}}
        del ys
        keep.clear()
        graph_mod.drop_plans(sde)
    torch.cuda.empty_cache()
    # ---- cfg4: latent-SDE-like training step, forward + backward ----
    B, D, T, dt = 32768, 128, 256, 2.0 ** -10
    sde = problems.LatentLike(D, hidden=128, seed=0).to(dev)
    ts = (torch.arange(T + 1, dtype=torch.float32) * dt).to(dev)
    y0 = torch.full((B, D), 0.1, device=dev)
    params = list(sde.parameters())

    def train_step(i):
        bm = tsde.BrownianInterval(0.0, T * dt, size=(B, D), dtype=torch.float32, device=dev, entropy=900 + i)
        bm.shard_rows(rank * B)
        ys = tsde.sdeint_adjoint(sde, y0, ts, bm=bm, method='reversible_heun', adjoint_method='adjoint_reversible_heun',
                                 dt=dt, options={'cuda_graph': True}, adjoint_options={'cuda_graph': True})
        loss = ys[-1].pow(2).sum(1).mean() / world
        for p in params:
            p.grad = None
        loss.backward()
        parallel.all_reduce_grads(params)   # the one collective of a batch-sharded adjoint (SURVEY §8e)
        return loss.detach()
    el, loss = _timed(train_step, 2, 3, dev, world)
    gn = float(sum(p.grad.float().norm() ** 2 for p in params) ** .5)
    res['cfg4_adjoint_reversible_heun'] = {
        "value": world * B * T / el, "unit": "traj-steps/s (forward + backward)", "ms_per_step": el * 1e3,
        "config": {"method": "reversible_heun", "adjoint_method": "adjoint_reversible_heun", "noise": "diagonal",
                   "model": "LatentLike MLP(129->128->128) softplus, g = 0.1 sigmoid(w*y+b)", "batch_per_gpu": B,
                   "state": D, "t_steps": T, "output": "full series (T+1,B,D)"},
        "collective": None if world == 1 else "one NCCL all_reduce(sum) of the parameter gradients per step",
        "solver_bytes_per_traj_step": (11 + 23) * D * 4,
        "solver_roofline_frac": world * B * T / el / world * (11 + 23) * D * 4 / 1e9 / peak,
        "loss": float(loss) * world, "grad_norm": gn, "finite": bool(np.isfinite(gn))}
    from torchsde_b200._core import adjoint as adjoint_mod
    graph_mod.drop_plans(sde)
    adjoint_mod.drop_plans(sde)
    del sde, params
    torch.cuda.empty_cache()
    # ---- cfg5: BrownianInterval sweeps, 64 sequential dt-spaced queries ----
    M, nq, h = 16, 64, 2.0 ** -6
    # (SURVEY §8d cfg5: sequential order, then a random permutation of the same 64 intervals — the counter-based
    # source answers a whole-cell query in one launch whatever was asked before it)
    perm = np.random.default_rng(5).permutation(nq).tolist()
    for levy, logb, order in (('none', 20, None), ('space-time', 20, None), ('space-time', 20, perm),
                              ('foster', 17, None), ('foster', 19, None), ('foster', 20, perm)):
        Bq = 1 << logb

        def sweep(i, levy=levy, Bq=Bq, order=order):
            bm = tsde.BrownianInterval(0.0, 1.0, size=(Bq, M), dtype=torch.float32, device=dev, entropy=700 + i, dt=h,
                                       levy_area_approximation=levy)
            bm.shard_rows(rank * Bq)
            for k in (order or range(nq)):
                r = bm(k * h, (k + 1) * h, return_U=levy != 'none', return_A=levy == 'foster')
            return r
        gc.collect()                # (intervals of the previous configuration: node <-> parent cycles hold their tensors)
        el, _ = _timed(sweep, 3, 5, dev, world)
        best = min(_timed(sweep, 0, 1, dev, world)[0] for _ in range(3))
        written = {'none': M * 4, 'space-time': 2 * M * 4, 'foster': (2 * M + M * M) * 4}[levy]
        v = world * Bq * nq / el
        name = f'cfg5_brownian_{levy}' + ('' if logb in (17, 20) and order is None else f'_b2e{logb}') + \
            ('_permuted' if order else '')
        res[name] = {"value": v, "unit": "row-queries/s", "ms_per_sweep": el * 1e3, "ms_per_sweep_best_of_3": best * 1e3,
                                        "config": {"batch_per_gpu": Bq, "channels": M, "queries": nq, "levy": levy,
                                                   "order": "random permutation" if order else "sequential"},
                                        "written_GBps_per_gpu": v / world * written / 1e9,
                                        "write_roofline_frac": v / world * written / 1e9 / peak}
    # batch sweep of the same 64-query pattern (SURVEY §8d: B in 2^10 .. 2^20): where the host's ~tens of microseconds
    # per Python-level query stop mattering
    sweep_res = {}
    for levy in ('none', 'space-time', 'foster'):
        for logb in (10, 12, 14, 16, 18):
            def sweep(i, levy=levy, Bq=1 << logb):
                bm = tsde.BrownianInterval(0.0, 1.0, size=(Bq, M), dtype=torch.float32, device=dev, entropy=800 + i,
                                           dt=h, levy_area_approximation=levy)
                bm.shard_rows(rank * Bq)
                for k in range(nq):
                    r = bm(k * h, (k + 1) * h, return_U=levy != 'none', return_A=levy == 'foster')
                return r
            el, _ = _timed(sweep, 2, 3, dev, world)
            sweep_res[f'{levy}_b2e{logb}'] = {"row_queries_per_s": world * (1 << logb) * nq / el,
                                              "us_per_query": el / nq * 1e6}
    res['cfg5_batch_sweep'] = sweep_res
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='cfg2', choices=sorted(WORKLOADS))
    ap.add_argument('--no-graph', action='store_true')
    ap.add_argument('--no-secondary', action='store_true', help='skip the cfg3/cfg4/cfg5 block')
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline sample')
    ap.add_argument('--row-split', type=int, default=1)
    ap.add_argument('--strong', action='store_true',
                    help='strong scaling: the workload batch is the GLOBAL batch, split over the ranks')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write the output of the last timed solve to DIR/*.npy '
                         '(see dump_outputs)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes the output of the GPU path (--impl ours)')
    w = dict(WORKLOADS[args.workload])
    if os.environ.get('TSDE_BENCH_B'):  # experiments only: override the batch size
        w['B'] = int(os.environ['TSDE_BENCH_B'])
    if args.strong:
        w['B'] = w['B'] // max(int(os.environ.get('WORLD_SIZE', '1')), 1)
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if args.impl == 'reference':
        run_reference(args, w, rank, world)
        return
    if os.environ.get('TSDE_BENCH_NO_PG') and world > 1:
        # bisecting aid (profiles/r02_multi_gpu_bisect.sh): N ranks under torchrun but NO process group — every rank
        # behaves like an independent single-GPU run on its own device and prints its own line
        world, rank = 1, 0
    group = world > 1 or bool(os.environ.get('TSDE_FORCE_PG'))  # (TSDE_FORCE_PG: bisecting aid, a 1-rank NCCL group)
    if group:
        import torch.distributed as dist
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        os.environ.setdefault('MASTER_PORT', '29512')
        os.environ.setdefault('RANK', '0')
        os.environ.setdefault('WORLD_SIZE', '1')
        torch.cuda.set_device(local_rank)
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
        if world == 1:
            dist.barrier()
    try:
        run_ours(args, w, rank, world, local_rank)
    finally:
        if group:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == '__main__':
    main()
