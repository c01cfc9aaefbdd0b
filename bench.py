#!/usr/bin/env python
"""bench.py - throughput of the CityLearn step path on B200 (driver contract: one JSON line on rank 0).

Workload (BASELINE.json configs[1]): citylearn_challenge_2022_phase_all, 17 buildings x 4096 parallel envs PER GPU
(weak scaling: envs shard across GPUs with no data-path collective, SURVEY.md §8e), synthetic uniform(-1, 1) actions.
A "step" is one environment time step of all 17 x 4096 units of a rank: actions in, state update, district sums, reward,
observation at t+1 out.  Metric: building-env steps / s (whole job, all ranks).

  value     device-resident: the timed region is exactly K = --steps steps, ONE `cl_rollout` launch after W = --warmup untimed
            steps (actions [K,E,A] already in HBM, every step writes its own observation / reward slab, so the launch's K * 7.8 MB
            output stream is larger than the 126 MB L2 for K >= 17), bracketed by CUDA events on the launch stream (max over
            ranks); both launches are queued behind ~10 ms of device writes, so the timed one runs under sustained memory load
            and host launch latency stays outside the bracket (see `timed_rollout`).
            `--dump-outputs DIR` writes what that launch computed for its last step (see `dump_outputs`).
  e2e       the public API with HOST buffers, K steps: env.step_host(ndarray) -> ONE native call per step (cl_step_host): this step's
            [E, A] actions wait in page-locked host memory and are read over PCIe by the step kernel, the rewards + the observation
            row (reference-parity observation rows are identical for every env, so one row crosses PCIe and the host gets a
            broadcast view) are written back to page-locked host memory by the kernels, then the stream is synchronised.
            `e2e_dma_copies` is the same loop with cudaMemcpyAsync H2D / D2H around the kernel, `e2e_full_observations` the loop with
            the full [E, L] observation copy, `e2e_rollout_host` one call of K steps.
  roofline  HBM: bytes a rollout launch MOVES (actions + observations + rewards + district sums; the unit state stays in
            registers between the steps of a launch) / launch duration.
  cpu_baseline  the UNMODIFIED reference (oracle/_ref, installed by oracle/build_ref.py) on one host core, when present; else the
            NumPy oracle port.
  extra     (N = 1, or --extras; C4 and C5 at every N) BASELINE configs[4] (C5: closed loop with an on-device policy, 32 768 envs in total),
            BASELINE configs[2] (C3: 3 LSTM buildings x 65 536 envs, MARL; LSTM cell on the tensor cores), configs[3] per-GPU share (C4: synthetic 1024 buildings x 1024 envs, full-year rollout) and configs[1] with
            stale_observations=False (fresh observations) ride on the same JSON line under "extra"; at N > 1 also the building-sharded
            district (district sums completed inside the step kernel over NVLink peer memory vs the NCCL two-phase variant).
            The extras keep their own fixed step counts; --steps sets those of configs[1] (value, e2e, fresh observations).

`--impl reference` times the reference's own CPU step on all host cores (one process per core, one env each; oracle/_ref when it
travelled with the snapshot, else the oracle port) and prints the same line with "impl": "reference".
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
for p in (ROOT, ROOT / 'oracle'):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

DATASET = 'citylearn_challenge_2022_phase_all'
ENVS_PER_GPU = 4096
METRIC = 'building_env_steps_per_sec'
UNIT = 'building-env steps/s'


def bytes_per_unit(precision: str, n_obs: float, n_act: float, n_buildings: int, rollout: bool = True, reward_dim: float = 1.0) -> float:
    """Algorithmic HBM bytes per (building, env) per step (SURVEY.md §8d): actions read, obs + reward + district written, and -
    for single-step launches only - the unit state read + written (fp64 flow: 20 B, fp32: 12 B).  A rollout launch keeps the
    state in registers between its steps, so those bytes do not move (rollout=True drops them)."""
    state = 0 if rollout else (20 if precision == 'fp64' else 12)
    return 4 * n_act + 2 * state + 4 * n_obs + 4 * reward_dim + 12.0 / n_buildings


class ClockSampler:
    """SM clocks / throttle reasons sampled DURING the timed regions through NVML in a background thread
    (same fields as the nvidia-smi line in B200_PROFILING.md, without spawning a process that perturbs the host loop)."""

    def __init__(self, index: int, period_s: float = 0.1):
        self.index, self.period = index, period_s
        self.sm, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self.thread = None
        self.ok = False

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            # NVML enumerates physical GPUs; honour CUDA_VISIBLE_DEVICES when it is a plain index list
            vis = os.environ.get('CUDA_VISIBLE_DEVICES')
            phys = self.index
            if vis:
                try:
                    phys = int(vis.split(',')[self.index])
                except Exception:
                    phys = self.index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.ok = False
            return self._start_smi()
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def _start_smi(self):
        """Fallback: the nvidia-smi line of B200_PROFILING.md at a low rate."""
        q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--id={self.index}', f'--query-gpu={q}', '--format=csv,noheader,nounits', '-lms', '250'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            return

        def read():
            for line in self.proc.stdout:
                r = [x.strip() for x in line.split(',')]
                try:
                    self.sm.append(float(r[0]))
                    self.max_mhz = float(r[1])
                    for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[2:6]):
                        if v.lower().startswith('active'):
                            self.reasons.add(name)
                except Exception:
                    pass
        self.thread = threading.Thread(target=read, daemon=True)
        self.thread.start()
        self.ok = True
        self.smi = True

    def _run(self):
        nv = self.nv
        names = {'hw_slowdown': nv.nvmlClocksEventReasonHwSlowdown, 'hw_thermal_slowdown': nv.nvmlClocksEventReasonHwThermalSlowdown,
                 'sw_thermal_slowdown': nv.nvmlClocksEventReasonSwThermalSlowdown, 'sw_power_cap': nv.nvmlClocksEventReasonSwPowerCap} \
            if hasattr(nv, 'nvmlClocksEventReasonHwSlowdown') else \
                {'hw_slowdown': nv.nvmlClocksThrottleReasonHwSlowdown, 'hw_thermal_slowdown': nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                 'sw_thermal_slowdown': nv.nvmlClocksThrottleReasonSwThermalSlowdown, 'sw_power_cap': nv.nvmlClocksThrottleReasonSwPowerCap}
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(self.period)

    def stop(self):
        if not self.ok:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable']}
        self._stop.set()
        if getattr(self, 'smi', False):
            self.proc.terminate()
        self.thread.join(timeout=2)
        sm = sorted(self.sm)
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons), 'samples': len(sm)}


def cpu_oracle_rate(n_envs: int, steps: int, seed: int = 0):
    """building-env steps / s of the NumPy oracle on ONE core for `steps` steps of `n_envs` envs."""
    import numpy as np
    from citylearn_b200 import schema as S
    from citylearn_oracle import OracleEnv
    spec = S.load(DATASET)
    env = OracleEnv(spec, n_envs)
    env.reset()
    rng = np.random.RandomState(seed)
    acts = rng.uniform(-1, 1, size=(steps + 1, n_envs, spec.action_dim)).astype('float32')
    env.step(acts[0])
    t0 = time.perf_counter()
    for k in range(steps):
        env.step(acts[k + 1])
    dt = time.perf_counter() - t0
    return spec.n_buildings * n_envs * steps / dt, dt


def effective_cpus() -> int:
    """Host cores this process may really use: min(affinity, cgroup CPU quota)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    for path in ('/sys/fs/cgroup/cpu.max', '/sys/fs/cgroup/cpu/cpu.cfs_quota_us'):
        try:
            txt = open(path).read().split()
            if path.endswith('cpu.max'):
                if txt[0] != 'max':
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]))))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
                    n = min(n, max(1, q // per))
            break
        except Exception:
            continue
    return n


REF_DIR = ROOT / 'oracle' / '_ref'


def reference_available() -> bool:
    return (REF_DIR / 'site' / 'citylearn' / 'citylearn.py').is_file() and (REF_DIR / 'data' / 'datasets' / DATASET / 'schema.json').is_file()


def cpu_reference_rate(steps: int, warm: int = 2, seed: int = 0):
    """building-env steps / s of the UNMODIFIED reference (oracle/_ref) on ONE core: its own `CityLearnEnv.step` loop, one env."""
    import shutil
    import logging
    import numpy as np
    os.environ['XDG_CACHE_HOME'] = str(REF_DIR / 'cache')          # DataSet()'s cache stays inside oracle/_ref (git-ignored)
    for q in (ROOT / 'oracle' / 'shims', REF_DIR / 'site'):
        if str(q) not in sys.path:
            sys.path.insert(0, str(q))
    from platformdirs import user_cache_dir
    d = Path(user_cache_dir(appname='citylearn', appauthor='intelligent-environments-lab', version='v2.4.2')) / 'misc'
    d.mkdir(parents=True, exist_ok=True)
    for f in ('battery_choices.yaml', 'lbl-tracking_the_sun-res-pv.csv'):      # CityLearnEnv._load asks DataSet() for them (citylearn.py:2055-2057)
        if not (d / f).is_file():
            shutil.copy(REF_DIR / 'data' / 'misc' / f, d / f)
    logging.getLogger().setLevel(logging.WARNING)
    from citylearn.citylearn import CityLearnEnv as RefEnv
    env = RefEnv(str(REF_DIR / 'data' / 'datasets' / DATASET / 'schema.json'))
    env.reset()
    B = len(env.buildings)
    rng = np.random.RandomState(seed)
    acts = [[[float(x)] for x in rng.uniform(-1, 1, B)] for _ in range(steps + warm)]
    for k in range(warm):
        env.step(acts[k])
    t0 = time.perf_counter()
    for k in range(warm, warm + steps):
        env.step(acts[k])
    dt = time.perf_counter() - t0
    return B * steps / dt, dt


def _ref_worker(args):
    kind, n_envs, steps, warm, seed = args
    os.environ.setdefault('OMP_NUM_THREADS', '1')
    if kind == 'reference':
        return cpu_reference_rate(steps, warm, seed)
    return cpu_oracle_rate(n_envs, steps + warm, seed)


def run_reference(args):
    """CPU arm on all host cores, one process per core: the UNMODIFIED reference (oracle/_ref, one env per process - it is
    single-threaded and single-env) when it travelled with the snapshot, else the oracle port (envs split evenly)."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import multiprocessing as mp
    procs = max(1, min(effective_cpus(), 128))
    steps, warm = args.steps, args.warmup
    real = reference_available()
    per = 1 if real else max(1, ENVS_PER_GPU // procs)
    ctx = mp.get_context('spawn' if real else 'fork')
    t0 = time.perf_counter()
    with ctx.Pool(procs) as pool:
        res = pool.map(_ref_worker, [('reference' if real else 'port', per, steps, warm, i) for i in range(procs)])
    wall = time.perf_counter() - t0
    # per-process rates exclude construction; sum over processes = whole-host throughput
    value = float(sum(r for r, _ in res))
    ms = 1e3 * max(dt for _, dt in res) / (steps if real else steps + warm)
    note = ('the UNMODIFIED reference (CityLearn v2.4.2 installed into oracle/_ref by oracle/build_ref.py): its own CityLearnEnv.step loop, '
            'one single-env process per host core') if real else \
           ('CPU port of the reference algorithm (oracle/citylearn_oracle.py, NumPy, float64 intermediates); oracle/_ref did not travel - '
            'BASELINE.md has the reference\'s measured 871.7 building-steps/s/core')
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': steps, 'warmup': warm,
        'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': f'{DATASET}: 17 buildings x {ENVS_PER_GPU} envs per GPU, observations 476/env, actions 17/env',
                   'sample': f'bounded sample: {procs} processes x {per} env(s) x {steps} steps', 'note': note},
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': procs, 'kind': 'reference' if real else 'port',
                         'sample': f'{procs} processes x {per} env(s) x {steps} timed steps (+{warm} warm-up), wall {wall:.1f}s incl. construction'},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


def timed_rollouts(env, torch, acts, obs, rew, dst, K: int, R: int, reset_every: int = 0):
    """R back-to-back K-step `cl_rollout` launches, each bracketed by CUDA events on the launch stream; nothing synchronises the
    host in between, so from the second launch on the GPU never waits for the host.  Returns per-launch milliseconds."""
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(R)]
    for i in range(R):
        if env.time_step + K > env.time_steps - 1:
            env.reset()                      # outside the brackets
        ev[i][0].record()
        env.rollout(acts, obs, rew, dst)
        ev[i][1].record()
    torch.cuda.synchronize(env.device)
    return [a.elapsed_time(b) for a, b in ev]


def timed_rollout(env, torch, acts, obs, rew, dst, K: int, W: int):
    """From a reset: W untimed warm-up steps in one launch, then ONE `cl_rollout` launch of exactly K steps bracketed by CUDA events on
    the launch stream.  Returns (milliseconds, kernel launches inside the bracket).

    Both launches are queued behind ~10 ms of writes to the output buffers and nothing synchronises the host in between, so the
    timed launch starts while the device is under sustained memory load, right after the warm-up launch, and the host's launch
    latency stays outside the bracket.  Measured on B200 (1000 W): after 1 ms of idle HBM the same launch runs 1.5 % slower
    (17 x 4096 envs, K = 100) than under sustained load, the state a training loop stepping the env sees."""
    env.reset()
    nbytes = sum(t.numel() * t.element_size() for t in (obs, rew, dst))
    for _ in range(min(2000, 1 + int(10e-3 * 6e12 / nbytes))):
        obs.zero_(); rew.zero_(); dst.zero_()
    env.rollout(acts[:W].contiguous(), obs[:W], rew[:W], dst[:W])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n0 = env.gpu_launches
    e0.record()
    env.rollout(acts[:K].contiguous(), obs[:K], rew[:K], dst[:K])
    e1.record()
    torch.cuda.synchronize(env.device)
    return e0.elapsed_time(e1), env.gpu_launches - n0


def dump_outputs(out_dir, arrays, budget=64 << 20, seed=0):
    """Write each [E, ...] array as `out_dir/<name>.npy`.  Above `budget` bytes in all, every array keeps the same rows: a fixed sample
    of the envs drawn with `seed`, in ascending order."""
    import numpy as np
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    n_envs = len(next(iter(arrays.values())))
    row_bytes = sum(a[0].nbytes for a in arrays.values())
    if n_envs * row_bytes > budget:
        keep = np.sort(np.random.default_rng(seed).choice(n_envs, budget // row_bytes, replace=False))
        arrays = {k: a[keep] for k, a in arrays.items()}
    for name, a in arrays.items():
        np.save(out / f'{name}.npy', a)


def median(xs):
    ys = sorted(xs)
    return ys[len(ys) // 2]


def timing_summary(ms, K):
    return {'repeats': len(ms), 'median_us_per_step': 1e3 * median(ms) / K, 'min_us_per_step': 1e3 * min(ms) / K,
            'max_us_per_step': 1e3 * max(ms) / K, 'first_launch_us_per_step': 1e3 * ms[0] / K}


def extra_fresh_c2(torch, dev, precision, K, W, peak):
    """BASELINE configs[1] with stale_observations=False: observations carry soc / net of the step (per-env row images)."""
    from citylearn_b200 import CityLearnEnv
    E = ENVS_PER_GPU
    env = CityLearnEnv(DATASET, num_envs=E, device=dev, precision=precision, stale_observations=False)
    B, A, L = env.spec.n_buildings, env.spec.action_dim, env._obs_dim
    N = max(K, W)
    acts = torch.rand((N, E, A), device=dev) * 2 - 1
    obs = torch.empty((N, E, L), device=dev); rew = torch.empty((N, E, B), device=dev); dst = torch.empty((N, E, 3), device=dev)
    m, _ = timed_rollout(env, torch, acts, obs, rew, dst, K, W)
    bpu = bytes_per_unit(precision, L / B, A / B, B)
    out = {'workload': f'{DATASET}: {B} x {E} envs, stale_observations=False (fresh observations)', 'ms_per_step': m / K,
           'value': B * E * K / (m * 1e-3), 'unit': UNIT, 'table_path': bool(env._h.geometry()),
           'roofline': {'bound': 'hbm', 'achieved': bpu * B * E * K / (m * 1e-3) / 1e9, 'peak': peak, 'unit': 'GB/s',
                        'frac': bpu * B * E * K / (m * 1e-3) / 1e9 / peak, 'bytes_per_unit': bpu}}
    env.close()
    return out


def extra_c3(torch, dev, precision, fma_peak):
    """BASELINE configs[2]: 2023 schema, 3 LSTM buildings x 65 536 envs, MARL per-building rewards, past the LSTM warm-up."""
    from citylearn_b200 import CityLearnEnv
    from citylearn_b200.data import DataSet
    src = DataSet.get_source('citylearn_challenge_2023_phase_2_local_evaluation')
    sch = src.schema()
    sch['reward_function'] = {'type': 'citylearn.reward_function.MARL', 'attributes': {}}
    E, K, W, R = 65536, 20, 16, 8
    env = CityLearnEnv(sch, data_source=src, central_agent=False, num_envs=E, device=dev, precision=precision)
    B, A, L = env.spec.n_buildings, env.spec.action_dim, env._obs_dim
    lo = torch.tensor([v for b in env.spec.buildings for v in b.action_low], device=dev)
    hi = torch.tensor([v for b in env.spec.buildings for v in b.action_high], device=dev)
    acts = lo + torch.rand((K, E, A), device=dev) * (hi - lo)
    obs = torch.empty((K, E, L), device=dev); rew = torch.empty((K, E, B), device=dev)
    env.reset()
    env.rollout(acts[:W].contiguous(), obs[:W], rew[:W], None)            # LSTM warm-up (12-step lookback)
    ms = timed_rollouts(env, torch, acts, obs, rew, None, K, R)
    m = median(ms)
    flop_unit = 93696.0 + 150.0                                            # SURVEY.md §8d: 46 848 LSTM MACs + device arithmetic
    tf = flop_unit * B * E * K / (m * 1e-3) / 1e12
    geo = env._h.geometry()
    tensor = os.environ.get('CL_B200_NO_LSTM_MMA') is None
    out = {'workload': f'citylearn_challenge_2023_phase_2_local_evaluation: {B} LSTM buildings x {E} envs, MARL, decentralised', 'ms_per_step': m / K,
           'value': B * E * K / (m * 1e-3), 'unit': UNIT, 'timing': timing_summary(ms, K), 'geometry': geo,
           'lstm_cell': ('tensor cores: mma.sync m16n8k8 TF32 operands, FP32 accumulate, 3 MMAs per product on hi / lo splits (float32-level accuracy)'
                         if tensor else 'scalar float32 FMAs, weights broadcast from shared memory'),
           # algorithmic FLOPs of the float32 cell (SURVEY.md §8d) against the measured FP32-FMA throughput: what a scalar cell could reach at best;
           # the tensor-core cell executes 3x the multiply-adds of the recurrent products on the (legacy) tensor path instead
           'roofline': {'bound': 'fp32_fma', 'achieved': tf, 'peak': fma_peak, 'unit': 'TFLOP/s', 'frac': tf / fma_peak if fma_peak else None,
                        'flop_per_unit': flop_unit, 'peak_source': 'cl_measure_fma_peak (independent FFMA chains, this device)'}}
    env.close()
    return out


def extra_c4(torch, dev, precision, peak, world, dist):
    """BASELINE configs[3], this GPU's share: synthetic 1024 buildings x 1024 envs, the FULL 8 759-step year as back-to-back
    32-step `cl_rollout` launches (observations + rewards + district sums written every step).  With N ranks the job is the
    configs[3] district at N x 1024 envs (env-sharded, no collective)."""
    from citylearn_b200 import CityLearnEnv, schema as S
    from citylearn_b200.synthetic import make_wide_district
    sch, src = make_wide_district(1024)
    spec = S.load(sch, data_source=src)
    E, K = 1024, 32                     # 32 steps per launch: observation slab 3.8 GB + rewards 134 MB per launch
    env = CityLearnEnv(spec, num_envs=E, device=dev, precision=precision)
    B, A, L = spec.n_buildings, spec.action_dim, env._obs_dim
    acts = torch.rand((K, E, A), device=dev) * 2 - 1
    obs = torch.empty((K, E, L), device=dev); rew = torch.empty((K, E, env._reward_dim), device=dev); dst = torch.empty((K, E, 3), device=dev)
    env.reset()
    timed_rollouts(env, torch, acts, obs, rew, dst, K, 2)
    env.reset()
    T1 = env.time_steps - 1
    n_full, rest = divmod(T1, K)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n_full):
        env.rollout(acts, obs, rew, dst)
    if rest:
        env.rollout(acts[:rest].contiguous(), obs[:rest], rew[:rest], dst[:rest])
    e1.record()
    torch.cuda.synchronize(dev)
    assert env.terminated
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    bpu = bytes_per_unit(precision, L / B, A / B, B)
    gbs = bpu * B * E * T1 / (ms * 1e-3) / 1e9
    out = {'workload': f'synthetic {B} buildings x {E} envs per GPU ({world * E} envs on {world} GPU(s)), full {T1}-step year', 'year_ms': ms,
           'ms_per_step': ms / T1, 'value': world * B * E * T1 / (ms * 1e-3), 'unit': UNIT, 'launches': n_full + (1 if rest else 0), 'geometry': env._h.geometry(),
           'roofline': {'bound': 'hbm', 'achieved': gbs, 'peak': peak, 'unit': 'GB/s', 'frac': gbs / peak, 'bytes_per_unit': bpu}}
    env.close()
    return out


def extra_c5(torch, dev, precision, world, dist, K_total=96, n_graph=8):
    """BASELINE configs[4]: SAC-style closed loop on 2022_phase_all, 32 768 envs in total (strong scaling: 32 768 / N per GPU),
    fresh observations.  Per step: a random-init per-building actor (17 x [28 -> 256 -> 256 -> 1], bf16 cuBLAS batched matmuls - the
    policy is the caller's, not part of the accelerated path) reads the observation slab on the device, writes the actions, and
    `cl_advance_device` steps the env - `n_graph` such steps captured as ONE CUDA graph and replayed (no host round trip); after every
    replay a parameter-sized float32 buffer is all-reduced over NCCL (stand-in for a DDP gradient exchange; skipped at N = 1)."""
    from citylearn_b200 import CityLearnEnv
    from citylearn_b200.closed_loop import ClosedLoop, PerBuildingMLP
    E = 32768 // world
    env = CityLearnEnv(DATASET, num_envs=E, device=dev, precision=precision, stale_observations=False)
    B, A, L = env.spec.n_buildings, env.spec.action_dim, env._obs_dim
    pol = PerBuildingMLP(B, L // B, A // B, hidden=256, dtype=torch.bfloat16, device=dev)
    grads = torch.zeros(pol.parameter_count(), dtype=torch.float32, device=dev)
    loop = ClosedLoop(env, pol, steps_per_replay=n_graph)

    def iterate(n_steps):
        for _ in range(n_steps // n_graph):
            loop.run(n_graph)
            if world > 1:
                dist.all_reduce(grads)
    iterate(2 * n_graph)                                   # warm-up
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); iterate(K_total); e1.record()
    torch.cuda.synchronize(dev)
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    # env-only share of the same loop: the identical graph with a policy that writes constant actions
    env2 = CityLearnEnv(DATASET, num_envs=E, device=dev, precision=precision, stale_observations=False)
    const = torch.zeros((E, A), device=dev)
    loop2 = ClosedLoop(env2, lambda o: const, steps_per_replay=n_graph)
    loop2.run(2 * n_graph)
    torch.cuda.synchronize(dev)
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record(); loop2.run(K_total); f1.record()
    torch.cuda.synchronize(dev)
    t2 = torch.tensor([f0.elapsed_time(f1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX); dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    ms, ms_env = float(t.item()), float(t2.item())
    out = {'workload': f'{DATASET}: {B} x {E} envs per GPU ({world * E} envs on {world} GPU(s)), stale_observations=False, closed loop with a per-building 2 x 256 MLP actor (bf16)',
           'ms_per_step': ms / K_total, 'value': world * B * E * K_total / (ms * 1e-3), 'unit': UNIT, 'steps': K_total, 'steps_per_graph_replay': n_graph,
           'policy_parameters': pol.parameter_count(), 'allreduce': None if world == 1 else f'{grads.numel() * 4} B float32 (NCCL) after every {n_graph} steps',
           'env_only_ms_per_step': ms_env / K_total, 'env_only_value': world * B * E * K_total / (ms_env * 1e-3),
           'policy_flop_per_step': 2.0 * E * B * ((L // B) * 256 + 256 * 256 + 256 * (A // B)), 'scaling': 'strong (32768 envs in total)'}
    env.close(); env2.close()
    return out


def extra_building_sharded(torch, dev, precision, world, dist, rank, K=40, R=8, E=4096):
    """SURVEY.md §8e "district all-reduce variant" (north_star: district-level reward terms across GPUs): 2022_phase_all with the 17
    buildings of EVERY env split over the N GPUs, MARL rewards (they read the district sum inside the step).  Three ways to complete
    the per-env district sums: (p2p_rollout) the fused path - K steps in ONE persistent launch per GPU, partial sums pushed into the
    peers' memory over NVLink and summed in the kernel; (p2p_step) the same exchange with one launch per step; (nccl_step) the
    two-phase baseline - kernel, `all_reduce` (NCCL), reward evaluation with tensor ops.  value = buildings x envs x steps / s of the
    whole district (17 x E), max over ranks."""
    import citylearn_b200.reward_function as rf
    from citylearn_b200.distributed import BuildingShardedEnv
    out = {'workload': f'{DATASET}: 17 buildings split over {world} GPUs x {E} envs, MARL (district sum inside the step)', 'unit': UNIT}

    def timed(fn, n_steps, reps):
        ms = []
        for _ in range(reps):
            torch.cuda.synchronize(dev); dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record(); torch.cuda.synchronize(dev)
            ms.append(e0.elapsed_time(e1))
        t = torch.tensor([median(ms)], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / n_steps

    sh = BuildingShardedEnv(DATASET, E, device=dev, exchange='p2p', reward_function=rf.MARL, precision=precision)
    env = sh.env
    Bl, A, L = env.spec.n_buildings, env.spec.action_dim, env._obs_dim
    acts = torch.rand((K, E, A), device=dev) * 2 - 1
    obs = torch.empty((K, E, L), device=dev); rew = torch.empty((K, E, Bl), device=dev); dst = torch.empty((K, E, 3), device=dev)
    sh.reset(); sh.rollout(acts, obs, rew, dst)
    ms = timed(lambda: sh.rollout(acts, obs, rew, dst), K, R)
    out['p2p_rollout'] = {'ms_per_step': ms, 'value': 17 * E / (ms * 1e-3), 'steps_per_launch': K, 'buildings_on_rank0': Bl}

    def steps_p2p():
        for k in range(K):
            sh.step(acts[k])
    sh.reset(); steps_p2p()
    ms = timed(steps_p2p, K, 3)
    out['p2p_step'] = {'ms_per_step': ms, 'value': 17 * E / (ms * 1e-3)}
    st = sh.exchange_status()
    out['exchange'] = st
    checksum = float(dst[-1].double().sum().item())
    sh.close()

    sn = BuildingShardedEnv(DATASET, E, device=dev, exchange='nccl', reward_function=rf.MARL, precision=precision)

    def steps_nccl():
        for k in range(K):
            sn.step(acts[k])
    sn.reset(); steps_nccl()
    ms = timed(steps_nccl, K, 3)
    out['nccl_step'] = {'ms_per_step': ms, 'value': 17 * E / (ms * 1e-3)}
    sn.close()
    # the same district env-sharded (no exchange at all): this rank's E / N envs of all 17 buildings
    from citylearn_b200 import CityLearnEnv
    Es = E // world
    es = CityLearnEnv(DATASET, num_envs=Es, device=dev, precision=precision, central_agent=False, reward_function=rf.MARL)
    a2 = torch.rand((K, Es, 17), device=dev) * 2 - 1
    o2 = torch.empty((K, Es, es._obs_dim), device=dev); r2 = torch.empty((K, Es, 17), device=dev); d2 = torch.empty((K, Es, 3), device=dev)
    es.reset(); es.rollout(a2, o2, r2, d2)
    ms = timed(lambda: es.rollout(a2, o2, r2, d2), K, R)
    out['env_sharded_rollout'] = {'ms_per_step': ms, 'value': 17 * E / (ms * 1e-3)}
    es.close()
    out['district_checksum'] = checksum
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=100)
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--precision', default='fp64', choices=['fp64', 'fp32'])
    ap.add_argument('--envs', type=int, default=ENVS_PER_GPU, help='parallel envs per GPU')
    ap.add_argument('--extras', default='auto', choices=['auto', 'all', 'none'], help="C3 / C4 / fresh-observation numbers under 'extra' (auto: N = 1 all, N > 1 C4 only)")
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', help='after the timed steps, write the observations [E, L], rewards [E, B] and district '
                    'sums [E, 3] of the last timed step (rank 0, float32) as DIR/<name>.npy; above 64 MB in all, a fixed seeded sample of the envs')
    args = ap.parse_args()
    if args.impl == 'reference':
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    from citylearn_b200 import CityLearnEnv, _native

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    assert torch.cuda.is_available(), 'bench.py needs a CUDA device'
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    K, W, E = args.steps, max(args.warmup, 3), args.envs
    env = CityLearnEnv(DATASET, num_envs=E, device=dev, precision=args.precision)
    B, A, L = env.spec.n_buildings, env.spec.action_dim, env._obs_dim
    T1 = env.time_steps - 1
    assert W + K <= T1, 'steps + warmup must fit in one episode'

    # ---------------- device-resident throughput ----------------
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    acts = torch.rand((max(K, W), E, A), device=dev, generator=g) * 2 - 1
    obs = torch.empty((max(K, W), E, L), device=dev)
    rew = torch.empty((max(K, W), E, B), device=dev)
    dst = torch.empty((max(K, W), E, 3), device=dev)
    peaks = {}
    try:
        peaks = json.loads((ROOT / 'MEASURED_PEAKS.json').read_text())
    except Exception:
        pass
    peak = float(peaks.get('hbm_gbs', 6650.0))
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    torch.cuda.synchronize(dev)
    ms_launch, launches = timed_rollout(env, torch, acts, obs, rew, dst, K, W)    # W untimed warm-up steps, then ONE launch of K steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {'observations': obs[K - 1].cpu().numpy(), 'rewards': rew[K - 1].cpu().numpy(),
                                         'district': dst[K - 1].cpu().numpy()})
    t = torch.tensor([ms_launch], device=dev, dtype=torch.float64)
    if world > 1:
        dist.barrier()
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    checksum = float(rew[:K].sum().item())            # reads the result back: the step's rewards
    units_per_step = B * E
    value = world * units_per_step * K / (ms_max * 1e-3)

    # ---------------- end to end through the public API with host buffers ----------------
    env_host_mode = env._host_in_place

    def e2e_loop(full, in_place=True):
        env.reset()
        env._host_in_place = env_host_mode if in_place else 0
        # this step's actions wait in page-locked host memory (the contract's "host->device copy ... from pinned host memory"): a host-side
        # policy writes them there; every step copies ITS OWN [E, A] block to the device inside the timed region
        host_pinned = torch.empty((W + K, E, A), dtype=torch.float32).pin_memory()
        host_acts = host_pinned.numpy()
        host_acts[...] = np.random.RandomState(7 + rank).uniform(-1, 1, size=(W + K, E, A)).astype('float32')
        for k in range(W):
            env.step_host(host_acts[k], full_observations=full)
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        acc = 0.0
        for k in range(W, W + K):
            o, r, term = env.step_host(host_acts[k], full_observations=full)
            acc += float(r[0, 0]) + float(o[E - 1, 0])
        ev1.record()
        torch.cuda.synchronize(dev)
        tt = torch.tensor([ev0.elapsed_time(ev1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.barrier()
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item()), acc
    e2e_ms, e2e_sum = e2e_loop(None)                   # shared observation row (reference-parity rows are env-independent)
    e2e_full_ms, _ = e2e_loop(True)                    # full [E, L] copy, for comparison
    e2e_dma_ms, _ = e2e_loop(None, in_place=False)     # same as e2e, but DMA copies before / after the kernel instead of in-place access
    env._host_in_place = env_host_mode
    # K steps as ONE host call: one H2D of [K, E, A], one launch, one D2H of rewards + K rows
    env.reset()
    blk = np.random.RandomState(9 + rank).uniform(-1, 1, size=(K, E, A)).astype('float32')
    env.rollout_host(blk)
    torch.cuda.synchronize(dev)
    if env.time_step + K > T1:
        env.reset()
    t0 = time.perf_counter(); env.rollout_host(blk)
    blk_s = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(blk_s, op=dist.ReduceOp.MAX)
    e2e_value = world * units_per_step * K / (e2e_ms * 1e-3)
    clocks = sampler.stop() if rank == 0 else None

    # ---------------- other BASELINE configs on the same line ----------------
    extra = {}
    want = args.extras
    fma_peak = None
    def hard_exit():
        # (multi-rank runs) leave without tearing the process group down: ranks finish at different times (rank 0 still times the CPU
        # baseline), and a communicator teardown that waits for a peer which is already gone has hung a 2-GPU run for minutes AFTER
        # the result line was out.  Everything is flushed; exit code 0.
        sys.stdout.flush(); sys.stderr.flush()
        os._exit(0)

    def guarded(name, fn):          # an extra must never take the headline (or another extra) down
        try:
            extra[name] = fn()
        except Exception as e:
            extra[name] = {'error': repr(e)[:300]}
    if want == 'all' or (want == 'auto' and world == 1):
        if rank == 0:
            with torch.cuda.device(dev):
                fma_peak = _native.measure_fma_peak()
            guarded('fresh_observations_c2', lambda: extra_fresh_c2(torch, dev, args.precision, K, W, peak))
            guarded('c3_lstm_marl', lambda: extra_c3(torch, dev, args.precision, fma_peak))
    if want != 'none':
        guarded('c4_wide_year', lambda: extra_c4(torch, dev, args.precision, peak, world, dist))
        guarded('c5_closed_loop', lambda: extra_c5(torch, dev, args.precision, world, dist))
        if world > 1:
            guarded('building_sharded_district', lambda: extra_building_sharded(torch, dev, args.precision, world, dist, rank))

    if rank != 0:
        hard_exit()

    bpu = bytes_per_unit(args.precision, L / B, A / B, B, rollout=True)
    bpu_step = bytes_per_unit(args.precision, L / B, A / B, B, rollout=False)
    # the timed region is one launch of the rollout kernel, K steps: algorithmic bytes per launch = K steps x bytes a step moves;
    # duration = CUDA events on the launch stream
    bytes_per_launch = bpu * units_per_step * K
    achieved = bytes_per_launch / (ms_launch * 1e-3) / 1e9
    traffic = None
    traffic_note = None
    try:
        # measured DRAM bytes (ncu --set full: dram__bytes_read.sum + dram__bytes_write.sum) of ONE launch of this exact configuration
        # (precision, envs, steps per launch); absent for other configurations
        rec = json.loads((ROOT / 'profiles' / 'step_kernel_traffic.json').read_text())
        hit = rec.get(f'{args.precision}:{E}:{K}')
        if hit:
            traffic = hit['dram_read_bytes'] + hit['dram_write_bytes']
            traffic_note = hit.get('source')
    except Exception:
        pass
    cpu = None
    if not args.no_cpu_baseline:
        if reference_available():
            rate, dt = cpu_reference_rate(600, 3)       # ~12-20 s of the reference's own single-core step loop
            cpu = {'value': rate, 'unit': UNIT, 'cores': 1, 'kind': 'reference',
                   'sample': f'UNMODIFIED reference (oracle/_ref), 17 buildings x 1 env x 600 steps in {dt:.1f}s on 1 core'}
        else:
            rate, dt = cpu_oracle_rate(512, 1200)       # ~10-20 s of single-core NumPy work
            cpu = {'value': rate, 'unit': UNIT, 'cores': 1, 'kind': 'port',
                   'sample': f'NumPy oracle, 17 buildings x 512 envs x 1200 steps in {dt:.1f}s on 1 core '
                             f'(reference itself: 871.7 building-steps/s/core, BASELINE.md)'}
    line = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': K, 'warmup': W, 'ms_per_step': ms_max / K,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f64' if args.precision == 'fp64' else 'f32', 'data': 'synthetic',
        'config': {'workload': f'{DATASET}: {B} buildings x {E} envs per GPU, observations {L}/env, actions {A}/env',
                   'precision': args.precision + (' (float64 intermediates, float32 storage: the reference\'s own flow, bit-exact)' if args.precision == 'fp64'
                                                  else ' (plain float arithmetic: within 1e-4 scaled-relative of the reference, not the 1e-5 target)'),
                   'mode': f'cl_rollout: ONE persistent kernel launch advances all K = {K} steps (state in registers, TMA row ring), actions pre-resident in HBM',
                   'timed_region': 'one launch of exactly K steps after the warm-up, one CUDA-event pair on the launch stream; max over ranks',
                   'l2': f'every step writes its own obs/reward slab: {K} x {bpu * units_per_step / 1e6:.1f} MB per launch vs 126 MB L2',
                   'envs_sharded_across_gpus': True, 'collectives_on_step_path': 0},
        'roofline': {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak, 'traffic': traffic, 'traffic_source': traffic_note,
                     'kernel': 'advance_kernel', 'bytes_per_unit': bpu, 'bytes_per_unit_single_step_launch': bpu_step,
                     'bytes_per_step': bpu * units_per_step, 'bytes_per_launch': bytes_per_launch, 'steps_per_launch': K,
                     'avg_launch_us': ms_launch * 1e3, 'peak_source': 'MEASURED_PEAKS.json hbm_gbs' if peaks else 'fallback 6650'},
        'cpu_baseline': cpu,
        'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': E * A * 4, 'd2h_bytes_per_step': L * 4 + E * B * 4,
                'ms_per_step': e2e_ms / K, 'api': 'CityLearnEnv.step_host(ndarray) -> cl_step_host, one native call per step: the step kernel reads the [E, A] actions from page-locked host memory and writes the rewards + the observation row all envs share back to it over PCIe (in place), stream sync'},
        'e2e_full_observations': {'value': world * units_per_step * K / (e2e_full_ms * 1e-3), 'unit': UNIT, 'ms_per_step': e2e_full_ms / K,
                                  'd2h_bytes_per_step': E * L * 4 + E * B * 4},
        'e2e_dma_copies': {'value': world * units_per_step * K / (e2e_dma_ms * 1e-3), 'unit': UNIT, 'ms_per_step': e2e_dma_ms / K,
                           'api': 'the same call with cudaMemcpyAsync H2D / D2H around the kernel instead of in-place PCIe access'},
        'e2e_rollout_host': {'value': world * units_per_step * K / float(blk_s.item()), 'unit': UNIT, 'ms_per_step': 1e3 * float(blk_s.item()) / K,
                             'api': 'CityLearnEnv.rollout_host(ndarray [K, E, A]): one H2D, one launch, one D2H (wall clock incl. host memcpy)'},
        'gpu_launches': int(launches),
        'clocks': clocks,
        'extra': extra,
        'checksum': checksum + e2e_sum * 0.0,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        hard_exit()


if __name__ == '__main__':
    main()
