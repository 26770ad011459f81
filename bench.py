#!/usr/bin/env python
"""bench.py — NCMC steps/s on the T4 lysozyme L99A – toluene workload (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--replicas R] [--workload NAME] [--impl reference]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path — one NCMC integrator step (H V R O R V H with work accumulation) of every
walker held by the GPU.  N > 1 is launched by torchrun, one rank per GPU; walkers are independent (weak scaling,
no data-path collective), only work/acceptance statistics are gathered over NCCL after the timed region.

Printed JSON (one line, rank 0):
  value        walker-steps/s with the state resident in HBM: K consecutive steps per window, CUDA events on the engine
               stream, barrier + synchronize on both sides of every window; `windows` windows per rank, the rank's
               figure is its median window, the job's figure the MAX over ranks of those medians (per-rank medians
               and the spread are printed under `timing`)
  e2e          the same metric through the public Context API with host buffers (H2D of positions + velocities, K
               steps with the on-device move, D2H of positions + protocol work, Metropolis test), wall clock
  roofline     dominant kernel from live per-kernel CUDA-event timing (direct-launch profiling pass) against the FP32
               FMA peak measured on this GPU by the library's own microbenchmark
  cpu_baseline the oracle's C twin (reference semantics, all host cores) on a bounded sample; `cpu_optimised` the same
               code with one force evaluation per step (the lambda-separable trick the engine uses), for context
  m3           BASELINE configs[2]: 64 walkers in total, 64 / N per GPU (same timed region)
`--dump-outputs DIR` also writes what the timed path computed in its last step as DIR/<name>.npy (see dump_outputs), so
that two builds can be compared output for output on identical inputs.
`--impl reference` times the CPU implementation alone (the reference stack — OpenMM/openmmtools/parmed — is not
installable here; rank 0 only, all host cores whatever OMP_NUM_THREADS the launcher exported).
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_PAIR = 60            # SURVEY.md §8(d)
FP32_PEAK_NOMINAL_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12
SEED = 20261017
DUMP_LIMIT_BYTES = 64 << 20


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def make_config(wl, replicas, world):
    """The `config` object of the JSON line — identical in the native and the reference arm."""
    return {'workload': wl['text'], 'replicas_per_gpu': replicas, 'global_walkers': world * replicas,
            'l2': 'not flushed between steps: the walker state (~2 MB per walker) is the step\'s own working set and '
                  'stays L2-resident in production exactly as here',
            'timed_region': 'windows of K consecutive device-resident NCMC steps (CUDA-graph replay), CUDA events on the '
                            'engine stream, median window per rank, max over ranks'}


def protocol_warmup(W, K, nsteps_nc):
    """Warm-up and window length actually used: a window must fit inside one protocol after the warm-up, so short
    protocols (M1) shorten the warm-up and, without --steps (K None), the window; a K given is never changed, and one
    that cannot fit is an error."""
    W = max(W, 3)
    if (K or 1000) + W >= nsteps_nc:
        W = min(W, max(3, nsteps_nc // 5))
    if K is None:
        K = min(1000, nsteps_nc - W - 2)
    if K < 1 or K + W + 2 > nsteps_nc:
        raise SystemExit('bench: --steps %d does not fit in one %d-step protocol after %d warm-up steps (1 to %d)'
                         % (K, nsteps_nc, W, nsteps_nc - W - 2))
    return W, K


def make_move(wl):
    """The move object of the workload and its on-device descriptor."""
    from blues_b200 import unit
    from blues_b200.moves import RandomLigandRotationMove, WaterTranslationMove
    if wl['move'] == 'water':
        mv = WaterTranslationMove(wl['structure'], protein_selection=wl['selection'], radius=wl['radius_nm'] * unit.nanometers)
        mv.atom_indices = list(wl['alch'])
        return mv
    return RandomLigandRotationMove(wl['base_structure'], 'LIG')     # tiled boxes: the first copy's toluene


class ClockSampler(object):
    """SM clock and throttle reasons of one GPU sampled through NVML inside this process while the timed windows run
    (no fork of nvidia-smi next to the measurement; falls back to nvidia-smi, at a slower rate, if NVML is missing)."""

    REASONS = [('hw_slowdown', 0x8), ('sw_power_cap', 0x4), ('hw_thermal_slowdown', 0x40), ('sw_thermal_slowdown', 0x20)]

    def __init__(self, index, period=0.05):
        self.index, self.period = index, period
        self.sm, self.mx, self.mask = [], [], 0
        self._stop = threading.Event()
        self._t = None
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get('CUDA_VISIBLE_DEVICES')
            phys = index
            if visible:
                ids = [v for v in visible.split(',') if v.strip() != '']
                if index < len(ids) and ids[index].strip().isdigit():
                    phys = int(ids[index])
            self._h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self._nvml = pynvml
        except Exception:
            self._nvml = None

    def _sample_nvml(self):
        n = self._nvml
        self.sm.append(float(n.nvmlDeviceGetClockInfo(self._h, n.NVML_CLOCK_SM)))
        self.mx.append(float(n.nvmlDeviceGetMaxClockInfo(self._h, n.NVML_CLOCK_SM)))
        fn = getattr(n, 'nvmlDeviceGetCurrentClocksEventReasons', None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
        self.mask |= int(fn(self._h))

    def _sample_smi(self):
        import subprocess
        q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
            'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
        out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + q, '--format=csv,noheader,nounits'],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        c = [v.strip() for v in out.split(',')]
        self.sm.append(float(c[0]))
        self.mx.append(float(c[1]))
        for bit, v in zip((0x8, 0x40, 0x20, 0x4), c[2:6]):
            if v.lower().startswith('active'):
                self.mask |= bit

    def _run(self):
        while not self._stop.is_set():
            try:
                if self._nvml is not None:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            self._stop.wait(self.period if self._nvml is not None else 0.5)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        return {'sm_mhz': statistics.median(self.sm) if self.sm else None, 'sm_max_mhz': max(self.mx) if self.mx else None,
                'reasons': sorted(n for n, bit in self.REASONS if self.mask & bit), 'samples': len(self.sm),
                'source': 'nvml (in-process)' if self._nvml is not None else 'nvidia-smi'}


def dump_outputs(out_dir, ctx, integ, n_atoms, n_rep):
    """What a caller of the timed path receives after its last step, as <out_dir>/<name>.npy in float64: positions (nm),
    velocities (nm/ps) and forces (kJ/mol/nm) of every walker as (walker, atom, xyz), and per walker the potential and
    kinetic energy (kJ/mol) and the protocol work (kT).  Where that would exceed 64 MB, the same fixed, seeded sample of
    atoms is kept in every run and its indices are written as atom_index.npy."""
    eng = ctx._engine
    atoms = slice(None)
    per_atom = 3 * 3 * 8 * n_rep + 8
    budget = DUMP_LIMIT_BYTES - 3 * 8 * n_rep - 4096           # less the per-walker scalars and the .npy headers
    if per_atom * n_atoms > budget:
        keep = budget // per_atom
        atoms = np.sort(np.random.default_rng(SEED).choice(n_atoms, keep, replace=False))
    ep, ek = eng.get_energy()
    out = {'positions': [eng.get_positions(r)[atoms] for r in range(n_rep)],
           'velocities': [eng.get_velocities(r)[atoms] for r in range(n_rep)],
           'forces': [eng.get_forces(r)[atoms] for r in range(n_rep)],
           'potential_energy': ep, 'kinetic_energy': ek,
           'protocol_work': [integ.get_protocol_work(dimensionless=True, replica=r) for r in range(n_rep)]}
    if not isinstance(atoms, slice):
        out['atom_index'] = atoms
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + '.npy'), np.asarray(a, dtype=np.float64))


def cpu_relax(topo, x, iters=60, max_disp=0.005):
    """Capped steepest descent with the constraints re-imposed (CPU oracle): the TOL-parm start coordinates carry
    the type-index quirk documented in DESIGN.md §8 and, like the reference's tests, need minimising before dynamics."""
    from oracle.c_oracle import COracle
    from oracle.ncmc_oracle import Constraints
    c = COracle(topo)
    cons = Constraints(topo)
    mobile = (np.asarray(topo['mass']) > 0)[:, None]
    x = cons.apply_positions(np.asarray(x, float), np.asarray(x, float), tol=1e-10)
    e, f = c.energy_forces(x)[:2]
    step = 1e-5
    for _ in range(iters):
        d = step * f * mobile
        n = np.linalg.norm(d, axis=1, keepdims=True)
        d *= np.minimum(1.0, max_disp / np.maximum(n, 1e-30))
        xn = cons.apply_positions(x + d, x, tol=1e-10)
        en, fn = c.energy_forces(xn)[:2]
        if np.isfinite(en) and en < e:
            x, e, f, step = xn, en, fn, step * 1.3
        else:
            step *= 0.4
    return x


def cpu_reference_run(wl, steps, warmup, budget_s, x=None, mode='reference'):
    """The path on the host cores: oracle C twin, all cores (set explicitly: launchers export OMP_NUM_THREADS=1).
    mode 'reference' = the reference's semantics (3 full evaluations per step); 'optimised' = one evaluation per step."""
    from oracle import c_oracle
    from blues_b200.workloads import lambda_tables, CASES
    cores = c_oracle.set_threads(host_cores())
    ls, le = lambda_tables(wl['nsteps_nc'])
    c = c_oracle.COracle(wl['topo'], ls, le, 'H V R O R V H', 300.0, 1.0, wl['dt'], wl['nsteps_nc'], 1, 0.2, 0.8, seed=SEED)
    if mode == 'optimised':
        c.set_fast(True)
    if x is None and wl['case'] == 'tol_parm':
        # relax one periodic image on the CPU, then tile the relaxed coordinates
        base = wl['base_structure']
        kw = dict(CASES['tol_parm']['kw'])
        xb = cpu_relax(base.createSystem(**kw).flatten(), base.coordinates * 0.1)
        reps = wl.get('tile') or (1, 1, 1)
        box = np.asarray(base.box[:3], float) * 0.1
        x = np.concatenate([xb + np.asarray((i, j, k)) * box for i in range(reps[0]) for j in range(reps[1])
                            for k in range(reps[2])])
    c.set_state(wl['x'] if x is None else x)
    c.velocities_to_temperature(300.0)
    t0 = time.time()
    warmed = 0
    while warmed < warmup and (time.time() - t0) < 0.4 * budget_s:
        c.step(1)
        warmed += 1
    t0 = time.time()
    done = 0
    while done < steps and (time.time() - t0) < budget_s:
        c.step(1)
        done += 1
    dt = time.time() - t0
    return done / dt, done, dt, cores, warmed


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    from blues_b200.workloads import load_workload
    wl = load_workload(args.workload)
    W, K = protocol_warmup(args.warmup, args.steps, wl['nsteps_nc'])
    R = args.replicas or wl['replicas']
    rate, done, dt, cores, warmed = cpu_reference_run(wl, K, W, 150.0)
    line = {'metric': 'NCMC steps/s (aggregate)', 'value': rate, 'unit': 'steps/s', 'n_gpus': args.gpus, 'steps': done,
            'warmup': W, 'ms_per_step': 1e3 * dt / done, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic', 'impl': 'reference',
            'config': make_config(wl, R, max(1, args.gpus)),
            'cpu_baseline': {'value': rate, 'unit': 'steps/s', 'cores': cores, 'kind': 'port',
                             'sample': '%d NCMC steps of one walker after %d warm-up steps (time-budgeted), CPU restatement '
                                       'of BLUES+OpenMM semantics: 3 full evaluations per step, float64, OpenMP on %d cores; '
                                       'not OpenMM itself' % (done, warmed, cores)},
            'e2e': {'value': rate, 'unit': 'steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'ns_per_day': rate * wl['dt'] * 86.4}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=None,
                    help='timed steps per window (default 1000, or as many as fit in a shorter protocol)')
    ap.add_argument('--warmup', type=int, default=200)
    ap.add_argument('--windows', type=int, default=20, help='timed windows of K steps per rank (median reported)')
    ap.add_argument('--replicas', type=int, default=0, help='independent walkers per GPU (0 = the workload\'s own)')
    ap.add_argument('--workload', default='t4l',
                    help='t4l = BASELINE configs[1] (default, the line the driver reads); t4l_frozen = the example\'s '
                         'freeze_radius variant; t4l_tol5e4; tolparm = M1; water = M4; m5 / m5_t4l = 250k atoms')
    ap.add_argument('--impl', default='native')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--batched', type=int, default=8, help='also report a batched run with this many walkers (0 = skip)')
    ap.add_argument('--m3-walkers', type=int, default=64, help='BASELINE configs[2]: total walkers of the m3 block (0 = skip)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the timed path computed in its last step as DIR/<name>.npy (rank 0\'s walkers)')
    args = ap.parse_args()
    if args.impl == 'reference':
        return run_reference(args)

    import torch
    import torch.distributed as dist
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))

    from blues_b200 import mm, unit, _native
    from blues_b200.integrators import AlchemicalExternalLangevinIntegrator
    from blues_b200.workloads import load_workload, DEFAULT_FUNCS

    wl = load_workload(args.workload)
    system, topo, x = wl['system'], wl['topo'], wl['x']
    NSTEPS_NC, DT_PS = wl['nsteps_nc'], wl['dt']
    W, K = protocol_warmup(args.warmup, args.steps, NSTEPS_NC)
    R = args.replicas or wl['replicas']

    def make_context(n_rep, seed):
        integ = AlchemicalExternalLangevinIntegrator(DEFAULT_FUNCS, splitting='H V R O R V H', temperature=300 * unit.kelvin,
                                                     timestep=DT_PS * unit.picoseconds, nsteps_neq=NSTEPS_NC,
                                                     nprop=1, prop_lambda=0.3)
        integ.setRandomNumberSeed(seed)
        ctx = mm.Context(system, integ, mm.Platform.getPlatformByName('CUDA'), {'DeviceIndex': local_rank},
                         n_replicas=n_rep)
        ctx.setPositions(x * unit.nanometers)
        ctx._engine.minimize(100, 10.0)                 # the surrogate force field needs a short relaxation
        ctx.setVelocitiesToTemperature(300 * unit.kelvin)
        return ctx, integ

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # A walker can blow up (the engine then raises OpenMM's "Particle coordinate is nan", BLUES rejects the move and goes
    # on): on the T4L surrogate force field that happens about once in 2e5 steps.  The bench does what BLUES does — the
    # protocol is abandoned and the next one starts from the relaxed state — and keeps the window out of the timings.
    nan_events = [0]

    def step_or_flag(integ, n):
        try:
            integ.step(n)
            return True
        except _native.EngineError as e:
            if 'nan' not in str(e).lower():
                raise
            nan_events[0] += 1
            if os.environ.get('BLUES_BENCH_VERBOSE'):
                sys.stderr.write('[bench] blown-up walker in a %d-step call (engine step now %s): %s\n'
                                 % (n, integ._context._engine.get_global('step'), str(e)[:80]))
            return False

    def timed_windows(ctx, integ, n_rep, warm, k, n_windows, budget_s=25.0):
        """`n_windows` windows of `k` steps, each bracketed by barrier + synchronize and timed with CUDA events on the
        engine stream.  A protocol is nstepsNC steps long: when the next window would not fit, a new protocol is started
        from the relaxed start state and warmed up again (outside the timed windows)."""
        eng = ctx._engine
        x0 = eng.get_positions(0)
        v0 = [eng.get_velocities(r) for r in range(n_rep)]
        stream = torch.cuda.ExternalStream(eng.lib.bl_stream(eng.h))

        def restart():
            # a new protocol starts at lambda = 0 from the relaxed coordinates (as every BLUES iteration starts from an
            # equilibrated MD state): restarting from the end of a cut-short protocol would switch a half-decoupled
            # ligand back on inside the solvent
            for attempt in range(4):
                integ.reset()
                ctx.setPositions(x0 * unit.nanometers)
                for r in range(n_rep):
                    ctx.setVelocities(v0[r] * (unit.nanometers / unit.picoseconds), replica=r)
                if step_or_flag(integ, warm):
                    break
            eng.synchronize()
            return warm

        done = restart()
        times, launches = [], 0
        t_begin = time.time()
        for w in range(n_windows):
            if done + k + 1 >= NSTEPS_NC:
                done = restart()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            l0 = eng.launch_count()
            e0.record(stream)
            ok = step_or_flag(integ, k)                  # k steps, no host round-trip inside
            e1.record(stream)
            barrier()
            if ok:
                times.append(e0.elapsed_time(e1))
                launches = eng.launch_count() - l0
                done += k
            else:
                done = restart()                         # a walker blew up: the window does not count
            # every rank must run the same number of windows (barriers): the budget decision is made collectively
            stop = torch.tensor([1.0 if (time.time() - t_begin > budget_s and w + 1 >= 5) else 0.0], device='cuda')
            if world > 1:
                dist.all_reduce(stop, op=dist.ReduceOp.MAX)
            if stop.item() > 0:
                break
        if not times:
            raise SystemExit('bench: every timed window ended in a blown-up walker')
        return times, launches, restart

    ctx, integ = make_context(R, SEED + 1000 * rank)
    eng = ctx._engine
    x_relaxed = eng.get_positions(0)                     # start of the CPU leg: same relaxed coordinates
    move = make_move(wl)
    dmove = move.device_move()

    # ---- device-resident throughput (value) --------------------------------------------------------------------
    with ClockSampler(local_rank) as clocks:
        t_load = time.time()
        step_or_flag(integ, W)
        while time.time() - t_load < 0.5:                # bring the clocks up before the first window
            ok = step_or_flag(integ, min(50, max(1, NSTEPS_NC // 8)))
            eng.synchronize()
            if not ok or eng.get_global('step') + 120 >= NSTEPS_NC:
                # positions AND velocities: resetting only the coordinates to the minimised structure would turn its
                # relaxation into kinetic energy once per cycle and hand the timed windows a walker at thousands of K
                integ.reset()
                ctx.setPositions(x_relaxed * unit.nanometers)
                ctx.setVelocitiesToTemperature(300 * unit.kelvin)
        integ.reset()
        ctx.setPositions(x_relaxed * unit.nanometers)
        ctx.setVelocitiesToTemperature(300 * unit.kelvin)
        times, launches, restart = timed_windows(ctx, integ, R, W, K, args.windows)
    if launches <= 0:
        raise SystemExit('bench: the timed region launched no kernels')
    med = statistics.median(times)
    t = torch.tensor([med, min(times), max(times)], device='cuda', dtype=torch.float64)
    per_rank = [t.clone() for _ in range(world)]
    if world > 1:
        dist.all_gather(per_rank, t)
    else:
        per_rank = [t]
    per_rank = [p.cpu().tolist() for p in per_rank]
    ms_max = max(p[0] for p in per_rank)
    slow_rank = int(np.argmax([p[0] for p in per_rank]))
    value = world * R * K / (ms_max * 1e-3)

    # ---- end to end through the public API with host buffers (e2e) ---------------------------------------------
    restart()
    pos_h = [torch.from_numpy(eng.get_positions(r)).pin_memory() for r in range(R)]
    vel_h = [torch.from_numpy(eng.get_velocities(r)).pin_memory() for r in range(R)]
    # the K timed steps are the middle slice of the nstepsNC protocol, so that the rotation move happens at
    # lambda = 0.5 (ligand fully decoupled) exactly as in a BLUES iteration (moveStep = nstepsNC / 2)
    first = max(0, NSTEPS_NC // 2 - K // 2)
    move_at = NSTEPS_NC // 2 - first
    e2e_times = []
    works, logp, acc = [], None, None
    for rep in range(5):
        integ.reset()
        integ.setGlobalVariableByName('step', first)
        integ.setGlobalVariableByName('lambda_step', 2 * first)
        integ.setGlobalVariableByName('lambda', 2.0 * first / (2 * NSTEPS_NC))
        barrier()
        t0 = time.perf_counter()
        for r in range(R):
            ctx.setPositions(pos_h[r].numpy() * unit.nanometers, replica=r)
            ctx.setVelocities(vel_h[r].numpy() * (unit.nanometers / unit.picoseconds), replica=r)
        if wl['move'] == 'water':
            move.beforeMove(ctx)                             # swap with a water inside the sphere (device, every walker)
        integ._scheduled_move = dict(dmove, step=move_at) if move_at < K else None
        e2e_ok = step_or_flag(integ, K)                      # a blown-up walker reads work = NaN and is rejected below
        integ._scheduled_move = None
        if wl['move'] == 'water':
            move.afterMove(ctx)                              # out of the sphere -> protocol_work = 999999 (device)
        out_pos = [ctx.getState(getPositions=True, replica=r).getPositions(asNumpy=True) for r in range(R)]
        works = [integ.get_protocol_work(dimensionless=True, replica=r) for r in range(R)]
        acc, logp, logu = eng.accept_reject()
        barrier()
        if e2e_ok or not e2e_times:
            e2e_times.append(time.perf_counter() - t0)
    del out_pos
    t = torch.tensor([statistics.median(e2e_times)], device='cuda', dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * R * K / float(t.item())
    nbytes = topo['n_atoms'] * 3 * 8
    h2d = 2 * nbytes * R / K
    d2h = (nbytes + 8 + 4 + 16) * R / K

    # ---- statistics gather (the only collective; outside the data path) ------------------------------------------
    from blues_b200 import parallel
    local_ids = [rank + world * r for r in range(R)]           # walker w lives on rank w % world
    gathered = parallel.gather_walker_stats(local_ids, works, logp, acc, device='cuda')
    stats = np.stack([gathered['work_kT'], gathered['accepted'].astype(float)], axis=1)

    # ---- BASELINE configs[2]: 64 walkers in total, 64 / N per GPU --------------------------------------------------
    m3 = None
    if args.m3_walkers and args.workload == 't4l' and args.m3_walkers % world == 0:
        r3 = args.m3_walkers // world
        if r3 == R:
            m3 = {'walkers_total': args.m3_walkers, 'replicas_per_gpu': r3, 'value': value, 'unit': 'steps/s',
                  'ms_per_step': ms_max / K, 'note': 'same as the main line'}
        else:
            ctx3, integ3 = make_context(r3, SEED + 7 + 1000 * rank)
            k3 = max(20, min(K, 100))
            t3, _, _ = timed_windows(ctx3, integ3, r3, 10, k3, 7, budget_s=15.0)
            tt = torch.tensor([statistics.median(t3)], device='cuda', dtype=torch.float64)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            m3 = {'walkers_total': args.m3_walkers, 'replicas_per_gpu': r3, 'steps': k3, 'windows': len(t3),
                  'value': args.m3_walkers * k3 / (float(tt.item()) * 1e-3), 'unit': 'steps/s',
                  'ms_per_step': float(tt.item()) / k3}
            del ctx3, integ3

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- per-kernel timing (roofline) on rank 0: direct launches bracketed by CUDA events ---------------------
    restart()
    eng.set_profiling(True)
    n_prof = min(K, 200)
    if not step_or_flag(integ, n_prof):                  # (a blow-up here: once more from the relaxed state)
        eng.set_profiling(False)
        restart()
        eng.set_profiling(True)
        integ.step(n_prof)
    eng.synchronize()
    ktimes = {}
    for name in _native.KERNEL_IDS:
        tot, n = eng.kernel_time(name)
        ktimes[name] = {'us_per_step': 1e3 * tot / n_prof, 'us_per_launch': 1e3 * tot / max(n, 1), 'launches': n}
    eng.set_profiling(False)
    pair_us = ktimes['pair']['us_per_launch']
    P_IN_PAIRS = wl['p_in']
    if P_IN_PAIRS is None:                               # pairs inside the cutoff, counted through the engine's list
        P_IN_PAIRS = int(len(eng.neighbor_pairs(0)))     # (bit-exact against the oracle's O(N^2) set in tests/)
    achieved_tflops = FLOP_PER_PAIR * P_IN_PAIRS * R / (pair_us * 1e-6) / 1e12
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    try:
        fp32_peak = _native.measure_fp32_peak(local_rank)
        fp32_src = 'measured on this GPU: bl_measure_fp32_peak (16 independent FFMA chains per thread, 8 CTAs x 256 ' \
                   'threads per SM, best of 10 launches); nominal 148 SM x 128 lanes x 2 x 1.965 GHz = %.1f' % FP32_PEAK_NOMINAL_TFLOPS
    except Exception as err:                              # pragma: no cover
        fp32_peak, fp32_src = FP32_PEAK_NOMINAL_TFLOPS, 'nominal (microbenchmark failed: %s)' % err
    hbm_peak = peaks.get('hbm_gbs', 6650.0)
    integ_bytes = 80 * topo['n_atoms'] * R           # SURVEY.md §8(d): 80 B/atom/launch
    integ_us = ktimes['integrate']['us_per_launch']
    # DRAM traffic per launch of the dominant kernels from the committed `ncu --set full` capture (1 walker)
    traffic = {}
    try:
        traffic = json.load(open(os.path.join(ROOT, 'profiles', 'ncu_traffic.json')))
    except Exception:
        pass
    roofline = {'kernel': 'k_pair4 (direct-space LJ + polynomial Ewald over the full Verlet list, packed FP32 FFMA2/FMUL2/'
                          'FADD2; the one energy evaluation per call uses k_pair2)', 'bound': 'fp32',
                'achieved': achieved_tflops, 'peak': fp32_peak, 'unit': 'TFLOP/s', 'frac': achieved_tflops / fp32_peak,
                'traffic': traffic.get('k_pair', {}).get('dram_bytes_per_launch'),
                'traffic_source': traffic.get('source'), 'peak_source': fp32_src,
                'algorithmic_flops_per_launch': FLOP_PER_PAIR * P_IN_PAIRS * R, 'us_per_launch': pair_us}
    roofline_hbm = {'kernel': 'k_integrate (V/R/O + SHAKE/RATTLE + work bookkeeping)', 'bound': 'hbm',
                    'achieved': integ_bytes / (integ_us * 1e-6) / 1e9, 'peak': hbm_peak, 'unit': 'GB/s',
                    'frac': integ_bytes / (integ_us * 1e-6) / 1e9 / hbm_peak,
                    'traffic': traffic.get('k_integrate', {}).get('dram_bytes_per_launch'),
                    'peak_source': 'MEASURED_PEAKS.json hbm_gbs' if 'hbm_gbs' in peaks else 'fallback 6650',
                    'algorithmic_bytes_per_launch': integ_bytes, 'us_per_launch': integ_us}

    # ---- batched walkers on one GPU (per-GPU share of configs[2] at 8 GPUs) ---------------------------------------
    batched = None
    if args.batched and args.batched != R and world == 1 and args.workload == 't4l':
        ctx_b, integ_b = make_context(args.batched, 777)
        kb = max(20, min(K, 200))
        tb, _, _ = timed_windows(ctx_b, integ_b, args.batched, 10, kb, 7, budget_s=10.0)
        bms = statistics.median(tb)
        batched = {'replicas_per_gpu': args.batched, 'steps': kb, 'windows': len(tb),
                   'value': args.batched * kb / (bms * 1e-3), 'unit': 'steps/s', 'ms_per_step': bms / kb}
        del ctx_b, integ_b

    # ---- CPU baseline (bounded sample) ---------------------------------------------------------------------------
    cpu = cpu_opt = None
    if not args.no_cpu_baseline and world == 1:
        rate, done, dt, cores, _ = cpu_reference_run(wl, min(40, NSTEPS_NC - 4), 2, 15.0, x=x_relaxed)
        cpu = {'value': rate, 'unit': 'steps/s', 'cores': cores, 'kind': 'port',
               'sample': '%d NCMC steps of one walker in %.1f s; CPU restatement of the reference step program (3 full '
                         'evaluations/step, float64, OpenMP) — not OpenMM itself, which is not installable here' % (done, dt)}
        try:
            rate, done, dt, cores, _ = cpu_reference_run(wl, min(60, NSTEPS_NC - 4), 2, 10.0, x=x_relaxed, mode='optimised')
            cpu_opt = {'value': rate, 'unit': 'steps/s', 'cores': cores, 'kind': 'port',
                       'sample': '%d NCMC steps in %.1f s; the same CPU code with ONE force evaluation per step (the '
                                 'lambda-separable evaluation the engine uses), float64 — the fair "optimised CPU" row of '
                                 'BASELINE.md §2; the reference itself pays three' % (done, dt)}
        except Exception as err:
            cpu_opt = {'unavailable': str(err)}

    # ---- outputs of the timed path ------------------------------------------------------------------------------------
    dump = None
    if args.dump_outputs:
        # The timed windows are not reproducible step for step: the clock warm-up and the window budget are wall-clock
        # bounded, and the thermostat's noise stream runs on across protocol restarts.  So the timed path is run once more
        # on a fresh context with the timed run's seed and start (minimised coordinates, velocities drawn at 300 K, the
        # same W warm-up steps, one window of K steps) and the state after its last step is written: an equivalent run
        # with identical inputs in every run, not a copy of the last timed window.  A blown-up walker leaves NaN in the
        # files and ok = false in the JSON line.
        ctx_d, integ_d = make_context(R, SEED + 1000 * rank)
        ok = step_or_flag(integ_d, W) and step_or_flag(integ_d, K)
        dump_outputs(args.dump_outputs, ctx_d, integ_d, topo['n_atoms'], R)
        dump = {'dir': args.dump_outputs, 'warmup': W, 'steps': K, 'replicas': R, 'ok': bool(ok),
                'what': 'state after the last of K steps of a fresh context with the timed run\'s seed and start, after W '
                        'warm-up steps'}
        del ctx_d, integ_d

    line = {'metric': 'NCMC steps/s (aggregate)', 'value': value, 'unit': 'steps/s', 'n_gpus': world, 'steps': K,
            'warmup': W, 'ms_per_step': ms_max / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32 pair math / f64 integration / i64 fixed-point accumulation', 'data': 'synthetic',
            'config': make_config(wl, R, world),
            'ns_per_day': value * DT_PS * 86.4,
            'timing': {'windows': len(times), 'window_steps': K,
                       'per_rank_ms_per_step': [{'median': p[0] / K, 'min': p[1] / K, 'max': p[2] / K} for p in per_rank],
                       'slowest_rank': slow_rank},
            'e2e': {'value': e2e_value, 'unit': 'steps/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                    'windows': len(e2e_times),
                    'what': 'Context.setPositions/setVelocities from pinned host arrays, K steps (the slice of the protocol '
                            'around lambda = 0.5) incl. the on-device move, getState positions + protocol work '
                            '+ Metropolis test, wall clock, median of the windows, max over ranks'},
            'gpu_launches': int(launches), 'clocks': clocks.summary(), 'roofline': roofline, 'roofline_hbm': roofline_hbm,
            'kernels_us_per_step': {k: round(v['us_per_step'], 2) for k, v in ktimes.items()},
            'cpu_baseline': cpu, 'cpu_optimised': cpu_opt, 'batched': batched, 'm3': m3,
            'blown_up_walkers': nan_events[0], 'dump': dump,
            'walker_stats': {'n': int(len(stats)), 'mean_work_kT': float(np.nanmean(stats[:, 0])),
                             'accepted': int(stats[:, 1].sum())}}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    # stdout carries exactly one JSON line: libraries that print to fd 1 (e.g. NCCL's version banner) go to stderr
    _real_stdout = os.dup(1)
    os.dup2(2, 1)
    _out = os.fdopen(_real_stdout, 'w')
    _print = print

    def print(*a, **k):          # noqa: A001  (only the final JSON line is printed through this)
        k.setdefault('file', _out)
        _print(*a, **k)
        _out.flush()

    main()
