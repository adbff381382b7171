#!/usr/bin/env python
"""bench.py — env agent-steps/s of the vectorised QuadSwarm env step on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--config c2|c3|c4] [--impl reference] [--dump-outputs DIR]

One "step" = one control step (2 physics sub-steps + collisions + observations, auto-reset included) of every env
of the workload.  Default workload = BASELINE.json configs[2] ("c3"): 8 drones x 4096 envs PER GPU (weak scaling),
12 pillars, K=2 neighbour obs, floor obs, downwash — the configuration the north-star target is quoted on.

JSON keys (one line, rank 0):
  value        whole-job agent-steps/s with actions/observations resident in HBM; one kernel launch per control step,
               replayed from a CUDA graph; inputs (action ring) and outputs (observation rollout ring) are larger than L2.
  e2e          the same metric through the reference-facing call with HOST numpy buffers (qs_step_host: H2D actions,
               kernel, D2H observations / rewards / dones inside the timed region).
  roofline     algorithmic bytes per launch (SURVEY.md §8d: 292 + 4 D + 8 M / N per agent-step) / mean launch time.
  cpu_baseline the UNMODIFIED reference (oracle/_ref, numba path) on one host core, bounded sample.
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

CONFIGS = {
    # SURVEY.md §8: BASELINE configs -> (E per GPU, env kwargs, scenario, reward coefficients)
    'c2': dict(E=1024, kw=dict(num_agents=8, neighbor_visible_num=6, obs_repr='xyz_vxyz_R_omega'),
               mode='static_same_goal', rew=dict(quadcol_bin=5.0, quadcol_bin_smooth_max=10.0),
               desc='8 drones x 1024 envs, obstacle-free, K=6, static_same_goal'),
    'c3': dict(E=4096, kw=dict(num_agents=8, neighbor_visible_num=2, obs_repr='xyz_vxyz_R_omega_floor',
                               use_obstacles=True, obst_density=0.2, obst_size=0.6, obst_spawn_area=(8.0, 8.0),
                               use_downwash=True),
               mode='o_random', rew=dict(quadcol_bin=5.0, quadcol_bin_smooth_max=4.0, quadcol_bin_obst=5.0),
               desc='8 drones x 4096 envs, 12 pillars (8x8 m, density 0.2, size 0.6), K=2, floor obs, downwash, o_random'),
    'c4': dict(E=2048, kw=dict(num_agents=32, neighbor_visible_num=6, obs_repr='xyz_vxyz_R_omega'),
               mode='swarm_vs_swarm', rew=dict(quadcol_bin=5.0, quadcol_bin_smooth_max=10.0),
               desc='32 drones x 2048 envs, all-pairs collisions, K=6, swarm_vs_swarm'),
    'c5': dict(E=4096, kw=dict(num_agents=8, neighbor_visible_num=6, obs_repr='xyz_vxyz_R_omega'),
               mode='static_same_goal', rew=dict(quadcol_bin=5.0, quadcol_bin_smooth_max=10.0),
               desc='8 drones x 4096 envs per GPU, obstacle-free, K=6'),
}


def measured_traffic(config):
    """dram__bytes_read.sum + dram__bytes_write.sum of the step kernel per launch, from the committed ncu --set full
    capture of this workload (profiles/r01_traffic.json), or None."""
    for name in ('r02_traffic.json', 'r01_traffic.json'):
        try:
            v = json.load(open(os.path.join(ROOT, 'profiles', name))).get(config, {}).get('dram_bytes_per_launch')
            if v is not None:
                return v
        except Exception:
            pass
    return None


def hbm_peak():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        try:
            return float(json.load(open(p))['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
        except Exception:
            pass
    return 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler:
    """nvidia-smi clock / throttle-reason samples during the timed region."""

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.samples = []
        self.proc = None

    def start(self):
        q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.gpu), f'--query-gpu={q}', '--format=csv,noheader,nounits',
                                          '-lms', '100'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        time.sleep(0.12)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for s in self.samples:
            f = [x.strip() for x in s.split(',')]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


def make_episode_tables(cfg, E, seed):
    """Synthetic episode tables of the workload's scenario, generated once on the host (scenarios.py)."""
    from quad_swarm_rl_b200.scenarios import create_scenario, obstacle_map_given_density
    kw = cfg['kw']
    N = kw['num_agents']
    use_obst = kw.get('use_obstacles', False)
    rs = np.random.RandomState(seed)
    goals = np.zeros((E, N, 3), np.float32)
    spawn = np.zeros((E, N, 3), np.float32)
    M = int(kw.get('obst_density', 0.2) * 64) if use_obst else 0
    obst = np.zeros((E, max(M, 1), 2), np.float32)
    sc = create_scenario(cfg['mode'], N, rng=rs, use_obstacles=use_obst)
    for e in range(E):
        if use_obst:
            obst_map, pos_arr, cells = obstacle_map_given_density(rs, kw['obst_spawn_area'], kw['obst_density'])
            sc.reset(obst_map=obst_map, cell_centers=cells)
            obst[e, :M] = np.asarray(pos_arr)[:, :2]
        else:
            sc.reset()
        goals[e] = sc.goals
        spawn[e] = sc.goals if sc.spawn_points is None else sc.spawn_points
    return goals, spawn, (obst[:, :M] if use_obst else None)


# ------------------------------------------------------------------------------------------
# reference CPU arm
# ------------------------------------------------------------------------------------------
def _ref_kwargs(cfg):
    kw = dict(cfg['kw'])
    rew = dict(pos=1.0, effort=0.05, spin=0.1, vel=0.0, crash=1.0, orient=1.0, yaw=0.0,
               quadcol_bin=0.0, quadcol_bin_smooth_max=0.0, quadcol_bin_obst=0.0)
    rew.update(cfg['rew'])
    return dict(num_agents=kw['num_agents'], neighbor_visible_num=kw['neighbor_visible_num'],
                obs_repr=kw['obs_repr'], use_obstacles=kw.get('use_obstacles', False),
                obst_density=kw.get('obst_density', 0.2), obst_size=kw.get('obst_size', 0.6),
                obst_spawn_area=kw.get('obst_spawn_area', (8.0, 8.0)), use_downwash=kw.get('use_downwash', False),
                quads_mode=cfg['mode'], rew_coeff=rew, use_numba=True)


def effective_cpus():
    """Host cores this process may actually use: cpu_count, capped by the affinity mask and the cgroup CPU quota."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        quota, period = open('/sys/fs/cgroup/cpu.max').read().split()[:2]                  # cgroup v2
        if quota != 'max':
            n = min(n, max(1, int(float(quota) / float(period))))
    except Exception:
        try:
            q = int(open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us').read())                    # cgroup v1
            per = int(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
            if q > 0:
                n = min(n, max(1, q // per))
        except Exception:
            pass
    return n


def _ref_worker(args, barrier=None):
    """One process = one reference env (how Sample Factory's rollout workers run it)."""
    cfg_name, n_warm, n_steps, seed = args
    from oracle import ref_harness as rh
    cfg = CONFIGS[cfg_name]
    kind = 'reference' if rh.reference_available() else 'port'
    N = cfg['kw']['num_agents']
    rs = np.random.RandomState(seed)
    if kind == 'reference':
        env = rh.make_reference_env(**_ref_kwargs(cfg))
        env.reset()
        step = lambda: env.step([a for a in rs.uniform(-1, 1, (N, 4)).astype(np.float32)])
    else:
        from tests.parity_util import cfg_to_oracle, make_tables
        from oracle import quadswarm_oracle as qo
        ocfg = cfg_to_oracle(cfg['kw'])
        t = make_tables(rs, 1, N, ocfg.num_obstacles, ocfg.use_obstacles, episodes=1)[0]
        src = qo.TableEpisodeSource([dict(goals=t['goals'][0], spawn=t['spawn'][0],
                                          obst_xy=None if t['obst'] is None else t['obst'][0])])
        env = qo.OracleEnv(ocfg, qo.PhiloxRng(seed), src)
        env.reset()
        step = lambda: env.step(rs.uniform(-1, 1, (N, 4)))
    for _ in range(n_warm):
        step()
    if barrier is not None:
        barrier.wait()                 # every process has imported, JIT-compiled and warmed up before any of them is timed
    t0 = time.perf_counter()
    for _ in range(n_steps):
        step()
    return time.perf_counter() - t0, kind


def _ref_proc(args, barrier, q):
    os.environ.setdefault('OMP_NUM_THREADS', '1')
    try:
        q.put(_ref_worker(args, barrier))
    except Exception as e:             # never leave the others waiting at the barrier
        try:
            barrier.abort()
        except Exception:
            pass
        q.put((float('nan'), f'error: {e!r}'))


def cpu_baseline_single(cfg_name, budget_s=12.0):
    """Reference on ONE host core, bounded sample (about budget_s seconds)."""
    dt, kind = _ref_worker((cfg_name, 30, 50, 0))
    per = dt / 50
    n = int(max(100, min(5000, budget_s / per)))
    dt, kind = _ref_worker((cfg_name, 0, n, 1))
    N = CONFIGS[cfg_name]['kw']['num_agents']
    return dict(value=N * n / dt, unit='agent-steps/s', cores=1, kind=kind,
                sample=f'1 env x {n} control steps of workload {cfg_name}, random actions, 1 process (numba path)')


def obs_dim_of(cfg):
    """D = S + 6 K (+ 9 with obstacles), quadrotor_single.py:311-316."""
    kw = cfg['kw']
    S = {'xyz_vxyz_R_omega': 18, 'xyz_vxyz_R_omega_floor': 19, 'xyz_vxyz_R_omega_wall': 24}[kw['obs_repr']]
    K = kw['num_agents'] - 1 if kw['neighbor_visible_num'] == -1 else kw['neighbor_visible_num']
    return S + 6 * K + (9 if kw.get('use_obstacles', False) else 0)


def bench_config(args, world):
    """The `config` object of the JSON line — identical for the CUDA arm and the reference arm (same workload, same keys)."""
    cfg = CONFIGS[args.config]
    E = args.envs or cfg['E']
    N = cfg['kw']['num_agents']
    return {'workload': f"{args.config}: {cfg['desc']}", 'envs_per_gpu': E, 'drones': N, 'obs_dim': obs_dim_of(cfg),
            'agents_per_gpu': E * N, 'ep_len': int(args.ep_time / 0.01), 'actions': 'i.i.d. U(-1,1)^4 per agent and step',
            'parallelism': f'dp{world} (envs sharded, no step-time collective)'}


def run_reference_arm(args):
    """--impl reference: the reference's own CPU implementation on all host cores (one env per process, the way Sample
    Factory's rollout workers run it).  The K bench steps are a BOUNDED SAMPLE of the workload: every process advances
    its env by n_proc = clamp(K, 100, 2500) control steps in total (so the run ends within minutes whatever K is);
    the rate, not the step count, is what is compared."""
    import multiprocessing as mp
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    N = cfg['kw']['num_agents']
    P = effective_cpus()
    n_proc = int(min(max(args.steps, 100), 2500))
    n_warm = int(min(max(args.warmup, 3), 50))
    for k in ('OMP_NUM_THREADS', 'OPENBLAS_NUM_THREADS', 'MKL_NUM_THREADS', 'NUMBA_NUM_THREADS'):
        os.environ.setdefault(k, '1')  # one env per process, one thread per process (inherited by the workers)
    ctx = mp.get_context('spawn')
    barrier, q = ctx.Barrier(P), ctx.Queue()
    procs = [ctx.Process(target=_ref_proc, args=((args.config, n_warm, n_proc, 100 + r), barrier, q)) for r in range(P)]
    for pr in procs:
        pr.start()
    res = [q.get() for _ in procs]
    for pr in procs:
        pr.join()
    bad = [r for r in res if not (r[0] == r[0])]
    if bad:
        raise RuntimeError(f'reference worker failed: {bad[0][1]}')
    wall = max(r[0] for r in res)
    kind = res[0][1]
    value = P * N * n_proc / wall
    line = {
        'impl': 'reference', 'metric': 'env agent-steps/sec', 'value': value, 'unit': 'agent-steps/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup,
        # one "step" of this arm = every one of the P reference envs advances one control step (P x N agent-steps)
        'ms_per_step': 1e3 * wall / n_proc, 'sample_steps': n_proc, 'sample_envs': P,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': bench_config(args, world),
        'sample_note': (f'bounded sample of the workload: {P} processes (= usable host cores of {os.cpu_count()} logical) x 1 reference env '
                        f'each x {n_proc} control steps (numba path), timed after all processes warmed up; ms_per_step = wall / {n_proc}; '
                        f'the rate (agent-steps/s) is what compares with the CUDA arm'),
        'cpu_baseline': {'value': value, 'unit': 'agent-steps/s', 'cores': P, 'kind': kind,
                         'sample': f'{P} processes x 1 env x {n_proc} control steps of workload {args.config}'},
        'e2e': {'value': value, 'unit': 'agent-steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------
# CUDA arm
# ------------------------------------------------------------------------------------------
L2_BYTES = 140e6          # rings are sized past this (B200 L2 = 126 MB)


class StepRunner:
    """E envs of one workload on one GPU, stepped from CUDA graphs of K consecutive launches (chained step grids).

    Rings: P = NG * K slots of actions / observations / rewards / dones, each ring larger than L2, so consecutive
    replays never find their inputs or outputs in cache; graph j covers ring slots [j K, (j+1) K)."""

    def __init__(self, torch, cfg, E, args, local_rank, rank, K, graph=True, stagger=True, wrapped=False):
        from quad_swarm_rl_b200.engine import QuadSwarmEngine
        self.torch = torch
        kw = cfg['kw']
        self.E, self.N = E, kw['num_agents']
        dev = self.dev = torch.device('cuda', local_rank)
        dev_scn = None if args.host_tables else cfg['mode']
        self.dev_scn = dev_scn
        from quad_swarm_rl_b200.sharding import shard_range
        world = int(os.environ.get('WORLD_SIZE', '1'))
        lo, hi = shard_range(world * E, world, rank)                 # contiguous block of global env ids of this rank
        assert hi - lo == E
        eng = self.eng = QuadSwarmEngine(num_envs=E, seed=args.seed, device=local_rank, env_id_offset=lo, rew_coeff=cfg['rew'],
                                         ep_time=args.ep_time, device_scenario=dev_scn, **kw)
        if dev_scn is None:
            goals, spawn, obst = make_episode_tables(cfg, E, seed=1000 + rank * 64)
            eng.set_next_episode(goals, spawn, obst)
        eng.reset()
        self.stagger = stagger
        if stagger:
            # every env starts at its own point of the episode (tick ~ U{0..ep_len}): each control step then carries
            # E / (ep_len + 1) auto-resets, as in training, where the replay wrapper de-synchronises the envs
            st = eng.get_state()
            g = torch.Generator(device=dev)
            g.manual_seed(1234 + rank)
            st['env_i32'][:, 0] = torch.randint(0, eng.ep_len + 1, (E,), device=dev, generator=g, dtype=torch.int32)
            eng.set_state(st)
        self.wrapped = wrapped
        if wrapped:
            # the reference's default training stack (replay p = 0.75 + reward shaping) as the kernel behind every step;
            # the can_drones_fly gate is bypassed: random actions never learn to fly, and the point is to time the full path
            eng.wrap_enable(use_replay=os.environ.get('QS_WRAP_REPLAY', '1') != '0', replay_buffer_size=20, replay_prob=0.75, replay_always_active=True)
        eng.set_chained(True)           # the step grids of a graph follow each other directly on the stream
        A, D = E * self.N, eng.D
        self.A, self.D, self.M = A, D, eng.M
        per_step = A * (16 + 4 * D + 4 + 1)
        # launches per graph: K itself when it fits, else the largest divisor of K that does (no eager launches inside a
        # timed block); ring memory bounded to ~8 GB
        kg_max = int(max(1, min(2048, 8e9 // per_step)))
        self.Kg = max(d for d in range(1, kg_max + 1) if K % d == 0) if K > kg_max else K
        if self.Kg < min(64, K):
            self.Kg = min(K, kg_max)
        need = int(np.ceil(L2_BYTES / (A * 16)))                            # slots until the ACTION ring alone exceeds L2
        self.NG = max(1, int(np.ceil(need / self.Kg)))
        while self.NG > 1 and self.NG * self.Kg * per_step > 8e9:           # bound the ring memory
            self.NG -= 1
        self.P = P = self.NG * self.Kg
        g = torch.Generator(device=dev)
        g.manual_seed(args.seed * 1000 + rank)
        self.act = (torch.rand((P, E, self.N, 4), device=dev, generator=g) * 2 - 1).contiguous()
        self.obs = torch.empty((P, E, self.N, D), device=dev)
        self.rew = torch.empty((P, E, self.N), device=dev)
        self.done = torch.empty((P, E, self.N), dtype=torch.uint8, device=dev)
        self.counter = 0
        self.stream = torch.cuda.Stream(device=dev)
        self.stream.wait_stream(torch.cuda.current_stream(dev))       # set_state / the action ring were enqueued on the default stream
        self.graphs = []
        with torch.cuda.stream(self.stream):
            for _ in range(3):
                self._one()
            self.stream.synchronize()
            if graph:
                self.counter = 0
                for j in range(self.NG):
                    gr = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(gr, stream=self.stream):
                        for _ in range(self.Kg):
                            self._one()
                    self.graphs.append(gr)
                self.counter = 0

    def _one(self):
        k = self.counter % self.P
        if self.wrapped:
            self.eng.wrap_step(self.act[k], obs_out=self.obs[k], rewards_out=self.rew[k], dones_out=self.done[k])
        else:
            self.eng.step(self.act[k], obs_out=self.obs[k], rewards_out=self.rew[k], dones_out=self.done[k])
        self.counter += 1

    def run(self, n):
        """n control steps on self.stream (call inside `with torch.cuda.stream(self.stream)`)."""
        done = 0
        if self.graphs:
            while n - done >= self.Kg and self.counter % self.Kg == 0:
                self.graphs[(self.counter // self.Kg) % self.NG].replay()
                done += self.Kg
                self.counter += self.Kg
        while done < n:
            self._one()
            done += 1

    def align(self):
        if self.graphs and self.counter % self.Kg:
            self.run(self.Kg - self.counter % self.Kg)

    def close(self):
        self.graphs = []
        self.eng.close()


def time_blocks(torch, dist, runner, K, R, world, side=None, metrics=None, gather_every=100, lead=0):
    """R back-to-back blocks of exactly K control steps, each bracketed by its own pair of CUDA events on the launching
    stream, behind `lead` untimed steps enqueued without a synchronise in between: they keep the device busy while the
    host enqueues the first block, so no launch latency falls inside it.  Returns the (start, end) event pairs and
    leaves the ring slot of the last timed step in runner.last_slot.  The optional cross-GPU metrics gather (NCCL
    all-reduce of a small vector every `gather_every` steps) runs on a side stream that only WAITS for the step stream —
    it is never an edge of the step chain — and is joined after the last block."""
    st = runner.stream
    pairs = []
    since = 0
    with torch.cuda.stream(st):
        runner.align()
        st.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        runner.run(lead)
        for b in range(R):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            runner.run(K)
            e1.record(st)
            runner.last_slot = (runner.counter - 1) % runner.P
            pairs.append((e0, e1))
            since += K
            if side is not None and since >= gather_every:
                since = 0
                side.wait_event(e1)
                with torch.cuda.stream(side):
                    metrics[0] = runner.rew[(runner.counter - 1) % runner.P].sum()
                    metrics[1] += 1
                    dist.all_reduce(metrics[:1], async_op=True)
            runner.align()                      # K > steps per graph: untimed steps up to the next graph boundary
        st.synchronize()
        if side is not None:
            side.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    return pairs


def block_times(torch, dist, pairs, world, dev):
    from quad_swarm_rl_b200.sharding import reduce_metrics
    ms = [a.elapsed_time(b) for a, b in pairs]
    if world > 1:
        ms = reduce_metrics(torch.tensor(ms, device=dev, dtype=torch.float64), op='max').tolist()      # max over ranks per block
    return ms


def measure_workload(torch, dist, name, args, local_rank, rank, world, K, target_s=None, clocks=None, side=None, metrics=None, wrapped=False):
    """Device-resident agent-steps/s of one workload.  target_s None: one timed window of exactly K chained step
    launches.  Otherwise R blocks of K, R chosen from two pilot blocks so that about target_s seconds are timed, median
    block."""
    cfg = CONFIGS[name]
    E = (args.envs if name == args.config and args.envs else cfg['E'])
    runner = StepRunner(torch, cfg, E, args, local_rank, rank, K, graph=not args.no_graph, stagger=not args.lockstep, wrapped=wrapped)
    dev = runner.dev
    with torch.cuda.stream(runner.stream):
        runner.run(max(3, args.warmup))
        runner.align()
        runner.stream.synchronize()
    if target_s is None:
        # the lead-in walks the whole ring once: every graph has been replayed (uploaded) before the window
        R, lead = 1, runner.P
    else:
        # pilot blocks: estimate the block time, warm the graphs
        evp = time_blocks(torch, dist, runner, K, 2, world)
        est_ms = max(1e-3, evp[1][0].elapsed_time(evp[1][1]))
        R, lead = int(min(5000, max(1, np.ceil(target_s * 1e3 / est_ms)))), 0
    if world > 1:
        t = torch.tensor([R], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        R = int(t.item())
    if side is not None:                       # NCCL's lazy channel / connection setup happens here, not in the window
        with torch.cuda.stream(side):
            metrics[0] = runner.rew[0].sum()
            dist.all_reduce(metrics[:1])
        side.synchronize()
    launches0 = runner.eng.launch_count
    if clocks is not None:
        clocks.start()
    K_eff = K
    pairs = time_blocks(torch, dist, runner, K, R, world, side=side, metrics=metrics, lead=lead)
    clk = clocks.stop() if clocks is not None else None
    ms = block_times(torch, dist, pairs, world, dev)
    if runner.eng.handover_timeouts:
        raise RuntimeError("a per-block hand-over between step grids timed out: results of this run are invalid")
    med = float(np.median(ms))
    D, M, N, A = runner.D, runner.M, runner.N, runner.A
    b_alg = 292 + 4 * D + (8.0 * M / N if M else 0.0)
    peak, peak_src = hbm_peak()
    launch_s = med * 1e-3 / K_eff
    res = dict(runner=runner, med_ms=med, blocks=R, block_ms_min=float(np.min(ms)), block_ms_max=float(np.max(ms)),
               us_per_step=launch_s * 1e6, value=world * A * K_eff / (med * 1e-3), b_alg=b_alg, D=D, M=M, N=N, A=A, E=E,
               frac=b_alg * A / launch_s / 1e9 / peak, achieved=b_alg * A / launch_s / 1e9, peak=peak, peak_src=peak_src,
               clk=clk, launches_host=runner.eng.launch_count - launches0, ring_slots=runner.P,
               ring_mb=dict(actions=runner.P * A * 16 / 1e6, observations=runner.P * A * D * 4 / 1e6), graphs=runner.NG,
               steps_per_graph=runner.Kg)
    return res


DUMP_BYTES = 64 << 20


def dump_outputs(torch, runner, out_dir):
    """What the last timed step returned to its caller (observations, rewards, dones of every env of this rank) as
    float32 DIR/<name>.npy.  Above DUMP_BYTES in all, the same fixed sample of envs (seeded, in env order) of each."""
    k = runner.last_slot
    out = dict(observations=runner.obs[k], rewards=runner.rew[k], dones=runner.done[k])
    per_env = 4 * sum(v[0].numel() for v in out.values())
    if per_env * runner.E > DUMP_BYTES:
        keep = np.sort(np.random.RandomState(0).choice(runner.E, DUMP_BYTES // per_env, replace=False))
        idx = torch.from_numpy(keep).to(runner.dev)
        out = {name: v.index_select(0, idx) for name, v in out.items()}
    os.makedirs(out_dir, exist_ok=True)
    for name, v in out.items():
        np.save(os.path.join(out_dir, f'{name}.npy'), v.float().cpu().numpy())


def run_cuda_arm(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    K = max(1, args.steps)
    cfg = CONFIGS[args.config]

    # optional cross-GPU metrics gather (north star: NCCL only for this): side stream, every 100 steps (SURVEY 8d)
    side = torch.cuda.Stream(device=dev) if world > 1 else None
    metrics = torch.zeros(64, device=dev) if world > 1 else None
    clocks = ClockSampler(local_rank) if rank == 0 else None
    main = measure_workload(torch, dist, args.config, args, local_rank, rank, world, K, clocks=clocks,
                            side=side, metrics=metrics, wrapped=args.wrapped_main)
    runner = main['runner']
    if args.dump_outputs and rank == 0:
        dump_outputs(torch, runner, args.dump_outputs)
    E, N, A, D, M = main['E'], main['N'], main['A'], main['D'], main['M']
    gathers = int(metrics[1].item()) if metrics is not None else 0
    runner.close()
    del runner
    torch.cuda.empty_cache()

    # ---- e2e: reference-facing call with HOST buffers (one engine holding all E envs of this GPU)
    from quad_swarm_rl_b200.engine import QuadSwarmEngine
    kw = cfg['kw']
    dev_scn = None if args.host_tables else cfg['mode']
    eng = QuadSwarmEngine(num_envs=E, seed=args.seed, device=local_rank, env_id_offset=rank * E, rew_coeff=cfg['rew'],
                          ep_time=args.ep_time, device_scenario=dev_scn, **kw)
    if dev_scn is None:
        goals, spawn, obst = make_episode_tables(cfg, E, seed=1000 + rank)
        eng.set_next_episode(goals, spawn, obst)
    eng.reset()
    n_e2e = max(10, min(max(args.steps, 100), args.e2e_steps))
    # page-locked host buffers (numpy views of pinned torch tensors): the DMA engine reads / writes them directly
    a_pin = torch.empty((8, E, N, 4), dtype=torch.float32).pin_memory()
    a_pin.copy_(torch.from_numpy(np.random.RandomState(5 + rank).uniform(-1, 1, (8, E, N, 4)).astype(np.float32)))
    a_host = a_pin.numpy()
    obs_h = torch.zeros((E, N, D), dtype=torch.float32).pin_memory().numpy()
    rew_h = torch.zeros((E, N), dtype=torch.float32).pin_memory().numpy()
    done_h = torch.zeros((E, N), dtype=torch.uint8).pin_memory().numpy()

    def host_loop(n):
        for k in range(3):
            eng.step_host(a_host[k % 8], obs_h, rew_h, done_h)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for k in range(n):
            eng.step_host(a_host[k % 8], obs_h, rew_h, done_h)
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    e2e_s = host_loop(n_e2e)
    # the same loop with explicit cudaMemcpyAsync H2D / D2H around the kernel (QS_ZERO_COPY=0) instead of the default, in
    # which the kernel reads / writes the mapped page-locked host buffers itself; reported beside it
    os.environ['QS_ZERO_COPY'] = '0'
    e2e_copy_s = host_loop(n_e2e)
    os.environ.pop('QS_ZERO_COPY', None)
    # the same envs as TWO halves stepped double-buffered (qs_step_host_async / qs_wait): the kernel of one half overlaps the
    # PCIe traffic of the other, the way Sample Factory's double-buffered sampling would drive it
    eng.close()
    Eh = E // 2
    halves = []
    for gi in range(2):
        e_ = QuadSwarmEngine(num_envs=Eh, seed=args.seed, device=local_rank, env_id_offset=rank * E + gi * Eh, rew_coeff=cfg['rew'],
                             ep_time=args.ep_time, device_scenario=dev_scn, **kw)
        if dev_scn is None:
            goals, spawn, obst = make_episode_tables(cfg, Eh, seed=1000 + rank * 2 + gi)
            e_.set_next_episode(goals, spawn, obst)
        e_.reset()
        halves.append(e_)

    def pipe_loop(n):
        sl = [slice(0, Eh), slice(Eh, 2 * Eh)]
        for k in range(3):
            for gi, e_ in enumerate(halves):
                e_.step_host_async(a_host[k % 8, sl[gi]], obs_h[sl[gi]], rew_h[sl[gi]], done_h[sl[gi]])
            for e_ in halves:
                e_.wait()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        halves[0].step_host_async(a_host[0, sl[0]], obs_h[sl[0]], rew_h[sl[0]], done_h[sl[0]])
        for k in range(n):
            halves[1].step_host_async(a_host[k % 8, sl[1]], obs_h[sl[1]], rew_h[sl[1]], done_h[sl[1]])
            halves[0].wait()                                    # A's observations are on the host: the policy would run here
            if k + 1 < n:
                halves[0].step_host_async(a_host[(k + 1) % 8, sl[0]], obs_h[sl[0]], rew_h[sl[0]], done_h[sl[0]])
            halves[1].wait()
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    pipe_s = pipe_loop(n_e2e)
    os.environ['QS_ZERO_COPY'] = '0'
    pipe_copy_s = pipe_loop(n_e2e)
    os.environ.pop('QS_ZERO_COPY', None)
    for e_ in halves:
        e_.close()
    # PCIe reference: one cudaMemcpyAsync of 64 MiB between page-locked host memory and the device, each direction
    big_d = torch.empty(64 << 20, dtype=torch.uint8, device=dev)
    big_h = torch.empty(64 << 20, dtype=torch.uint8).pin_memory()
    pcie = {}
    for name, (dst, src) in (('d2h', (big_h, big_d)), ('h2d', (big_d, big_h))):
        best = 0.0
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); dst.copy_(src, non_blocking=True); e1.record()
            torch.cuda.synchronize()
            best = max(best, (64 << 20) / (e0.elapsed_time(e1) * 1e-3) / 1e9)
        pcie[name] = best
    del big_d, big_h
    eng = None
    if world > 1:
        t = torch.tensor([e2e_s, e2e_copy_s, pipe_s, pipe_copy_s], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s, e2e_copy_s, pipe_s, pipe_copy_s = [float(x) for x in t.tolist()]

    # ---- extras: they explain the headline, they are not the headline
    extra = {}
    if not args.no_extras:
        if world == 1:
            def _events(fn, reps):
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); [fn() for _ in range(reps)]; e1.record()
                torch.cuda.synchronize()
                return e0.elapsed_time(e1) * 1e-3 / reps
            # (a) the same kernel, T steps per launch (qs_rollout: env block stays in registers, every observation written)
            T = 64
            g = torch.Generator(device=dev); g.manual_seed(3)
            acts = (torch.rand((T, E, N, 4), device=dev, generator=g) * 2 - 1).contiguous()
            o = torch.empty((T, E, N, D), device=dev); r = torch.empty((T, E, N), device=dev)
            d_ = torch.empty((T, E, N), dtype=torch.uint8, device=dev)
            eng_r = QuadSwarmEngine(num_envs=E, seed=args.seed, device=local_rank, env_id_offset=rank * E, rew_coeff=cfg['rew'],
                                    ep_time=args.ep_time, device_scenario=dev_scn, **kw)
            if dev_scn is None:
                goals, spawn, obst = make_episode_tables(cfg, E, seed=1000 + rank)
                eng_r.set_next_episode(goals, spawn, obst)
            eng_r.reset()
            eng_r.rollout(acts, obs_out=o, rewards_out=r, dones_out=d_)
            sec = _events(lambda: eng_r.rollout(acts, obs_out=o, rewards_out=r, dones_out=d_), 8)
            eng_r.close()
            extra['rollout'] = {'steps_per_launch': T, 'us_per_step': sec / T * 1e6, 'agent_steps_per_s': A * T / sec,
                                'roofline_frac': main['b_alg'] * A * T / sec / 1e9 / main['peak'],
                                'note': 'qs_rollout: T control steps per launch, all observations written'}
            del o, r, d_, acts
            # (a') the headline workload with the reference's default wrapper stack behind every step (csrc/qs_wrap.cuh)
            sub = argparse.Namespace(**vars(args))
            m = measure_workload(torch, dist, args.config, sub, local_rank, rank, world, min(K, 2000), 0.15, wrapped=True)
            agg = m['runner'].eng.wrap_read(reset=False)
            from quad_swarm_rl_b200 import _lib as L_
            extra['wrapped'] = {'us_per_step': m['us_per_step'], 'agent_steps_per_s': m['value'], 'vs_bare_step': m['us_per_step'] / main['us_per_step'],
                                'launches_per_step': 2, 'episodes_finished': float(agg[L_.WA['EPISODES_TOTAL']]),
                                'checkpoints': float(agg[L_.WA['CHECKPOINTS']]), 'events_stored': float(agg[L_.WA['EVENTS_STORED']]),
                                'events_replayed': float(agg[L_.WA['REPLAYED_EVENTS']]),
                                'note': 'qs_wrap_step: step kernel + the wrapper kernel, chained block by block (reward-shaping accumulators and episode statistics, '
                                        'checkpoint every 0.5 s, collision events, replay p = 0.75 with the can_drones_fly gate open); no host sync'}
            m['runner'].close()
            torch.cuda.empty_cache()
            # (b) the other BASELINE configs and a 4x batch of the headline workload, same protocol (blocks of K chained launches)
            per_cfg = {}
            sub = argparse.Namespace(**vars(args))
            sub.envs = 0
            for name in ('c2', 'c4', 'c5'):
                if name == args.config:
                    continue
                m = measure_workload(torch, dist, name, sub, local_rank, rank, world, min(K, 2000), 0.12)
                per_cfg[name] = {'workload': CONFIGS[name]['desc'], 'us_per_step': m['us_per_step'], 'agent_steps_per_s': m['value'],
                                 'roofline_frac': m['frac'], 'alg_bytes_per_agent_step': m['b_alg'], 'blocks': m['blocks']}
                m['runner'].close()
                torch.cuda.empty_cache()
            extra['configs'] = per_cfg
            sub.envs = 4 * E
            m = measure_workload(torch, dist, args.config, sub, local_rank, rank, world, min(K, 2000), 0.12)
            extra['large_batch'] = {'envs': 4 * E, 'agents': 4 * A, 'us_per_step': m['us_per_step'], 'agent_steps_per_s': m['value'],
                                    'roofline_frac': m['frac'],
                                    'note': 'same kernel, one launch per control step, 4x the envs of the headline workload'}
            m['runner'].close()
        else:
            # BASELINE config c5 (8 drones x 4096 envs per GPU, obstacle-free, K=6) over all ranks, same protocol
            sub = argparse.Namespace(**vars(args))
            sub.envs = 0
            m = measure_workload(torch, dist, 'c5', sub, local_rank, rank, world, min(K, 2000), 0.12, side=side, metrics=metrics)
            extra['c5'] = {'workload': CONFIGS['c5']['desc'], 'n_gpus': world, 'envs_total': world * CONFIGS['c5']['E'],
                           'us_per_step': m['us_per_step'], 'agent_steps_per_s': m['value'], 'roofline_frac_per_gpu': m['frac']}
            m['runner'].close()

    if rank == 0:
        cpu = cpu_baseline_single(args.config) if (world == 1 and not args.no_cpu_baseline) else None
        conf = bench_config(args, world)
        line = {
            'metric': 'env agent-steps/sec', 'value': main['value'], 'unit': 'agent-steps/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': main['med_ms'] / K, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': conf,
            'timing': {'protocol': (f'one window of exactly {K} control steps bracketed by CUDA events on the launching stream, enqueued '
                                    f'behind {main["ring_slots"]} untimed steps; value / ms_per_step are that window (max over ranks)'),
                       'window_ms': main['med_ms'],
                       'episodes': ('generated on the device at every auto-reset' if dev_scn else 'host-generated tables, uploaded once'),
                       'auto_resets': ('envs start at staggered ticks: every control step carries E / (ep_len + 1) auto-resets' if not args.lockstep
                                       else 'envs in lock-step: all envs reset in the same step every ep_len + 1 steps'),
                       'l2': (f'inputs and outputs larger than L2: rings of {main["ring_slots"]} slots, actions {main["ring_mb"]["actions"]:.0f} MB, '
                              f'observations {main["ring_mb"]["observations"]:.0f} MB ({main["graphs"]} CUDA graphs of {main["steps_per_graph"]} launches '
                              f'walk them in turn); env state ({A * 192 / 1e6:.1f} MB) is L2-resident by nature'),
                       'launch': 'one kernel per control step, chained step grids replayed from CUDA graphs' if not args.no_graph else 'one kernel per control step, eager launches',
                       'metrics_gather': (f'NCCL all-reduce of a 64-float vector every 100 steps on a side stream ({gathers} issued)' if world > 1 else 'n/a (1 GPU)')},
            'clocks': main['clk'],
            'e2e': {'value': world * A * n_e2e / e2e_s, 'unit': 'agent-steps/s', 'h2d_bytes_per_step': A * 16,
                    'd2h_bytes_per_step': A * (4 * D + 4 + 1), 'steps': n_e2e,
                    'explicit_copies_value': world * A * n_e2e / e2e_copy_s,
                    'pipelined_value': world * A * n_e2e / pipe_s, 'pipelined_explicit_copies_value': world * A * n_e2e / pipe_copy_s,
                    'pcie_measured_gbs': pcie,
                    'd2h_gbs_achieved': {'value': A * (4 * D + 4 + 1) * n_e2e / e2e_s / 1e9, 'pipelined': A * (4 * D + 4 + 1) * n_e2e / pipe_s / 1e9},
                    'frac_of_pcie_d2h': {'value': A * (4 * D + 4 + 1) * n_e2e / e2e_s / 1e9 / pcie['d2h'],
                                         'pipelined': A * (4 * D + 4 + 1) * n_e2e / pipe_s / 1e9 / pcie['d2h']},
                    'note': 'qs_step_host with page-locked numpy buffers, stream sync every step.  value: the kernel reads the '
                            'actions from and writes obs/rewards/dones to the mapped host buffers itself (zero-copy: the bytes '
                            'listed cross PCIe inside the timed region, no separate copy launches); explicit_copies_value: '
                            'cudaMemcpyAsync H2D actions, step kernel, cudaMemcpyAsync D2H obs/rewards/dones (QS_ZERO_COPY=0); '
                            'pipelined_value: the envs as two halves with their own handles, qs_step_host_async / qs_wait, the kernel '
                            'of one half overlapping the PCIe traffic of the other; pcie_measured_gbs: one 64 MiB cudaMemcpyAsync per '
                            'direction on this box'},
            'gpu_launches': int(K),
            'roofline': {'bound': 'hbm', 'achieved': main['achieved'], 'peak': main['peak'], 'unit': 'GB/s', 'frac': main['frac'],
                         'traffic': measured_traffic(args.config) if E == cfg['E'] else None, 'peak_source': main['peak_src'],
                         'alg_bytes_per_agent_step': main['b_alg'], 'alg_bytes_per_launch': main['b_alg'] * A,
                         'launch_us': main['us_per_step']},
            'cpu_baseline': cpu,
        }
        line.update(extra)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=100000)
    ap.add_argument('--warmup', type=int, default=1024)
    ap.add_argument('--impl', default='cuda', choices=['cuda', 'reference'])
    ap.add_argument('--config', default='c3', choices=sorted(CONFIGS))
    ap.add_argument('--envs', type=int, default=0, help='envs per GPU (default: the config\'s)')
    ap.add_argument('--ep-time', type=float, default=15.0)
    ap.add_argument('--seed', type=int, default=0)
    ap.add_argument('--e2e-steps', type=int, default=300)
    ap.add_argument('--wrapped-main', action='store_true', help='tuning: time the headline workload WITH the training wrappers (the line is then not the BASELINE metric)')
    ap.add_argument('--no-extras', action='store_true', help='skip the rollout / large-batch explanatory measurements')
    ap.add_argument('--lockstep', action='store_true', help='start all envs at tick 0 (all auto-resets fall into the same step)')
    ap.add_argument('--no-graph', action='store_true')
    ap.add_argument('--host-tables', action='store_true', help='use host-generated episode tables even where a device generator exists')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write the observations / rewards / dones of the last timed step (rank 0) '
                         'as float32 DIR/<name>.npy, at most 64 MB in all (a fixed sample of envs beyond that)')
    args = ap.parse_args()
    if args.impl == 'reference':
        run_reference_arm(args)
    else:
        run_cuda_arm(args)


if __name__ == '__main__':
    main()
