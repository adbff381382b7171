"""Generate tests/golden/ref_*.npz by running the UNMODIFIED reference — TEST INFRASTRUCTURE ONLY.

Run in the build container (where /root/reference is mounted):
    python -m oracle.gen_golden
The fixtures pin the CPU oracle (oracle/quadswarm_oracle.py) to the reference: they hold seeds, actions,
planted states and the reference's own observations / rewards / dones / reward terms / state snapshots.
/root/reference does not exist on the GPU box, so the fixtures (not the reference) travel.
"""
import json
import os
import sys

import numpy as np

from . import ref_harness as rh

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests', 'golden')

INFO_KEYS = ['rew_main', 'rew_pos', 'rew_action', 'rew_crash', 'rew_orient', 'rew_spin',
             'rewraw_main', 'rewraw_pos', 'rewraw_action', 'rewraw_crash', 'rewraw_orient', 'rewraw_spin',
             'rew_quadcol', 'rew_proximity', 'rewraw_quadcol', 'rew_quadcol_obstacle', 'rewraw_quadcol_obstacle']


def rotz(a):
    c, s = np.cos(a), np.sin(a)
    return np.array([[c, -s, 0.], [s, c, 0.], [0., 0., 1.]])


def rotx(a):
    c, s = np.cos(a), np.sin(a)
    return np.array([[1., 0., 0.], [0., c, -s], [0., s, c]])


def _plants_cluster(n, rs, center=(0.5, -0.3, 2.0), spread=0.12, speed=0.6):
    """Drones packed inside ~2 collision radii, flying at each other: collisions, proximity, downwash."""
    plants = []
    c = np.array(center)
    for i in range(n):
        off = rs.uniform(-spread, spread, 3)
        off[2] = rs.uniform(-0.45, 0.45)          # stacked vertically -> downwash cylinders overlap
        pos = c + off
        vel = -speed * off / (np.linalg.norm(off) + 1e-9) + rs.uniform(-0.1, 0.1, 3)
        plants.append(dict(i=i, pos=pos, vel=vel, rot=rotz(rs.uniform(-3, 3)) @ rotx(rs.uniform(-0.3, 0.3)),
                           omega=rs.uniform(-1, 1, 3)))
    return plants


def _plants_room(rs):
    """One drone per room surface: +x wall, -y wall, corner, ceiling, floor upright, floor upside-down."""
    P = []
    P.append(dict(i=0, pos=[4.995, 1.0, 3.0], vel=[2.5, 0.2, 0.1], rot=rotz(0.3), omega=[0.1, 0.2, 0.3]))
    P.append(dict(i=1, pos=[-1.0, -4.99, 2.0], vel=[0.3, -3.0, 0.0], rot=rotz(-1.0), omega=[0., 0., 0.]))
    P.append(dict(i=2, pos=[-4.99, 4.99, 4.0], vel=[-2.0, 2.0, 0.5], rot=rotz(2.0), omega=[1., 0., 0.]))
    P.append(dict(i=3, pos=[0.5, 0.5, 9.99], vel=[0.1, 0.0, 4.0], rot=rotz(0.0), omega=[0., 0.5, 0.]))
    P.append(dict(i=4, pos=[2.0, -2.0, 0.06], vel=[0.5, 0.3, -1.5], rot=rotz(1.2) @ rotx(0.2), omega=[0.3, 0., 0.]))
    P.append(dict(i=5, pos=[-2.0, 2.0, 0.07], vel=[-0.2, 0.4, -2.0], rot=rotz(0.4) @ rotx(np.pi - 0.2),
                  omega=[0., 0.2, 0.1]))
    return P


CASES = [
    # name, env kwargs, T steps, seeds, planted states, obs stride in the fixture, state-snapshot stride (default: the
    # obs stride; 2 where every-step snapshots would take the fixture past 1 MB)
    dict(name='single_1', kw=dict(num_agents=1, neighbor_visible_num=0, neighbor_obs_type='none', ep_time=1.0,
                                  quads_mode='static_same_goal'), T=230, seed=11, obs_stride=1),
    dict(name='c2_same_goal_8', kw=dict(num_agents=8, neighbor_visible_num=6, ep_time=1.0,
                                        quads_mode='static_same_goal'), T=230, seed=21, obs_stride=1, state_stride=2),
    dict(name='all_neighbors_8', kw=dict(num_agents=8, neighbor_visible_num=-1, ep_time=0.6,
                                         quads_mode='static_diff_goal', obs_repr='xyz_vxyz_R_omega_wall'),
         T=130, seed=31, obs_stride=1),
    dict(name='cluster_8_downwash', kw=dict(num_agents=8, neighbor_visible_num=2, ep_time=1.0, use_downwash=True,
                                            quads_mode='static_same_goal', obs_repr='xyz_vxyz_R_omega_floor'),
         T=120, seed=41, obs_stride=1, plant='cluster', plant_at=[0, 40, 80]),
    dict(name='room_6', kw=dict(num_agents=6, neighbor_visible_num=2, ep_time=1.0, quads_mode='static_diff_goal'),
         T=110, seed=51, obs_stride=1, plant='room', plant_at=[0, 50]),
    dict(name='c3_obstacles_8', kw=dict(num_agents=8, neighbor_visible_num=2, ep_time=1.0, use_obstacles=True,
                                        use_downwash=True, quads_mode='o_random', obs_repr='xyz_vxyz_R_omega_floor',
                                        rew_coeff=dict(pos=1.0, effort=0.05, spin=0.1, vel=0.0, crash=1.0, orient=1.0,
                                                       yaw=0.0, quadcol_bin=5.0, quadcol_bin_smooth_max=4.0,
                                                       quadcol_bin_obst=5.0)),
         T=230, seed=61, obs_stride=1, state_stride=2, plant='obst', plant_at=[5, 120]),
    dict(name='c4_swarm_vs_swarm_16', kw=dict(num_agents=16, neighbor_visible_num=6, ep_time=4.5,
                                              quads_mode='swarm_vs_swarm'), T=500, seed=71, obs_stride=10),
    dict(name='dynamic_formations_8', kw=dict(num_agents=8, neighbor_visible_num=6, ep_time=0.8,
                                              quads_mode='dynamic_formations'), T=180, seed=81, obs_stride=4),
    # the remaining scenario classes: timed goal events (4-6 s periods need episodes > 6 s), per-tick goal motion,
    # obstacle scenarios with the largest-free-square goal
    dict(name='dynamic_same_goal_4', kw=dict(num_agents=4, neighbor_visible_num=2, ep_time=6.3,
                                             quads_mode='dynamic_same_goal'), T=700, seed=91, obs_stride=20),
    dict(name='dynamic_diff_goal_4', kw=dict(num_agents=4, neighbor_visible_num=2, ep_time=6.3,
                                             quads_mode='dynamic_diff_goal'), T=700, seed=92, obs_stride=20),
    dict(name='swap_goals_4', kw=dict(num_agents=4, neighbor_visible_num=2, ep_time=6.3,
                                      quads_mode='swap_goals'), T=700, seed=93, obs_stride=20),
    dict(name='lissajous_3', kw=dict(num_agents=3, neighbor_visible_num=2, ep_time=1.0,
                                     quads_mode='ep_lissajous3D'), T=160, seed=94, obs_stride=8),
    dict(name='run_away_5', kw=dict(num_agents=5, neighbor_visible_num=2, ep_time=2.6,
                                    quads_mode='run_away'), T=300, seed=95, obs_stride=10),
    dict(name='o_static_same_goal_4', kw=dict(num_agents=4, neighbor_visible_num=2, ep_time=1.0, use_obstacles=True,
                                              quads_mode='o_static_same_goal', obs_repr='xyz_vxyz_R_omega_floor'),
         T=230, seed=96, obs_stride=10),
    dict(name='o_dynamic_same_goal_4', kw=dict(num_agents=4, neighbor_visible_num=2, ep_time=6.3, use_obstacles=True,
                                               quads_mode='o_dynamic_same_goal', obs_repr='xyz_vxyz_R_omega_floor'),
         T=700, seed=97, obs_stride=20),
    dict(name='o_swap_goals_4', kw=dict(num_agents=4, neighbor_visible_num=2, ep_time=6.3, use_obstacles=True,
                                        quads_mode='o_swap_goals', obs_repr='xyz_vxyz_R_omega_floor'),
         T=700, seed=98, obs_stride=20),
    # goal following quadratic Bezier segments re-drawn every 5 s (third-party `bezier` restated in oracle/stubs/bezier)
    dict(name='ep_rand_bezier_3', kw=dict(num_agents=3, neighbor_visible_num=2, ep_time=10.4,
                                          quads_mode='ep_rand_bezier'), T=1100, seed=99, obs_stride=25),
    dict(name='o_ep_rand_bezier_4', kw=dict(num_agents=4, neighbor_visible_num=2, ep_time=6.4, use_obstacles=True,
                                            quads_mode='o_ep_rand_bezier', obs_repr='xyz_vxyz_R_omega_floor'),
         T=700, seed=104, obs_stride=20),
    # more drones than one warp: pins the oracle for the N > 32 work (48 drones converging on one goal and a planted
    # cluster: collision rows wider than 32 bits, K-nearest among 47 candidates, the flattened-id novelty quirk)
    dict(name='swarm_48_downwash', kw=dict(num_agents=48, neighbor_visible_num=6, ep_time=0.7, use_downwash=True,
                                           quads_mode='static_same_goal'), T=100, seed=111, obs_stride=5,
         plant='cluster', plant_at=[30]),
    # other physical models (SURVEY 8f-4): per-drone constants derived by the reference are stored in the fixture
    dict(name='defaultquad_4', kw=dict(num_agents=4, neighbor_visible_num=2, ep_time=1.0, quads_mode='static_diff_goal',
                                       dynamics_params='DefaultQuad'), T=130, seed=101, obs_stride=1, plant='room4', plant_at=[30]),
    dict(name='mediumquad_3', kw=dict(num_agents=3, neighbor_visible_num=2, ep_time=0.8, quads_mode='static_same_goal',
                                      dynamics_params='MediumQuad'), T=100, seed=102, obs_stride=1),
    dict(name='randomquad_relsampler_5', kw=dict(num_agents=5, neighbor_visible_num=2, ep_time=0.6, quads_mode='static_diff_goal',
                                                 dynamics_params='RandomQuad', use_downwash=True,
                                                 dyn_sampler_1={'class': 'RelativeSampler', 'noise_ratio': 0.05, 'sampler': 'normal'},
                                                 dynamics_randomize_every=1),
         T=140, seed=103, obs_stride=1, plant='room4', plant_at=[20, 90], construct_seed=777),
]


def _plants_obst(env, rs):
    """Drones flying into pillars (and one already inside a pillar's footprint)."""
    obst = np.array(env.obstacles.pos_arr)
    P = []
    for k in range(min(4, len(obst))):
        o = obst[k]
        ang = rs.uniform(-np.pi, np.pi)
        r = 0.3 + 0.046 + 0.01 if k else 0.2
        pos = np.array([o[0] + r * np.cos(ang), o[1] + r * np.sin(ang), rs.uniform(1.0, 3.0)])
        vel = np.array([-1.2 * np.cos(ang), -1.2 * np.sin(ang), 0.1])
        P.append(dict(i=k, pos=pos, vel=vel, rot=rotz(rs.uniform(-3, 3)), omega=rs.uniform(-0.5, 0.5, 3)))
    return P


def run_reference_case(case):
    kw = dict(case['kw'])
    if 'construct_seed' in case:
        np.random.seed(case['construct_seed'])     # RandomQuad / samplers draw from numpy's global stream at construction
    env = rh.make_reference_env(**kw)
    n = kw['num_agents']
    seed = case['seed']
    spawn_seeds = [seed + 100 + i for i in range(n)]
    rh.seed_reference(env, seed, seed + 1, spawn_seeds)
    act_rs = np.random.RandomState(seed + 7)
    plant_rs = np.random.RandomState(seed + 9)
    T = case['T']
    obs0 = np.array(env.reset(), dtype=np.float64)
    D = obs0.shape[1]
    out = dict(obs0=np.array(obs0, dtype=np.float64), goals0=np.array([e.goal for e in env.envs]))
    actions = np.zeros((T, n, 4))
    obs = []
    rewards = np.zeros((T, n))
    dones = np.zeros((T, n), dtype=bool)
    infos = np.full((T, n, len(INFO_KEYS)), np.nan)
    goals = np.zeros((T, n, 3))
    state_keys = ['pos', 'vel', 'rot', 'omega', 'thrust_rot_damp', 'thrust_cmds_damp', 'ou', 'on_floor']
    states = {k: [] for k in state_keys}
    plants_log = []
    ep_stats = []
    obst_log = []
    from quad_swarm_rl_b200.quad_models import DYN_FIELDS
    # constants in force after the first reset() (with dynamics_randomize_every the reset itself resamples them)
    dyn_log = [(0, np.array([[r[k] for k in DYN_FIELDS] for r in rh.dynamics_rows(env)]))]
    out['env_arm'] = np.array(float(env.quad_arm))
    if kw.get('use_obstacles'):
        obst_log.append((0, np.array(env.obstacles.pos_arr)[:, :2].copy()))
    for t in range(T):
        if case.get('plant') and t in case.get('plant_at', []):
            if case['plant'] == 'cluster':
                plants = _plants_cluster(n, plant_rs)
            elif case['plant'] == 'room':
                plants = _plants_room(plant_rs)
            elif case['plant'] == 'room4':
                plants = [p for p in _plants_room(plant_rs) if p['i'] in (0, 3, 4, 5)]
                for k, p in enumerate(plants):
                    p['i'] = k % n
            else:
                plants = _plants_obst(env, plant_rs)
            for p in plants:
                rh.plant_state(env, p['i'], p['pos'], p['vel'], p['rot'], p['omega'])
                plants_log.append((t, p['i'], np.array(p['pos'], float), np.array(p['vel'], float),
                                   np.array(p['rot'], float), np.array(p['omega'], float)))
        scale = 1.3 if t % 7 == 3 else 1.0            # some out-of-range actions to exercise the clip
        a = (scale * act_rs.uniform(-1, 1, size=(n, 4))).astype(np.float32).astype(np.float64)
        actions[t] = a
        o, r, d, inf = env.step([a[i] for i in range(n)])
        if t % case['obs_stride'] == 0 or d[0]:
            obs.append((t, np.array(o, dtype=np.float64)))
        rewards[t] = np.array(r, dtype=np.float64)
        dones[t] = d
        for i in range(n):
            for k, key in enumerate(INFO_KEYS):
                if key in inf[i]['rewards']:
                    infos[t, i, k] = float(inf[i]['rewards'][key])
        goals[t] = np.array([e.goal for e in env.envs])
        snap = rh.snapshot(env)
        for k in state_keys:
            states[k].append(snap[k])
        if d[0]:
            ep_stats.append((t, {k: float(v) for k, v in inf[0]['episode_extra_stats'].items()}))
            dyn_log.append((t + 1, np.array([[r[k] for k in DYN_FIELDS] for r in rh.dynamics_rows(env)])))
            if kw.get('use_obstacles'):
                obst_log.append((t + 1, np.array(env.obstacles.pos_arr)[:, :2].copy()))
    out.update(actions=actions, rewards=rewards, dones=dones, infos=infos, goals=goals,
               obs_t=np.array([t for t, _ in obs]), obs=np.array([o for _, o in obs]),
               plant_t=np.array([p[0] for p in plants_log], dtype=int), plant_i=np.array([p[1] for p in plants_log], dtype=int),
               plant_pos=np.array([p[2] for p in plants_log]).reshape(-1, 3),
               plant_vel=np.array([p[3] for p in plants_log]).reshape(-1, 3),
               plant_rot=np.array([p[4] for p in plants_log]).reshape(-1, 3, 3),
               plant_omega=np.array([p[5] for p in plants_log]).reshape(-1, 3),
               ep_stats_json=np.array(json.dumps(ep_stats)),
               dyn_t=np.array([t for t, _ in dyn_log], dtype=int), dyn_rows=np.array([r for _, r in dyn_log]),
               obst_t=np.array([t for t, _ in obst_log], dtype=int),
               obst_xy=np.array([o for _, o in obst_log]),
               case_json=np.array(json.dumps(dict(name=case['name'], kw=kw, T=T, seed=seed, obs_stride=case['obs_stride'],
                                                  state_stride=case.get('state_stride', case['obs_stride']), D=int(D)))))
    stride = max(1, case.get('state_stride', case['obs_stride']))
    for k in state_keys:
        arr = np.array(states[k])
        out['state_' + k] = arr[::stride]
    out['state_t'] = np.arange(T)[::stride]
    return out


def dump_constants():
    rh._ensure_path()
    env = rh.make_reference_env(num_agents=1, neighbor_visible_num=0, neighbor_obs_type='none')
    d = env.envs[0].dynamics
    sn = env.envs[0].sense_noise
    c = dict(mass=float(d.mass), inertia=[float(x) for x in d.inertia], thrust_max=float(d.thrust_max[0]),
             torque_max=float(d.torque_max[0]), motor_linearity=float(d.motor_linearity),
             prop_crossproducts=[[float(x) for x in r] for r in d.prop_crossproducts],
             prop_ccw=[float(x) for x in d.prop_ccw], arm=float(d.arm), motor_tau_up=float(d.motor_tau_up),
             motor_tau_down=float(d.motor_tau_down), omega_max=float(d.omega_max),
             damp_omega_quadratic=float(d.damp_omega_quadratic), vel_damp=float(d.vel_damp),
             since_last_svd_limit=float(d.since_last_svd_limit), mu=float(d.mu), dt=float(d.dt),
             ou_theta=float(d.thrust_noise.theta), ou_sigma=float(d.thrust_noise.sigma), ou_mu=float(d.thrust_noise.mu),
             pos_norm_std=float(sn.pos_norm_std), vel_norm_std=float(sn.vel_norm_std),
             gyro_noise_density=float(sn.gyro_noise_density), C_rot_drag=float(d.C_rot_drag),
             C_rot_roll=float(d.C_rot_roll), ep_len_15s=int(env.envs[0].ep_len), control_freq=float(env.control_freq),
             collision_threshold=float(env.collision_threshold),
             collision_falloff_threshold=float(env.collision_falloff_threshold))
    with open(os.path.join(GOLDEN_DIR, 'crazyflie_constants.json'), 'w') as f:
        json.dump(c, f, indent=1, sort_keys=True)


def main(argv=None):
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    only = set(sys.argv[1:] if argv is None else argv)
    dump_constants()
    for case in CASES:
        if only and case['name'] not in only:
            continue
        out = run_reference_case(case)
        path = os.path.join(GOLDEN_DIR, f"ref_{case['name']}.npz")
        np.savez_compressed(path, **out)
        print(f"{case['name']}: T={case['T']} D={out['obs0'].shape[1]} -> {path} ({os.path.getsize(path) / 1e3:.0f} kB)")


if __name__ == '__main__':
    main()
