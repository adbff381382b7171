"""Run the UNMODIFIED reference (Zhehui-Huang/quad-swarm-rl) as a black box — TEST INFRASTRUCTURE ONLY.

The reference is pure Python and needs three packages this image lacks at import time
(gymnasium, pyglet, bezier); `oracle/stubs/` supplies inert stand-ins.  The reference tree is looked up
in this order: $QS_REFERENCE_ROOT, oracle/_ref (a `pip install --target` of the reference made by
`__graft_entry__.build()` when /root/reference is present; git-ignored), /root/reference.
Nothing here is imported by the product package.
"""
import os
import shutil
import stat
import sys
import contextlib
import io

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_MIRROR = os.path.join(_HERE, '_ref')
MIRROR_PACKAGES = ('gym_art', 'swarm_rl')


def mirror_reference():
    """Mirror the reference's two python packages into oracle/_ref (git-ignored), so that a copy of this tree taken to
    a machine without the reference still runs it (bench.py's CPU arms).  The source is the reference tree
    `reference_root()` finds other than the mirror itself; without one, an existing mirror is kept.  The trees are
    copied as they are: `pip install --target` of the reference drops its namespace sub-packages, e.g.
    scenarios/obstacles."""
    src = reference_root(mirror=False)
    if src is None:
        return
    for pkg in MIRROR_PACKAGES:
        target = os.path.join(_MIRROR, pkg)
        if os.path.isdir(target):
            # copytree keeps the modes of a read-only checkout; without write permission on its directories the
            # previous mirror could not be removed by anyone but root
            for dirpath, _, _ in os.walk(target):
                os.chmod(dirpath, os.stat(dirpath).st_mode | stat.S_IWUSR)
            shutil.rmtree(target)
        shutil.copytree(os.path.join(src, pkg), target,
                        ignore=shutil.ignore_patterns('*.gif', '*.png', '*.pdf', '__pycache__', '*.pyc'))


def reference_root(mirror=True):
    """The first reference tree in the order of the module docstring; mirror=False passes over oracle/_ref."""
    for cand in (os.environ.get('QS_REFERENCE_ROOT'), os.path.join(_HERE, '_ref'), '/root/reference'):
        if cand and (mirror or os.path.abspath(cand) != _MIRROR) and os.path.isdir(os.path.join(cand, 'gym_art', 'quadrotor_multi')):
            return cand
    return None


def reference_available():
    return reference_root() is not None


def _ensure_path():
    root = reference_root()
    if root is None:
        raise RuntimeError("reference tree not found (looked in $QS_REFERENCE_ROOT, oracle/_ref, /root/reference)")
    stubs = os.path.join(_HERE, 'stubs')
    for p in (root, stubs):
        if p not in sys.path:
            sys.path.insert(0, p)
    return root


# keyword set of swarm_rl/env_wrappers/quad_utils.py:36-65 (the factory every run script goes through)
def make_reference_env(num_agents=8, ep_time=15.0, obs_repr='xyz_vxyz_R_omega', neighbor_visible_num=6,
                       neighbor_obs_type='pos_vel', use_obstacles=False, obst_density=0.2, obst_size=0.6,
                       obst_spawn_area=(8.0, 8.0), use_downwash=False, use_numba=True, quads_mode='static_same_goal',
                       room_dims=(10., 10., 10.), rew_coeff=None, collision_hitbox_radius=2.0,
                       collision_falloff_radius=4.0, sense_noise='default', quiet=True, dynamics_params='Crazyflie',
                       dyn_sampler_1=None, dynamics_change=None, dynamics_randomize_every=None):
    _ensure_path()
    from gym_art.quadrotor_multi.quadrotor_multi import QuadrotorEnvMulti
    if rew_coeff is None:
        rew_coeff = dict(pos=1.0, effort=0.05, spin=0.1, vel=0.0, crash=1.0, orient=1.0, yaw=0.0,
                         quadcol_bin=5.0, quadcol_bin_smooth_max=10.0, quadcol_bin_obst=5.0)
    ctx = contextlib.redirect_stdout(io.StringIO()) if quiet else contextlib.nullcontext()
    with ctx:
        env = QuadrotorEnvMulti(
            num_agents=num_agents, ep_time=ep_time, rew_coeff=rew_coeff, obs_repr=obs_repr,
            neighbor_visible_num=neighbor_visible_num, neighbor_obs_type=neighbor_obs_type,
            collision_hitbox_radius=collision_hitbox_radius, collision_falloff_radius=collision_falloff_radius,
            use_obstacles=use_obstacles, obst_density=obst_density, obst_size=obst_size,
            obst_spawn_area=list(obst_spawn_area), use_downwash=use_downwash, use_numba=use_numba,
            quads_mode=quads_mode, room_dims=list(room_dims), use_replay_buffer=False,
            quads_view_mode=['topdown'], quads_render=False, dynamics_params=dynamics_params, raw_control=True,
            raw_control_zero_middle=True, dynamics_randomize_every=dynamics_randomize_every,
            dynamics_change=(dynamics_change if dynamics_change is not None else
                             dict(noise=dict(thrust_noise_ratio=0.05), damp=dict(vel=0, omega_quadratic=0))),
            dyn_sampler_1=dyn_sampler_1, sense_noise=sense_noise, init_random_state=False)
    return env


_numba_seed = None


def seed_reference(env, seed_py, seed_nb, spawn_seeds):
    """Seed the three generators the hot path draws from (SURVEY.md Appendix F)."""
    global _numba_seed
    if _numba_seed is None:
        from numba import njit

        @njit
        def _seed(s):
            np.random.seed(s)
        _numba_seed = _seed
    np.random.seed(seed_py)
    _numba_seed(seed_nb)
    for e, s in zip(env.envs, spawn_seeds):
        e._seed(int(s))


def plant_state(env, i, pos, vel, rot, omega):
    """Overwrite drone i's rigid-body state between steps (QuadrotorDynamics.set_state, quadrotor_dynamics.py:178)."""
    d = env.envs[i].dynamics
    d.set_state(np.array(pos, dtype=np.float64), np.array(vel, dtype=np.float64),
                np.array(rot, dtype=np.float64), np.array(omega, dtype=np.float64))


def snapshot(env):
    dyn = [e.dynamics for e in env.envs]
    return dict(
        pos=np.array([d.pos for d in dyn]), vel=np.array([d.vel for d in dyn]),
        rot=np.array([d.rot for d in dyn]), omega=np.array([np.float64(d.omega) for d in dyn]),
        thrust_rot_damp=np.array([d.thrust_rot_damp for d in dyn]),
        thrust_cmds_damp=np.array([d.thrust_cmds_damp for d in dyn]),
        ou=np.array([d.thrust_noise.state for d in dyn]),
        on_floor=np.array([bool(d.on_floor) for d in dyn]),
        goal=np.array([e.goal for e in env.envs]),
        tick=np.array([e.tick for e in env.envs]),
    )


def dynamics_rows(env):
    """Per-drone derived constants of the reference env (QuadrotorDynamics.update_model, quadrotor_dynamics.py:104-166) as
    dicts in the layout of quad_swarm_rl_b200.quad_models.DYN_FIELDS."""
    rows = []
    for e in env.envs:
        d = e.dynamics
        c = dict(mass=float(d.mass), inv_mass=1.0 / float(d.mass), ixx=float(d.inertia[0]), iyy=float(d.inertia[1]),
                 izz=float(d.inertia[2]), inv_ixx=1.0 / float(d.inertia[0]), inv_iyy=1.0 / float(d.inertia[1]),
                 inv_izz=1.0 / float(d.inertia[2]), tau_up=float(d.motor_tau_up), tau_down=float(d.motor_tau_down),
                 linearity=float(d.motor_linearity), ou_sigma=float(d.thrust_noise.sigma), c_drag=float(d.C_rot_drag),
                 c_roll=float(d.C_rot_roll), vel_damp=float(d.vel_damp), omega_quadratic=float(d.damp_omega_quadratic),
                 arm=float(d.arm), reserved0=0., reserved1=0., reserved2=0.)
        pp = np.asarray(d.model.prop_pos)
        for m in range(4):
            c[f'thrust_max{m}'], c[f'torque_max{m}'] = float(d.thrust_max[m]), float(d.torque_max[m])
            c[f'px{m}'], c[f'py{m}'], c[f'pz{m}'] = float(pp[m, 0]), float(pp[m, 1]), float(pp[m, 2])
        rows.append(c)
    return rows
