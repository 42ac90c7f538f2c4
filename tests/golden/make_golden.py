"""Regenerates tests/golden/*.npz by running the UNMODIFIED reference (tier-1 oracle).

Run in the build container only (needs /root/reference):
    python tests/golden/make_golden.py
The reference's Physics.DYN path is executed through the stand-in modules of
oracle/standins/ (see oracle/ref_loader.py); everything recorded here is float64
output of the reference's own code.  The fixtures travel to the GPU box, the
reference does not.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle.ref_loader import load_reference, quiet  # noqa: E402

R = load_reference()
import pybullet as pb  # the stand-in  # noqa: E402


def snap(env):
    return dict(pos=env.pos.copy(), quat=env.quat.copy(), rpy=env.rpy.copy(), vel=env.vel.copy(),
                ang_v=env.ang_v.copy(), rpy_rates=env.rpy_rates.copy())


def run_env(env, actions, record_obs_every=1):
    """Steps `env` through `actions` [T, D, A]; returns stacked per-step records."""
    rec = {k: [] for k in ("pos", "quat", "rpy", "vel", "ang_v", "rpy_rates", "reward", "terminated", "truncated")}
    has_pid = hasattr(env, "ctrl")
    if has_pid:     # embedded DSLPIDControl state after each step (for teacher-forced parity checks)
        rec.update({k: [] for k in ("pid_integral_pos_e", "pid_integral_rpy_e", "pid_last_rpy")})
    obs_rec = []
    obs0, _ = env.reset()
    for t in range(actions.shape[0]):
        obs, rew, term, trunc, _ = env.step(actions[t])
        s = snap(env)
        for k, v in s.items():
            rec[k].append(v)
        rec["reward"].append(float(rew)); rec["terminated"].append(bool(term)); rec["truncated"].append(bool(trunc))
        if has_pid:
            rec["pid_integral_pos_e"].append(np.array([c.integral_pos_e for c in env.ctrl]))
            rec["pid_integral_rpy_e"].append(np.array([c.integral_rpy_e for c in env.ctrl]))
            rec["pid_last_rpy"].append(np.array([c.last_rpy for c in env.ctrl]))
        if t % record_obs_every == 0:
            obs_rec.append(np.asarray(obs, dtype=np.float64))
    out = {k: np.asarray(v) for k, v in rec.items()}
    out["obs"] = np.asarray(obs_rec)
    out["obs0"] = np.asarray(obs0, dtype=np.float64)
    out["actions"] = actions
    return out


def save(name, **arrs):
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **arrs)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


def flat(prefix, d):
    return {prefix + "_" + k: v for k, v in d.items()}


def main():
    A = R.ActionType
    DYN = R.Physics.DYN
    # ---- constants of the three drone models (BaseAviary.py:116-128) -------------------
    consts = {}
    for dm in (R.DroneModel.CF2X, R.DroneModel.CF2P, R.DroneModel.RACE):
        with quiet():
            e = R.CtrlAviary(drone_model=dm, physics=DYN)
        names = ["M", "L", "KF", "KM", "THRUST2WEIGHT_RATIO", "GRAVITY", "HOVER_RPM", "MAX_RPM", "MAX_THRUST",
                 "MAX_XY_TORQUE", "MAX_Z_TORQUE", "GND_EFF_COEFF", "PROP_RADIUS", "GND_EFF_H_CLIP", "DW_COEFF_1",
                 "DW_COEFF_2", "DW_COEFF_3", "MAX_SPEED_KMH", "COLLISION_H", "COLLISION_Z_OFFSET"]
        consts[dm.value + "_names"] = np.array(names)
        consts[dm.value + "_values"] = np.array([float(getattr(e, n)) for n in names])
        consts[dm.value + "_J"] = np.diag(e.J).copy()
        consts[dm.value + "_DRAG_COEFF"] = np.asarray(e.DRAG_COEFF)
    for dm in (R.DroneModel.CF2X, R.DroneModel.CF2P, R.DroneModel.RACE):
        with quiet():
            consts[dm.value + "_INIT_XYZS3"] = np.asarray(R.CtrlAviary(drone_model=dm, num_drones=3, physics=DYN).INIT_XYZS)
    save("constants", **consts)

    # ---- config 1: HoverAviary, 1 drone, DYN, RPM, 1000 steps, S=1 and S=8 -----------------
    T = 1000
    tt = np.arange(T)[:, None, None] / 240.0
    streams = {
        "zeros": np.zeros((T, 1, 4), np.float32),
        # constant differential thrust spins the body up without bound (the explicit-Euler
        # gyroscopic term diverges after ~4 s): keep 400 substeps of it
        "const": np.tile(np.array([[1, -1, 0.5, -0.5]], np.float32), (400, 1, 1)),
        "rand": np.random.default_rng(0).uniform(-1, 1, (T, 1, 4)).astype(np.float32),
        "sine": (0.25 * np.sin(2 * np.pi * tt * np.array([0.9, 1.3, 1.7, 2.3]) + np.array([0, 1, 2, 3]))).astype(np.float32),
    }
    out = {}
    for cf in (240, 30):
        for nm, acts in streams.items():
            if nm == "const" and cf == 30:
                acts = acts[:50]
            with quiet():
                env = R.HoverAviary(physics=DYN, pyb_freq=240, ctrl_freq=cf, act=A.RPM)
                rec = run_env(env, acts, record_obs_every=50)
            out.update(flat("cf%d_%s" % (cf, nm), rec))
    save("hover_rpm_1000", **out)

    # ---- learn.py config: HoverAviary ONE_D_RPM 240/30, action 0, one episode --------------
    with quiet():
        env = R.HoverAviary(physics=DYN, act=A.ONE_D_RPM)
        rec = run_env(env, np.zeros((250, 1, 1), np.float32))
    save("hover_one_d_rpm_episode", **rec)

    # ---- MultiHover, 2 and 3 drones, RPM / ONE_D_RPM, random actions ------------------------
    out = {}
    for nd, act in ((2, A.ONE_D_RPM), (2, A.RPM), (3, A.RPM)):
        aw = 1 if act == A.ONE_D_RPM else 4
        acts = np.random.default_rng(10 + nd + aw).uniform(-1, 1, (300, nd, aw)).astype(np.float32)
        with quiet():
            env = R.MultiHoverAviary(num_drones=nd, physics=DYN, act=act)
            tp = np.asarray(env.TARGET_POS)
            rec = run_env(env, acts, record_obs_every=10)
        rec["TARGET_POS"] = tp
        out.update(flat("d%d_%s" % (nd, act.value), rec))
    save("multihover_rand_300", **out)

    # ---- RL envs with the embedded PID: PID / VEL / ONE_D_PID -------------------------------
    # At the RL default 240/30 Hz the reference's cascaded PID chatters chaotically (a 1e-12 perturbation
    # grows to 1e-2 in ~3 s, measured), so the 30 Hz vectors are for TEACHER-FORCED one-step checks; the
    # 240/120 Hz vectors are contractive and are compared as whole trajectories.
    for cf, T in ((30, 240), (120, 480)):
        out = {}
        for cls, nd, act in ((R.HoverAviary, 1, A.PID), (R.HoverAviary, 1, A.VEL), (R.HoverAviary, 1, A.ONE_D_PID),
                             (R.MultiHoverAviary, 2, A.PID)):
            aw = {A.PID: 3, A.VEL: 4, A.ONE_D_PID: 1}[act]
            rng = np.random.default_rng(20 + aw + nd)
            seg = rng.uniform(-1, 1, (4, nd, aw)).astype(np.float32)     # piecewise-constant commands
            if act == A.PID:      # set-points inside the truncation box (SURVEY 8d config 2)
                seg = (np.array([0, 0, 1.0], np.float32) + 0.5 * seg).astype(np.float32)
            acts = np.repeat(seg, T // 4, axis=0)
            with quiet():
                kw = dict(physics=DYN, act=act, pyb_freq=240, ctrl_freq=cf)
                env = cls(**kw) if cls is R.HoverAviary else cls(num_drones=nd, **kw)
                rec = run_env(env, acts, record_obs_every=10)
            out.update(flat("%s_d%d_%s" % ("hover" if cls is R.HoverAviary else "multi", nd, act.value), rec))
        save("rl_pid_cf%d" % cf, **out)

    # ---- pid.py workload: CtrlAviary(DYN, 240/48) x 3 drones + DSLPIDControl, 576 ticks -----
    for dm in (R.DroneModel.CF2X, R.DroneModel.CF2P):
        nd, cf = 3, 48
        H, H_STEP, RAD = .1, .05, .3
        INIT_XYZS = np.array([[RAD * np.cos((i / 6) * 2 * np.pi + np.pi / 2), RAD * np.sin((i / 6) * 2 * np.pi + np.pi / 2) - RAD, H + i * H_STEP] for i in range(nd)])
        INIT_RPYS = np.array([[0, 0, i * (np.pi / 2) / nd] for i in range(nd)])
        NUM_WP = cf * 10
        TARGET_POS = np.zeros((NUM_WP, 3))
        for i in range(NUM_WP):
            TARGET_POS[i, :] = RAD * np.cos((i / NUM_WP) * (2 * np.pi) + np.pi / 2) + INIT_XYZS[0, 0], RAD * np.sin((i / NUM_WP) * (2 * np.pi) + np.pi / 2) - RAD + INIT_XYZS[0, 1], 0
        wp = np.array([int((i * NUM_WP / 6) % NUM_WP) for i in range(nd)])
        with quiet():
            env = R.CtrlAviary(drone_model=dm, num_drones=nd, initial_xyzs=INIT_XYZS, initial_rpys=INIT_RPYS,
                               physics=DYN, pyb_freq=240, ctrl_freq=cf)
            ctrl = [R.DSLPIDControl(drone_model=dm) for _ in range(nd)]
        action = np.zeros((nd, 4))
        rec = {k: [] for k in ("obs", "action", "target", "pos_e", "yaw_e", "rpy_rates", "pid_integral_pos_e", "pid_integral_rpy_e", "pid_last_rpy")}
        for i in range(12 * cf):
            obs, _, _, _, _ = env.step(action)
            tg = np.zeros((nd, 3)); pe = np.zeros((nd, 3)); ye = np.zeros(nd)
            for j in range(nd):
                tg[j] = np.hstack([TARGET_POS[wp[j], 0:2], INIT_XYZS[j, 2]])
                action[j, :], pe[j], ye[j] = ctrl[j].computeControlFromState(control_timestep=env.CTRL_TIMESTEP, state=obs[j],
                                                                           target_pos=tg[j], target_rpy=INIT_RPYS[j, :])
            for j in range(nd):
                wp[j] = wp[j] + 1 if wp[j] < (NUM_WP - 1) else 0
            rec["obs"].append(obs.copy()); rec["action"].append(action.copy()); rec["target"].append(tg)
            rec["pos_e"].append(pe); rec["yaw_e"].append(ye); rec["rpy_rates"].append(env.rpy_rates.copy())
            rec["pid_integral_pos_e"].append(np.array([c.integral_pos_e for c in ctrl]))
            rec["pid_integral_rpy_e"].append(np.array([c.integral_rpy_e for c in ctrl]))
            rec["pid_last_rpy"].append(np.array([c.last_rpy for c in ctrl]))
        rec = {k: np.asarray(v) for k, v in rec.items()}
        rec["INIT_XYZS"], rec["INIT_RPYS"] = INIT_XYZS, INIT_RPYS
        rec["final_integral_pos_e"] = np.array([c.integral_pos_e for c in ctrl])
        rec["final_integral_rpy_e"] = np.array([c.integral_rpy_e for c in ctrl])
        rec["final_last_rpy"] = np.array([c.last_rpy for c in ctrl])
        save("pid_circle_%s" % dm.value, **rec)

    # ---- DSLPIDControl known answers on random states (stateful: 3 consecutive calls) ------
    rng = np.random.default_rng(7)
    n = 256
    out = {}
    for dm in (R.DroneModel.CF2X, R.DroneModel.CF2P):
        pos = rng.uniform(-1, 1, (n, 3)); vel = rng.uniform(-1, 1, (n, 3))
        q = rng.normal(size=(n, 4)); q[:, 3] = np.abs(q[:, 3]) + 1.0; q /= np.linalg.norm(q, axis=1, keepdims=True)
        tpos = rng.uniform(-1, 1, (n, 3)); trpy = np.zeros((n, 3)); trpy[:, 2] = rng.uniform(-1, 1, n)
        tvel = rng.uniform(-.3, .3, (n, 3)); trr = rng.uniform(-.1, .1, (n, 3))
        res = {k: [] for k in ("rpm", "pos_e", "yaw_e", "integral_pos_e", "integral_rpy_e", "last_rpy")}
        with quiet():
            ctrls = [R.DSLPIDControl(drone_model=dm) for _ in range(n)]
        for call in range(3):
            rpm = np.zeros((n, 4)); pe = np.zeros((n, 3)); ye = np.zeros(n)
            for i in range(n):
                rpm[i], pe[i], ye[i] = ctrls[i].computeControl(1 / 48, pos[i] + 0.01 * call, q[i], vel[i], np.zeros(3), tpos[i], trpy[i], tvel[i], trr[i])
            res["rpm"].append(rpm); res["pos_e"].append(pe); res["yaw_e"].append(ye)
            res["integral_pos_e"].append(np.array([c.integral_pos_e for c in ctrls]))
            res["integral_rpy_e"].append(np.array([c.integral_rpy_e for c in ctrls]))
            res["last_rpy"].append(np.array([c.last_rpy for c in ctrls]))
        d = dict(pos=pos, quat=q, vel=vel, target_pos=tpos, target_rpy=trpy, target_vel=tvel, target_rpy_rates=trr)
        d.update({k: np.asarray(v) for k, v in res.items()})
        out.update(flat(dm.value, d))
    save("pid_kat", **out)

    # ---- other drone models through CtrlAviary(DYN): random RPM around hover -----------------
    out = {}
    for dm in (R.DroneModel.CF2P, R.DroneModel.RACE):
        with quiet():
            env = R.CtrlAviary(drone_model=dm, num_drones=2, physics=DYN, pyb_freq=240, ctrl_freq=120)
        rng = np.random.default_rng(33)
        acts = env.HOVER_RPM * (1 + 0.1 * rng.uniform(-1, 1, (300, 2, 4)))
        acts[::50] = env.MAX_RPM * 1.2          # exercises CtrlAviary's clip to MAX_RPM
        acts[25::50] = -5.0                     # ... and to 0
        rec = run_env(env, acts, record_obs_every=1)
        out.update(flat(dm.value, rec))
    save("ctrl_models_300", **out)

    # ---- VelocityAviary (examples/pid_velocity.py shape): 2 drones, 240/240 Hz, piecewise-constant velocity commands ----
    with quiet():
        env = R.VelocityAviary(num_drones=2, physics=DYN, pyb_freq=240, ctrl_freq=240)
    rng = np.random.default_rng(44)
    seg = rng.uniform(-1, 1, (5, 2, 4)).astype(np.float32)
    seg[..., 3] = np.abs(seg[..., 3])
    seg[2, 1, 0:3] = 0                                   # zero direction -> zero unit vector branch (VelocityAviary.py:150-153)
    acts = np.repeat(seg, 96, axis=0)
    rec = run_env(env, acts, record_obs_every=1)
    save("velocity_aviary_480", **rec)

    # ---- formula-level pins for the PYB-only aerodynamic models ---------------------------------
    rng = np.random.default_rng(5)
    out = {}
    for dm in (R.DroneModel.CF2X, R.DroneModel.CF2P):
        nd = 24
        xyz = np.stack([rng.uniform(-1.5, 1.5, nd), rng.uniform(-1.5, 1.5, nd), rng.uniform(0.02, 1.2, nd)], axis=1)
        xyz[0, 2] = 0.01; xyz[1, 2] = 0.03
        rpys = rng.uniform(-0.6, 0.6, (nd, 3)); rpys[2, 0] = 1.7; rpys[3, 1] = -1.56
        with quiet():
            env = R.CtrlAviary(drone_model=dm, num_drones=nd, initial_xyzs=xyz, initial_rpys=rpys, physics=R.Physics.PYB_GND_DRAG_DW)
        env.vel[:] = rng.uniform(-2, 2, (nd, 3))
        rpm = env.HOVER_RPM * (1 + 0.2 * rng.uniform(-1, 1, (nd, 4)))
        gnd = np.zeros((nd, 4)); drag_body = np.zeros((nd, 3)); dw = np.zeros(nd)
        for i in range(nd):
            pb.APPLIED.clear(); env._groundEffect(rpm[i], i)
            for (_, b, link, f, fl) in pb.APPLIED:
                assert fl == pb.LINK_FRAME and f[0] == 0 and f[1] == 0
                gnd[i, link] += f[2]
            pb.APPLIED.clear(); env._drag(rpm[i], i)
            (_, b, link, f, fl), = pb.APPLIED
            assert link == 4 and fl == pb.LINK_FRAME
            drag_body[i] = f
            pb.APPLIED.clear(); env._downwash(i)
            for (_, b, link, f, fl) in pb.APPLIED:
                assert link == 4 and fl == pb.LINK_FRAME and f[0] == 0 and f[1] == 0
                dw[i] += f[2]
        out.update(flat(dm.value, dict(pos=env.pos.copy(), quat=env.quat.copy(), rpy=env.rpy.copy(), vel=env.vel.copy(), rpm=rpm,
                                       gnd_thrust=gnd, drag_body=drag_body, downwash_body_z=dw)))
    save("effects_formula", **out)
    adjacency_fixture()
    logger_fixture()


def adjacency_fixture():
    """BaseAviary._getAdjacencyMatrix (BaseAviary.py:658-675) on random swarms, three neighbourhood radii."""
    rng = np.random.default_rng(77)
    out = {}
    for k, (nd, radius) in enumerate([(40, 0.8), (33, 2.5), (7, 1e-3)]):
        xyz = rng.uniform(-1.5, 1.5, (nd, 3)).astype(np.float32).astype(np.float64)
        xyz[:, 2] += 2.0
        with quiet():
            env = R.CtrlAviary(num_drones=nd, neighbourhood_radius=radius, initial_xyzs=xyz, physics=R.Physics.DYN)
        out.update(flat("case%d" % k, dict(pos=env.pos.copy(), radius=np.float64(radius), adjacency=env._getAdjacencyMatrix())))
    save("adjacency", **out)


def logger_fixture():
    """utils/Logger.py: the arrays the reference's Logger holds after 7 ticks of 3 drones, logged one drone at a time."""
    import tempfile
    import types
    for name in ("matplotlib", "matplotlib.pyplot", "cycler"):          # plotting deps of the reference module; unused here
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["cycler"].cycler = lambda *a, **k: None
    from gym_pybullet_drones.utils.Logger import Logger
    T, nd = 7, 3
    rng = np.random.default_rng(1)
    timestamp, state, control = np.arange(T) / 48, np.zeros((T, nd, 20)), np.zeros((T, nd, 12))
    with tempfile.TemporaryDirectory() as tmp:
        lg = Logger(logging_freq_hz=48, output_folder=os.path.join(tmp, "r"), num_drones=nd)
        for t in range(T):
            for j in range(nd):
                state[t, j], control[t, j] = rng.normal(size=20), rng.normal(size=12)
                lg.log(drone=j, timestamp=timestamp[t], state=state[t, j], control=control[t, j])
    save("logger_reference", timestamp=timestamp, state=state, control=control,
         timestamps=lg.timestamps, states=lg.states, controls=lg.controls)


if __name__ == "__main__":
    main()
