"""Seeded synthetic inputs of the BASELINE.json shapes (SURVEY.md section 8d).

Input generation only - no GP arithmetic.  Every window is generated from a counter-based hash of
(seed, window id, sample id), so any shard of windows can be produced independently and 1-GPU and N-GPU runs see
identical data.

Slip series (scale matches core_navigation/script/slipVal.csv: std 0.071, range +-0.19):
    x_j = 20 + j  (0.1 s odometry counts as recorded at CoreNav.cpp:286),
    y_j = 0.02 + 0.05 sin(2 pi j / 37) + 0.03 j / N + eps_j,  eps ~ N(0, 0.03^2), clipped to (-1, 1).
Test grid: x*_k = x_{N-1} + 1 + k, k < M, M = 600 (gp_slip_node.py:45).

Look-ahead context: Phi and Q restate the pure functions CoreNav::insErrorStateModel_LNF / CoreNav::calc_Q
(core_navigation/src/CoreNav.cpp:411-527) at a fixed operating point; H is the 4x15 odometry measurement matrix of
CoreNav.cpp:217-220 with the time-averaged integrals replaced by instantaneous values, packed with the reference's
aliasing index Hvec[r*4+c] (CoreNav.cpp:669-673).
"""
from __future__ import annotations

import numpy as np

T0 = 20.0
M_DEFAULT = 600
SEED = 1234

# fixed hyper-parameters of the predict configs (SURVEY.md 8d)
SE_VAR, SE_LS = 0.01, 10.0
PER_VAR, PER_LS, PER_P = 0.0025, 1.0, 37.0
NOISE = 1e-3

INIT_LLH = np.array([0.693457963620326, -1.39498384275845, 334.993517334743])     # config/init_params.yaml:13-16
INIT_ECEF = np.array([859153.015300000, -4836303.72660000, 4055378.50100000])      # config/init_params.yaml:9-12
INIT_ATT = np.array([0.0, 0.0, -0.733038286])                                      # config/init_params.yaml:17-20


def theta_for(kernel: str) -> np.ndarray:
    """Fixed hyper-parameters (noise last) for the kernels the configs name."""
    k = kernel.replace(" ", "").lower()
    table = {
        "rbf": [SE_VAR, SE_LS],
        "se": [SE_VAR, SE_LS],
        "rbf+stdperiodic": [SE_VAR, SE_LS, PER_VAR, PER_P, PER_LS],
        "se+periodic": [SE_VAR, SE_LS, PER_VAR, PER_P, PER_LS],
        "rbf*brownian": [SE_VAR, SE_LS, 0.05],
    }
    if k not in table:
        raise KeyError(kernel)
    return np.array(table[k] + [NOISE])


def _splitmix64(z: np.ndarray) -> np.ndarray:
    z = (z + np.uint64(0x9E3779B97F4A7C15)).astype(np.uint64)
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def _normals(window_ids: np.ndarray, n: int, seed: int, stream: int = 0) -> np.ndarray:
    """Standard normals [len(window_ids), n] from a counter hash (Box-Muller)."""
    with np.errstate(over="ignore"):
        w = window_ids.astype(np.uint64)[:, None]
        j = np.arange(n, dtype=np.uint64)[None, :]
        ctr = (np.uint64(seed) << np.uint64(40)) ^ (np.uint64(stream) << np.uint64(56)) ^ (w << np.uint64(16)) ^ j
        a = _splitmix64(ctr)
        b = _splitmix64(a)
    u1 = ((a >> np.uint64(11)).astype(np.float64) + 1.0) * (1.0 / 9007199254740993.0)
    u2 = (b >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)
    return np.sqrt(-2.0 * np.log(u1)) * np.cos(2.0 * np.pi * u2)


def _uniforms(window_ids: np.ndarray, seed: int, stream: int) -> np.ndarray:
    with np.errstate(over="ignore"):
        ctr = (np.uint64(seed) << np.uint64(40)) ^ (np.uint64(stream) << np.uint64(56)) ^ window_ids.astype(np.uint64)
        a = _splitmix64(ctr)
    return (a >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)


def slip_windows(first: int, count: int, N: int, seed: int = SEED):
    """x [count,N], y [count,N] for windows first .. first+count-1."""
    ids = np.arange(first, first + count, dtype=np.int64)
    j = np.arange(N, dtype=np.float64)
    x = np.broadcast_to(T0 + j, (count, N)).copy()
    y = 0.02 + 0.05 * np.sin(2.0 * np.pi * j / 37.0) + 0.03 * (j / N) + 0.03 * _normals(ids, N, seed)
    return x, np.clip(y, -0.999999, 0.999999)


def test_grid(x: np.ndarray, M: int = M_DEFAULT) -> np.ndarray:
    """x*_k = x_{N-1} + 1 + k (shared by every window when the windows share their time stamps)."""
    last = x[..., -1:]
    return last + 1.0 + np.arange(M, dtype=np.float64)


test_grid.__test__ = False  # not a pytest test


# ----------------------------------------------------------------------------------------------------------
# look-ahead context
# ----------------------------------------------------------------------------------------------------------
OMEGA_IE = 7.292115e-5
R0 = 6378137.0
ECC = 0.0818191909425
FLAT = 1.0 / 298.257223563
T_CONST = (1.0 - FLAT) ** 2
PI_INS = 3.14159265358979


def _skew(v):
    return np.array([[0.0, -v[2], v[1]], [v[2], 0.0, -v[0]], [-v[1], v[0], 0.0]])


def eul_to_dcm(phi, theta, psi):
    """CoreNav::eul_to_dcm (CoreNav.cpp:561-581): nav -> body."""
    cpsi, spsi = np.cos(psi), np.sin(psi)
    cthe, sthe = np.cos(theta), np.sin(theta)
    cphi, sphi = np.cos(phi), np.sin(phi)
    c1 = np.array([[cpsi, spsi, 0.0], [-spsi, cpsi, 0.0], [0.0, 0.0, 1.0]])
    c2 = np.array([[cthe, 0.0, -sthe], [0.0, 1.0, 0.0], [sthe, 0.0, cthe]])
    c3 = np.array([[1.0, 0.0, 0.0], [0.0, cphi, sphi], [0.0, -sphi, cphi]])
    return (c3 @ c2) @ c1


def radii(lat):
    """R_N, R_E as in CoreNav::Propagate (CoreNav.cpp:63-66)."""
    s2 = np.sin(lat) ** 2
    R_N = R0 * (1.0 - ECC ** 2) / (1.0 - ECC ** 2 * s2) ** 1.5
    R_E = R0 / np.sqrt(1.0 - ECC ** 2 * s2)
    return R_N, R_E


def stm_lnf(llh, vel, dt, Cbn, omega_n_in, f_ib_b):
    """Restatement of CoreNav::insErrorStateModel_LNF (CoreNav.cpp:411-470), quirks included."""
    lat, lon, h = llh
    R_N, R_E = radii(lat)
    geo_lat = np.arctan2(T_CONST * np.sin(lat * 180.0 / PI_INS), np.cos(lat * 180.0 / PI_INS))
    r_geo = np.sqrt(R0 ** 2 / (1.0 + (1.0 / (1.0 - FLAT) ** 2 - 1.0) * np.sin(geo_lat) ** 2))
    g0 = 9.780318 * (1.0 + 5.3024e-3 * np.sin(lat) ** 2 - 5.9e-6 * np.sin(2 * lat) ** 2)
    F11 = -_skew(omega_n_in)
    F12 = np.array([[0.0, -1.0 / (R_E + h), 0.0], [1.0 / (R_N + h), 0.0, 0.0], [0.0, np.tan(lat) / (R_E + h), 0.0]])
    F13 = np.array([[OMEGA_IE * np.sin(lat), 0.0, vel[1] / (R_E + h) ** 2],
                    [0.0, 0.0, -vel[0] / (R_N + h) ** 2],
                    [OMEGA_IE * np.cos(lat) + vel[1] / ((R_E + h) * np.cos(lat) ** 2), 0.0,
                     -vel[1] * np.tan(lat) / (R_E + h) ** 2]])
    F21 = -_skew(Cbn @ f_ib_b)
    F22 = np.array([
        [vel[2] / (R_N + h), -(2.0 * vel[1] * np.tan(lat) / (R_E + h)) - 2.0 * OMEGA_IE * np.sin(lat), vel[0] / (R_N + h)],
        [vel[1] * np.tan(lat) / (R_E + h) + 2.0 * OMEGA_IE * np.sin(lat), (vel[0] * np.tan(lat) + vel[2]) / (R_E + h),
         vel[1] / (R_E + h) + 2.0 * OMEGA_IE * np.cos(lat)],
        [-2.0 * vel[0] / (R_N + h), -2.0 * (vel[1] / (R_E + h)) - 2.0 * OMEGA_IE * np.cos(lat), 0.0]])
    sec2 = 1.0 / np.cos(lat) ** 2
    F23 = np.array([
        [-(vel[1] ** 2 * sec2 / (R_E + h)) - 2.0 * vel[1] * OMEGA_IE * np.cos(lat), 0.0,
         vel[1] ** 2 * np.tan(lat) / (R_E + h) ** 2 - vel[0] * vel[2] / (R_N + h) ** 2],
        [vel[0] * vel[1] * sec2 / (R_E + h) + 2.0 * vel[0] * OMEGA_IE * np.cos(lat) - 2.0 * vel[2] * OMEGA_IE * np.sin(lat),
         0.0, -((vel[0] * vel[1] * np.tan(lat) + lon * h) / (R_E + h) ** 2)],
        [2.0 * vel[1] * OMEGA_IE * np.sin(lat), 0.0,
         vel[1] ** 2 / (R_E + h) ** 2 + vel[0] ** 2 / (R_N + h) ** 2 - 2.0 * g0 / r_geo]])
    F32 = np.diag([1.0 / (R_N + h), 1.0 / ((R_E + h) * np.cos(lat)), -1.0])
    F33 = np.array([[0.0, 0.0, -vel[0] / (R_N + h) ** 2],
                    [vel[1] * np.sin(lat) / ((R_E + h) * np.cos(lat) ** 2), 0.0, -vel[1] / ((R_E + h) ** 2 * np.cos(lat))],
                    [0.0, 0.0, 0.0]])
    I3, Z3 = np.eye(3), np.zeros((3, 3))
    return np.block([
        [I3 + F11 * dt, F12 * dt, F13 * dt, Z3, Cbn * dt],
        [F21 * dt, I3 + F22 * dt, F23 * dt, Cbn * dt, Z3],
        [Z3, F32 * dt, I3 + F33 * dt, Z3, Z3],
        [Z3, Z3, Z3, I3, Z3],
        [Z3, Z3, Z3, Z3, I3]])


def calc_q(llh, dt, Cbn, f_ib_b):
    """Restatement of CoreNav::calc_Q (CoreNav.cpp:471-527)."""
    lat, _, h = llh
    R_N, R_E = radii(lat)
    F21 = -_skew(Cbn @ f_ib_b)
    T = np.diag([1.0 / (R_N + h), 1.0 / ((R_E + h) * np.cos(lat)), -1.0])
    gg = 9.80665
    sig_gyro = 1.6 * PI_INS / 180 / 3600
    sig_arw = .1 * (PI_INS / 180) * np.sqrt(3600) / 3600
    sig_acc = 3.2e-6 * gg
    sig_vrw = 0.008 * np.sqrt(3600) / 3600
    Srg, Sra = sig_arw ** 2 * dt, sig_vrw ** 2 * dt
    Sbad, Sbgd = sig_acc ** 2 / dt, sig_gyro ** 2 / dt
    I3, Z3 = np.eye(3), np.zeros((3, 3))
    FF = F21 @ F21.T
    Q11 = (Srg * dt + Sbgd * dt ** 3 / 3.0) * I3
    Q21 = (Srg * dt ** 2 / 2.0 + Sbgd * dt ** 4 / 4.0) * F21
    Q31 = (Srg * dt ** 3 / 3.0 + Sbgd * dt ** 5 / 5.0) * T @ F21
    Q15 = Sbgd * dt ** 2 / 2.0 * Cbn
    Q22 = (Sra * dt + Sbad * dt ** 3 / 3.0) * I3 + (Srg * dt ** 3 / 3.0 + Sbgd * dt ** 5 / 5.0) * FF
    Q32 = (Sra * dt ** 2 / 2.0 + Sbad * dt ** 4 / 4.0) * T + (Srg * dt ** 4 / 4.0 + Sbgd * dt ** 6 / 6.0) * T @ FF
    Q24 = Sbad * dt ** 2 / 2.0 * Cbn
    Q25 = Sbgd * dt ** 3 / 3.0 * F21 @ Cbn
    Q33 = (Sra * dt ** 3 / 3.0 + Sbad * dt ** 5 / 5.0) * (T @ T) + (Srg * dt ** 5 / 5.0 + Sbgd * dt ** 7 / 7.0) * T @ FF @ T
    Q34 = Sbad * dt ** 3 / 3.0 * T @ Cbn
    Q35 = Sbgd * dt ** 4 / 4.0 * T @ F21 @ Cbn
    Q42 = Sbad * dt ** 2 / 2.0 * Cbn.T
    Q44 = Sbad * dt * I3
    Q51 = Sbgd * dt ** 2 / 2.0 * Cbn.T
    Q52 = Sbgd * dt ** 3 / 3.0 * F21.T @ Cbn.T
    Q55 = Sbgd * dt * I3
    return np.block([
        [Q11, Q21.T, Q31.T, Z3, Q15],
        [Q21, Q22, Q32.T, Q24, Q25],
        [Q31, Q32, Q33, Q34, Q35],
        [Z3, Q42, Q34.T, Q44, Z3],
        [Q51, Q52, Q35.T, Z3, Q55]])


def pack_hvec(H: np.ndarray) -> np.ndarray:
    """CoreNav::setStopping_ (CoreNav.cpp:669-673): HvecData[r*4+c] = H(r,c), r<4, c<15 - later writes win."""
    v = np.zeros(60)
    for r in range(4):
        for c in range(15):
            v[r * 4 + c] = H[r, c]
    return v


def lookahead_context(horizontal_sigma=0.5, velocity_sigma=None):
    """Shared context of the look-ahead configs: dict(P [225] or [B,225], Q, STM, Hvec, pos).

    horizontal_sigma: scalar or array [B] of the initial horizontal 1-sigma position error in metres.
    velocity_sigma:   scalar or array [B] of the initial 1-sigma velocity error in m/s (default sqrt(1e-3) = 0.0316).
        With the reference's H packing the odometry update barely constrains the velocity states, so the 3-sigma
        horizontal error grows like 3 sqrt(s^2 + (v t)^2): the default reaches the 3 m threshold after ~30 s whatever s
        is; a Monte-Carlo batch in which some windows never trigger inside the 60 s horizon needs smaller v too."""
    att = INIT_ATT
    psi = att[2]
    llh = INIT_LLH.copy()
    vel = 0.8 * np.array([np.cos(psi), np.sin(psi), 0.0])
    f_ib_b = np.array([0.0, 0.0, -9.80665])
    dt = 0.02
    C = eul_to_dcm(*att)           # nav -> body
    Cbn = C.T
    R_N, R_E = radii(llh[0])
    omega_n_ie = np.array([OMEGA_IE * np.cos(llh[0]), 0.0, -OMEGA_IE * np.sin(llh[0])])
    omega_n_en = np.array([vel[1] / (R_E + llh[2]), -vel[0] / (R_N + llh[2]), -vel[1] * np.tan(llh[0]) / (R_E + llh[2])])
    STM = stm_lnf(llh, vel, dt, Cbn, omega_n_en + omega_n_ie, f_ib_b)
    Q = calc_q(llh, dt, Cbn, f_ib_b)
    vss = _skew(vel)
    H = np.zeros((4, 15))
    H[0, 0:3] = -(C @ vss)[0]
    H[0, 3:6] = -C[0]
    H[1, 9:12] = -(np.cos(att[1]) * C.T[2]) / 0.1
    H[2, 0:3] = -(C @ vss)[1]
    H[2, 3:6] = -C[1]
    H[3, 0:3] = -(C @ vss)[2]
    H[3, 3:6] = -C[2]
    s = np.atleast_1d(np.asarray(horizontal_sigma, dtype=np.float64))
    vv = 1e-3 if velocity_sigma is None else np.atleast_1d(np.asarray(velocity_sigma, dtype=np.float64)) ** 2
    if np.ndim(vv) and np.size(vv) != s.size:
        s, vv = np.broadcast_arrays(s, vv)
    d = np.zeros((s.size, 15))
    d[:, 0:3] = 1.218e-6
    d[:, 3:6] = vv[:, None] if np.ndim(vv) else vv
    d[:, 6] = (s / (R_N + llh[2])) ** 2
    d[:, 7] = (s / ((R_E + llh[2]) * np.cos(llh[0]))) ** 2
    d[:, 8] = s ** 2
    d[:, 9:12] = 1e-4
    d[:, 12:15] = 1e-8
    P = np.zeros((s.size, 15, 15))
    idx = np.arange(15)
    P[:, idx, idx] = d
    P = P.reshape(s.size, 225)
    if np.ndim(horizontal_sigma) == 0 and (velocity_sigma is None or np.ndim(velocity_sigma) == 0):
        P = P[0]
    return dict(P=P, Q=Q.reshape(225), STM=STM.reshape(225), Hvec=pack_hvec(H), pos=llh, H=H)


def window_sigmas(first: int, count: int, seed: int = SEED, lo: float = 0.2, hi: float = 0.8) -> np.ndarray:
    """Per-window initial horizontal sigma ~ U[lo, hi] m (configs[3]) so that some windows trigger and some never do."""
    ids = np.arange(first, first + count, dtype=np.int64)
    return lo + (hi - lo) * _uniforms(ids, seed, stream=7)


def monte_carlo_contexts(first: int, count: int, seed: int = SEED, decades: float = 4.5):
    """Per-window SetStopping contexts of the Monte-Carlo config (BASELINE.json configs[3]): dict(P [B,225], Q [B,225],
    STM, Hvec, pos shared).

    With the reference's own P0 / Q (lookahead_context) EVERY window reaches the 3 m threshold after 25-30 s of the 60 s
    horizon - the velocity, attitude and bias states are barely constrained by the odometry update under the reference's
    H packing - which makes a poor Monte-Carlo: no window runs the full 2995 steps.  Here each window draws a "filter
    quality" u ~ U[0,1]: the variances of the attitude / velocity / bias states of P0 and the whole of Q are scaled by
    10^(-decades u), the horizontal position sigma is window_sigmas' U[0.2, 0.8] m.  Windows with a well-converged filter
    (u near 1) never trigger inside the horizon; the fraction is reported by tools/bench_configs.py next to the
    throughput (about a seventh of the windows at decades = 4.5)."""
    ids = np.arange(first, first + count, dtype=np.int64)
    base = lookahead_context(window_sigmas(first, count, seed))
    u = _uniforms(ids, seed, stream=8)
    f = 10.0 ** (-decades * u)
    P = base["P"].reshape(count, 15, 15).copy()
    for i in list(range(0, 6)) + list(range(9, 15)):
        P[:, i, i] *= f
    Q = base["Q"][None, :] * f[:, None]
    return dict(P=P.reshape(count, 225), Q=np.ascontiguousarray(Q), STM=base["STM"], Hvec=base["Hvec"], pos=base["pos"],
                quality=u)


def drives(first: int, count: int, T: int = 400, seed: int = SEED, stop_events: bool = True, pauses: bool = False):
    """Synthetic odometry logs for the slip recorder (SURVEY.md 8f row N1): dict(joint [B,T,4], att [B,T,3],
    vel [B,T,3], cmd [B,T], stop_cmd [B,T]).  10 Hz updates: standstill for a per-drive lead-in, then a 0.8 m/s drive at
    the survey heading with wheel slip of the slipVal.csv scale on the right/left wheel pairs, an occasional stuck phase
    (slip clamps to 1) and, on some drives, a stop command shortly after the first window closes.

    pauses: the drive command is released (cmd = 0) for 0-134 updates at a per-drive place inside the first window, so
    the recorder's windows hold different numbers of samples (from a few up to the window length) with gaps in their
    stamps - the ragged GP_Input a real drive produces (CoreNav.cpp:264-300)."""
    ids = np.arange(first, first + count, dtype=np.int64)
    k = np.arange(T)[None, :]
    lead = (5 + 40 * _uniforms(ids, seed, stream=11)).astype(np.int64)[:, None]
    driving = k >= lead
    psi = INIT_ATT[2] + 0.05 * (_uniforms(ids, seed, stream=12)[:, None] - 0.5) + 0.002 * np.sin(k / 23.0)
    the = 0.03 * np.sin(k / 31.0 + 6.0 * _uniforms(ids, seed, stream=13)[:, None])
    phi = 0.01 * np.cos(k / 17.0) + 0.0 * psi
    stuck = (_uniforms(ids, seed, stream=17)[:, None] < 0.3) & (k > lead + 60) & (k < lead + 70)
    v = np.where(stuck, -0.05, np.where(driving, 0.8, 0.0))      # stuck: wheels spin, the rover creeps backwards
    vel = np.stack([v * np.cos(psi) * np.cos(the), v * np.sin(psi) * np.cos(the), -v * np.sin(the)], axis=-1)
    vel = vel + 0.002 * _normals(ids, 3 * T, seed, stream=14).reshape(count, T, 3)
    slip_r = 0.02 + 0.05 * np.sin(2 * np.pi * k / 37.0) + 0.03 * _normals(ids, T, seed, stream=15)
    slip_l = slip_r + 0.01 * _normals(ids, T, seed, stream=16)
    wr = np.where(stuck, 1.0, v / (1.0 - slip_r))       # wheel speed (m/s): slip = (v_wheel - v) / v_wheel
    wl = np.where(stuck, 1.0, v / (1.0 - slip_l))
    R = 0.11
    joint = np.stack([-wl / R, wr / R, -wl / R * 0.999, wr / R * 1.001], axis=-1)
    cmd = np.where(driving, 1.0, 0.0)
    if pauses:
        p0 = lead + 12 + np.floor(140.0 * _uniforms(ids, seed, stream=19)).astype(np.int64)[:, None]
        plen = np.floor(135.0 * _uniforms(ids, seed, stream=20)).astype(np.int64)[:, None]
        cmd = np.where((k >= p0) & (k < p0 + plen), 0.0, cmd)
    stop_cmd = np.full((count, T), np.nan)
    if stop_events:
        has = _uniforms(ids, seed, stream=18) < 0.5
        at = np.minimum(T - 1, lead[:, 0] + 10 + 150 + 3)
        stop_cmd[np.where(has)[0], at[has]] = 2.3
    return dict(joint=joint, att=np.stack([phi, the, psi], axis=-1), vel=vel, cmd=cmd, stop_cmd=stop_cmd)


def operating_points(first: int, count: int, seed: int = SEED):
    """Operating points for the EKF context generator (SURVEY.md 8f row N4): dict(llh, vel, att, f_ib_b), each [B,3] -
    positions scattered ~100 m around the survey origin, 0.8 m/s drives at scattered headings and small tilts, the
    specific force of a rover at rest on that tilt plus accelerometer noise."""
    ids = np.arange(first, first + count, dtype=np.int64)
    u = lambda st: _uniforms(ids, seed, stream=st)
    llh = INIT_LLH[None, :] + np.stack([(u(21) - 0.5) * 3e-5, (u(22) - 0.5) * 3e-5, (u(23) - 0.5) * 10.0], axis=-1)
    att = np.stack([(u(24) - 0.5) * 0.1, (u(25) - 0.5) * 0.2, (u(26) - 0.5) * 2 * np.pi], axis=-1)
    speed = 0.4 + 0.8 * u(27)
    vel = np.stack([speed * np.cos(att[:, 2]) * np.cos(att[:, 1]), speed * np.sin(att[:, 2]) * np.cos(att[:, 1]),
                    -speed * np.sin(att[:, 1])], axis=-1)
    g = 9.80665
    f = np.stack([g * np.sin(att[:, 1]), -g * np.sin(att[:, 0]) * np.cos(att[:, 1]),
                  -g * np.cos(att[:, 0]) * np.cos(att[:, 1])], axis=-1)
    f = f + 0.05 * _normals(ids, 3, seed, stream=28)
    return dict(llh=llh, vel=vel, att=att, f_ib_b=f)
