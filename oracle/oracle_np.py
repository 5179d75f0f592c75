"""CPU ORACLE (numpy) for the batched BlueROV2 / legacy-AUV env-step path.

TEST INFRASTRUCTURE ONLY.  This file restates the reference's algorithm in
numpy so that the CUDA path can be checked on machines where /root/reference
does not exist.  Only ``tests/``, ``__graft_entry__.smoke()`` and
``bench.py``'s CPU-baseline legs may import it; the product package never does
(the product fails loudly when its CUDA library is missing).

Parity pin: the reference ships no tests and no golden vectors for this path
(SURVEY.md section 4; the single in-repo vector, example_temp.py:19-28, is
checked in tests/test_oracle_golden.py).  The oracle is therefore pinned
against outputs of the UNMODIFIED reference executed in the build container:
``tests/golden/golden_*.npz`` written by ``tests/golden/gen_golden_*.py``.

Every function is vectorised over a leading batch axis ``N`` (array-of-structs
``[N, k]`` - the natural numpy layout; the CUDA library uses ``[k][N]``).
Reference citations are ``file:line`` relative to the reference root, with
``6DoF.py`` = dynamicsModel_BlueROV2_Heavy_6DoF.py, ``3DoF.py`` =
dynamicsModel_BlueROV2_Heavy_3DoF.py, ``legacy/`` =
tag_00_Dec2023_simpleControlTurbulence/.
"""
from dataclasses import dataclass, field

import numpy as np

TWO_PI = 2.0 * np.pi


# ==========================================================================
# resources.py helpers
# ==========================================================================
def compute_thrust_allocation(positions, normals, x0=None):
    """resources.py:19-35 - A[:, i] = [n_i ; (r_i - x0) x n_i], Ainv = pinv(A)."""
    positions = np.asarray(positions, dtype=float)
    normals = np.asarray(normals, dtype=float)
    if x0 is None:
        x0 = np.zeros(3)
    A = np.zeros((6, positions.shape[0]))
    for i in range(positions.shape[0]):
        A[:3, i] = normals[i]
        A[3:, i] = np.cross(positions[i] - x0, normals[i])
    return A, np.linalg.pinv(A)


def angle_error(psi_d, psi):
    """resources.py:75-95 (== legacy/resources.py:26-46).  Python-modulo
    semantics; returns -0.0 for equal angles and -pi for a == b == pi."""
    psi_d = np.asarray(psi_d, dtype=float)
    psi = np.asarray(psi, dtype=float)
    a = np.mod(psi_d - psi, TWO_PI)
    b = np.mod(psi - psi_d, TWO_PI)
    return np.where(a < b, a, -b)


def coordinate_transform6(phi, theta, psi):
    """resources.py:115-141 -> [N, 6, 6].  Bug-compatible: J1[0,2] carries
    sin(phi) in its second term (Fossen has cos(phi)); cos(theta) in J2's
    denominators is clamped away from zero as at resources.py:116-120."""
    phi, theta, psi = (np.atleast_1d(np.asarray(v, dtype=float)) for v in (phi, theta, psi))
    sph, cph = np.sin(phi), np.cos(phi)
    sth, cth = np.sin(theta), np.cos(theta)
    sps, cps = np.sin(psi), np.cos(psi)
    den = np.where(np.abs(cth) < 1e-12, 1e-6, np.where(np.abs(cth) < 1e-6, 1e-6 * np.sign(cth), cth))
    J = np.zeros(phi.shape + (6, 6))
    J[..., 0, 0] = cps * cth
    J[..., 0, 1] = -sps * cph + cps * sth * sph
    J[..., 0, 2] = sps * sph + cps * sth * sph
    J[..., 1, 0] = sps * cth
    J[..., 1, 1] = cps * cph + sps * sth * sph
    J[..., 1, 2] = -cps * sph + sps * sth * cph
    J[..., 2, 0] = -sth
    J[..., 2, 1] = cth * sph
    J[..., 2, 2] = cth * cph
    J[..., 3, 3] = 1.0
    J[..., 3, 4] = sph * sth / den
    J[..., 3, 5] = cph * sth / den
    J[..., 4, 4] = cph
    J[..., 4, 5] = -sph
    J[..., 5, 4] = sph / den
    J[..., 5, 5] = cph / den
    return J


def coordinate_transform3(psi):
    """resources.py:108-113 -> [N, 3, 3] planar rotation."""
    psi = np.atleast_1d(np.asarray(psi, dtype=float))
    J = np.zeros(psi.shape + (3, 3))
    J[..., 0, 0] = np.cos(psi)
    J[..., 0, 1] = -np.sin(psi)
    J[..., 1, 0] = np.sin(psi)
    J[..., 1, 1] = np.cos(psi)
    J[..., 2, 2] = 1.0
    return J


# ==========================================================================
# 6DoF model
# ==========================================================================
@dataclass
class Rov6Params:
    """6DoF.py:83-218.  Attribute names are the reference's."""
    rho_f: float = 1000.
    m: float = 11.4
    Length: float = 0.457
    Width: float = 0.338
    CB: np.ndarray = field(default_factory=lambda: np.array([0., 0., 0.]))
    CG: np.ndarray = field(default_factory=lambda: np.array([0., 0., 0.05]))
    I: np.ndarray = field(default_factory=lambda: np.diag([0.16, 0.16, 0.16]))
    Xudot: float = -5.5
    Yvdot: float = -12.7
    Zwdot: float = -14.57
    Kpdot: float = -0.12
    Mqdot: float = -0.12
    Nrdot: float = -0.12
    Yrdot: float = 0.
    Zvdot: float = 0.
    Nvdot: float = 0.
    Xuu: float = -18.18
    Yvv: float = -21.66
    Zww: float = -36.99
    Kpp: float = -1.55
    Mqq: float = -1.55
    Nrr: float = -1.55
    Yrr: float = 0.
    Ypp: float = 0.
    Zqq: float = 0.
    Kvv: float = 0.
    Krr: float = 0.
    Mww: float = -1.55
    Nvv: float = 0.
    Npp: float = 0.
    Xu: float = -4.03
    Yv: float = -6.22
    Zw: float = -5.18
    Kp: float = -0.07
    Mq: float = -0.07
    Nr: float = -0.07
    Yr: float = 0.
    Yp: float = 0.
    Zq: float = 0.
    Kv: float = 0.
    Kr: float = 0.
    Mw: float = 0.
    Nv: float = 0.
    Np: float = 0.
    D_thruster: float = 0.1
    alphaThruster: float = 33. / 180. * np.pi
    l_x: float = 0.1475
    l_y: float = 0.101
    l_z: float = 0.068
    l_x_v: float = 0.120
    l_y_v: float = 0.22
    l_z_v: float = 0.0

    def __post_init__(self):
        self.dispVol = self.m / self.rho_f
        self.Kt_thruster = 40. / (1000. * (3500. / 60.) ** 2. * self.D_thruster ** 4.)
        a = self.alphaThruster
        self.thrusterPositions = np.array([
            [self.l_x, self.l_y, self.l_z], [self.l_x, -self.l_y, self.l_z],
            [-self.l_x, self.l_y, self.l_z], [-self.l_x, -self.l_y, self.l_z],
            [self.l_x_v, self.l_y_v, self.l_z_v], [self.l_x_v, -self.l_y_v, self.l_z_v],
            [-self.l_x_v, self.l_y_v, self.l_z_v], [-self.l_x_v, -self.l_y_v, self.l_z_v]])
        self.thrusterNormals = np.array([
            [np.cos(a), -np.sin(a), 0.], [np.cos(a), np.sin(a), 0.],
            [-np.cos(a), -np.sin(a), 0.], [-np.cos(a), np.sin(a), 0.],
            [0., 0., -1.], [0., 0., 1.], [0., 0., 1.], [0., 0., -1.]])
        self.A, self.Ainv = compute_thrust_allocation(self.thrusterPositions, self.thrusterNormals)

    # 6DoF.py:286-299.  NB Ma[2,2] uses Zvdot (= 0), not Zwdot.
    def mass_matrix(self):
        m, (xg, yg, zg) = self.m, self.CG
        Mrb = np.array([
            [m, 0., 0., 0., m * zg, -m * yg],
            [0., m, 0., -m * zg, 0., m * xg],
            [0., 0., m, m * yg, -m * xg, 0.],
            [0., -m * zg, m * yg, 0., 0., 0.],
            [m * zg, 0., -m * xg, 0., 0., 0.],
            [-m * yg, m * xg, 0., 0., 0., 0.]])
        Mrb[3:, 3:] = self.I
        Ma = -1. * np.diag([self.Xudot, self.Yvdot, self.Zvdot, self.Kpdot, self.Mqdot, self.Nrdot])
        return Mrb + Ma


PID6_WINDUP = np.array([2., 2., 2., 90. / 180. * np.pi, 90. / 180. * np.pi, 90. / 180. * np.pi])
PID6_MAX = np.array([50., 50., 50., 1., 1., 2.])
PID6_KP = np.array([25., 25., 25., 10., 10., 1.])
PID6_KI = np.array([2., 2., 2., 0.1, 0.1, 0.2])
PID6_KD = np.array([20., 20., 20., 5., 5., 0.65])


def _track_margin(ctrl, e, e_old, dtc):
    """NOT part of the algorithm - a conditioning diagnostic for the parity tests, kept only when the caller put a
    "margin" array into ``ctrl``: the smallest non-zero |e - eOld| seen by a call with t - tOld < 1e-9, where
    dedt = (e - eOld) / 1e-9 turns the SIGN of that difference into a saturated demand (RK4 stages 1 and 3)."""
    if "margin" not in ctrl:
        return
    d = np.abs(e - e_old)
    d = np.where((d > 0.) & (dtc < 1e-9)[:, None], d, np.inf).min(axis=1)
    ctrl["margin"] = np.minimum(ctrl["margin"], d)


def pid6_new_state(n):
    """6DoF.py:37-41: eOld=None, eInt=0, tOld=0."""
    return {"eOld": np.zeros((n, 6)), "has_old": np.zeros(n, dtype=bool),
            "eInt": np.zeros((n, 6)), "tOld": np.zeros(n)}


def pid6_control(ctrl, set_point, pose, t):
    """6DoF.py:43-73 - mutates ``ctrl`` exactly like the reference mutates the
    controller on EVERY call.  Roll/pitch errors are raw differences, yaw is
    wrapped; dedt divides by max(1e-9, t - tOld)."""
    set_point = np.asarray(set_point, dtype=float)
    pose = np.asarray(pose, dtype=float)
    t = np.broadcast_to(np.asarray(t, dtype=float), pose.shape[:1])
    e = np.empty_like(pose)
    e[:, 0:3] = set_point[:, 0:3] - pose[:, 0:3]
    e[:, 3] = set_point[:, 3] - pose[:, 3]
    e[:, 4] = set_point[:, 4] - pose[:, 4]
    e[:, 5] = angle_error(set_point[:, 5], pose[:, 5])
    e_old = np.where(ctrl["has_old"][:, None], ctrl["eOld"], e)
    dtc = t - ctrl["tOld"]
    _track_margin(ctrl, e, e_old, dtc)
    dedt = (e - e_old) / np.maximum(1e-9, dtc)[:, None]
    e_int = ctrl["eInt"] + 0.5 * (e_old + e) * dtc[:, None]
    e_int = np.where(np.abs(e) > PID6_WINDUP, 0., e_int)
    u = PID6_KP * e + PID6_KD * dedt + PID6_KI * e_int
    u = np.maximum(-PID6_MAX, np.minimum(PID6_MAX, u))
    ctrl["eOld"] = e
    ctrl["has_old"] = np.ones_like(ctrl["has_old"])
    ctrl["eInt"] = e_int
    ctrl["tOld"] = t.copy()
    return u


def body_axes(angles):
    """6DoF.py:238-242: rows of R^T for the intrinsic-XYZ rotation
    R = Rx(phi) Ry(theta) Rz(psi) (closed form of scipy's
    Rotation.from_euler('XYZ')) -> iHat, jHat, kHat, each [N, 3]."""
    phi, th, psi = angles[:, 0], angles[:, 1], angles[:, 2]
    sph, cph, sth, cth, sps, cps = np.sin(phi), np.cos(phi), np.sin(th), np.cos(th), np.sin(psi), np.cos(psi)
    i_hat = np.stack([cth * cps, cph * sps + sph * sth * cps, sph * sps - cph * sth * cps], axis=1)
    j_hat = np.stack([-cth * sps, cph * cps - sph * sth * sps, sph * cps + cph * sth * sps], axis=1)
    k_hat = np.stack([sth, -sph * cth, cph * cth], axis=1)
    return i_hat, j_hat, k_hat


def global_to_vehicle(axes, v):
    """6DoF.py:244-248."""
    return np.stack([np.sum(v * axes[0], axis=1), np.sum(v * axes[1], axis=1), np.sum(v * axes[2], axis=1)], axis=1)


def allocate_thrust6(p, axes, gcf):
    """6DoF.py:220-231: earth-frame forces AND moments are rotated like
    vectors into the body frame, then rpm = sign(c) sqrt(|c|/(rho D^4 Kt)) 60."""
    body = np.concatenate([global_to_vehicle(axes, gcf[:, :3]), global_to_vehicle(axes, gcf[:, 3:])], axis=1)
    cv = body @ p.Ainv.T
    return np.sign(cv) * np.sqrt(np.abs(cv) / (p.rho_f * p.D_thruster ** 4. * p.Kt_thruster)) * 60.


# NOT part of the algorithm - conditioning diagnostic for the parity tests.  A test may set DIAG["dbmargin"] to an
# array [n] of +inf; limit_rpm then keeps in it the smallest relative distance | |rpm| - 300 | / 300 of a thruster demand
# from the dead-band edge, where the thrust jumps from 0 to 0.29 N (an environment that comes within rounding distance
# of the edge cannot agree between two precisions).
DIAG = {"dbmargin": None}


def limit_rpm(rpm):
    """6DoF.py:271-275: saturate at +-3500, zero inside the 300 rpm deadband."""
    r = np.maximum(-3500., np.minimum(3500., rpm))
    if DIAG["dbmargin"] is not None and np.ndim(r) == 2 and r.shape[0] == DIAG["dbmargin"].shape[0]:
        DIAG["dbmargin"] = np.minimum(DIAG["dbmargin"], (np.abs(np.abs(r) - 300.) / 300.).min(axis=1))
    return np.where(np.abs(r) < 300, 0., r)


def thruster_force6(p, rpm):
    """6DoF.py:233-236."""
    return p.rho_f * (rpm / 60.) ** 2. * np.sign(rpm) * p.D_thruster ** 4. * p.Kt_thruster


def force_components6(p, angles, vel, rpm):
    """6DoF.py:253-404 -> (-Crb v, -Ca v, -D v, G, H), each [N, 6]."""
    m = p.m
    xg, yg, zg = p.CG
    Im = p.I
    phi, theta = angles[:, 0], angles[:, 1]
    u, v, w, pp, q, r = (vel[:, i] for i in range(6))

    H = thruster_force6(p, limit_rpm(rpm)) @ p.A.T  # 6DoF.py:278-282

    # Crb v, 6DoF.py:303-332
    a1 = m * (yg * q + zg * r); a2 = m * (xg * q - w); a3 = m * (xg * r + v)
    b1 = m * (yg * pp + w); b2 = m * (zg * r + xg * pp); b3 = m * (yg * r - u)
    c1 = m * (zg * pp - v); c2 = m * (zg * q + u); c3 = m * (xg * pp + yg * q)
    i1 = -Im[1, 2] * q - Im[0, 2] * pp + Im[2, 2] * r
    i2 = Im[1, 2] * r + Im[0, 1] * pp - Im[1, 1] * q
    i3 = -Im[0, 2] * r - Im[0, 1] * q + Im[0, 0] * pp
    crb = np.stack([
        a1 * pp - a2 * q - a3 * r,
        -b1 * pp + b2 * q - b3 * r,
        -c1 * pp - c2 * q + c3 * r,
        -a1 * u + b1 * v + c1 * w + i1 * q + i2 * r,
        a2 * u - b2 * v + c2 * w - i1 * pp + i3 * r,
        a3 * u + b3 * v - c3 * w - i2 * pp - i3 * q], axis=1)

    # Ca v, 6DoF.py:334-341 (uses Zwdot although Ma uses Zvdot)
    Xd, Yd, Zd, Kd, Md, Nd = p.Xudot, p.Yvdot, p.Zwdot, p.Kpdot, p.Mqdot, p.Nrdot
    ca = np.stack([
        -Zd * w * q + Yd * v * r,
        Zd * w * pp - Xd * u * r,
        -Yd * v * pp + Xd * u * q,
        -Zd * w * v + Yd * v * w - Nd * r * q + Md * q * r,
        Zd * w * u - Xd * u * w + Nd * r * pp - Kd * pp * r,
        -Yd * v * u + Xd * u * v - Md * q * pp + Kd * pp * q], axis=1)

    # -D v, 6DoF.py:345-370 (D = -(Dl + Dq|v|), so -D v = +(coef) v)
    au, av, aw, ap, aq, ar = (np.abs(x) for x in (u, v, w, pp, q, r))
    mdv = np.stack([
        (p.Xu + p.Xuu * au) * u,
        (p.Yv + p.Yvv * av) * v + (p.Yp + p.Ypp * ap) * pp + (p.Yr + p.Yrr * ar) * r,
        (p.Zw + p.Zww * aw) * w + (p.Zq + p.Zqq * aq) * q,
        (p.Kv + p.Kvv * av) * v + (p.Kp + p.Kpp * ap) * pp + (p.Kr + p.Krr * ar) * r,
        (p.Mw + p.Mww * aw) * w + (p.Mq + p.Mqq * aq) * q,
        (p.Nv + p.Nvv * av) * v + (p.Np + p.Npp * ap) * pp + (p.Nr + p.Nrr * ar) * r], axis=1)

    # G, 6DoF.py:374-388
    W = p.m * 9.81
    B = p.dispVol * p.rho_f * 9.81
    xb, yb, zb = p.CB
    sth, cth, sph, cph = np.sin(theta), np.cos(theta), np.sin(phi), np.cos(phi)
    G = np.stack([
        (W - B) * sth,
        -(W - B) * cth * sph,
        -(W - B) * cth * cph,
        -(yg * W - yb * B) * cth * cph + (zg * W - zb * B) * cth * sph,
        (zg * W - zb * B) * sth + (xg * W - xb * B) * cth * cph,
        -(xg * W - xb * B) * cth * sph - (yg * W - yb * B) * sth], axis=1)
    return -crb, -ca, mdv, G, H


def rhs6(p, angles, vel, rpm):
    """6DoF.py:396 with velCurrent = 0 and E = 0."""
    mcrb, mca, mdv, G, H = force_components6(p, angles, vel, rpm)
    return mcrb + mca + mdv - G + H


def _eta_dot6(angles, vel):
    J = coordinate_transform6(angles[:, 0], angles[:, 1], angles[:, 2])
    return np.einsum("nij,nj->ni", J, vel)


def derivs6_rpm(p, state, rpm):
    """6DoF.py:424-442 with the thruster rpm given directly."""
    state = np.atleast_2d(np.asarray(state, dtype=float))
    rpm = np.atleast_2d(np.asarray(rpm, dtype=float))
    angles, vel = state[:, 3:6], state[:, 6:12]
    acc = np.linalg.solve(p.mass_matrix(), rhs6(p, angles, vel, rpm).T).T
    return np.concatenate([_eta_dot6(angles, vel), acc], axis=1)


def derivs6_force(p, state, gcf, return_cv=False):
    """6DoF.py:406-442 with a stateless controller returning ``gcf``."""
    state = np.atleast_2d(np.asarray(state, dtype=float))
    gcf = np.atleast_2d(np.asarray(gcf, dtype=float))
    cv = allocate_thrust6(p, body_axes(state[:, 3:6]), gcf)
    d = derivs6_rpm(p, state, cv)
    return (d, cv) if return_cv else d


def derivs6_pid(p, t, state, ctrl, set_point, return_aux=False):
    """6DoF.py:406-442 with the reference's stateful PID (mutates ``ctrl``)."""
    state = np.atleast_2d(np.asarray(state, dtype=float))
    gcf = pid6_control(ctrl, set_point, state[:, 0:6], t)
    d, cv = derivs6_force(p, state, gcf, return_cv=True)
    return (d, gcf, cv) if return_aux else d


# ==========================================================================
# fixed-step RK4 (the integrator both sides of every parity test use)
# ==========================================================================
def rk4_substep(f, t, y, h):
    k1 = f(t, y)
    k2 = f(t + 0.5 * h, y + 0.5 * h * k1)
    k3 = f(t + 0.5 * h, y + 0.5 * h * k2)
    k4 = f(t + h, y + h * k3)
    return y + (h / 6.0) * (k1 + 2.0 * k2 + 2.0 * k3 + k4)


def rk4_advance(f, t0, y, dt, n_sub):
    h = dt / n_sub
    for j in range(n_sub):
        y = rk4_substep(f, t0 + j * h, y, h)
    return y


# ==========================================================================
# counter-based RNG used for auto-reset (Philox4x32-10; new in the build -
# the reference draws from the unseeded global numpy RNG, 6DoF.py:497-498)
# ==========================================================================
_PH_M0, _PH_M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_PH_W0, _PH_W1 = 0x9E3779B9, 0xBB67AE85
_MASK32 = np.uint64(0xFFFFFFFF)


def philox4x32(counter, key):
    """counter: [N, 4] uint32, key: (k0, k1) -> [N, 4] uint32."""
    c = [np.asarray(counter[:, i], dtype=np.uint64) for i in range(4)]
    k0, k1 = int(key[0]) & 0xFFFFFFFF, int(key[1]) & 0xFFFFFFFF
    for _ in range(10):
        p0 = _PH_M0 * c[0]
        p1 = _PH_M1 * c[2]
        hi0, lo0 = p0 >> np.uint64(32), p0 & _MASK32
        hi1, lo1 = p1 >> np.uint64(32), p1 & _MASK32
        c = [(hi1 ^ c[1] ^ np.uint64(k0)) & _MASK32, lo1, (hi0 ^ c[3] ^ np.uint64(k1)) & _MASK32, lo0]
        k0 = (k0 + _PH_W0) & 0xFFFFFFFF
        k1 = (k1 + _PH_W1) & 0xFFFFFFFF
    return np.stack(c, axis=1).astype(np.uint32)


def philox_uniform(seed, env_id, episode, n_values, stream=0):
    """n_values uniforms in [0,1) with 24-bit resolution (exact in fp32 and
    fp64) for each env: value j comes from word j%4 of block j//4, counter =
    (env_lo, env_hi, episode, stream*65536 + block), key = (seed_lo, seed_hi)."""
    env_id = np.asarray(env_id, dtype=np.uint64)
    episode = np.asarray(episode, dtype=np.uint64)
    n = env_id.shape[0]
    out = np.empty((n, n_values))
    key = (seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    for blk in range((n_values + 3) // 4):
        ctr = np.stack([env_id & _MASK32, env_id >> np.uint64(32), episode & _MASK32,
                        np.full(n, stream * 65536 + blk, dtype=np.uint64)], axis=1).astype(np.uint32)
        w = philox4x32(ctr, key)
        for j in range(4):
            if blk * 4 + j < n_values:
                out[:, blk * 4 + j] = (w[:, j] >> np.uint32(8)).astype(np.float64) * (1.0 / 16777216.0)
    return out


def normal_pair_u1(k1):
    """The radius uniform of the actor's Box-Muller pair from the 24-bit word k1, rounded as the kernel rounds it: a
    float32 add of 0.5, then the float32 multiply by 2^-24.  So u1 lies in [2^-25, 1]: for k1 >= 2^23 the add rounds to
    even, the upper half takes only 2^22 + 1 values, and k1 = 2^24 - 1 gives u1 = 1 exactly."""
    return (np.asarray(k1, dtype=np.uint32).astype(np.float32) + np.float32(0.5)) * np.float32(1.0 / 16777216.0)


def philox_normal_pair(seed, env_ids, step, blk, stream):
    """Pair ``blk`` (action dimensions 2 blk and 2 blk + 1) of the fused actor's standard normals; stream 7 is the
    policy's eps, stream 8 the squashed head's action noise.  Counter (env lo, env hi, step, stream * 65536 + blk), key
    (seed lo, seed hi).  ``step`` and ``blk`` broadcast against ``env_ids``.  Returns (k1, k2, z0, z1): the 24-bit words
    k1 = w.x >> 8 and k2 = w.y >> 8, and in fp64 z0 = r cos(theta), z1 = r sin(theta) with r = sqrt(-2 ln u1),
    u1 = ``normal_pair_u1(k1)``, theta = 2 pi k2 2^-24."""
    env_ids = np.atleast_1d(np.asarray(env_ids, dtype=np.uint64))
    step, blk = (np.broadcast_to(np.asarray(v, dtype=np.uint64), env_ids.shape) for v in (step, blk))
    ctr = np.stack([env_ids & _MASK32, env_ids >> np.uint64(32), step & _MASK32, np.uint64(stream * 65536) + blk],
                   axis=1).astype(np.uint32)
    w = philox4x32(ctr, (seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF))
    k1, k2 = w[:, 0] >> np.uint32(8), w[:, 1] >> np.uint32(8)
    r = np.sqrt(-2.0 * np.log(normal_pair_u1(k1).astype(np.float64)))
    theta = TWO_PI * (k2.astype(np.float64) * (1.0 / 16777216.0))
    return k1, k2, r * np.cos(theta), r * np.sin(theta)


# ==========================================================================
# 6DoF env (vectorised; 6DoF.py:445-594)
# ==========================================================================
MODE_RPM, MODE_FORCE, MODE_PID = 0, 1, 2


class Rov6EnvOracle:
    """Vectorised restatement of BlueROV2Heavy6DoFEnv with the integrator fixed
    to RK4 x n_sub.  ``mode``: 0 = action is 8 thruster rpm, 1 = action is a
    6-vector of earth-frame generalised forces, 2 = the reference's Gym
    semantics (action -> PID set-point, 6DoF.py:545-552).  Auto-reset (SB3
    VecEnv convention) is a build addition; with ``auto_reset=False`` the env
    behaves like the reference (state keeps integrating past ``done``)."""

    def __init__(self, n, params=None, dt=0.2, max_steps=250, n_sub=8, mode=MODE_PID, seed=0,
                 auto_reset=False, env_id0=0):
        self.n, self.p = n, (params or Rov6Params())
        self.dt, self.max_steps, self.n_sub, self.mode, self.seed = dt, max_steps, n_sub, mode, seed
        self.auto_reset = auto_reset
        self.env_ids = np.arange(env_id0, env_id0 + n, dtype=np.uint64)
        self.episode = np.zeros(n, dtype=np.uint64)
        self.fixed_sp = False
        self.Minv = np.linalg.inv(self.p.mass_matrix())

    # -- reset ------------------------------------------------------------
    def _draw(self, idx):
        """Random branch of reset (6DoF.py:493-501).  The reference's own line
        raises (shape (2,3) minus (2,)); the build defines it as the 3-component
        analogue of 3DoF.py:423: path = (U[0,1)^(2x3) - 0.5) * 10 and
        targetOrientation = U[0,1)^3 * 2 pi, drawn from Philox."""
        u = philox_uniform(self.seed, self.env_ids[idx], self.episode[idx], 9)
        path = (u[:, :6] - 0.5) * 10.
        orient = u[:, 6:9] * TWO_PI
        return path, orient

    def reset(self, initial_setpoint=None):
        n = self.n
        self.i_step = np.zeros(n, dtype=np.int64)
        self.time = np.zeros(n)
        self.state = np.zeros((n, 12))
        self.path = np.zeros((n, 6))
        if initial_setpoint is None:
            path, orient = self._draw(np.arange(n))
            self.path[:] = path
            self.set_point = np.concatenate([path[:, :3], orient], axis=1)
            self.fixed_sp = False
        else:
            sp = np.broadcast_to(np.asarray(initial_setpoint, dtype=float), (n, 6)).copy()
            self.path[:, :3] = sp[:, :3]
            self.path[:, 3:] = sp[:, :3]
            self.set_point = sp
            self.fixed_sp = True
        self.ctrl = pid6_new_state(n)
        self.gcf = np.zeros((n, 6))
        self.cv = np.zeros((n, 8))
        return self.observe()

    def _reset_rows(self, idx):
        self.episode[idx] += np.uint64(1)
        self.i_step[idx] = 0
        self.time[idx] = 0.
        self.state[idx] = 0.
        if not self.fixed_sp:
            path, orient = self._draw(idx)
            self.path[idx] = path
            self.set_point[idx] = np.concatenate([path[:, :3], orient], axis=1)
        for k in ("eOld", "eInt"):
            self.ctrl[k][idx] = 0.
        self.ctrl["has_old"][idx] = False
        self.ctrl["tOld"][idx] = 0.
        self.gcf[idx] = 0.
        self.cv[idx] = 0.

    # -- observation, 6DoF.py:467-483 (iWp is always 0) ------------------------
    def observe(self):
        s, L3 = self.state, self.p.Length * 3.
        obs = np.concatenate([
            (self.path[:, 0:3] - s[:, 0:3]) / L3,
            (self.path[:, 3:6] - s[:, 0:3]) / L3,
            angle_error(self.set_point[:, 3:6], s[:, 3:6]) / (45. / 180. * np.pi)], axis=1)
        return np.clip(obs, -1., 1.)

    # -- one derivative evaluation in the configured mode ------------------
    def _f(self, action):
        if self.mode == MODE_RPM:
            def f(t, y):
                self.cv = action
                return derivs6_rpm(self.p, y, action)
        elif self.mode == MODE_FORCE:
            def f(t, y):
                self.gcf = action
                d, self.cv = derivs6_force(self.p, y, action, return_cv=True)
                return d
        else:
            def f(t, y):
                d, self.gcf, self.cv = derivs6_pid(self.p, t, y, self.ctrl, self.set_point, return_aux=True)
                return d
        return f

    def step(self, action):
        action = np.atleast_2d(np.asarray(action, dtype=float))
        self.i_step += 1
        self.time = self.time + self.dt
        if self.mode == MODE_PID and not self.fixed_sp:  # 6DoF.py:545-552
            L2 = 2. * self.p.Length
            scale = np.array([L2, L2, L2, 45. / 180. * np.pi, 45. / 180. * np.pi, 45. / 180. * np.pi])
            self.set_point = action * scale + self.state[:, :6]
        y = rk4_advance(self._f(action), self.time - self.dt, self.state, self.dt, self.n_sub)
        y[:, 3:6] = np.mod(y[:, 3:6], TWO_PI)  # 6DoF.py:560
        self.state = y
        obs = self.observe()
        done = self.i_step >= self.max_steps
        reward = np.zeros(self.n)
        info = {}
        if self.auto_reset and done.any():
            idx = np.nonzero(done)[0]
            info["terminal_observation"] = obs.copy()
            self._reset_rows(idx)
            obs = self.observe()
        return obs, reward, done, info

    def history_row(self):
        """The 33 columns the reference appends per step, 6DoF.py:578-580."""
        return np.concatenate([self.time[:, None], self.state, self.gcf, self.cv, self.set_point], axis=1)


# ==========================================================================
# 3DoF model (3DoF.py:25-296) and env (3DoF.py:375-514)
# ==========================================================================
@dataclass
class Rov3Params:
    """3DoF.py:39-112.  Attribute names are the reference's."""
    rho_f: float = 1000.
    m: float = 11.4
    Length: float = 0.457
    Width: float = 0.338
    CB: np.ndarray = field(default_factory=lambda: np.zeros(3))
    CG: np.ndarray = field(default_factory=lambda: np.array([0., 0., 0.02]))
    I: np.ndarray = field(default_factory=lambda: np.diag([0.16, 0.16, 0.16]))
    Xudot: float = -5.5
    Yvdot: float = -12.7
    Nrdot: float = -0.12
    Yrdot: float = 0.
    Nvdot: float = 0.
    Xuu: float = -18.18
    Yvv: float = -21.66
    Yrr: float = 0.
    Ypp: float = 0.
    Nvv: float = 0.
    Nrr: float = -1.55
    Npp: float = 0.
    Xu: float = -4.03
    Yv: float = -6.22
    Yr: float = 0.
    Yp: float = 0.
    Nv: float = 0.
    Nr: float = -0.07
    Np: float = 0.
    D_thruster: float = 0.1
    alphaThruster: float = 45. / 180. * np.pi
    l_x: float = 0.156
    l_y: float = 0.111

    def __post_init__(self):
        self.dispVol = self.m / self.rho_f
        self.Kt_thruster = 40. / (1000. * (3500. / 60.) ** 2. * self.D_thruster ** 4.)
        A = np.array([[1., 1., -1., -1.], [1., -1., 1., -1.], [1., 1., 1., 1.]])
        A[0, :] = A[0, :] * np.cos(self.alphaThruster)
        A[1, :] = A[1, :] * np.sin(self.alphaThruster)
        A[2, :] = A[2, :] * np.sin(self.alphaThruster) * self.Length / 2.  # allocation uses Length/2 arms (3DoF.py:111)
        self.A = A
        self.Ainv = np.linalg.pinv(A)

    def mass_matrix(self):
        """3DoF.py:198-206."""
        m, xg, yg = self.m, self.CG[0], self.CG[1]
        Mrb = np.array([[m, 0., -m * yg], [0., m, m * xg], [-m * yg, m * xg, self.I[2, 2]]])
        return Mrb + -1. * np.diag([self.Xudot, self.Yvdot, self.Nrdot])


PID3_WINDUP = np.array([2., 2., 90. / 180. * np.pi])
PID3_KP = np.array([20., 20., 20.])
PID3_KI = np.array([0.1, 0.1, 0.1])
PID3_KD = np.array([5., 5., 0.5])
PID3_MAX = np.array([150., 150., 100.])


def pid3_new_state(n):
    """3DoF.py:33-35."""
    return {"eOld": np.zeros((n, 3)), "has_old": np.zeros(n, dtype=bool), "eInt": np.zeros((n, 3)), "tOld": np.zeros(n)}


def pid3_control(ctrl, set_point, pose, t):
    """3DoF.py:141-157 (mutates ``ctrl`` on every call)."""
    t = np.broadcast_to(np.asarray(t, dtype=float), pose.shape[:1])
    e = np.stack([set_point[:, 0] - pose[:, 0], set_point[:, 1] - pose[:, 1], angle_error(set_point[:, 2], pose[:, 2])], axis=1)
    e_old = np.where(ctrl["has_old"][:, None], ctrl["eOld"], e)
    dtc = t - ctrl["tOld"]
    _track_margin(ctrl, e, e_old, dtc)
    dedt = (e - e_old) / np.maximum(1e-9, dtc)[:, None]
    e_int = ctrl["eInt"] + 0.5 * (e_old + e) * dtc[:, None]
    e_int = np.where(np.abs(e) > PID3_WINDUP, 0., e_int)
    u = PID3_KP * e + PID3_KD * dedt + PID3_KI * e_int
    u = np.maximum(-PID3_MAX, np.minimum(PID3_MAX, u))
    ctrl["eOld"], ctrl["eInt"], ctrl["tOld"] = e, e_int, t.copy()
    ctrl["has_old"] = np.ones_like(ctrl["has_old"])
    return u


def thruster_model3(p, u, rpm):
    """3DoF.py:114-126 -> (Fthruster, Xthruster) with the jet-velocity drag augment."""
    F = p.rho_f * (rpm / 60.) ** 2. * np.sign(rpm) * p.D_thruster ** 4. * p.Kt_thruster
    u_jet = np.sqrt(np.abs(F) / (0.5 * p.rho_f * np.pi * p.D_thruster ** 2))
    den = np.maximum(1e-5, u_jet)
    d_cd = 0.56599 * np.exp(-7.60891 * np.abs(u) / den) + 0.05654 * np.exp(-0.89679 * np.abs(u) / den)
    X = d_cd * -0.5 * p.rho_f * np.abs(u) * u * p.dispVol ** (2. / 3.)
    return F, X


def allocate_thrust3(p, psi, control_values):
    """3DoF.py:159-168 -> (generalisedControlForces in the body frame, rpm)."""
    Xd = control_values[:, 0] * np.cos(psi) + control_values[:, 1] * np.sin(psi)
    Yd = -control_values[:, 0] * np.sin(psi) + control_values[:, 1] * np.cos(psi)
    gcf = np.stack([Xd, Yd, control_values[:, 2]], axis=1)
    cv = gcf @ p.Ainv.T
    cv = np.sign(cv) * np.sqrt(np.abs(cv) / (p.rho_f * p.D_thruster ** 4. * p.Kt_thruster)) * 60.
    return gcf, cv


def derivs3_rpm(p, state, rpm):
    """3DoF.py:170-296 from the limited-rpm stage on (rpm given: FP, AP, FS, AS)."""
    state = np.atleast_2d(np.asarray(state, dtype=float))
    rpm = np.atleast_2d(np.asarray(rpm, dtype=float))
    psi, u, v, r = state[:, 2], state[:, 3], state[:, 4], state[:, 5]
    m, xg, yg = p.m, p.CG[0], p.CG[1]
    lim = limit_rpm(rpm)
    F, X = thruster_model3(p, u[:, None], lim)
    ca, sa = np.cos(p.alphaThruster), np.sin(p.alphaThruster)
    Xh = X[:, 0] + X[:, 1] + X[:, 2] + X[:, 3] + (F[:, 0] + F[:, 1] - F[:, 2] - F[:, 3]) * ca
    Yh = (F[:, 0] - F[:, 1] + F[:, 2] - F[:, 3]) * sa
    Nh = np.sqrt(p.l_x ** 2. + p.l_y ** 2.) * (F[:, 0] + F[:, 1] + F[:, 2] + F[:, 3])  # true moment arms, 3DoF.py:263
    crb = np.stack([-m * (xg * r + v) * r, -m * (yg * r - u) * r, m * (xg * r + v) * u + m * (yg * r - u) * v], axis=1)
    cav = np.stack([p.Yvdot * v * r, -p.Xudot * u * r, -p.Yvdot * v * u + p.Xudot * u * v], axis=1)
    dv = -np.stack([(p.Xu + p.Xuu * np.abs(u)) * u,
                    (p.Yv + p.Yvv * np.abs(v)) * v + (p.Yr + p.Yrr * np.abs(r)) * r,
                    (p.Nv + p.Nvv * np.abs(v)) * v + (p.Nr + p.Nrr * np.abs(r)) * r], axis=1)
    RHS = -crb - (cav + dv) + np.stack([Xh, Yh, Nh], axis=1)
    acc = np.linalg.solve(p.mass_matrix(), RHS.T).T
    vel = np.stack([np.cos(psi) * u - np.sin(psi) * v, np.sin(psi) * u + np.cos(psi) * v, r], axis=1)
    return np.concatenate([vel, acc], axis=1)


def derivs3_pid(p, t, state, ctrl, set_point, return_aux=False):
    """BlueROV2Heavy3DoF.derivs, 3DoF.py:128-296 (mutates ``ctrl``)."""
    state = np.atleast_2d(np.asarray(state, dtype=float))
    control_values = pid3_control(ctrl, set_point, state[:, 0:3], t)
    gcf, cv = allocate_thrust3(p, state[:, 2], control_values)
    d = derivs3_rpm(p, state, cv)
    return (d, gcf, cv) if return_aux else d


class Rov3EnvOracle:
    """Vectorised BlueROV2Heavy3DoFEnv (3DoF.py:375-514) with RK4 x n_sub.
    mode 0: action = 4 rpm (build addition, stateless); 2: the reference's
    set-point semantics."""

    def __init__(self, n, params=None, dt=0.2, max_steps=250, n_sub=8, mode=MODE_PID, seed=0, auto_reset=False, env_id0=0):
        self.n, self.p = n, (params or Rov3Params())
        self.dt, self.max_steps, self.n_sub, self.mode, self.seed = dt, max_steps, n_sub, mode, seed
        self.auto_reset = auto_reset
        self.env_ids = np.arange(env_id0, env_id0 + n, dtype=np.uint64)
        self.episode = np.zeros(n, dtype=np.uint64)
        self.fixed_sp = False

    def _draw(self, idx):
        """3DoF.py:423-424: path = (U^(2x2) - 0.5) * 10, heading = U * 2 pi (Philox instead of np.random)."""
        u = philox_uniform(self.seed, self.env_ids[idx], self.episode[idx], 5)
        return (u[:, :4] - 0.5) * 10., u[:, 4] * TWO_PI

    def reset(self, initial_setpoint=None):
        n = self.n
        self.i_step = np.zeros(n, dtype=np.int64)
        self.time = np.zeros(n)
        self.state = np.zeros((n, 6))
        self.path = np.zeros((n, 4))
        if initial_setpoint is None:
            path, head = self._draw(np.arange(n))
            self.path[:] = path
            self.set_point = np.concatenate([path[:, :2], head[:, None]], axis=1)
            self.fixed_sp = False
        else:
            sp = np.broadcast_to(np.asarray(initial_setpoint, dtype=float), (n, 3)).copy()
            self.path[:, :2] = sp[:, :2]
            self.path[:, 2:] = sp[:, :2]
            self.set_point = sp
            self.fixed_sp = True
        self.ctrl = pid3_new_state(n)
        self.gcf = np.zeros((n, 3))
        self.cv = np.zeros((n, 4))
        return self.observe()

    def _reset_rows(self, idx):
        self.episode[idx] += np.uint64(1)
        self.i_step[idx] = 0
        self.time[idx] = 0.
        self.state[idx] = 0.
        if not self.fixed_sp:
            path, head = self._draw(idx)
            self.path[idx] = path
            self.set_point[idx] = np.concatenate([path[:, :2], head[:, None]], axis=1)
        for k in ("eOld", "eInt"):
            self.ctrl[k][idx] = 0.
        self.ctrl["has_old"][idx] = False
        self.ctrl["tOld"][idx] = 0.
        self.gcf[idx] = 0.
        self.cv[idx] = 0.

    def observe(self):
        """3DoF.py:397-409."""
        s, L3 = self.state, self.p.Length * 3.
        obs = np.concatenate([(self.path[:, 0:2] - s[:, 0:2]) / L3, (self.path[:, 2:4] - s[:, 0:2]) / L3,
                              (angle_error(self.set_point[:, 2], s[:, 2]) / (45. / 180. * np.pi))[:, None]], axis=1)
        return np.clip(obs, -1., 1.)

    def step(self, action):
        action = np.atleast_2d(np.asarray(action, dtype=float))
        self.i_step += 1
        self.time = self.time + self.dt
        if self.mode == MODE_PID and not self.fixed_sp:  # 3DoF.py:469-472
            L2 = 2. * self.p.Length
            self.set_point = action * np.array([L2, L2, 45. / 180. * np.pi]) + self.state[:, :3]
        if self.mode == MODE_RPM:
            def f(t, y):
                self.cv = action
                return derivs3_rpm(self.p, y, action)
        else:
            def f(t, y):
                d, self.gcf, self.cv = derivs3_pid(self.p, t, y, self.ctrl, self.set_point, return_aux=True)
                return d
        y = rk4_advance(f, self.time - self.dt, self.state, self.dt, self.n_sub)
        y[:, 2] = np.mod(y[:, 2], TWO_PI)  # 3DoF.py:480
        self.state = y
        obs = self.observe()
        done = self.i_step >= self.max_steps
        info = {}
        if self.auto_reset and done.any():
            info["terminal_observation"] = obs.copy()
            self._reset_rows(np.nonzero(done)[0])
            obs = self.observe()
        return obs, np.zeros(self.n), done, info

    def history_row(self):
        """17 columns, 3DoF.py:498-507."""
        return np.concatenate([self.time[:, None], self.state, self.gcf, self.cv, self.set_point], axis=1)


# ==========================================================================
# legacy: ReconstructedFlow.scale / interp (legacy/flowGenerator.py:53-136)
# ==========================================================================
class FlowOracle:
    """Holds ``baseFlowData`` [Nt, Ny, Nx, 3] (u/Uinf, v/Uinf, Cp) on a uniform
    grid and reproduces ``scale`` and ``interp``.  The SPOD reconstruction of
    ``__init__`` (legacy/flowGenerator.py:15-23) needs blobs that are absent
    from the reference checkout; callers supply the base field."""

    def __init__(self, base_field, base_dx=0.005, base_dy=0.005, base_dt=0.002):
        self.baseFlowData = np.asarray(base_field, dtype=float)
        self.baseDx, self.baseDy, self.baseDt = float(base_dx), float(base_dy), float(base_dt)
        self.scale(1., 1., 1.)

    @staticmethod
    def reconstruct(modes, coeffs, lt_mean):
        """legacy/flowGenerator.py:20-23: ``baseFlowData[t] = Re(modes @ coeffs[:, t]) + lt_mean``, one time level after
        the other like the reference.  modes [Ny, Nx, 3, K], coeffs [K, Nt] (complex or real) -> [Nt, Ny, Nx, 3]."""
        modes, coeffs = np.asarray(modes), np.asarray(coeffs)
        base = np.zeros((coeffs.shape[1],) + modes.shape[:-1])
        for it in range(base.shape[0]):
            base[it] = np.real(np.matmul(modes, coeffs[:, it])) + lt_mean
        return base

    def intensity(self):
        """legacy/flowGenerator.py:47-51 (evaluated on ``flowData`` after ``scale(1, 1, 1)``): uPrime, vPrime, TI, baseTI."""
        f = self.baseFlowData
        up = np.sqrt(np.sum((f[:, :, :, 0] - 1.) ** 2., axis=0) / f.shape[0])
        vp = np.sqrt(np.sum((f[:, :, :, 1] - 0.) ** 2., axis=0) / f.shape[0])
        ti = np.sqrt(0.5 * (up + vp))
        return up, vp, ti, ti[ti.shape[0] // 2, ti.shape[1] // 2]

    def scale(self, sizeScale, velocityScale, turbScale, translate=(0, 0)):
        """legacy/flowGenerator.py:53-95.  ``translate`` only moves the plotting
        coordinates; ``interp`` ignores it (bug-compatible)."""
        self.dx = self.baseDx * sizeScale
        self.dy = self.baseDy * sizeScale
        f = self.baseFlowData.copy()
        f[..., 0] *= velocityScale
        f[..., 1] *= velocityScale
        f[..., 0] = (f[..., 0] - velocityScale) * turbScale + velocityScale
        f[..., 1] = (f[..., 1] - 0.) * turbScale
        f[..., 2] /= max(1e-6, (velocityScale * turbScale) ** 2.)
        self.flowData = f
        self.dt = self.baseDt * sizeScale / max(1e-6, velocityScale)
        self.time = np.array([i * self.dt for i in range(f.shape[0])])

    def interp(self, time, xy):
        """legacy/flowGenerator.py:97-136, vectorised: time [N], xy [N, 2] -> [N, 3].
        Indices are clamped to the grid, weights are NOT (extrapolation)."""
        time = np.atleast_1d(np.asarray(time, dtype=float))
        xy = np.atleast_2d(np.asarray(xy, dtype=float))
        nt, ny, nx, _ = self.flowData.shape
        tt, xx, yy = time / self.dt, xy[:, 0] / self.dx, xy[:, 1] / self.dy
        kk = np.minimum(nt - 2, np.maximum(0, np.floor(tt).astype(np.int64)))
        ii = np.minimum(nx - 2, np.maximum(0, np.floor(xx).astype(np.int64)))
        jj = np.minimum(ny - 2, np.maximum(0, np.floor(yy).astype(np.int64)))
        wt, wx, wy = tt - kk, xx - ii, yy - jj
        f = self.flowData
        res = np.zeros((time.shape[0], f.shape[3]))
        for dk, ct in ((0, 1. - wt), (1, wt)):
            c00, c01 = f[kk + dk, jj, ii], f[kk + dk, jj, ii + 1]
            c10, c11 = f[kk + dk, jj + 1, ii], f[kk + dk, jj + 1, ii + 1]
            row0 = c00 * (1. - wx)[:, None] + c01 * wx[:, None]       # F[jj, ii:ii+2] . xx
            row1 = c10 * (1. - wx)[:, None] + c11 * wx[:, None]
            res += ((1. - wy)[:, None] * row0 + wy[:, None] * row1) * ct[:, None]
        return res


# ==========================================================================
# legacy: AuvEnv (legacy/verySimpleAuv.py:76-410)
# ==========================================================================
class AuvEnvOracle:
    """Vectorised AuvEnv.  Random draws of ``reset`` come from Philox in the
    reference's order (8 coefficient multipliers, 3 actuation multipliers,
    position x/y, heading, headingTarget, flow time offset -
    legacy/verySimpleAuv.py:222-245); ``set_initial`` installs values drawn by
    the reference's own RNG for the golden-vector tests."""

    def __init__(self, n, flow, dt=0.02, noiseMagCoeffs=0.0, noiseMagActuation=0.0, stopOnBoundsExceeded=True,
                 max_steps=250, seed=0, auto_reset=False, env_id0=0):
        self.n, self.flow, self.dt = n, flow, dt
        self.noiseMagCoeffs, self.noiseMagActuation = noiseMagCoeffs, noiseMagActuation
        self.stop_on_bounds, self.max_steps = stopOnBoundsExceeded, max_steps
        self.seed, self.auto_reset = seed, auto_reset
        self.env_ids = np.arange(env_id0, env_id0 + n, dtype=np.uint64)
        self.episode = np.zeros(n, dtype=np.uint64)
        # legacy/verySimpleAuv.py:110-127
        self.xMinMax, self.yMinMax = [-1, 1], [-1, 1]
        self.m, self.Izz = 11.4, 0.16
        self.Xuu, self.Yvv, self.Nrr = -18.18 * 2.21, -21.66 * 4.87, -1.55
        self.Xu, self.Yv, self.Nr = -4.03 * 2.21, -6.22 * 4.87, -0.07
        self.maxForce, self.maxMoment = 150., 20.

    def _draw(self, idx, apply_noise=True):
        u = philox_uniform(self.seed, self.env_ids[idx], self.episode[idx], 16)
        mults = np.ones((len(idx), 11))
        if apply_noise:
            mults[:, :8] = 1. + self.noiseMagCoeffs / 2. - u[:, :8] * self.noiseMagCoeffs
            mults[:, 8:] = 1. + self.noiseMagActuation / 2. - u[:, 8:11] * self.noiseMagActuation
        pos = (u[:, 11:13] - 0.5) * 0.5 * np.array([self.xMinMax[1] - self.xMinMax[0], self.yMinMax[1] - self.yMinMax[0]])
        heading, target = u[:, 13] * TWO_PI, u[:, 14] * TWO_PI
        offset = u[:, 15] * self.flow.time[self.flow.time.shape[0] // 4]
        return mults, pos, heading, target, offset

    def _install(self, idx, mults, pos, heading, target, offset):
        self.mults[idx], self.position[idx], self.heading[idx] = mults, pos, heading
        self.heading_target[idx], self.t_offset[idx] = target, offset
        self.velocities[idx] = 0.
        self.time[idx] = 0.
        self.i_step[idx] = 0
        self.recent[idx] = 0.
        self.n_recent[idx] = 0
        # first dataToState after reset initialises herr_o / perr_o (legacy/verySimpleAuv.py:158-160)
        self.perr_o[idx] = -self.position[idx]
        self.herr_o[idx] = angle_error(self.heading_target[idx], self.heading[idx])

    def reset(self, applyNoise=True):
        n = self.n
        self.mults, self.position, self.heading = np.ones((n, 11)), np.zeros((n, 2)), np.zeros(n)
        self.heading_target, self.t_offset = np.zeros(n), np.zeros(n)
        self.velocities, self.time, self.i_step = np.zeros((n, 3)), np.zeros(n), np.zeros(n, dtype=np.int64)
        self.recent, self.n_recent = np.zeros((n, 10, 3)), np.zeros(n, dtype=np.int64)
        self.perr_o, self.herr_o = np.zeros((n, 2)), np.zeros(n)
        idx = np.arange(n)
        self._install(idx, *self._draw(idx, applyNoise))
        return self.observe()

    def set_initial(self, mults, pos, heading, target, offset):
        self._install(np.arange(self.n), np.asarray(mults, float), np.asarray(pos, float), np.asarray(heading, float),
                      np.asarray(target, float), np.asarray(offset, float))
        return self.observe()

    def observe(self):
        """dataToState V3, legacy/verySimpleAuv.py:147-214 (uses herr_o / perr_o of the previous call)."""
        perr = -self.position
        herr = angle_error(self.heading_target, self.heading)
        c = lambda x: np.minimum(1., np.maximum(-1., x))
        return np.stack([c(perr[:, 0]), c(perr[:, 1]), c(herr / (45. / 180. * np.pi)), c(herr - self.herr_o),
                         c(perr[:, 0] - self.perr_o[:, 0]), c(perr[:, 1] - self.perr_o[:, 1]),
                         c(self.velocities[:, 0]), c(self.velocities[:, 1]), c(self.velocities[:, 2]),
                         np.zeros(self.n), np.zeros(self.n)], axis=1)

    def _errors(self, position, heading):
        """perr, herr of legacy/verySimpleAuv.py:344-346 (positionTarget = 0)."""
        return -position, angle_error(self.heading_target, heading)

    def step(self, action):
        """legacy/verySimpleAuv.py:264-410."""
        action = np.atleast_2d(np.asarray(action, dtype=float))
        n = self.n
        self.i_step += 1
        self.time = self.time + self.dt
        done = self.i_step >= self.max_steps
        self.recent = np.concatenate([action[:, None, :], self.recent[:, :9]], axis=1)  # deque.appendleft, maxlen 10
        self.n_recent = np.minimum(10, self.n_recent + 1)
        mm = self.mults
        Fset = action[:, :2] * self.maxForce * mm[:, 8:10]
        Nset = action[:, 2] * self.maxMoment * mm[:, 10]
        c, s = np.cos(self.heading), np.sin(self.heading)
        vel_current = self.flow.interp(self.time + self.t_offset, self.position)[:, :2]
        d = self.velocities[:, :2] - vel_current
        vr0, vr1 = c * d[:, 0] + s * d[:, 1], -s * d[:, 0] + c * d[:, 1]          # inverse of the planar rotation
        r = self.velocities[:, 2]
        Fh = np.stack([(self.Xu * mm[:, 5] + self.Xuu * mm[:, 2] * np.abs(vr0)) * vr0,
                       (self.Yv * mm[:, 6] + self.Yvv * mm[:, 3] * np.abs(vr1)) * vr1,
                       (self.Nr * mm[:, 7] + self.Nrr * mm[:, 4] * np.abs(r)) * r], axis=1)
        Fh = np.stack([c * Fh[:, 0] - s * Fh[:, 1], s * Fh[:, 0] + c * Fh[:, 1], Fh[:, 2]], axis=1)
        acc = np.stack([(Fh[:, 0] + Fset[:, 0]) / (self.m * mm[:, 0]), (Fh[:, 1] + Fset[:, 1]) / (self.m * mm[:, 0]),
                        (Fh[:, 2] + Nset) / (self.Izz * mm[:, 1])], axis=1)
        # explicit Euler; position advances with the OLD velocity (legacy/verySimpleAuv.py:321-326)
        position = self.position + self.velocities[:, :2] * self.dt
        heading = np.mod(self.heading + self.velocities[:, 2] * self.dt, TWO_PI)
        velocities = self.velocities + acc * self.dt
        self.position, self.heading, self.velocities = position, heading, velocities
        obs = self.observe()
        bonus = np.zeros(n)
        out_x = (position[:, 0] < self.xMinMax[0]) | (position[:, 0] > self.xMinMax[1])
        out_y = (position[:, 1] < self.yMinMax[0]) | (position[:, 1] > self.yMinMax[1])
        bonus += -100. * out_x + -100. * out_y
        if self.stop_on_bounds:
            done = done | out_x | out_y
        perr, herr = self._errors(position, heading)
        self.herr_o, self.perr_o = herr, perr
        # population std of the <= 10 most recent actions, mean over the 3 components (:353-355)
        cnt = self.n_recent[:, None, None]
        valid = (np.arange(10)[None, :, None] < cnt)
        mean = (self.recent * valid).sum(axis=1) / self.n_recent[:, None]
        var = (((self.recent - mean[:, None, :]) ** 2.) * valid).sum(axis=1) / self.n_recent[:, None]
        rms_ac = np.sqrt(var).mean(axis=1)
        herr_deg = np.abs(herr / np.pi * 180.)
        terms = np.stack([np.exp(-5. * np.sqrt(perr[:, 0] ** 2 + perr[:, 1] ** 2)),
                          np.where(np.abs(herr) < np.pi / 2., np.exp(-0.1 * herr_deg), -np.exp(-0.1 * (180. - herr_deg))),
                          np.exp(-0.6 * rms_ac), -0.1 * np.sum(action ** 2., axis=1) / 3., bonus], axis=1)
        reward = terms.sum(axis=1)
        self.last = {"Fhydro": Fh, "Fset": Fset, "Nset": Nset, "vel_current": vel_current, "rmsAc": rms_ac, "terms": terms}
        info = {}
        if self.auto_reset and done.any():
            idx = np.nonzero(done)[0]
            info["terminal_observation"] = obs.copy()
            self.episode[idx] += np.uint64(1)
            self._install(idx, *self._draw(idx, True))
            obs[idx] = self.observe()[idx]  # only the reset envs: the others keep the obs taken before herr_o / perr_o moved on
        return obs, reward, done, info


# ==========================================================================
# action producers in front of the env step: LOS navigation (3DoF.py:517-607)
# ==========================================================================
def line_of_sight(p0, p1, rnav):
    """``lineOfSight`` (3DoF.py:517-583), vectorised: p0, p1 [N, 2] way-points relative to the vehicle,
    rnav [N] or scalar -> target point [N, 2].  Branch order and NaN behaviour (all comparisons false) as
    in the reference."""
    p0 = np.atleast_2d(np.asarray(p0, dtype=float)); p1 = np.atleast_2d(np.asarray(p1, dtype=float))
    rnav = np.broadcast_to(np.asarray(rnav, dtype=float), p0.shape[:1])
    with np.errstate(all="ignore"):
        d_to_wp = np.sqrt(np.sum(p1 ** 2., axis=1))
        path = p1 - p0
        d_seg = np.sqrt(np.sum(path ** 2., axis=1))
        p_hat = path / d_seg[:, None]                      # np.linalg.norm(pathVec): same value as dSegment
        det = p0[:, 0] * p1[:, 1] - p1[:, 0] * p0[:, 1]
        delta = rnav ** 2. * d_seg ** 2. - det ** 2.
        # delta < 0: project the vehicle onto the segment
        d_along = np.sum(-p0 * p_hat, axis=1)
        t_neg = np.where((d_along > d_seg)[:, None], p1, np.where((d_along < 0)[:, None], p0, p0 + d_along[:, None] * p_hat))
        # delta >= 0: the two intersections of the LOS circle with the line
        sy = np.sign(path[:, 1]); sy = np.where(np.abs(sy) < 1e-12, 1., sy)
        den = np.maximum(1e-6, d_seg) ** 2.
        sq = np.sqrt(delta)
        pp0 = np.stack([(det * path[:, 1] + sy * path[:, 0] * sq) / den, (-det * path[:, 0] + np.abs(path[:, 1]) * sq) / den], axis=1)
        pp1 = np.stack([(det * path[:, 1] - sy * path[:, 0] * sq) / den, (-det * path[:, 0] - np.abs(path[:, 1]) * sq) / den], axis=1)
        s0 = np.sum(p_hat * (pp0 - p0), axis=1) / np.maximum(1e-6, d_seg)
        s1 = np.sum(p_hat * (pp1 - p0), axis=1) / np.maximum(1e-6, d_seg)
        n0, n1 = np.sqrt(np.sum(p0 ** 2., axis=1)), np.sqrt(np.sum(p1 ** 2., axis=1))
        t_pos = np.where(((s0 >= 0.) & (s0 <= 1.) & (s0 > s1))[:, None], pp0,
                         np.where(((s1 >= 0.) & (s1 <= 1.))[:, None], pp1, np.where((n1 < n0)[:, None], p1, p0)))
        # the reference tests `delta < 0` and `delta >= 0` separately: NaN delta leaves targetPoint unassigned
        # (UnboundLocalError upstream); the build returns NaN there
        t_far = np.where((delta < 0)[:, None], t_neg, np.where((delta >= 0)[:, None], t_pos, np.nan))
        return np.where((d_to_wp < rnav)[:, None], p1, t_far)


def los_navigation_predict(obs, rnav=0.5):
    """``LOSNavigation.predict`` (3DoF.py:586-607): obs [N, 5] -> actions [N, 3] = (target point, heading error)."""
    obs = np.atleast_2d(np.asarray(obs, dtype=float))
    tp = line_of_sight(obs[:, 0:2], obs[:, 2:4], rnav)
    return np.concatenate([tp, obs[:, 4:5]], axis=1)


# ==========================================================================
# legacy: AuvEnvCyl (legacy/verySimpleAuv_cyl.py:22-345) - way-point following around a cylinder
# ==========================================================================
def cyl_waypoints(Rcyl=1.33, xCyl=(2.5, 0.)):
    """legacy/verySimpleAuv_cyl.py:29-41 -> ([21, 3] way-points x, y, target heading; switch threshold)."""
    Rwp = Rcyl * 1.3
    t = np.linspace(-30, 30, 21) * np.pi / 180.
    return np.vstack([-Rwp * np.cos(t) + xCyl[0], Rwp * np.sin(t) + xCyl[1], -t]).T, Rcyl * 0.05


class AuvCylEnvOracle(AuvEnvOracle):
    """Differences to AuvEnv: position / heading targets follow a way-point list (the index ``iWp`` advances when
    the vehicle is within ``wpThreshold`` and is NOT reset between episodes - it lives in ``__init__`` only,
    :41), V0 observation scaling (:99-112), bounds +-2 (:69-70), 1200-step episodes (:44), and reset draws no
    heading target (:155-160), i.e. 15 uniforms instead of 16."""

    def __init__(self, n, flow, max_steps=1200, **kw):
        super().__init__(n, flow, max_steps=max_steps, **kw)
        self.xMinMax, self.yMinMax = [-2, 2], [-2, 2]
        self.waypoints, self.wp_threshold = cyl_waypoints()
        self.i_wp = np.zeros(n, dtype=np.int64)

    def _draw(self, idx, apply_noise=True):
        u = philox_uniform(self.seed, self.env_ids[idx], self.episode[idx], 15)
        mults = np.ones((len(idx), 11))
        if apply_noise:
            mults[:, :8] = 1. + self.noiseMagCoeffs / 2. - u[:, :8] * self.noiseMagCoeffs
            mults[:, 8:] = 1. + self.noiseMagActuation / 2. - u[:, 8:11] * self.noiseMagActuation
        pos = (u[:, 11:13] - 0.5) * 0.5 * np.array([self.xMinMax[1] - self.xMinMax[0], self.yMinMax[1] - self.yMinMax[0]])
        heading = u[:, 13] * TWO_PI
        offset = u[:, 14] * self.flow.time[self.flow.time.shape[0] // 4]
        return mults, pos, heading, self.waypoints[self.i_wp[idx], 2], offset

    def _install(self, idx, mults, pos, heading, target, offset):
        super()._install(idx, mults, pos, heading, self.waypoints[self.i_wp[idx], 2], offset)
        self.perr_o[idx] = self.waypoints[self.i_wp[idx], :2] - self.position[idx]

    def observe(self):
        """legacy/verySimpleAuv_cyl.py:84-115 (V0 scaling)."""
        perr = self.waypoints[self.i_wp, :2] - self.position
        herr = angle_error(self.heading_target, self.heading)
        c = lambda x: np.minimum(1., np.maximum(-1., x))
        return np.stack([c(perr[:, 0] / 0.2), c(perr[:, 1] / 0.2), c(herr / (45. / 180. * np.pi)),
                         c((herr - self.herr_o) / (2. / 180 * np.pi)), c((perr[:, 0] - self.perr_o[:, 0]) / 0.025),
                         c((perr[:, 1] - self.perr_o[:, 1]) / 0.025), c(self.velocities[:, 0] / 0.2), c(self.velocities[:, 1] / 0.2),
                         c(self.velocities[:, 2] / (30. / 180. * np.pi)), np.zeros(self.n), np.zeros(self.n)], axis=1)

    def _errors(self, position, heading):
        """perr / herr against the CURRENT way-point, then the way-point switch (:243-254)."""
        perr = self.waypoints[self.i_wp, :2] - position
        herr = angle_error(self.heading_target, heading)
        reached = np.sqrt(perr[:, 0] ** 2 + perr[:, 1] ** 2) < self.wp_threshold
        self.i_wp = np.where(reached, np.minimum(self.waypoints.shape[0] - 1, self.i_wp + 1), self.i_wp)
        self.heading_target = self.waypoints[self.i_wp, 2].copy()
        return perr, herr


# ==========================================================================
# legacy: CustomReplayBuffer.add (legacy/main_02_sbl_contrib_customBuffer.py:57-160)
# ==========================================================================
class ReplayBufferOracle:
    """The symmetry-augmenting replay buffer.  Storage as set up by stable_baselines3's ``ReplayBuffer.__init__`` (the
    base class, not in the reference checkout; 2.x ``common/buffers.py``): ``max(buffer_size // n_envs, 1)`` slots of
    ``n_envs`` transitions.  ``add`` follows main_02...:75-160 line by line."""
    T_OBS = np.array([[1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1], [-1, -1, 1, 1, -1, -1, -1, -1, 1, 1, 1], [-1, 1, 1, 1, -1, 1, -1, 1, 1, 1, 1],
                      [1, -1, 1, 1, 1, -1, 1, -1, 1, 1, 1], [1, 1, -1, 1, 1, 1, 1, 1, -1, 1, 1]], dtype=float)   # :107-118
    T_ACT = np.array([[1, 1, 1], [-1, -1, 1], [-1, 1, 1], [1, -1, 1], [1, 1, -1]], dtype=float)                    # :119-125

    def __init__(self, buffer_size, n_envs, dtype=np.float32):
        self.n_envs = int(n_envs)
        self.buffer_size = max(int(buffer_size) // self.n_envs, 1)
        z = lambda *shape: np.zeros(shape, dtype=dtype)
        self.observations, self.next_observations = z(self.buffer_size, n_envs, 11), z(self.buffer_size, n_envs, 11)
        self.actions, self.rewards = z(self.buffer_size, n_envs, 3), z(self.buffer_size, n_envs)
        self.dones, self.timeouts = z(self.buffer_size, n_envs), z(self.buffer_size, n_envs)
        self.pos, self.full, self.nRollovers = 0, False, 0

    def add(self, obs, next_obs, action, reward, done, timeouts=None):
        for i in range(5):
            if self.nRollovers > 2 and i != 0:      # :143-145: no mirror images after the third roll-over
                continue
            p = self.pos
            self.observations[p] = np.asarray(obs) * self.T_OBS[i]
            self.next_observations[p] = np.asarray(next_obs) * self.T_OBS[i]
            self.actions[p] = np.asarray(action) * self.T_ACT[i]
            self.rewards[p], self.dones[p] = reward, done
            self.timeouts[p] = 0 if timeouts is None else timeouts
            self.pos += 1
            if self.pos == self.buffer_size:        # :155-158
                self.full, self.pos = True, 0
                self.nRollovers += 1
