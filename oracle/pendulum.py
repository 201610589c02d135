"""Oracle: pendulum dynamics and its analytic linearisation (test infrastructure).

step()       follows env_dx/pendulum.py:65-102 (PendulumDx.forward, `simple` and full models)
linearize()  replaces mpc/approximate.py:77-119 (n_state chainer.grad calls per timestep)
             by the closed-form Jacobian; F_t = [R S], f_t = x' - R x - S u (:111-114).
             F.clip's sub-gradient at |u| == max_torque is taken as 1 (inclusive) -
             parity unpinned there (Chainer 6.3.0 source is not in the reference tree).
"""
import numpy as np

DT = 0.05
MAX_TORQUE = 2.0


def step(x, u, params=(10.0, 1.0, 1.0), dt=DT, max_torque=MAX_TORQUE):
    """x[B,3]=(cos th, sin th, dth), u[B,1] -> x'[B,3]; dt, max_torque = PendulumDx.dt / .max_torque."""
    g, m, l = params[0], params[1], params[2]
    simple = len(params) == 3
    uc = np.clip(u, -max_torque, max_torque)[:, 0]
    cos_th, sin_th, dth = x[:, 0], x[:, 1], x[:, 2]
    th = np.arctan2(sin_th, cos_th)
    if simple:
        newdth = dth + dt * (-3.0 * g / (2.0 * l) * (-sin_th) + 3.0 * uc / (m * l ** 2))
    else:
        d, b = params[3], params[4]
        newdth = dth + dt * (-3.0 * g / (2.0 * l) * (-np.sin(th + b)) + 3.0 * uc / (m * l ** 2) - d * th)
    newth = th + newdth * dt
    return np.stack((np.cos(newth), np.sin(newth), newdth), axis=1)


def jacobian(x, u, params=(10.0, 1.0, 1.0), dt=DT, max_torque=MAX_TORQUE):
    """Returns (x', R[B,3,3], S[B,3,1]) for the `simple` model."""
    assert len(params) == 3
    g, m, l = params
    B = x.shape[0]
    c, s, w = x[:, 0], x[:, 1], x[:, 2]
    r2 = c * c + s * s
    dth_dc, dth_ds = -s / r2, c / r2                      # d atan2(s,c)
    a = 3.0 * g / (2.0 * l)
    bu = 3.0 / (m * l ** 2)
    uraw = u[:, 0]
    inside = (uraw >= -max_torque) & (uraw <= max_torque)
    uc = np.clip(uraw, -max_torque, max_torque)
    th = np.arctan2(s, c)
    nw = w + dt * (a * s + bu * uc)
    nth = th + nw * dt
    # d nw / d(c,s,w,u)
    dnw = np.stack((np.zeros(B), dt * a * np.ones(B), np.ones(B), dt * bu * inside), axis=1)
    dnth = np.stack((dth_dc, dth_ds, np.zeros(B), np.zeros(B)), axis=1) + dt * dnw
    J = np.stack((-np.sin(nth)[:, None] * dnth, np.cos(nth)[:, None] * dnth, dnw), axis=1)  # [B,3,4]
    xn = np.stack((np.cos(nth), np.sin(nth), nw), axis=1)
    return xn, J[:, :, :3], J[:, :, 3:]


def linearize(x0, u, params=(10.0, 1.0, 1.0), dt=DT, max_torque=MAX_TORQUE):
    """Roll out from x0 under u[T,B,1]; returns (F[T-1,B,3,4], f[T-1,B,3])."""
    T = u.shape[0]
    Fs, fs = [], []
    x = x0
    for t in range(T - 1):
        xn, R, S = jacobian(x, u[t], params, dt, max_torque)
        Fs.append(np.concatenate((R, S), axis=2))
        fs.append(xn - (R @ x[:, :, None])[:, :, 0] - (S @ u[t][:, :, None])[:, :, 0])
        x = xn
    return np.stack(Fs), np.stack(fs)
