"""ORACLE — test infrastructure only.  numpy restatements of the reference's vehicle models
(/root/reference/Vehicle_Dynamics/vehicle_models.py):
  dynamics_model     Vehicle_Dynamics.get_dynamics_model (:52-340): Pacejka lateral tyres, analytic Jacobians,
                     forward-Euler discretisation
  dynamics_step      Vehicle_Dynamics.update_dynamics_model (:343-482): one explicit Euler step of the same nonlinear model
  kinematics_model   Vehicle_Kinematics.get_kinematics_model (:835-863)
  kinematics_step    Vehicle_Kinematics.update_kinematics_model (:866-882)
Checked against the reference itself through tests/golden/vehicle_models.npz (tests/test_oracle.py)."""
import math

import numpy as np


def _dynamics_terms(x, u, m, l_f, l_r, width, length, C_d, A_f, C_roll):
    """The low-speed guards, the tyre and longitudinal forces and the state derivative f(x, u) that both
    get_dynamics_model and update_dynamics_model evaluate; the guards modify the state and input they start from."""
    x = np.array(x, dtype=np.float64).ravel().copy(); u = np.array(u, dtype=np.float64).ravel().copy()
    wb = l_f + l_r
    Iz = 1 / 12 * m * (width ** 2 + length ** 2)
    roh = 1.23
    a = [-22.1, 1011, 1078, 1.82, 0.208]
    C = 1.30

    def tyre(Fz):
        D = a[0] * Fz ** 2 + a[1] * Fz
        BCD = a[2] * math.sin(a[3] * math.atan(a[4] * Fz))
        return D, BCD / (C * D) * 180 / np.pi

    Df, Bf = tyre(9.81 * (m * l_r / wb) * 0.001)
    Dr, Br = tyre(9.81 * (m * l_f / wb) * 0.001)
    if 0 <= x[3] < 0.5:                                   # vehicle_models.py:143-150 (:416-424)
        x[4] = 0.; x[5] = 0.; u[0] = 0.
        if x[3] < 0.3:
            x[3] = 0.3
    if -0.5 < x[3] < 0:                                   # :152-159 (:426-433)
        x[4] = 0.; x[5] = 0.; u[0] = 0.
        if x[3] > -0.3:
            x[3] = -0.3
    yaw, vx, vy, wz = x[2], x[3], x[4], x[5]
    st, acc = u
    af = -math.atan2(l_f * wz + vy, vx) + st
    ar = -math.atan2(-l_r * wz + vy, vx)
    Fyf = Df * math.sin(C * math.atan(Bf * af)); Fyr = Dr * math.sin(C * math.atan(Br * ar))
    sg = np.sign(vx)
    Fxf = m * acc - 0.5 * roh * C_d * A_f * vx ** 2 * sg - C_roll * m * 9.81 * sg
    sy, cy, ss, cs = math.sin(yaw), math.cos(yaw), math.sin(st), math.cos(st)
    f = np.array([vx * cy - vy * sy, vy * cy + vx * sy, wz,
                  1. / m * (Fxf * cs - Fyf * ss + m * vy * wz),
                  1. / m * (Fxf * ss + Fyr + Fyf * cs - m * vx * wz),
                  1. / Iz * (Fxf * l_f * ss + Fyf * l_f * cs - Fyr * l_r)])
    return dict(x=x, u=u, Iz=Iz, roh=roh, C=C, Df=Df, Bf=Bf, Dr=Dr, Br=Br, af=af, ar=ar, Fyf=Fyf, Fyr=Fyr, Fxf=Fxf,
                sy=sy, cy=cy, ss=ss, cs=cs, f=f)


def dynamics_model(x, u, m=1300., l_f=1.25, l_r=1.40, width=1.78, length=4.25, C_d=0.34, A_f=2.0, C_roll=0.015, dt=0.02):
    t = _dynamics_terms(x, u, m, l_f, l_r, width, length, C_d, A_f, C_roll)
    x, u, Iz, C = t["x"], t["u"], t["Iz"], t["C"]
    Df, Bf, Dr, Br, af, ar = t["Df"], t["Bf"], t["Dr"], t["Br"], t["af"], t["ar"]
    Fyf, Fxf, sy, cy, ss, cs = t["Fyf"], t["Fxf"], t["sy"], t["cy"], t["ss"], t["cs"]
    vx, vy, wz = x[3], x[4], x[5]
    dFx = -t["roh"] * C_d * A_f * vx
    kf = (Bf * C * Df * math.cos(C * math.atan(Bf * af))) / (1 + Bf ** 2 * af ** 2)
    kr = (Br * C * Dr * math.cos(C * math.atan(Br * ar))) / (1 + Br ** 2 * ar ** 2)
    nf, nr = l_f * wz + vy, -l_r * wz + vy
    df, dr = nf ** 2 + vx ** 2, nr ** 2 + vx ** 2
    dFyf = np.array([kf * nf / df, kf * (-vx / df), kf * (-l_f * vx) / df]); dFyf_ds = kf
    dFyr = np.array([kr * nr / dr, kr * (-vx) / dr, kr * (l_r * vx) / dr])
    Ac = np.zeros((6, 6)); Bc = np.zeros((6, 2))
    Ac[0, 2:5] = [-vx * sy - vy * cy, cy, -sy]
    Ac[1, 2:5] = [-vy * sy + vx * cy, sy, cy]
    Ac[2, 5] = 1.
    Ac[3, 3:] = [1 / m * (dFx * cs - dFyf[0] * ss), 1 / m * (-dFyf[1] * ss + m * wz), 1 / m * (-dFyf[2] * ss + m * vy)]
    Ac[4, 3:] = [1 / m * (dFx * ss + dFyr[0] + dFyf[0] * cs - m * wz), 1 / m * (dFyr[1] + dFyf[1] * cs),
                 1 / m * (dFyr[2] + dFyf[2] * cs - m * vx)]
    Ac[5, 3:] = [1 / Iz * (dFx * l_f * ss + dFyf[0] * l_f * cs - dFyr[0] * l_r), 1 / Iz * (dFyf[1] * l_f * cs - dFyr[1] * l_r),
                 1 / Iz * (dFyf[2] * l_f * cs - dFyr[2] * l_r)]
    Bc[3] = [1 / m * (-Fxf * ss - dFyf_ds * ss - Fyf * cs), 1 / m * (m * cs)]
    Bc[4] = [1 / m * (Fxf * cs + dFyf_ds * cs - Fyf * ss), 1 / m * (m * ss)]
    Bc[5] = [1 / Iz * (Fxf * l_f * cs + dFyf_ds * l_f * cs - Fyf * l_f * ss), 1 / Iz * (m * l_f * ss)]
    gc = t["f"] - Ac @ x - Bc @ u
    return np.eye(6) + Ac * dt, Bc * dt, gc * dt


def dynamics_step(x, u, m=1300., l_f=1.25, l_r=1.40, width=1.78, length=4.25, C_d=0.34, A_f=2.0, C_roll=0.015, dt=0.02):
    """One explicit Euler step x + f(x, u) dt from the guarded state; returns (x_next (6,), alpha_f, alpha_r), the
    front and rear side-slip angles of that state."""
    t = _dynamics_terms(x, u, m, l_f, l_r, width, length, C_d, A_f, C_roll)
    return t["x"] + t["f"] * dt, t["af"], t["ar"]


def kinematics_model(x, u, wheelbase=1.25 + 1.40, dt=0.02):
    """Linearisation of the kinematic bicycle (state [x, y, v, yaw], input [steer, acceleration]) about (x, u):
    A (4,4), B (4,2) and the affine term C (4,)."""
    x = np.asarray(x, dtype=np.float64).ravel(); u = np.asarray(u, dtype=np.float64).ravel()
    v, yaw, st = x[2], x[3], u[0]
    sy, cy, ct = math.sin(yaw), math.cos(yaw), math.cos(st)
    A = np.array([[1., 0., dt * cy, -dt * v * sy],
                  [0., 1., dt * sy, dt * v * cy],
                  [0., 0., 1., 0.],
                  [0., 0., dt * math.tan(st) / wheelbase, 1.]])
    B = np.array([[0., 0.], [0., 0.], [0., dt], [dt * v / (wheelbase * ct * ct), 0.]])
    C = np.array([dt * v * sy * yaw, -dt * v * cy * yaw, 0., -dt * v * st / (wheelbase * ct * ct)])
    return A, B, C


def kinematics_step(x, u, wheelbase=1.25 + 1.40, dt=0.02):
    """One Euler step, updated in place in the reference's order: position with the old speed and yaw, then the speed,
    then the yaw with the NEW speed."""
    x = np.array(x, dtype=np.float64).ravel().copy(); u = np.asarray(u, dtype=np.float64).ravel()
    st, acc = u[0], u[1]
    x[0] = x[0] + x[2] * math.cos(x[3]) * dt
    x[1] = x[1] + x[2] * math.sin(x[3]) * dt
    x[2] = x[2] + acc * dt
    x[3] = x[3] + x[2] / wheelbase * math.tan(st) * dt
    return x
