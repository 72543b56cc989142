"""Chain descriptions for the oracle / golden generator -- TEST INFRASTRUCTURE ONLY.

An independent restatement (numpy only) of the reference's model tables and of
the ET marshalling its Python layer performs, so that golden fixtures do not
depend on the product's own `models/` tables:

* constant ET matrices: ``trotx/troty/trotz/transl`` with plain cos/sin, i.e.
  Rx(pi/2) keeps cos = 6.1e-17 (reference ET.py:610-760 via spatialmath.base)
* Panda ETS  -- reference models/ETS/Panda.py:32-54 (spelled out in tests/test_ETS.py:267-293)
* DH -> ETS expansion -- reference DHLink.py:173-225
* UR10 DH    -- reference models/DH/UR10.py:56-59
* Puma560 DH -- reference models/DH/Puma560.py:92-179 (kinematic + dynamic)
* Panda MDH  -- reference models/DH/Panda.py:36-160
* frne packing (24 doubles/link) -- reference DHRobot.py:1340-1358, inertia 6-vector
  -> 3x3 reference Link.py:733-742
"""
from __future__ import annotations

import math

import numpy as np

RX, RY, RZ, TX, TY, TZ = 0, 1, 2, 3, 4, 5


def trotx(t):
    c, s = math.cos(t), math.sin(t)
    return np.array([[1, 0, 0, 0], [0, c, -s, 0], [0, s, c, 0], [0, 0, 0, 1.0]])


def troty(t):
    c, s = math.cos(t), math.sin(t)
    return np.array([[c, 0, s, 0], [0, 1, 0, 0], [-s, 0, c, 0], [0, 0, 0, 1.0]])


def trotz(t):
    c, s = math.cos(t), math.sin(t)
    return np.array([[c, -s, 0, 0], [s, c, 0, 0], [0, 0, 1, 0], [0, 0, 0, 1.0]])


def transl(x, y, z):
    T = np.eye(4)
    T[:3, 3] = [x, y, z]
    return T


_CONST = {RX: trotx, RY: troty, RZ: trotz, TX: lambda e: transl(e, 0, 0),
          TY: lambda e: transl(0, e, 0), TZ: lambda e: transl(0, 0, e)}


class Builder:
    """Accumulates ETs into a chain description dict."""

    def __init__(self):
        self.rows = []

    def const(self, axis, eta):
        self.rows.append((0, axis, 0, 0, _CONST[axis](eta), (-math.pi, math.pi) if axis < 3 else (0.0, 1.0)))
        return self

    def se3(self, T):
        self.rows.append((0, 0, 0, 0, np.array(T, dtype=float), (0.0, 1.0)))  # axis "SE3" is not "R..": ET.py:109-115
        return self

    def joint(self, axis, flip=False, jindex=None, qlim=None):
        if qlim is None:
            qlim = (-math.pi, math.pi) if axis < 3 else (0.0, 1.0)  # ET.py:109-115
        self.rows.append((1, axis, int(flip), jindex, np.eye(4), tuple(qlim)))
        return self

    def desc(self):
        rows = self.rows
        j = 0
        jidx = []
        for r in rows:  # sequential jindex assignment, ETS.py:803-840
            if r[0]:
                jidx.append(j if r[3] is None else r[3])
                j += 1
            else:
                jidx.append(0)
        return {
            "isjoint": np.array([r[0] for r in rows], dtype=np.int32),
            "axis": np.array([r[1] for r in rows], dtype=np.int32),
            "flip": np.array([r[2] for r in rows], dtype=np.int32),
            "jindex": np.array(jidx, dtype=np.int32),
            "T": np.stack([r[4] for r in rows]).astype(np.float64),
            "qlim": np.array([r[5] for r in rows], dtype=np.float64),
            "n": j,
        }


def panda_ets():
    deg = math.pi / 180
    b = Builder()
    b.const(TZ, 0.333).joint(RZ)
    b.const(RX, -90 * deg).joint(RZ)
    b.const(RX, 90 * deg).const(TZ, 0.316).joint(RZ)
    b.const(TX, 0.0825).const(RX, 90 * deg).joint(RZ)
    b.const(TX, -0.0825).const(RX, -90 * deg).const(TZ, 0.384).joint(RZ)
    b.const(RX, 90 * deg).joint(RZ)
    b.const(TX, 0.088).const(RX, 90 * deg).const(TZ, 0.107).joint(RZ)
    b.const(TZ, 103 * 1e-3).const(RZ, -math.pi / 4)  # tool_offset = (103) * mm, Panda.py:32
    return b.desc()


def dh_link_to_ets(b: Builder, sigma, theta, d, alpha, a, offset, flip, mdh, qlim=None):
    """reference DHLink._to_ets, DHLink.py:173-225 (zero terms omitted)."""
    revolute = not sigma
    if mdh:
        if a != 0:
            b.const(TX, a)
        if alpha != 0:
            b.const(RX, alpha)
        if revolute:
            if offset != 0:
                b.const(RZ, offset)
            if d != 0:
                b.const(TZ, d)
            b.joint(RZ, flip, qlim=qlim)
        else:
            if theta != 0:
                b.const(RZ, theta)
            if offset != 0:
                b.const(TZ, offset)
            b.joint(TZ, flip, qlim=qlim)
    else:
        if revolute:
            if offset != 0:
                b.const(RZ, offset)
            b.joint(RZ, flip, qlim=qlim)
            if d != 0:
                b.const(TZ, d)
        else:
            if theta != 0:
                b.const(RZ, theta)
            if offset != 0:
                b.const(TZ, offset)
            b.joint(TZ, flip, qlim=qlim)
        if a != 0:
            b.const(TX, a)
        if alpha != 0:
            b.const(RX, alpha)
    return b


def dh_to_ets(links, mdh=False, base=None, tool=None):
    """links: list of dicts(sigma,theta,d,alpha,a,offset,flip,qlim); reference DHRobot.ets 878-918."""
    b = Builder()
    if base is not None:
        b.se3(base)
    for L in links:
        dh_link_to_ets(b, L.get("sigma", 0), L.get("theta", 0.0), L.get("d", 0.0), L.get("alpha", 0.0),
                       L.get("a", 0.0), L.get("offset", 0.0), L.get("flip", False), mdh, L.get("qlim"))
    if tool is not None:
        b.se3(tool)
    return b.desc()


def dh_A(L, q, mdh=False):
    """Link transform A(q), reference DHLink.py:633-673 -- independent FK check for DH models."""
    sa, ca = math.sin(L.get("alpha", 0.0)), math.cos(L.get("alpha", 0.0))
    q = (-q if L.get("flip", False) else q) + L.get("offset", 0.0)
    if not L.get("sigma", 0):
        st, ct, d = math.sin(q), math.cos(q), L.get("d", 0.0)
    else:
        st, ct, d = math.sin(L.get("theta", 0.0)), math.cos(L.get("theta", 0.0)), q
    a = L.get("a", 0.0)
    if not mdh:
        return np.array([[ct, -st * ca, st * sa, a * ct], [st, ct * ca, -ct * sa, a * st],
                         [0, sa, ca, d], [0, 0, 0, 1.0]])
    return np.array([[ct, -st, 0, a], [st * ca, ct * ca, -sa, -sa * d],
                     [st * sa, ct * sa, ca, ca * d], [0, 0, 0, 1.0]])


def ur10_links():
    pi = math.pi
    a = [0, -0.612, -0.5723, 0, 0, 0]
    d = [0.1273, 0, 0, 0.163941, 0.1157, 0.0922]
    alpha = [pi / 2, 0.0, 0.0, pi / 2, -pi / 2, 0.0]
    mass = [7.1, 12.7, 4.27, 2.000, 2.000, 0.365]
    com = [[0.021, 0, 0.027], [0.38, 0, 0.158], [0.24, 0, 0.068], [0.0, 0.007, 0.018],
           [0.0, 0.007, 0.018], [0, 0, -0.026]]
    inertia = [
        [[0.0341, 0, -0.0043], [0, 0.0353, 0.0001], [-0.0043, 0.0001, 0.0216]],
        [[0.0281, 0.0001, -0.0156], [0.0001, 0.7707, 0], [-0.0156, 0, 0.7694]],
        [[0.0101, 0.0001, 0.0092], [0.0001, 0.3093, 0], [0.0092, 0, 0.3065]],
        [[0.0030, -0.0000, 0], [-0.0000, 0.0022, -0.0002], [0, -0.0002, 0.0026]],
        [[0.0030, -0.0000, 0], [-0.0000, 0.0022, -0.0002], [0, -0.0002, 0.0026]],
        [[0, 0, 0], [0, 0.0004, 0], [0, 0, 0.0003]],
    ]
    return [dict(d=d[j], a=a[j], alpha=alpha[j], m=mass[j], r=com[j], I=inertia[j], G=1.0)
            for j in range(6)]


def puma560_links():
    pi = math.pi
    deg = pi / 180
    inch = 0.0254
    return [
        dict(d=26.45 * inch, a=0, alpha=pi / 2, I=[0, 0.35, 0, 0, 0, 0], r=[0, 0, 0], m=0, Jm=200e-6,
             G=-62.6111, B=1.48e-3, Tc=[0.395, -0.435], qlim=[-160 * deg, 160 * deg]),
        dict(d=0, a=0.4318, alpha=0.0, I=[0.13, 0.524, 0.539, 0, 0, 0], r=[-0.3638, 0.006, 0.2275],
             m=17.4, Jm=200e-6, G=107.815, B=0.817e-3, Tc=[0.126, -0.071], qlim=[-110 * deg, 110 * deg]),
        dict(d=0.15005, a=0.0203, alpha=-pi / 2, I=[0.066, 0.086, 0.0125, 0, 0, 0],
             r=[-0.0203, -0.0141, 0.070], m=4.8, Jm=200e-6, G=-53.7063, B=1.38e-3, Tc=[0.132, -0.105],
             qlim=[-135 * deg, 135 * deg]),
        dict(d=0.4318, a=0, alpha=pi / 2, I=[1.8e-3, 1.3e-3, 1.8e-3, 0, 0, 0], r=[0, 0.019, 0], m=0.82,
             Jm=33e-6, G=76.0364, B=71.2e-6, Tc=[11.2e-3, -16.9e-3], qlim=[-266 * deg, 266 * deg]),
        dict(d=0, a=0, alpha=-pi / 2, I=[0.3e-3, 0.4e-3, 0.3e-3, 0, 0, 0], r=[0, 0, 0], m=0.34,
             Jm=33e-6, G=71.923, B=82.6e-6, Tc=[9.26e-3, -14.5e-3], qlim=[-100 * deg, 100 * deg]),
        dict(d=0, a=0, alpha=0.0, I=[0.15e-3, 0.15e-3, 0.04e-3, 0, 0, 0], r=[0, 0, 0.032], m=0.09,
             Jm=33e-6, G=76.686, B=36.7e-6, Tc=[3.96e-3, -10.5e-3], qlim=[-266 * deg, 266 * deg]),
    ]


PUMA_QN = np.array([0, math.pi / 4, math.pi, 0, math.pi / 4, 0])


def panda_mdh_links():
    pi = math.pi
    P = [
        (0.0, 0.333, 0.0, [-2.8973, 2.8973], 4.970684, [7.03370e-01, 7.06610e-01, 9.11700e-03, -1.39000e-04, 1.91690e-02, 6.77200e-03]),
        (0.0, 0.0, -pi / 2, [-1.7628, 1.7628], 0.646926, [7.96200e-03, 2.81100e-02, 2.59950e-02, -3.92500e-03, 7.04000e-04, 1.02540e-02]),
        (0.0, 0.316, pi / 2, [-2.8973, 2.8973], 3.228604, [3.72420e-02, 3.61550e-02, 1.08300e-02, -4.76100e-03, -1.28050e-02, -1.13960e-02]),
        (0.0825, 0.0, pi / 2, [-3.0718, -0.0698], 3.587895, [2.58530e-02, 1.95520e-02, 2.83230e-02, 7.79600e-03, 8.64100e-03, -1.33200e-03]),
        (-0.0825, 0.384, -pi / 2, [-2.8973, 2.8973], 1.225946, [3.55490e-02, 2.94740e-02, 8.62700e-03, -2.11700e-03, 2.29000e-04, -4.03700e-03]),
        (0.0, 0.0, pi / 2, [-0.0175, 3.7525], 1.666555, [1.96400e-03, 4.35400e-03, 5.43300e-03, 1.09000e-04, 3.41000e-04, -1.15800e-03]),
        (0.088, 107 * 1e-3, pi / 2, [-2.8973, 2.8973], 7.35522e-01, [1.25160e-02, 1.00270e-02, 4.81500e-03, -4.28000e-04, -7.41000e-04, -1.19600e-03]),
    ]
    return [dict(a=a, d=d, alpha=al, qlim=ql, m=m, I=I, G=1.0) for a, d, al, ql, m, I in P]


def panda_mdh_tool():
    return transl(0, 0, 103 * 1e-3) @ trotz(-math.pi / 4)


def inertia3(I):
    I = np.asarray(I, dtype=float)
    if I.shape == (3, 3):
        return I
    if I.size == 6:  # Link.py:733-742
        return np.array([[I[0], I[3], I[5]], [I[3], I[1], I[4]], [I[5], I[4], I[2]]])
    if I.size == 3:
        return np.diag(I)
    raise ValueError("bad inertia")


def pack_rne(links, mdh=False):
    """24 doubles per link, reference DHRobot.py:1340-1358."""
    L = np.zeros(24 * len(links))
    for i, l in enumerate(links):
        j = 24 * i
        L[j] = l.get("alpha", 0.0)
        L[j + 1] = l.get("a", 0.0)
        L[j + 2] = l.get("theta", 0.0)
        L[j + 3] = l.get("d", 0.0)
        L[j + 4] = l.get("sigma", 0)
        L[j + 5] = l.get("offset", 0.0)
        L[j + 6] = l.get("m", 0.0)
        L[j + 7:j + 10] = np.asarray(l.get("r", [0, 0, 0]), dtype=float)
        L[j + 10:j + 19] = inertia3(l.get("I", np.zeros((3, 3)))).flatten()
        L[j + 19] = l.get("Jm", 0.0)
        L[j + 20] = l.get("G", 0.0)
        L[j + 21] = l.get("B", 0.0)
        Tc = np.asarray(l.get("Tc", [0.0, 0.0]), dtype=float)
        L[j + 22:j + 24] = Tc
    return L


def random_se3(rng, reach=0.5):
    """A general rigid transform: rotations about all three axes and a translation in [-reach, reach]^3."""
    return (trotz(rng.uniform(-math.pi, math.pi)) @ troty(rng.uniform(-math.pi, math.pi))
            @ trotx(rng.uniform(-math.pi, math.pi)) @ transl(*rng.uniform(-reach, reach, 3)))


DH_ALPHAS = (0.0, math.pi / 2, -math.pi / 2, None)  # None: alpha drawn from U(-pi, pi)


def dh_like_chain(rng, n, tail=True):
    """A random chain of the shape the kernels treat as DH-like: a general SE(3) head A_0, n unflipped Rz joints,
    inter-joint constants transl(x, y, z) @ trotx(alpha) and, with `tail`, a general SE(3) tail.  Without it nothing
    follows the last joint.  The alphas cycle from a random start through 0 (a pure translation), +-pi/2 (cos(alpha)
    stays 6.1e-17, not 0) and a random angle, so every kind appears once a chain has four inter-joint constants."""
    b = Builder()
    b.se3(random_se3(rng))
    k0 = int(rng.integers(0, len(DH_ALPHAS)))
    for j in range(n):
        if j > 0:
            alpha = DH_ALPHAS[(k0 + j) % len(DH_ALPHAS)]
            if alpha is None:
                alpha = float(rng.uniform(-math.pi, math.pi))
            b.se3(transl(*rng.uniform(-0.5, 0.5, 3)) @ trotx(alpha))
        b.joint(RZ)
    if tail:
        b.se3(random_se3(rng))
    return b.desc()


def perturb_joint(desc, k, flip=None, axis=None):
    """A copy of a chain description with the k-th joint flipped and/or moved to another axis."""
    d = {key: (v.copy() if isinstance(v, np.ndarray) else v) for key, v in desc.items()}
    i = int(np.flatnonzero(d["isjoint"])[k])
    if flip is not None:
        d["flip"][i] = int(flip)
    if axis is not None:
        d["axis"][i] = int(axis)
    return d


def chain_reach(desc, *extra):
    """Sum of the translation lengths of a chain's constants and of any extra 4x4 transforms (base, tool): a bound on
    how far the end effector can be from the origin, the scale of the absolute errors of poses and Jacobians."""
    Ts = [T for T, j in zip(desc["T"], desc["isjoint"]) if not j] + [T for T in extra if T is not None]
    return float(sum(np.linalg.norm(np.asarray(T)[:3, 3]) for T in Ts))


def random_chain(rng, n_joints=6, with_flips=True, extra_consts=True):
    """A random serial chain exercising all six ET kinds, flips, constant runs and SE3 constants."""
    b = Builder()
    for _ in range(n_joints):
        if extra_consts:
            for _ in range(int(rng.integers(0, 3))):
                ax = int(rng.integers(0, 6))
                b.const(ax, float(rng.uniform(-1.0, 1.0)))
            if rng.random() < 0.2:
                T = trotx(rng.uniform(-3, 3)) @ troty(rng.uniform(-3, 3)) @ transl(*rng.uniform(-0.5, 0.5, 3))
                b.se3(T)
        ax = int(rng.integers(0, 6))
        flip = bool(with_flips and rng.random() < 0.3)
        lo = float(rng.uniform(-3.0, -0.5))
        hi = float(rng.uniform(0.5, 3.0))
        b.joint(ax, flip, qlim=(lo, hi))
    if extra_consts and rng.random() < 0.7:
        b.const(int(rng.integers(0, 6)), float(rng.uniform(-1, 1)))
    return b.desc()
