"""Oracles of the step with solid obstacles (test infrastructure).

- `lib()` builds tests/obstacle_oracle.c (the reference oracle plus smk_oracle_jacobi_obst / smk_oracle_step_obst) with gcc
  -ffp-contract=off into a temporary directory, keyed by the sources' hash, and binds it.
- `jacobi_obst`, `step_obst`: the C oracle on dense numpy arrays.
- `np_jacobi_obst`, `np_step_obst`: a numpy restatement of the same semantics, checked bit-equal to the C oracle; the physics
  checks of tests/test_obstacles_host.py use it.
- `faces`, `demo_mask`: closed-face masks of a cell mask, and the box + partial wall + single cell mask of DESIGN.md s5.7.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "obstacle_oracle.c")
_REF = os.path.join(_HERE, "..", "oracle", "smoke_oracle.c")
_lib = None
f32 = np.float32

f32p = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
u8p = np.ctypeslib.ndpointer(dtype=np.uint8, flags="C_CONTIGUOUS")


def lib():
    global _lib
    if _lib is None:
        key = hashlib.sha256(open(_SRC, "rb").read() + open(_REF, "rb").read()).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), "smk_obstacle_oracle_%s_%d.so" % (key, os.getuid()))
        if not os.path.exists(so):
            tmp = so + ".%d" % os.getpid()
            subprocess.check_call(["gcc", "-O2", "-std=gnu11", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-shared",
                                   "-o", tmp, _SRC, "-lm", "-lpthread"])
            os.replace(tmp, so)
        L = C.CDLL(so)
        i, f, v = C.c_int, C.c_float, C.c_void_p
        L.smk_oracle_jacobi_obst.argtypes = [f32p, f32p, u8p, f32p, i, i, i]
        L.smk_oracle_step_obst.argtypes = [f32p, f32p, f32p, f32p, i, i, f, f, f, i, f32p, v, v, u8p]
        L.smk_oracle_step.argtypes = [f32p, f32p, f32p, f32p, i, i, f, f, f, i, f32p, v, v]
        L.smk_oracle_work_floats.argtypes = [i, i]
        L.smk_oracle_work_floats.restype = C.c_long
        for fn in (L.smk_oracle_jacobi_obst, L.smk_oracle_step_obst, L.smk_oracle_step):
            fn.restype = None
        _lib = L
    return _lib


def mask_u8(solid):
    return np.ascontiguousarray(np.asarray(solid) != 0, dtype=np.uint8)


def jacobi_obst(p, div, solid, K):
    p = np.ascontiguousarray(p, dtype=f32).copy()
    div = np.ascontiguousarray(div, dtype=f32)
    tmp = np.empty_like(p)
    lib().smk_oracle_jacobi_obst(p, div, mask_u8(solid), tmp, p.shape[0], p.shape[1], int(K))
    return p


def coefs(dt, visc):
    return f32(dt), oracle.coef(dt, visc), f32(float(dt) * (float(visc) * 0.1))


def step_obst(u, v, p, d, solid, dt, visc, K, want_norms=False):
    """One step in place on dense (u, v, p, d) with solid cells `solid` (None: smk_oracle_step); -> (frame, norms or None)."""
    h, w = d.shape
    work = np.empty(lib().smk_oracle_work_floats(h, w), f32)
    frame = np.empty((h, w), f32)
    norms = np.zeros(2)
    args = (u, v, p, d, h, w) + coefs(dt, visc) + (int(K), work, frame.ctypes.data, norms.ctypes.data if want_norms else None)
    if solid is None:
        lib().smk_oracle_step(*args)
    else:
        lib().smk_oracle_step_obst(*args, mask_u8(solid))
    return frame, (tuple(norms) if want_norms else None)


class ObstacleSolver(oracle.OracleSolver):
    """OracleSolver (dense twin of NavierStokesSimulator) whose step applies the solid cells `solid` [h, w]."""

    def __init__(self, grid_size, dt, viscosity, jacobi_iters, solid):
        self.solid = mask_u8(solid)
        super().__init__(grid_size, dt, viscosity, jacobi_iters)

    def step(self, want_norms=False):
        for k in ("u", "v", "p", "density"):
            setattr(self, k, np.ascontiguousarray(getattr(self, k), dtype=f32))
        frame, norms = step_obst(self.u, self.v, self.p, self.density, self.solid, self.dt, self.viscosity, self.jacobi_iters,
                                 want_norms)
        if want_norms:
            self.last_div_norms = norms
        return frame


# ---- numpy restatement -----------------------------------------------------------------------------------------------------
def faces(S):
    """(closed u faces [h+1, w], closed v faces [h, w+1]) of the solid cells S [h, w]."""
    S = np.asarray(S) != 0
    h, w = S.shape
    cu = np.zeros((h + 1, w), bool)
    cv = np.zeros((h, w + 1), bool)
    cu[:-1] |= S
    cu[1:] |= S
    cv[:, :-1] |= S
    cv[:, 1:] |= S
    return cu, cv


def np_jacobi_obst(P, D, S, K):
    S = np.asarray(S) != 0
    P = np.asarray(P, f32)
    h, w = P.shape
    for _ in range(K):
        Q = np.zeros_like(P)
        if h >= 3 and w >= 3:
            c = P[1:-1, 1:-1]
            s = np.where(S[:-2, 1:-1], c, P[:-2, 1:-1]) + np.where(S[2:, 1:-1], c, P[2:, 1:-1])
            s = s + np.where(S[1:-1, :-2], c, P[1:-1, :-2])
            s = s + np.where(S[1:-1, 2:], c, P[1:-1, 2:])
            s = s - D[1:-1, 1:-1]
            Q[1:-1, 1:-1] = np.where(S[1:-1, 1:-1], f32(0), f32(0.25) * s)
        P = Q
    return P


def np_div(U, V, dt):
    s = U[1:] - U[:-1]
    s = s + V[:, 1:]
    s = s - V[:, :-1]
    return (s / f32(dt)).astype(f32)


def np_step_obst(u, v, p, d, S, dt, visc, K):
    """Returns the new (u, v, p, d); the phases the obstacles leave alone are the reference oracle's own."""
    S = np.asarray(S) != 0
    cu, cv = faces(S)
    dt32, c_uv, c_d = coefs(dt, visc)
    h, w = d.shape
    v = oracle.buoyancy(v, d, dt)
    u = oracle.diffusion_step(u, dt, visc)
    v = oracle.diffusion_step(v, dt, visc)
    d = _diffuse(d, c_d)
    u = np.where(cu, f32(0), u)                                                 # O1
    v = np.where(cv, f32(0), v)
    div = np_div(u, v, dt32)
    p = np_jacobi_obst(p, div, S, K)
    g = (p[1:] - p[:-1]) * dt32
    u = u.copy()
    u[1:-1] = np.where(cu[1:-1], u[1:-1], u[1:-1] - g)
    g = (p[:, 1:] - p[:, :-1]) * dt32
    v = v.copy()
    v[:, 1:-1] = np.where(cv[:, 1:-1], v[:, 1:-1], v[:, 1:-1] - g)
    u_new = oracle.advection_step(u, u, v, dt32)
    v_new = oracle.advection_step(v, u_new, v, dt32)
    u_new = np.where(cu, f32(0), u_new)                                         # O4
    v_new = np.where(cv, f32(0), v_new)
    d = oracle.advection_step(d, u_new, v_new, dt32) * f32(0.995)
    d = np.where(S, f32(0), d).astype(f32)                                      # O3
    return u_new.astype(f32), v_new.astype(f32), p.astype(f32), d


def _diffuse(F, c):
    """diffusion_step with the coefficient already rounded (c_d is float32(dt * (viscosity * 0.1)), formed in double)."""
    F = np.ascontiguousarray(F, dtype=f32)
    out = np.empty_like(F)
    oracle.lib().smk_oracle_diffuse(F, out, F.shape[0], F.shape[1], c)
    return out


def demo_mask(h, w):
    """The box of rows 20-29 x columns 25-39, a wall of rows h/2 .. h/2 + 2 over the first w/3 columns, and the cell (5, 5)."""
    S = np.zeros((h, w), bool)
    S[20:30, 25:40] = True
    S[h // 2:h // 2 + 3, :w // 3] = True
    S[5, 5] = True
    return S


def interior_fluid(S):
    S = np.asarray(S) != 0
    fl = ~S
    fl[0] = fl[-1] = False
    fl[:, 0] = fl[:, -1] = False
    return fl
