"""oracle/hp_reference.py — TEST INFRASTRUCTURE ONLY.

An extended-precision restatement of the operations the CUDA kernels implement, with a per-point error yardstick.

Every stage mirrors a section of ``rhs_element`` in oracle/caar_oracle.c (A pressure, B horizontal operators,
C virtual temperature, D/E the two vertical integrals, the Eulerian block, F accumulate, G tendencies, H apply), plus
the tracer step (``caar_oracle_euler_step``) and the weak-form operators (``caar_oracle_sphere_wk``). The stages are
vectorised over elements, levels and points; only the vertical scans loop, over levels. The code is generic over the
dtype of its inputs: ``from_state(s)`` runs it in ``np.longdouble`` (x86-64: 64-bit mantissa, eps = 2^-63, about
2000 times finer than FP64), ``from_state(s, np.float64)`` runs the same expressions in FP64.

The yardstick
-------------
Every value is an ``HP``: the value ``v`` and a magnitude ``M`` from a first-order (Wilkinson-style) running error
analysis of the same expression. An input ``x`` has ``M = |x|`` (constants such as rrearth, Dvv, dt2, eta_ave_w and
Rgas are inputs like any other), and

    a +- b : M = M_a + M_b        a * b : M = M_a * M_b        a / b : M = M_a / |b| + |a| M_b / b^2.

An FP64 evaluation of the expression in ANY order -- any association of a sum, any FMA contraction, any factoring or
premultiplication of a product (Dinv * rrearth), a reciprocal in place of a division -- whose longest chain of
dependent roundings has K operations is within ``K u M`` of the exact value, u = 2^-53, to first order: each rounding
is a relative perturbation of at most u of one node, and a perturbation of a node changes the result by at most the
node's share of M. A sum of n terms evaluated in any order is a chain of at most n - 1 additions. ``gate(g, ref, K)``
checks ``|g - v| <= K u M`` at every point; where M == 0 (nothing but zeros entered) it demands equality. The error
of the longdouble evaluation itself is about K 2^-64 M, 2048 times below the gate.

K of each operation (sums flattened: a sum of n terms counts n - 1; multiplications by 0.5 and 2 counted too)
-----------------------------------------------------------------------------------------------------------
Weak-form operators (``caar_oracle_sphere_wk``), one level of one element:
  gradient_sphere   Dvv*s 1, sum of 4: 3, *rrearth 1, Dinv* 1, sum of 2: 1                        =  7
  tensorVisc.g      tv* 1, sum of 2: 1                                                              =  2
  div_sphere_wk     Dinv* 1, sum of 2: 1, spheremp* 1, Dvv* 1, sum of 8: 7, *rrearth 1            = 12
  K_DIVWK = 12,  K_LAPLACE_SIMPLE = 7 + 12 = 19,  K_LAPLACE_TENSOR = 7 + 2 + 12 = 21.
Tracer step: vstar*Qdp 1, Dinv* 1, sum of 2: 1, metdet* 1, Dvv* 1, sum of 8: 7, *rmetdet 1, *rrearth 1,
  (-dt)* 1, Qdp + 1                                                                                 K_EULER = 16.
compute_and_apply_rhs, one call, nlev = L; depth of each intermediate:
  p[k]       hyai0*ps0 1, then a sum of 2k+2 terms                                      <= 2L
  div_sphere (divdp) vdp 1, Dinv* 1, sum of 2: 1, metdet* 1, Dvv* 1, sum of 8: 7, *rmetdet 1, *rrearth 1 = 14
  grad_sphere of a depth-d field                                                        d + 7
  T_v        Rwv/Rgas 1, -1 1, *(Qdp/dp) 1, 1+ 1, T* 1                                      5
  phi[k]     hkk = 0.5*dp/p: 2L + 2, Rgas*T_v*hkk: 2L + 4, then phis + a sum over <= L levels:  3L + 4
  Ephi       a sum of 4 with phi (its inner sum flattened in): 0.5*|v|^2, phi, pecnd        3L + 7
  vt1, vt2   grad(Ephi): 3L + 14, then a sum of 4 (v_vadv, v*(fcor+vort), gE, glnps): 3L + 17
  v(np1)     dt2* 1, v(nm1) + 1, spheremp* 1                                                3L + 20
  omega      suml: divdp summed over <= L-1 levels: L + 12; ckl*suml with ckl = 2*(0.5/p): 2L + 4;
             vgrad_p/p: grad(p) 2L + 7, v* 1, sum of 2: 1, /p 1 = 2L + 10; sum of 3: 2L + 12
  omega_p    eta_ave_w* 1, + 1                                                              2L + 14
  T(np1)     kappa*T_v*omega 2L + 14, sum of 3 (T_vadv, vgrad_T, that): 2L + 16, apply 3     2L + 19
  Eulerian   sdot: divdp summed over L levels: L + 13; eta = hybi*sdot - partial sum: L + 15;
             facp = 0.5*(1/dp)*eta: L + 17; *(T[k+1]-T[k]): L + 18; T_vadv, sum of 2: L + 19;
             T(np1): sum of 3: L + 21, apply 3: L + 24;  dp(np1): divdp + eta - eta, sum of 3: L + 17, apply: L + 20;
             eta_dot_dpdn: eta_ave_w* 1, + 1: L + 17
  The longest is max(3L + 20, 2L + 19, L + 24) <= 3L + 24 = K_RHS(L) for every L >= 2.
  Over ncalls calls the state and the accumulators carry their error into the next call: first order, an input
  error of k u M_in moves the output by at most k u M_out (the propagation rules above bound every partial
  derivative times its input's M), so call n is within n K_RHS(L) u M. ``k_rhs(L, ncalls) = ncalls * (3L + 24)``.
"""
from __future__ import annotations

import numpy as np

U64 = 2.0 ** -53            # unit roundoff of FP64

K_DIVWK = 12
K_LAPLACE_SIMPLE = 19
K_LAPLACE_TENSOR = 21
K_EULER = 16


def k_rhs(nlev, ncalls=1):
    return ncalls * (3 * nlev + 24)


K_SPHERE_WK = {"divergence_sphere_wk": K_DIVWK, "laplace_simple": K_LAPLACE_SIMPLE, "laplace_tensor": K_LAPLACE_TENSOR}


class HP:
    """A value and its first-order error magnitude (see the module docstring). Plain numbers are inputs (M = |x|)."""
    __slots__ = ("v", "M")

    def __init__(self, v, M):
        self.v, self.M = v, M

    @staticmethod
    def input(x, dtype):
        v = np.array(x, dtype=dtype)
        return HP(v, np.abs(v))

    def _lift(self, o):
        return o if isinstance(o, HP) else HP.input(o, self.v.dtype)

    def __add__(self, o):
        o = self._lift(o)
        return HP(self.v + o.v, self.M + o.M)

    def __sub__(self, o):
        o = self._lift(o)
        return HP(self.v - o.v, self.M + o.M)

    def __mul__(self, o):
        o = self._lift(o)
        return HP(self.v * o.v, self.M * o.M)

    def __truediv__(self, o):
        o = self._lift(o)
        return HP(self.v / o.v, self.M / np.abs(o.v) + np.abs(self.v) * o.M / (o.v * o.v))

    def __radd__(self, o):
        return self._lift(o) + self

    def __rsub__(self, o):
        return self._lift(o) - self

    def __rmul__(self, o):
        return self._lift(o) * self

    def __rtruediv__(self, o):
        return self._lift(o) / self

    def __neg__(self):
        return HP(-self.v, self.M)

    def __getitem__(self, idx):
        return HP(self.v[idx], self.M[idx])

    def __setitem__(self, idx, o):
        self.v[idx] = o.v
        self.M[idx] = o.M

    def copy(self):
        return HP(self.v.copy(), self.M.copy())

    @staticmethod
    def stack(xs, axis):
        return HP(np.stack([x.v for x in xs], axis), np.stack([x.M for x in xs], axis))

    @staticmethod
    def concat(xs, axis):
        return HP(np.concatenate([x.v for x in xs], axis), np.concatenate([x.M for x in xs], axis))


def contract(spec, c, x):
    """einsum of a constant matrix with a field: a sum of products, so M is the same sum over the magnitudes."""
    return HP(np.einsum(spec, c.v, x.v), np.einsum(spec, c.M, x.M))


class _Arrays(dict):
    """name -> HP, converted from the state's array on first use (the level-local operators read geometry only)."""

    def __init__(self, src, dtype):
        super().__init__()
        self.src, self.dtype = src, dtype

    def __missing__(self, name):
        self[name] = HP.input(self.src[name], self.dtype)
        return self[name]


class HPState:
    """A harness.State as HP arrays (pointers_only layout) plus HP scalars."""

    def __init__(self, s, dtype=np.longdouble):
        self.dtype = dtype
        self.nelem, self.nlev, self.qsize_d, self.ntl = s.nelem, s.nlev, s.qsize_d, s.ntl
        self.arrays = _Arrays(s.arrays, dtype)
        self.nets, self.nete, self.n0, self.np1, self.nm1, self.qn0 = (int(x) for x in s.ctl)
        inp = lambda x: HP.input(x, dtype)
        self.dt2 = inp(s.dt2)
        self.rrearth, self.eta_ave_w, self.cp, self.Rwv, self.Rgas, self.kappa = (inp(x) for x in s.consts)
        self.dvv = inp(s.dvv)
        self.ps0, self.hyai0 = inp(s.ps0), inp(s.hyai[0])

    def geo(self, name, per_level=True):
        """Geometry of elements [nets,nete), with a level axis to broadcast over when per_level."""
        g = self.arrays[name][self.nets:self.nete]
        return HP(g.v[:, None], g.M[:, None]) if per_level else g


def from_state(s, dtype=np.longdouble):
    return HPState(s, dtype)


# ---- sphere operators: fields (..., 4, 4) [i][j], vectors as (x0, x1); geometry broadcasts over the leading axes ----

def gradient_sphere(s, dvv, dinv, rrearth):
    """PO/sphere_operators.cpp:21-47 (caar_oracle.c grad_sphere)."""
    a = contract("il,...ij->...lj", dvv, s) * rrearth
    b = contract("il,...ji->...jl", dvv, s) * rrearth
    return dinv[..., 0, 0] * a + dinv[..., 1, 0] * b, dinv[..., 0, 1] * a + dinv[..., 1, 1] * b


def divergence_sphere(v0, v1, dvv, dinv, metdet, rmetdet, rrearth):
    """PO/sphere_operators.cpp:62-88 (caar_oracle.c div_sphere)."""
    g0 = metdet * (dinv[..., 0, 0] * v0 + dinv[..., 0, 1] * v1)
    g1 = metdet * (dinv[..., 1, 0] * v0 + dinv[..., 1, 1] * v1)
    return (contract("ki,...kj->...ij", dvv, g0) + contract("kj,...ik->...ij", dvv, g1)) * rmetdet * rrearth


def vorticity_sphere(v0, v1, dvv, d, rmetdet, rrearth):
    """PO/sphere_operators.cpp:102-128 (caar_oracle.c vort_sphere)."""
    c0 = d[..., 0, 0] * v0 + d[..., 1, 0] * v1
    c1 = d[..., 0, 1] * v0 + d[..., 1, 1] * v1
    return (contract("ki,...kj->...ij", dvv, c1) - contract("kj,...ik->...ij", dvv, c0)) * rmetdet * rrearth


def divergence_sphere_wk(v0, v1, dvv, dinv, spheremp, rrearth):
    """LV/SphereOperators.hpp:493-535 (caar_oracle.c div_sphere_wk)."""
    u0 = spheremp * (dinv[..., 0, 0] * v0 + dinv[..., 0, 1] * v1)
    u1 = spheremp * (dinv[..., 1, 0] * v0 + dinv[..., 1, 1] * v1)
    return -((contract("mj,...jn->...mn", dvv, u0) + contract("nj,...mj->...mn", dvv, u1)) * rrearth)


def laplace_wk(s, dvv, dinv, spheremp, tensorvisc, rrearth):
    """laplace_simple (tensorvisc None) / laplace_tensor, LV/SphereOperators.hpp:537-636 (caar_oracle.c laplace_wk)."""
    g0, g1 = gradient_sphere(s, dvv, dinv, rrearth)
    if tensorvisc is not None:
        g0, g1 = (tensorvisc[..., 0, 0] * g0 + tensorvisc[..., 0, 1] * g1,
                  tensorvisc[..., 1, 0] * g0 + tensorvisc[..., 1, 1] * g1)
    return divergence_sphere_wk(g0, g1, dvv, dinv, spheremp, rrearth)


# ---- compute_and_apply_rhs, section by section (caar_oracle.c rhs_element); fields are (E, L, 4, 4) ----------------

def _levels(x):
    return [x[:, k] for k in range(x.v.shape[1])]


def pressure(hyai0, ps0, dp):
    """A: mid-level pressure, top-down."""
    dp = _levels(dp)
    p = [hyai0 * ps0 + 0.5 * dp[0]]
    for k in range(1, len(dp)):
        p.append(p[k - 1] + 0.5 * dp[k - 1] + 0.5 * dp[k])
    return HP.stack(p, 1)


def horizontal(hs, p, v0, v1, dp):
    """B: level-local horizontal operators -> grad_p (2), vgrad_p, vdp (2), divdp, vort."""
    Dinv, D = hs.geo("elem_Dinv"), hs.geo("elem_D")
    gp = gradient_sphere(p, hs.dvv, Dinv, hs.rrearth)
    vgrad_p = v0 * gp[0] + v1 * gp[1]
    vdp = (v0 * dp, v1 * dp)
    divdp = divergence_sphere(vdp[0], vdp[1], hs.dvv, Dinv, hs.geo("elem_metdet"), hs.geo("elem_rmetdet"), hs.rrearth)
    vort = vorticity_sphere(v0, v1, hs.dvv, D, hs.geo("elem_rmetdet"), hs.rrearth)
    return gp, vgrad_p, vdp, divdp, vort


def virtual_temperature(hs, T, Qdp, dp):
    """C: T_v; Qdp is None when qn0 == -1 (dry)."""
    if Qdp is None:
        return T
    return T * (1.0 + (hs.Rwv / hs.Rgas - 1.0) * (Qdp / dp))


def hydrostatic(phis, T_v, p, dp, Rgas):
    """D: preq_hydrostatic, the reverse (bottom-up) sum."""
    T_v, p, dp = _levels(T_v), _levels(p), _levels(dp)
    L = len(p)
    phi = [None] * L
    k = L - 1
    hkk = 0.5 * dp[k] / p[k]
    phii = Rgas * T_v[k] * (2.0 * hkk)
    phi[k] = phis + Rgas * T_v[k] * hkk
    for k in range(L - 2, 0, -1):
        hkk = 0.5 * dp[k] / p[k]
        phi[k] = phis + phii + Rgas * T_v[k] * hkk
        phii = phii + Rgas * T_v[k] * (2.0 * hkk)
    hkk = 0.5 * dp[0] / p[0]
    phi[0] = phis + phii + Rgas * T_v[0] * hkk
    return HP.stack(phi, 1)


def omega_ps(p, vgrad_p, divdp):
    """E: preq_omega_ps, the forward (top-down) running sum of divdp."""
    p, vgrad_p, divdp = _levels(p), _levels(vgrad_p), _levels(divdp)
    L = len(p)
    omega = [vgrad_p[0] / p[0] - (0.5 / p[0]) * divdp[0]]
    suml = divdp[0]
    for k in range(1, L):
        ckk = 0.5 / p[k]
        omega.append(vgrad_p[k] / p[k] - (2.0 * ckk) * suml - ckk * divdp[k])
        if k < L - 1:
            suml = suml + divdp[k]
    return HP.stack(omega, 1)


def eulerian_eta(divdp, hybi):
    """rsplit == 0: eta_dot_dpdn at the L+1 interfaces from the running sum of divdp and hybi; zero at both ends."""
    d = _levels(divdp)
    L = len(d)
    part = [d[0]]
    for k in range(1, L):
        part.append(part[k - 1] + d[k])
    sdot = part[L - 1]
    zero = HP.input(np.zeros_like(sdot.v), sdot.v.dtype)
    eta = [zero] + [hybi[k + 1] * sdot - part[k] for k in range(L - 1)] + [zero]
    return HP.stack(eta, 1)


def preq_vertadv(T, v0, v1, eta, rpdel):
    """Vertical advection of T and v (CaarFunctor.hpp:504-547, caar_oracle.c preq_vertadv). Needs L >= 2."""
    facp = 0.5 * rpdel * eta[:, 1:]
    facm = 0.5 * rpdel * eta[:, :-1]

    def adv(x):
        dx = x[:, 1:] - x[:, :-1]                     # dx[k] = x[k+1] - x[k]
        up = facp[:, :-1] * dx                        # levels 0 .. L-2
        down = facm[:, 1:] * dx                       # levels 1 .. L-1
        mid = up[:, 1:] + down[:, :-1]                # levels 1 .. L-2
        return HP.concat([up[:, :1], mid, down[:, -1:]], 1)

    return adv(T), (adv(v0), adv(v1))


def tendencies(hs, v0, v1, T, T_v, p, gp, vort, phi, pecnd, omega, T_vadv, v_vadv):
    """G: vt1, vt2, tt. On the Lagrangian branch T_vadv and v_vadv are zeros."""
    Dinv, fcor = hs.geo("elem_Dinv"), hs.geo("elem_fcor")
    Ephi = 0.5 * (v0 * v0 + v1 * v1) + phi + pecnd
    gT = gradient_sphere(T, hs.dvv, Dinv, hs.rrearth)
    vgrad_T = v0 * gT[0] + v1 * gT[1]
    gE = gradient_sphere(Ephi, hs.dvv, Dinv, hs.rrearth)
    gpterm = T_v / p
    glnps1 = hs.Rgas * gpterm * gp[0]
    glnps2 = hs.Rgas * gpterm * gp[1]
    vt1 = -v_vadv[0] + v1 * (fcor + vort) - gE[0] - glnps1
    vt2 = -v_vadv[1] - v0 * (fcor + vort) - gE[1] - glnps2
    tt = -T_vadv - vgrad_T + hs.kappa * T_v * omega
    return vt1, vt2, tt


def rhs(hs, hybi=None):
    """One compute_and_apply_rhs call on elements [nets,nete) of hs, in place. hybi: None = Lagrangian (rsplit > 0),
    else the Eulerian branch (rsplit == 0) with hybi[nlev+1]."""
    A = hs.arrays
    r = slice(hs.nets, hs.nete)
    if hs.nete <= hs.nets:
        return hs
    dp = A["elem_state_dp3d"][r, hs.n0].copy()
    v = A["elem_state_v"][r, hs.n0]
    v0, v1 = v[..., 0].copy(), v[..., 1].copy()
    T = A["elem_state_T"][r, hs.n0].copy()

    p = pressure(hs.hyai0, hs.ps0, dp)
    gp, vgrad_p, vdp, divdp, vort = horizontal(hs, p, v0, v1, dp)
    vn0 = A["elem_derived_vn0"]
    vn0[r, ..., 0] = vn0[r, ..., 0] + hs.eta_ave_w * vdp[0]
    vn0[r, ..., 1] = vn0[r, ..., 1] + hs.eta_ave_w * vdp[1]
    Qdp = None if hs.qn0 == -1 else A["elem_state_Qdp"][r, 0, hs.qn0]
    T_v = virtual_temperature(hs, T, Qdp, dp)
    phi = hydrostatic(hs.geo("elem_state_phis", per_level=False), T_v, p, dp, hs.Rgas)
    A["elem_derived_phi"][r] = phi
    omega = omega_ps(p, vgrad_p, divdp)

    zero = HP.input(np.zeros_like(T.v), hs.dtype)
    if hybi is None:
        eta = HP.input(np.zeros((T.v.shape[0], hs.nlev + 1, 4, 4)), hs.dtype)
        T_vadv, v_vadv = zero, (zero, zero)
    else:
        eta = eulerian_eta(divdp, HP.input(hybi, hs.dtype))
        T_vadv, v_vadv = preq_vertadv(T, v0, v1, eta, 1.0 / dp)

    # F: accumulate
    A["elem_derived_eta_dot_dpdn"][r] = A["elem_derived_eta_dot_dpdn"][r] + hs.eta_ave_w * eta
    A["elem_derived_omega_p"][r] = A["elem_derived_omega_p"][r] + hs.eta_ave_w * omega

    vt1, vt2, tt = tendencies(hs, v0, v1, T, T_v, p, gp, vort, phi, A["elem_derived_pecnd"][r], omega, T_vadv, v_vadv)
    apply(hs, vt1, vt2, tt, divdp if hybi is None else divdp + eta[:, 1:] - eta[:, :-1])
    return hs


def apply(hs, vt1, vt2, tt, dpdt):
    """H: the leapfrog update into np1 from nm1 (every read of this element happened before)."""
    A = hs.arrays
    r = slice(hs.nets, hs.nete)
    mp = hs.geo("elem_spheremp")
    v_nm1 = A["elem_state_v"][r, hs.nm1]
    T_nm1 = A["elem_state_T"][r, hs.nm1]
    dp_nm1 = A["elem_state_dp3d"][r, hs.nm1]
    v_np1_0 = mp * (v_nm1[..., 0] + hs.dt2 * vt1)
    v_np1_1 = mp * (v_nm1[..., 1] + hs.dt2 * vt2)
    T_np1 = mp * (T_nm1 + hs.dt2 * tt)
    dp_np1 = mp * (dp_nm1 - hs.dt2 * dpdt)
    A["elem_state_v"][r, hs.np1, ..., 0] = v_np1_0
    A["elem_state_v"][r, hs.np1, ..., 1] = v_np1_1
    A["elem_state_T"][r, hs.np1] = T_np1
    A["elem_state_dp3d"][r, hs.np1] = dp_np1


def compute_and_apply_rhs(hs, ncalls=1, hybi=None):
    """ncalls calls, the state and the accumulators carried between them in hs's precision."""
    for _ in range(ncalls):
        rhs(hs, hybi)
    return hs


# ---- level-local operators ------------------------------------------------------------------------------------------

def euler_step(hs, vstar, qn0, qsize, dt):
    """qtens = Qdp(qn0) - dt*div(vstar*Qdp(qn0)) (caar_oracle_euler_step) on [nets,nete) -> HP (E, qsize_d, L, 4, 4),
    zero outside the element range and past qsize. vstar: (E, L, 4, 4, 2) array."""
    E, Q, L = hs.nelem, hs.qsize_d, hs.nlev
    out = HP.input(np.zeros((E, Q, L, 4, 4)), hs.dtype)
    r = slice(hs.nets, hs.nete)
    if hs.nete <= hs.nets or qsize <= 0:
        return out
    vs = HP.input(vstar, hs.dtype)[r]
    q = hs.arrays["elem_state_Qdp"][r, :qsize, qn0]                     # (e, qsize, L, 4, 4)
    ex = lambda g: HP(g.v[:, None, None], g.M[:, None, None])           # geometry over tracers and levels
    div = divergence_sphere(HP(vs.v[:, None, ..., 0], vs.M[:, None, ..., 0]) * q,
                            HP(vs.v[:, None, ..., 1], vs.M[:, None, ..., 1]) * q, hs.dvv,
                            ex(hs.arrays["elem_Dinv"][r]), ex(hs.arrays["elem_metdet"][r]),
                            ex(hs.arrays["elem_rmetdet"][r]), hs.rrearth)
    out[r, :qsize] = q * 1.0 + (-HP.input(dt, hs.dtype)) * div
    return out


def sphere_wk(name, hs, field, tensorvisc=None, nets=None, nete=None):
    """divergence_sphere_wk (field (E, L, 4, 4, 2)) / laplace_simple / laplace_tensor (field (E, L, 4, 4), tensorvisc
    (E, 4, 4, 2, 2)) on [nets,nete) -> HP (E, L, 4, 4), zero outside (caar_oracle_sphere_wk)."""
    nets = hs.nets if nets is None else nets
    nete = hs.nete if nete is None else nete
    out = HP.input(np.zeros((hs.nelem, hs.nlev, 4, 4)), hs.dtype)
    if nete <= nets:
        return out
    r = slice(nets, nete)
    lv = lambda g: HP(g.v[:, None], g.M[:, None])
    f = HP.input(field, hs.dtype)[r]
    dinv, mp = lv(hs.arrays["elem_Dinv"][r]), lv(hs.arrays["elem_spheremp"][r])
    if name == "divergence_sphere_wk":
        out[r] = divergence_sphere_wk(f[..., 0], f[..., 1], hs.dvv, dinv, mp, hs.rrearth)
    else:
        tv = None if name == "laplace_simple" else lv(HP.input(tensorvisc, hs.dtype)[r])
        out[r] = laplace_wk(f, hs.dvv, dinv, mp, tv, hs.rrearth)
    return out


# ---- the gate -------------------------------------------------------------------------------------------------------

def ratio(g, ref):
    """|g - v| / (u M) per point, in longdouble; 0 where g == v, inf where M == 0 and g != v."""
    d = np.abs(np.asarray(g, dtype=np.longdouble) - ref.v.astype(np.longdouble))
    M = ref.M.astype(np.longdouble) * np.longdouble(U64)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(d == 0, np.longdouble(0), d / M)
    return np.where(np.isnan(r), np.inf, r)


def gate(g, ref, K):
    """True when |g - v| <= K u M at every point (equality where M == 0)."""
    return bool(np.all(ratio(g, ref) <= K))


def worst(g, ref):
    """(worst ratio, its index, |v|/M there) over the array."""
    r = ratio(g, ref)
    i = np.unravel_index(int(np.argmax(r)), r.shape)
    M = ref.M[i]
    return float(r[i]), tuple(int(x) for x in i), float(abs(ref.v[i]) / M) if M > 0 else float("nan")


def rel_err(a, b):
    """The field-normalised error max|a-b| / max|b| the parity tests gate on."""
    a, b = np.asarray(a, dtype=np.longdouble), np.asarray(b, dtype=np.longdouble)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), np.longdouble(1e-300)))
