"""Every pair kernel, particle by particle, against a float64 restatement of the reference formulas, across scene
parameters, particle counts and neighbourhood edges.

The fp32 oracle comparisons elsewhere divide the worst error by max|field|, so one dominant particle hides the
others.  Here each particle gets its own bound.

Reference (float64, numpy/scipy, in this file)
  * Inputs are the engine's fp32 state: positions, m_V, m, v and -- where a later kernel reads them -- the densities,
    factors and density changes the engine itself stored.
  * The neighbour set is the fp32 predicate of the engine and the reference: candidates from a cKDTree, kept when
    (rx*rx + ry*ry) + rz*rz < h2 evaluated in float32 without FMA (numpy rounds every float32 operation), h2 derived
    as derive_dev_params() derives it.  Neighbours in cell 0 are dropped: the reference's neighbour walk never sees
    cell 0 (SURVEY Q2).
  * Formulas: sph_base.py (W, grad W, Akinci volumes), WCSPH.py (density, Tait EOS, cohesion + viscosity, pressure
    and rigid reactions), DFSPH.py (factor, density change / advected density, Jacobi sweeps).

Bound.  For particle i with n_i neighbours the reference also returns a scale S_i: the sum of the absolute values of
the particle's terms with every kernel factor replaced by its bound over the support, |W| <= k and |grad W| <= k_dw / h
(k = 8 / (pi h^3), k_dw = 6 k), so that rounding inside (1 - q)^3 near q = 1 is covered.  Then

    |engine - ref64| <= (C0 + C1 n_i) u S_i + A_i,        u = 2^-24 (unit roundoff of float32).

  C0 (one term, relative to its bound): r_vec = x_i - x_j is one rounding (u), r2 three products and two sums (3u
  relative to r2, 1.5u on r), r = r2 * rsqrt_ftz(r2) and 1/r from MUFU.RSQ at ~2 ulp (4u), q = r * inv_h with a rounded
  inv_h (2u): |dq/q| <= ~10u.  |dW/dq| <= 2k and |d^2W/dq^2| <= 24k = 4 k_dw, so the kernel factors move by <= 20u k
  and <= 40u k_dw / h; evaluating the polynomials in float32 (<= 8 operations, constants k, k_dw, h rounded to float32)
  adds <= 12u of the bound; the products with m_V, rho0, the velocity dot product and the pressure / cohesion /
  viscosity coefficients (<= 8 roundings, __fdividef ~2 ulp) add <= 12u.  Sum <= 64u: C0 = 64.
  C1: the terms are accumulated one at a time in float32, in an order that differs from the reference's (centre
  column first, batched by four, atomics for the reactions); any order of recursive summation errs by at most
  (n - 1) u sum|terms|, and the final combination (the particle's own term, gravity, the clamp, v + dv) adds a few u
  more: C1 = 2.
  A_i carries the error of an fp32 input that the engine computed itself and the reference recomputes: the Tait EOS
  (below) and, in the fused step, the unclamped density of neighbours whose stored density was clamped.
Tait EOS: x = rho / rho0 is one rounding; x^gamma by the x^7 chain (4 multiplies), the integer loop (gamma - 1) or
powf (~4 ulp); then - 1 and * stiffness: |dp| <= (2 gamma + 16) u stiffness x^gamma.  The PRESSURE FIELD is compared
with p(rho_ref64) through dp/drho of the Tait law times the density bound, so (rho / rho0)^gamma is not counted twice.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
C0, C1 = 64.0, 2.0
GUARD = 1e-5  # r > 1e-5 gradient guard (sph_base.py:55); the engine's r2 > 1e-10f form agrees away from 1e-5 +- 1%


# ---------------------------------------------------------------------------------------------------------------
# scenes
# ---------------------------------------------------------------------------------------------------------------
def _scene(radius=0.01, fluid=(6, 6, 6), static=True, dynamic=True, cells=(15, 15, 15), dfsph=False,
           fluid_density=None, **cfg):
    """Fluid block next to a static and on top of it a dynamic rigid block, all sizes in particle diameters."""
    from sph_taichi_b200 import scene
    d = 2.0 * radius
    h = 2.0 * d
    sx, sy, sz = 2.5 * h, 1.5 * h, 2.5 * h
    sc = scene.dam_break_box(list(fluid), domain_end=[c * h for c in cells], start=[sx, sy, sz], radius=radius)
    blocks = []
    if static:
        x0 = sx + fluid[0] * d
        blocks.append({"objectId": 1, "start": [x0, sy, sz], "end": [x0 + 2.5 * d, sy + 5.5 * d, sz + 5.5 * d],
                       "translation": [0.0, 0.0, 0.0], "scale": [1, 1, 1], "velocity": [0.0, 0.0, 0.0],
                       "density": 1000.0, "color": [255, 255, 255], "isDynamic": False})
    if dynamic:
        y0 = sy + fluid[1] * d
        blocks.append({"objectId": 2, "start": [sx, y0, sz], "end": [sx + 3.5 * d, y0 + 2.5 * d, sz + 3.5 * d],
                       "translation": [0.0, 0.0, 0.0], "scale": [1, 1, 1], "velocity": [0.0, -0.5, 0.0],
                       "density": 600.0, "color": [255, 0, 0], "isDynamic": True})
    if blocks:
        sc["RigidBlocks"] = blocks
    if fluid_density is not None:
        sc["FluidBlocks"][0]["density"] = float(fluid_density)
    if dfsph:
        sc["Configuration"].update(simulationMethod=4, timeStepSize=0.004)
    sc["Configuration"].update(cfg)
    return sc


def _build(sc):
    from sph_taichi_b200 import ParticleSystem, SimConfig
    ps = ParticleSystem(SimConfig(sc))
    return ps, ps.build_solver()


def _perturb(ps, seed, amp=0.15, squeeze=0.93, vamp=0.5):
    """Jitter the dynamic particles by amp diameters, compress the fluid around its centre, random velocities."""
    rng = np.random.default_rng(seed)
    d = 2.0 * ps.particle_radius
    x, v = ps.x.to_numpy().copy(), ps.v.to_numpy().copy()
    dyn, fl = ps.is_dynamic.to_numpy().copy() != 0, ps.material.to_numpy().copy() == 1
    x[dyn] += (rng.uniform(-1, 1, size=(int(dyn.sum()), 3)) * amp * d).astype(np.float32)
    c = x[fl].mean(axis=0)
    x[fl] = ((x[fl] - c) * np.float32(squeeze) + c).astype(np.float32)
    v[dyn] += rng.uniform(-vamp, vamp, size=(int(dyn.sum()), 3)).astype(np.float32)
    ps.x.from_numpy(x)
    ps.v.from_numpy(v)


def _place(ps, x, seed=0, vamp=0.5):
    rng = np.random.default_rng(seed + 7919)  # not the stream the positions came from: v must not follow x
    ps.x.from_numpy(np.asarray(x, np.float32))
    ps.v.from_numpy(rng.uniform(-vamp, vamp, size=(len(x), 3)).astype(np.float32))


def _clusters(centres, counts, spread, seed):
    rng = np.random.default_rng(seed)
    return np.concatenate([np.asarray(c) + rng.uniform(-spread, spread, size=(k, 3))
                           for c, k in zip(centres, counts)]).astype(np.float32)


# ---------------------------------------------------------------------------------------------------------------
# fp64 reference
# ---------------------------------------------------------------------------------------------------------------
def _h2(h):
    """derive_dev_params: the smallest float32 t with sqrtf(t) >= h, so that r2 < h2 <=> sqrtf(r2) < h."""
    h = np.float32(h)
    t = np.float32(h * h)
    while np.sqrt(t) >= h:
        t = np.nextafter(t, np.float32(0))
    while np.sqrt(np.nextafter(t, np.float32(np.inf))) < h:
        t = np.nextafter(t, np.float32(np.inf))
    return np.nextafter(t, np.float32(np.inf))


def cells_of(x, h, g):
    c = (np.asarray(x, np.float32) / np.float32(h)).astype(np.int32)  # float32 division, truncation
    return (c[:, 0] * int(g[1]) + c[:, 1]) * int(g[2]) + c[:, 2]


class Pairs:
    """Directed neighbour pairs (i, j) under the fp32 predicate, j outside cell 0."""

    def __init__(self, x, h, g):
        from scipy.spatial import cKDTree
        x = np.ascontiguousarray(x, np.float32)
        n = len(x)
        self.cell = cells_of(x, h, g)
        p = cKDTree(x.astype(np.float64)).query_pairs(h * (1 + 1e-4), output_type="ndarray").reshape(-1, 2)
        I, J = np.concatenate([p[:, 0], p[:, 1]]), np.concatenate([p[:, 1], p[:, 0]])
        rv = x[I] - x[J]
        r2 = (rv[:, 0] * rv[:, 0] + rv[:, 1] * rv[:, 1]) + rv[:, 2] * rv[:, 2]
        keep = (r2 < _h2(h)) & (self.cell[J] != 0)
        I, J = I[keep], J[keep]
        o = np.lexsort((J, I))
        self.i, self.j = I[o], J[o]
        x64 = x.astype(np.float64)
        self.rv = x64[self.i] - x64[self.j]
        self.r = np.sqrt((self.rv ** 2).sum(axis=1))
        self.nn = np.bincount(self.i, minlength=n)
        self.n = n
        near = np.abs(self.r - GUARD) < 0.01 * GUARD
        assert not near.any(), "a pair sits on the gradient guard: the scene is ambiguous, move it"

    def sel(self, m):
        return self.i[m], self.j[m], self.rv[m], self.r[m]

    def sum(self, i, w):
        return np.bincount(i, weights=w, minlength=self.n)

    def vsum(self, i, w3):
        return np.stack([self.sum(i, w3[:, a]) for a in range(3)], axis=1)


class K:
    """Constants folded in double as the reference folds them (sph_base.py:11-21, WCSPH.py:9-14)."""

    def __init__(self, ps, solver):
        r = float(ps.particle_radius)
        self.h, self.d = 4.0 * r, 2.0 * r
        self.k = 8.0 / np.pi / self.h ** 3
        self.kdw = 6.0 * self.k
        self.gb = self.kdw / self.h  # bound of |grad W|
        self.rho0 = float(solver.density_0)
        self.ks = float(getattr(solver, "stiffness", 0.0))
        self.gam = float(getattr(solver, "exponent", 7.0))
        self.sigma = float(solver.surface_tension)
        self.dvisc = 2.0 * (3 + 2) * float(solver.viscosity)
        self.eps = 0.01 * self.h ** 2
        self.g = np.asarray(solver.g, np.float32).astype(np.float64).reshape(3)  # the engine's gravity is float32
        self.dt = float(solver.dt[None])
        self.grid = [int(v) for v in ps.grid_num]

    def W(self, r):
        q = r / self.h
        return np.where(q <= 0.5, self.k * (6.0 * q ** 3 - 6.0 * q ** 2 + 1.0), 2.0 * self.k * np.maximum(1.0 - q, 0.0) ** 3)

    def gs(self, r):
        """grad W = gs(r) * r_vec (sph_base.py:46-68)."""
        q = r / self.h
        s = np.where(q <= 0.5, self.kdw * q * (3.0 * q - 2.0), -self.kdw * np.maximum(1.0 - q, 0.0) ** 2)
        return np.where(r > GUARD, s / (np.where(r > 0, r, 1.0) * self.h), 0.0)

    def tait(self, rho):
        x = rho / self.rho0
        return self.ks * (x ** self.gam - 1.0)

    def tait_err(self, rho):
        """Absolute float32 error of the engine's EOS at a float32 density."""
        return (2.0 * self.gam + 16.0) * U * self.ks * (rho / self.rho0) ** self.gam

    def dtait(self, rho):
        return self.ks * self.gam * (rho / self.rho0) ** (self.gam - 1.0) / self.rho0


def _state(ps):
    f = lambda name: getattr(ps, name).to_numpy().copy()
    st = {k: f(k) for k in ("x", "v", "m", "m_V", "density", "material", "is_dynamic", "acceleration", "x_0",
                            "object_id")}
    st["fl"] = st["material"] == 1
    st["dyn_solid"] = (st["material"] == 0) & (st["is_dynamic"] != 0)
    st["static"] = (st["material"] == 0) & (st["is_dynamic"] == 0)
    return st


def ref_boundary_volume(c, P, st):
    """sph_base.py:91-113: m_V = 3 / (W(0) + sum_solid W)."""
    sol = ~st["fl"]
    i, j, _, r = P.sel(sol[P.i] & sol[P.j])
    D = c.k + P.sum(i, c.W(r))
    return 3.0 / D, 3.0 * c.k * (1.0 + P.nn) / D ** 2


def ref_density(c, P, st):
    """WCSPH.py:33-43 / DFSPH.py:39-47 (unclamped)."""
    mV = st["m_V"].astype(np.float64)
    rho = c.rho0 * (mV * c.k + P.sum(P.i, mV[P.j] * c.W(P.r)))
    S = c.rho0 * c.k * (mV + P.sum(P.i, mV[P.j]))
    return rho, S


def ref_non_pressure(c, P, st, vol, vol_rel=None):
    """WCSPH.py:88-140 (DFSPH.py:50-101): gravity + cohesion + viscosity over fluid neighbours.
    vol = m_j / rho_j (unclamped); vol_rel = relative uncertainty of vol where it is not an exact engine input."""
    fl = st["fl"]
    m, v = st["m"].astype(np.float64), st["v"].astype(np.float64)
    i, j, rv, r = P.sel(fl[P.i] & fl[P.j])
    coh = -(c.sigma / m[i] * m[j] * c.W(np.maximum(r, c.d)))[:, None] * rv
    vij = v[i] - v[j]
    vxy = (vij * rv).sum(axis=1)
    sv = c.dvisc * vol[j] * vxy / (r * r + c.eps) * c.gs(r)
    acc = c.g[None, :] + P.vsum(i, coh + sv[:, None] * rv)
    S = np.linalg.norm(c.g) + P.sum(i, c.sigma * m[j] / m[i] * c.k * r
                                    + c.dvisc * vol[j] * np.linalg.norm(vij, axis=1) * r / (r * r + c.eps) * c.gb)
    A = np.zeros(P.n) if vol_rel is None else P.sum(i, np.abs(sv) * r * vol_rel[j])
    acc[st["dyn_solid"]] = c.g
    acc[st["static"]] = 0.0
    return acc, S, A


def ref_pressure_acc(c, P, st, rho_c):
    """WCSPH.py:46-85: pressure acceleration of fluid particles (Akinci mirror for solid neighbours) and the reactions
    on dynamic rigid particles.  p comes from the engine's clamped float32 density through the fp64 EOS; A carries the
    engine's EOS rounding."""
    fl = st["fl"]
    mV = st["m_V"].astype(np.float64)
    rho_c = rho_c.astype(np.float64)
    p = np.where(fl, c.tait(rho_c), 0.0)
    dp = np.where(fl, p / rho_c ** 2, 0.0)
    ddp = np.where(fl, c.tait_err(rho_c) / rho_c ** 2, 0.0)
    m = fl[P.i]
    i, j, rv, r = P.sel(m)
    jf = fl[j]
    dpj = np.where(jf, dp[j], p[i] / c.rho0 ** 2)
    ddpj = np.where(jf, ddp[j], c.tait_err(rho_c[i]) / c.rho0 ** 2)
    gs = c.gs(r)
    coef = -c.rho0 * mV[j] * (dp[i] + dpj)
    f = (coef * gs)[:, None] * rv
    term_S = c.rho0 * mV[j] * (np.abs(dp[i]) + np.abs(dpj)) * c.gb
    term_A = c.rho0 * mV[j] * (ddp[i] + ddpj) * np.abs(gs) * r
    acc = P.vsum(i, f)
    S, A = P.sum(i, term_S), P.sum(i, term_A)
    # reactions: -f rho0 / rho_body on the dynamic rigid neighbour (WCSPH.py:66-68)
    dj = st["dyn_solid"][j]
    rb = st["density"].astype(np.float64)[j[dj]]
    react = P.vsum(j[dj], -f[dj] * (c.rho0 / rb)[:, None])
    nr = np.bincount(j[dj], minlength=P.n)
    SR = P.sum(j[dj], term_S[dj] * c.rho0 / rb)
    AR = P.sum(j[dj], term_A[dj] * c.rho0 / rb)
    return acc, S, A, react, SR, AR, nr


# ---------------------------------------------------------------------------------------------------------------
# comparison
# ---------------------------------------------------------------------------------------------------------------
def check(case, name, got, want, bound, mask):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    err = np.abs(got - want)
    if err.ndim == 2:
        err = err.max(axis=1)
    bound = np.broadcast_to(np.asarray(bound, np.float64), err.shape)
    mask = np.asarray(mask, bool)
    assert mask.any(), f"{case} {name}: no particle to check"
    ratio = np.where(mask, err / np.maximum(bound, 1e-300), 0.0)
    k = int(np.argmax(ratio))
    print(f"{case:28s} {name:22s} n={int(mask.sum()):5d}  worst error / bound = {ratio[k]:.3g}")
    assert ratio[k] <= 1.0, (f"{case} {name}: particle {k}: engine {got[k]} reference {want[k]} "
                             f"error {err[k]:.4g} > bound {bound[k]:.4g}")


def bnd(P, S, A=0.0):
    return (C0 + C1 * P.nn) * U * S + A


# ---------------------------------------------------------------------------------------------------------------
# WCSPH
# ---------------------------------------------------------------------------------------------------------------
def run_wcsph(case, ps, solver, fused):
    c = K(ps, solver)
    solver.initialize()
    st = _state(ps)
    P = Pairs(st["x"], c.h, c.grid)
    fl, dyn, static = st["fl"], st["dyn_solid"], st["static"]
    mv_ref, mv_S = ref_boundary_volume(c, P, st)
    rho64, rho_S = ref_density(c, P, st)
    rho_b = bnd(P, rho_S)
    # the volumes after initialize(); the fused step recomputes the moving ones on the same positions
    for kind, m in (("m_V static", static), ("m_V moving", dyn)):
        if m.any():
            check(case, kind, st["m_V"], mv_ref, bnd(P, mv_S), m)

    if not fused:
        solver.compute_densities()
        rho = ps.density.to_numpy().copy()
        check(case, "density", rho, rho64, rho_b, fl)
        solver.compute_non_pressure_forces()
        a_np = ps.acceleration.to_numpy().copy()
        vol = st["m"].astype(np.float64) / rho.astype(np.float64)  # m_j / rho_j: rho is the engine's own output
        np_ref, np_S, np_A = ref_non_pressure(c, P, st, vol)
        check(case, "non-pressure acc", a_np, np_ref, bnd(P, np_S, np_A), fl)
        assert np.array_equal(a_np[dyn], np.broadcast_to(c.g.astype(np.float32), a_np[dyn].shape))
        assert not a_np[static].any()
        solver.compute_pressure_forces()
        rho_c, p, a = ps.density.to_numpy().copy(), ps.pressure.to_numpy().copy(), ps.acceleration.to_numpy().copy()
        assert np.array_equal(rho_c[fl], np.maximum(rho[fl], np.float32(c.rho0)))
        pr, pr_S, pr_A, react, R_S, R_A, nr = ref_pressure_acc(c, P, st, rho_c)
        d_a = a.astype(np.float64) - a_np
        slack = 2 * U * np.abs(a).max(axis=1)
        check(case, "pressure acc", d_a, pr, bnd(P, pr_S, pr_A) + slack, fl)
    else:
        solver.step()
        assert ps._engine.check_status() == 0
        rho_c, p, a = ps.density.to_numpy().copy(), ps.pressure.to_numpy().copy(), ps.acceleration.to_numpy().copy()
        check(case, "density (clamped)", rho_c, np.maximum(rho64, c.rho0), rho_b, fl)
        mv = ps.m_V.to_numpy().copy()
        for kind, m in (("m_V static", static), ("m_V moving", dyn)):
            if m.any():
                check(case, kind + " (step)", mv, mv_ref, bnd(P, mv_S), m)
        # viscosity reads m / rho with the UNCLAMPED density; where the stored one was clamped, take the reference's
        clamped = rho_c <= np.float32(c.rho0)
        rho_u = np.where(clamped, rho64, rho_c.astype(np.float64))
        vol = st["m"].astype(np.float64) / rho_u
        vol_rel = np.where(clamped, rho_b / rho64, 0.0)
        np_ref, np_S, np_A = ref_non_pressure(c, P, st, vol, vol_rel)
        pr, pr_S, pr_A, react, R_S, R_A, nr = ref_pressure_acc(c, P, st, rho_c)
        check(case, "acceleration", a, np_ref + pr, bnd(P, np_S + pr_S, np_A + pr_A) + U * np.abs(a).max(axis=1), fl)
        # fused advect: v' = v + dt a (only particles the wall clamp left alone)
        pad, hi = np.float32(c.h), (np.asarray(ps.domain_size, np.float64) - c.h).astype(np.float32)
        x1 = ps.x.to_numpy().copy()
        inside = fl & (x1 > pad).all(axis=1) & (x1 < hi).all(axis=1)
        v1 = ps.v.to_numpy().copy()
        v0 = st["v"].astype(np.float64)
        a_b = bnd(P, np_S + pr_S, np_A + pr_A)
        v_b = c.dt * a_b + 2 * U * (np.abs(v0).max(axis=1) + c.dt * np.abs(a).max(axis=1))
        if inside.any():
            check(case, "velocity after advect", v1, v0 + c.dt * (np_ref + pr), v_b, inside)
    # pressure field: through dp/drho of the Tait law
    rho_hi = np.maximum(rho64 + rho_b, c.rho0)
    p_b = c.dtait(rho_hi) * rho_b + c.tait_err(rho_hi)
    check(case, "pressure", p, c.tait(np.maximum(rho64, c.rho0)), p_b, fl)
    if dyn.any():
        hit = dyn & (nr > 0)
        a_dyn = a.astype(np.float64) - c.g
        R_b = (C0 + C1 * nr) * U * R_S + R_A + 2 * U * np.abs(a).max(axis=1)
        check(case, "rigid reactions", a_dyn, react, R_b, dyn)
        assert hit.any() and np.abs(react[hit]).max() > 0.0
    return c, P, st


# parameter matrix: (case id, scene keyword arguments, solver attributes set after construction)
G = 9.81
PARAM_CASES = [
    ("base", {}, {}),
    ("radius_0.0125", {"radius": 0.0125}, {}),
    ("radius_0.007", {"radius": 0.007}, {}),
    ("exponent_1", {"exponent": 1}, {}),
    ("exponent_3", {"exponent": 3}, {}),
    ("exponent_7.5", {"exponent": 7.5}, {}),
    ("density0_800", {"density0": 800, "fluid_density": 800.0}, {}),
    ("gravity_-x", {"gravitation": [-G, 0.0, 0.0]}, {}),
    ("gravity_0", {"gravitation": [0.0, 0.0, 0.0]}, {}),
    ("stiffness_visc_tension", {"stiffness": 3000}, {"viscosity": 0.05, "surface_tension": 0.3}),
]


@pytest.mark.parametrize("fused", [False, True], ids=["methods", "fused_step"])
@pytest.mark.parametrize("case,kw,attrs", PARAM_CASES, ids=[p[0] for p in PARAM_CASES])
def test_wcsph_fp64_params(case, kw, attrs, fused):
    ps, solver = _build(_scene(**kw))
    _perturb(ps, seed=[p[0] for p in PARAM_CASES].index(case) + 1, squeeze=0.9)  # independent jitter per case
    for k, v in attrs.items():  # after construction, before the first engine call: must reach the (graph) step
        setattr(solver, k, v)
    run_wcsph(case, ps, solver, fused)


def test_wcsph_solver_attributes_reach_the_oracle():
    """solver.viscosity / surface_tension assigned after construction: the fused graph-replayed step against the fp32
    oracle given the same constants (the oracle pins the visiting order)."""
    from oracle.sph_oracle import OracleSim
    sc = _scene(stiffness=3000)
    ps, solver = _build(sc)
    _perturb(ps, seed=3)
    o = OracleSim(sc)
    o.x[:] = ps.x.to_numpy().copy()
    o.v[:] = ps.v.to_numpy().copy()
    solver.viscosity, solver.surface_tension = 0.05, 0.3
    o.P.viscosity, o.P.surface_tension = 0.05, 0.3
    solver.initialize(); o.initialize()
    solver.step(); o.step()
    assert np.array_equal(ps.x_0.to_numpy().copy(), o.x_0)
    a, ao = ps.acceleration.to_numpy().copy(), o.acceleration
    assert np.abs(a - ao).max() <= 1e-4 * np.abs(ao).max()
    assert np.abs(ps.density.to_numpy().copy() - o.density).max() <= 2e-5 * np.abs(o.density).max()


def test_wcsph_fp64_two_densities_general_kernel():
    """Non-uniform fluid masses: the fused step takes k_force_general."""
    sc = _scene(static=True, dynamic=True)
    second = dict(sc["FluidBlocks"][0])
    d = 0.02
    s = sc["FluidBlocks"][0]["start"]
    second.update({"objectId": 3, "start": [s[0], s[1], s[2] + 6 * d], "end": [s[0] + 5.5 * d, s[1] + 3.5 * d, s[2] + 9.5 * d],
                   "density": 800.0})
    sc["FluidBlocks"].append(second)
    for fused in (False, True):
        ps, solver = _build(sc)
        _perturb(ps, seed=21, squeeze=0.92)
        run_wcsph(f"two_densities_{'fused' if fused else 'methods'}", ps, solver, fused)
        assert len(np.unique(ps.m.to_numpy().copy()[ps.material.to_numpy().copy() == 1])) == 2


# ---------------------------------------------------------------------------------------------------------------
# integer edges
# ---------------------------------------------------------------------------------------------------------------
def _fluid_only(n, radius=0.01, cells=(12, 12, 12), **cfg):
    """n fluid particles (positions set by the caller)."""
    from sph_taichi_b200 import scene
    h = 4 * radius
    sc = scene.dam_break_box([n, 1, 1], domain_end=[max(c * h, (n + 8) * 2 * radius) if a == 0 else c * h
                                                    for a, c in enumerate(cells)], start=[3 * h, 3 * h, 3 * h],
                             radius=radius)
    sc["Configuration"].update(cfg)
    return sc


def _scatter(ps, n, seed, mean_nbrs=30.0):
    """n particles uniformly in a cube around the domain centre, at about mean_nbrs neighbours each."""
    h = 4 * ps.particle_radius
    side = max(h, (n * 4.19 / mean_nbrs) ** (1 / 3) * h)
    ctr = np.asarray(ps.domain_size, np.float64) * 0.5
    rng = np.random.default_rng(seed)
    return (ctr + rng.uniform(-0.5, 0.5, size=(n, 3)) * side).astype(np.float32)


@pytest.mark.parametrize("fused", [False, True], ids=["methods", "fused_step"])
@pytest.mark.parametrize("n", [1, 31, 33, 127, 129, 257])
def test_wcsph_fp64_particle_counts(n, fused):
    ps, solver = _build(_fluid_only(n))
    _place(ps, _scatter(ps, n, seed=n), seed=n)
    run_wcsph(f"fluid_only_n{n}", ps, solver, fused)


@pytest.mark.parametrize("fused", [False, True], ids=["methods", "fused_step"])
def test_wcsph_fp64_one_fluid_among_solids(fused):
    sc = _scene(fluid=(1, 1, 1))
    ps, solver = _build(sc)
    x = ps.x.to_numpy().copy()
    fl = ps.material.to_numpy().copy() == 1
    solid = ~fl
    d = 0.02
    # next to the static block's face, and touching the dynamic block
    x[fl] = x[solid & (ps.object_id.to_numpy().copy() == 1)].min(axis=0) + np.float32([-0.7 * d, 2.2 * d, 2.4 * d])
    _place(ps, x, seed=1)
    c, P, st = run_wcsph("one_fluid_among_solids", ps, solver, fused)
    assert int(P.nn[st["fl"]][0]) > 10 and (~st["fl"][P.j[st["fl"][P.i]]]).all()


@pytest.mark.parametrize("fused", [False, True], ids=["methods", "fused_step"])
def test_wcsph_fp64_unjittered_lattice(fused):
    """Exact lattice: many pairs at r = h (outside by the fp32 predicate or inside by a rounding) and at r = d, some
    of them with r2 == d2 exactly in float32, where cohesion switches between W(r) and W(d).

    The switch points r2 > d2 (cohesion) and q <= 1/2 (W) are continuous in value: at r = d, q = d / h = 1/2 and both
    branches of W give k / 4 (k (6/8 - 6/4 + 1) = 2k (1/2)^3, exactly, also in float32).  Moving either comparison by
    its equality case therefore changes results by rounding only (at most a few ulp of one term), which no bound that
    must absorb the MUFU.RSQ error of every other pair can see; a bit-exact check would have to predict the rsqrt
    approximation of each target.  What this test pins is that the neighbourhood of those switch points is
    evaluated to within the per-particle bound."""
    ps, solver = _build(_scene())
    c, P, st = run_wcsph("lattice", ps, solver, fused)
    at_d = np.abs(P.r - c.d) < 1e-6 * c.d
    at_h = np.abs(P.r - c.h) < 1e-6 * c.h
    print("lattice pairs at r = d:", int(at_d.sum()), " at r = h (inside by rounding):", int(at_h.sum()))
    assert at_d.sum() > 100
    x = st["x"]
    rv = x[P.i] - x[P.j]
    r2 = (rv[:, 0] * rv[:, 0] + rv[:, 1] * rv[:, 1]) + rv[:, 2] * rv[:, 2]
    fluid_pair = st["fl"][P.i] & st["fl"][P.j]
    assert (fluid_pair & (r2 == np.float32(c.d) * np.float32(c.d))).sum() > 10


@pytest.mark.parametrize("fused", [False, True], ids=["methods", "fused_step"])
def test_wcsph_fp64_close_pairs(fused):
    """Coincident pairs and pairs just inside and just outside the r > 1e-5 gradient guard."""
    ps, solver = _build(_scene())
    _perturb(ps, seed=8)
    x = ps.x.to_numpy().copy()
    fl = np.nonzero(ps.material.to_numpy().copy() == 1)[0]
    for (a, b), off in zip(((fl[0], fl[1]), (fl[10], fl[11]), (fl[20], fl[21]), (fl[30], fl[31])),
                           ([0, 0, 0], [0.6e-5, 0, 0], [0, 1.6e-5, 0], [0.3e-5, 0.3e-5, 0.3e-5])):
        x[a] = x[b] + np.float32(off)
    _place(ps, x, seed=8)
    c, P, st = run_wcsph("close_pairs", ps, solver, fused)
    assert (P.r == 0).sum() >= 2 and ((P.r > 0) & (P.r < GUARD)).sum() >= 4 and ((P.r > GUARD) & (P.r < 2e-5)).sum() >= 2


@pytest.mark.parametrize("fused", [False, True], ids=["methods", "fused_step"])
def test_wcsph_fp64_cell_zero_and_last_layers(fused):
    """Particles in cell 0 (invisible as neighbours, SURVEY Q2) and in the last cell layer of each axis (k_hi clamp)."""
    n = 60
    ps, solver = _build(_fluid_only(n, cells=(10, 9, 11)))
    h = 4 * ps.particle_radius
    g = np.asarray(ps.grid_num, np.float64)
    top = (g - 0.5) * h
    mid = g * h * 0.5
    centres = [[0.6 * h] * 3, [top[0], mid[1], mid[2]], [mid[0], top[1], mid[2]], [mid[0], mid[1], top[2]], top]
    x = _clusters(centres, [12] * 5, 0.45 * h, seed=4)
    x = np.minimum(np.maximum(x, 0.0), (g * h - 1e-4)).astype(np.float32)
    _place(ps, x, seed=4)
    c, P, st = run_wcsph("cell0_last_layers", ps, solver, fused)
    cell = P.cell
    assert (cell == 0).sum() >= 2 and (P.nn[cell == 0] > 0).any()
    ck = (st["x"] / np.float32(c.h)).astype(np.int32)
    for ax in range(3):
        assert (ck[:, ax] == c.grid[ax] - 1).sum() >= 3, ax


@pytest.mark.parametrize("fused", [False, True], ids=["methods", "fused_step"])
def test_wcsph_fp64_overflowed_lists(fused):
    """Fluid squeezed to ~3.7 rho0: most particles have more than NBR_CAP = 96 neighbours and take the 27-cell
    fallback of the list walk."""
    ps, solver = _build(_scene(dynamic=False, stiffness=5))
    _perturb(ps, seed=11, amp=0.1, squeeze=0.6)
    c, P, st = run_wcsph("overflowed_lists", ps, solver, fused)
    assert (P.nn[st["fl"]] > 96).sum() > 20
    if fused:
        assert ps._engine.neighbor_stats()["overflow"] > 20


def test_dfsph_fp64_overflowed_lists():
    ps, s = _build(_scene(dfsph=True))
    _perturb(ps, seed=12, amp=0.1, squeeze=0.6)
    run_dfsph("dfsph_overflowed_lists", ps, s)
    assert ps._engine.neighbor_stats()["overflow"] > 20


def _win_cap_column(dfsph=False):
    """A sparse column (one particle per z cell) next to a dense one (five per z cell): a warp of the sparse column
    spans 32 z cells, so its staged window over the dense column is ~34 * 5 > WIN_CAP = 128 particles, while no
    particle comes near NBR_CAP = 96 neighbours."""
    radius = 0.01
    h = 4 * radius
    nz = 70
    sc = _fluid_only(nz * 6, cells=(6, 6, nz + 2), **({"simulationMethod": 4, "timeStepSize": 0.004} if dfsph else {}))
    ps, solver = _build(sc)
    rng = np.random.default_rng(12)
    zc = np.arange(1, nz + 1)
    sparse = np.stack([np.full(nz, 2.5 * h), np.full(nz, 2.5 * h), (zc + 0.5) * h], 1)
    dense = np.repeat(np.stack([np.full(nz, 3.5 * h), np.full(nz, 2.5 * h), (zc + 0.5) * h], 1), 5, axis=0)
    x = np.concatenate([sparse, dense]) + rng.uniform(-0.3, 0.3, size=(6 * nz, 3)) * h
    _place(ps, x.astype(np.float32), seed=12)
    return ps, solver


def _max_union_window(ps):
    """Largest per-warp, per-column union of candidate ranges over the fluid lanes (the k_density_tma staging)."""
    x = ps.x.to_numpy().copy()
    fl = ps.material.to_numpy().copy() == 1
    ce = ps.grid_particles_num.to_numpy().copy()
    g = [int(v) for v in ps.grid_num]
    ci = np.clip((x / np.float32(4 * ps.particle_radius)).astype(np.int64), 0, np.array(g) - 1)
    best = 0
    for w0 in range(0, len(x), 32):
        lanes = [i for i in range(w0, min(w0 + 32, len(x))) if fl[i]]
        for dx in (-1, 0, 1):
            for dy in (-1, 0, 1):
                lo, hi = None, None
                for i in lanes:
                    a, b, k = ci[i, 0] + dx, ci[i, 1] + dy, ci[i, 2]
                    if not (0 <= a < g[0] and 0 <= b < g[1]):
                        continue
                    row = (a * g[1] + b) * g[2]
                    j0, j1 = ce[max(row + max(k - 1, 0) - 1, 0)], ce[row + min(k + 1, g[2] - 1)]
                    if j1 > j0:
                        lo = j0 if lo is None else min(lo, j0)
                        hi = j1 if hi is None else max(hi, j1)
                if lo is not None:
                    best = max(best, hi - lo)
    return best


def test_wcsph_fp64_window_longer_than_win_cap():
    ps, solver = _win_cap_column()
    c, P, st = run_wcsph("win_cap_column", ps, solver, fused=True)
    assert _max_union_window(ps) > 128
    assert ps._engine.neighbor_stats()["overflow"] == 0 and int(P.nn.max()) < 96


# ---------------------------------------------------------------------------------------------------------------
# DFSPH
# ---------------------------------------------------------------------------------------------------------------
def ref_dfsph_factor(c, P, st):
    """DFSPH.py:114-154: factor = -1 / (sum_fluid |grad_p_j|^2 + |sum_all grad_p_j|^2), 0 below 1e-6."""
    fl = st["fl"]
    mV = st["m_V"].astype(np.float64)
    gp = -(mV[P.j] * c.gs(P.r))[:, None] * P.rv
    sum_k = P.sum(P.i, np.where(fl[P.j], (gp ** 2).sum(axis=1), 0.0)) + (P.vsum(P.i, gp) ** 2).sum(axis=1)
    b = mV[P.j] * c.gb
    S_k = P.sum(P.i, b ** 2) + P.sum(P.i, b) ** 2 * 2.0  # |G|^2 error <= 2 |G| dG + dG^2 with |G| <= sum b
    f = np.where(sum_k > 1e-6, -1.0 / np.where(sum_k > 0, sum_k, 1.0), 0.0)
    err_k = (C0 + C1 * P.nn) * U * S_k
    # where the rounding of sum_k can decide the 1e-6 threshold either way, the factor is not defined to a bound
    sure = np.abs(sum_k - 1e-6) > err_k
    return f, err_k / np.maximum(sum_k - err_k, 1e-6) ** 2 + 2 * U * np.abs(f), sure


def ref_density_change(c, P, st, mode, rho=None, acc_in=None):
    """DFSPH.py:157-219.  mode 0: max(div, 0), zeroed below 20 neighbours; mode 1: max(rho / rho0 + dt div, 1)."""
    mV, v = st["m_V"].astype(np.float64), st["v"].astype(np.float64)
    vij = v[P.i] - v[P.j]
    acc = P.sum(P.i, mV[P.j] * (vij * P.rv).sum(axis=1) * c.gs(P.r))
    S = P.sum(P.i, mV[P.j] * np.linalg.norm(vij, axis=1) * c.gb)
    if mode == 0:
        return np.where(P.nn < 20, 0.0, np.maximum(acc, 0.0)), S, acc
    return np.maximum(rho / c.rho0 + c.dt * acc, 1.0), rho / c.rho0 + c.dt * S, acc


def ref_dfsph_sweep(c, P, st, factor, dadv, rho, mode):
    """DFSPH.py:278-311 (mode 0) / 354-389 (mode 1): v of fluid particles after one sweep, and the reactions."""
    fl = st["fl"]
    mV, v = st["m_V"].astype(np.float64), st["v"].astype(np.float64)
    boff = 0.0 if mode == 0 else 1.0
    kk = np.where(fl, (dadv.astype(np.float64) - boff) * factor, 0.0)
    i, j, rv, r = P.sel(fl[P.i])
    jf = fl[j]
    ksum = np.where(jf, kk[i] + kk[j], kk[i])
    on = np.where(jf, np.abs(ksum) > 1e-5, np.abs(kk[i]) > 1e-5)
    gradW = c.gs(r)[:, None] * rv
    dv = np.where(on[:, None], c.dt * (ksum * mV[j])[:, None] * gradW, 0.0)
    v1 = v + P.vsum(i, dv)
    S = np.abs(v).max(axis=1) + P.sum(i, np.where(on, c.dt * np.abs(ksum) * mV[j] * c.gb, 0.0))
    # reactions on dynamic rigid neighbours: -k_i rho_i m_V_j / rho_body grad W
    dj = st["dyn_solid"][j] & on
    rb = st["density"].astype(np.float64)[j[dj]]
    fr = -(kk[i[dj]] * rho[i[dj]] * mV[j[dj]] / rb)[:, None] * gradW[dj]
    react = P.vsum(j[dj], fr)
    SR = P.sum(j[dj], np.abs(kk[i[dj]] * rho[i[dj]]) * mV[j[dj]] / rb * c.gb)
    nr = np.bincount(j[dj], minlength=P.n)
    return v1, S, react, SR, nr


def run_dfsph(case, ps, s, check_nn_cut=False):
    c = K(ps, s)
    s.initialize()
    fl, dt = ps.material.to_numpy().copy() == 1, c.dt
    s.compute_densities()
    st = _state(ps)
    P = Pairs(st["x"], c.h, c.grid)
    rho64, rho_S = ref_density(c, P, st)
    rho = st["density"].astype(np.float64)
    check(case, "dfsph density", rho, rho64, bnd(P, rho_S), fl)
    s.compute_DFSPH_factor()
    f_ref, f_b, sure = ref_dfsph_factor(c, P, st)
    assert (fl & sure).sum() >= 0.9 * fl.sum(), "too many fluid particles on the 1e-6 factor threshold"
    check(case, "dfsph_factor", ps.dfsph_factor.to_numpy().copy(), f_ref, f_b, fl & sure)
    s.compute_density_change()
    dc_ref, dc_S, raw = ref_density_change(c, P, st, 0)
    check(case, "density_change", ps.density_adv.to_numpy().copy(), dc_ref, bnd(P, dc_S), fl)
    if check_nn_cut:
        for k in (19, 20, 21):  # the nn < 20 cut, from the fp32 pair set
            assert (fl & (P.nn == k)).sum() >= 5, k
        cut = fl & (P.nn == 19) & (raw > 10 * bnd(P, dc_S))
        kept = fl & (P.nn == 20) & (raw > 10 * bnd(P, dc_S))
        assert cut.any() and kept.any(), (np.bincount(P.nn[fl]), raw[fl & (P.nn == 19)], bnd(P, dc_S)[fl & (P.nn == 19)])
    s.multiply_time_step(ps.dfsph_factor, 1 / dt)
    factor = ps.dfsph_factor.to_numpy().copy().astype(np.float64)
    dadv = ps.density_adv.to_numpy().copy()
    s.divergence_solver_iteration_kernel()
    v1, S, _, _, _ = ref_dfsph_sweep(c, P, st, factor, dadv, rho, 0)
    check(case, "v divergence sweep", ps.v.to_numpy().copy(), v1, bnd(P, S), fl)
    s.multiply_time_step(ps.dfsph_factor, dt)
    s.compute_non_pressure_forces()
    st = _state(ps)  # v after the sweep
    vol = st["m"].astype(np.float64) / rho
    np_ref, np_S, np_A = ref_non_pressure(c, P, st, vol)
    a_np = ps.acceleration.to_numpy().copy()
    check(case, "dfsph non-pressure", a_np, np_ref, bnd(P, np_S, np_A), fl)
    s.predict_velocity()
    s.compute_density_adv()
    st = _state(ps)
    da_ref, da_S, _ = ref_density_change(c, P, st, 1, rho=rho)
    check(case, "density_adv", ps.density_adv.to_numpy().copy(), da_ref, bnd(P, da_S), fl)
    s.multiply_time_step(ps.dfsph_factor, 1 / dt ** 2)
    factor = ps.dfsph_factor.to_numpy().copy().astype(np.float64)
    dadv = ps.density_adv.to_numpy().copy()
    s.pressure_solve_iteration_kernel()
    v1, S, react, SR, nr = ref_dfsph_sweep(c, P, st, factor, dadv, rho, 1)
    check(case, "v pressure sweep", ps.v.to_numpy().copy(), v1, bnd(P, S), fl)
    dyn = st["dyn_solid"]
    if dyn.any():
        a = ps.acceleration.to_numpy().copy()
        R_b = (C0 + C1 * nr) * U * SR + 2 * U * np.abs(a).max(axis=1)
        check(case, "dfsph rigid reactions", a.astype(np.float64) - c.g, react, R_b, dyn)
        assert np.abs(react[dyn]).max() > 0.0
    return c, P, st


DFSPH_CASES = [("base", {}), ("radius_0.0125", {"radius": 0.0125}), ("density0_800", {"density0": 800, "fluid_density": 800.0}),
               ("gravity_-x", {"gravitation": [-G, 0.0, 0.0]})]


@pytest.mark.parametrize("case,kw", DFSPH_CASES, ids=[p[0] for p in DFSPH_CASES])
def test_dfsph_fp64_params(case, kw):
    ps, s = _build(_scene(dfsph=True, **kw))
    _perturb(ps, seed=5, squeeze=0.9)
    s.viscosity, s.surface_tension = 0.02, 0.05
    run_dfsph("dfsph_" + case, ps, s)


def test_dfsph_fp64_neighbour_count_cut():
    """A fluid-only scatter with particles of exactly 19, 20 and 21 neighbours: nn < 20 zeroes density_change."""
    n = 800
    ps, s = _build(_fluid_only(n, simulationMethod=4, timeStepSize=0.004))
    _place(ps, _scatter(ps, n, seed=19, mean_nbrs=20.0), seed=19, vamp=1.0)
    run_dfsph("dfsph_nn_19_20_21", ps, s, check_nn_cut=True)


def test_dfsph_fp64_close_pairs_and_win_cap_column():
    ps, s = _win_cap_column(dfsph=True)
    x = ps.x.to_numpy().copy()
    x[5] = x[400]
    x[6] = x[401] + np.float32([0.6e-5, 0, 0])
    _place(ps, x, seed=12)
    run_dfsph("dfsph_win_cap_close_pairs", ps, s)
    assert _max_union_window(ps) > 128 and ps._engine.neighbor_stats()["overflow"] == 0


# ---------------------------------------------------------------------------------------------------------------
# DFSPH loop controls: device loops, host loops and the oracle run the same sweeps
# ---------------------------------------------------------------------------------------------------------------
CONTROL_CASES = [
    ("max_iterations_0", {"m_max_iterations_v": 0, "m_max_iterations": 0}),
    ("max_iterations_1", {"m_max_iterations_v": 1, "m_max_iterations": 1}),
    ("max_iterations_2", {"m_max_iterations_v": 2, "m_max_iterations": 2}),
    ("no_divergence_solver", {"enable_divergence_solver": False}),
]


def _control_run(sc, attrs, mode, guess=None, steps=4):
    from oracle.sph_oracle import OracleSim
    if mode == "oracle":
        o = OracleSim(sc)
        _perturb_arrays(o.x, o.v, o.material, o.is_dynamic, sc)
        for k, v in attrs.items():
            if k == "enable_divergence_solver":
                if not v:
                    o.divergence_solve = lambda: setattr(o, "last_iterations_v", 0)
            else:
                setattr(o, k, v)
        o.last_iterations_v = 0
        o.initialize()
        counts = []
        for _ in range(steps):
            o.step()
            counts.append((o.last_iterations_v, o.last_iterations))
        return counts, None
    from sph_taichi_b200 import ParticleSystem, SimConfig
    ps = ParticleSystem(SimConfig(sc))
    s = ps.build_solver()
    x, v = ps.x.to_numpy().copy(), ps.v.to_numpy().copy()
    _perturb_arrays(x, v, ps.material.to_numpy().copy(), ps.is_dynamic.to_numpy().copy(), sc)
    ps.x.from_numpy(x); ps.v.from_numpy(v)
    s.device_side_loops = mode == "device"
    for k, val in attrs.items():
        setattr(s, k, val)
    s.initialize()
    counts = []
    for _ in range(steps):
        if guess is not None:
            s._sweeps_guess = list(guess)
        s.step()
        counts.append((s.last_iterations_v, s.last_iterations))
    assert ps._engine.check_status() == 0
    return counts, (ps.x.to_numpy().copy(), ps.v.to_numpy().copy(), ps.density.to_numpy().copy())


def _perturb_arrays(x, v, material, is_dynamic, sc):
    rng = np.random.default_rng(31)
    dyn = np.asarray(is_dynamic) != 0
    fl = np.asarray(material) == 1
    x[dyn] += (rng.uniform(-1, 1, size=(int(dyn.sum()), 3)) * 0.002).astype(x.dtype)
    c = x[fl].mean(axis=0)
    x[fl] = ((x[fl] - c) * 0.9 + c).astype(x.dtype)
    v[dyn] += rng.uniform(-0.5, 0.5, size=(int(dyn.sum()), 3)).astype(v.dtype)


def _control_scene():
    from sph_taichi_b200 import scene
    sc = scene.dam_break_box([10, 12, 9], domain_end=[0.6, 0.6, 0.5], start=[0.06, 0.06, 0.06])
    sc["Configuration"].update(simulationMethod=4, timeStepSize=0.004)
    return sc


@pytest.mark.parametrize("case,attrs", CONTROL_CASES, ids=[p[0] for p in CONTROL_CASES])
def test_dfsph_loop_controls(case, attrs):
    sc = _control_scene()
    dev, sd = _control_run(sc, attrs, "device")
    host, sh = _control_run(sc, attrs, "host")
    orc, _ = _control_run(sc, attrs, "oracle")
    print(case, "iterations (divergence, pressure) per step:", dev)
    assert dev == host == orc, (dev, host, orc)
    if attrs.get("enable_divergence_solver", True) is False:
        assert all(cv == 0 for cv, _ in dev)
    cap = attrs.get("m_max_iterations")
    if cap is not None:
        assert all(cp <= max(cap, 1) for _, cp in dev) and max(cp for _, cp in dev) == max(cap, 1)
    for a, b in zip(sd, sh):
        assert np.array_equal(a, b)


def test_dfsph_oversized_first_batch_leaves_the_state_unchanged():
    """Sweeps queued behind the converged one (first batch 64) return at once: same counts, bit-identical state."""
    sc = _control_scene()
    big, sb = _control_run(sc, {}, "device", guess=(64, 64))
    one, so = _control_run(sc, {}, "device", guess=(1, 1))
    assert big == one and max(cp for _, cp in big) < 64
    for a, b in zip(sb, so):
        assert np.array_equal(a, b)
