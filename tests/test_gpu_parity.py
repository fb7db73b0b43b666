"""GPU parity: the CUDA path (through the C ABI, csrc/liblfr_b200.so) against
the CPU oracle on identical inputs.

Tolerance: BASELINE.json north_star asks for keypoint displacements within
1e-4 px of the reference solve; 1 solver unit = 16 px
(reconstruction-scripts/colmap_utils.py:135-136), so 6.25e-6 units.  The
trajectory (per-component LM iteration count and termination reason) must be
identical as well.
"""
import sys

import numpy as np
import pytest

from conftest import get_problem

TOL_UNITS = 1e-4 / 16.0   # 1e-4 px

pytestmark = pytest.mark.gpu


def _compare(b200, oracle, p, **opts):
    pos_g, st_g = b200.solve(p, b200.default_options(**opts))
    pos_o, st_o = oracle.solve(p, oracle.default_options(n_threads=8, **opts))
    err = np.abs(pos_g - pos_o).max() if pos_g.size else 0.0
    assert err <= TOL_UNITS, "max |dx| = %.3e units (%.3e px)" % (err, err * 16)
    np.testing.assert_array_equal(st_g["termination"], st_o["termination"])
    np.testing.assert_array_equal(st_g["iterations"], st_o["iterations"])
    np.testing.assert_allclose(st_g["initial_cost"], st_o["initial_cost"], rtol=1e-10, atol=1e-14)
    np.testing.assert_allclose(st_g["final_cost"], st_o["final_cost"], rtol=1e-8, atol=1e-14)
    assert st_g["total_iterations"] == st_o["total_iterations"]
    assert st_g["n_solved"] == st_o["n_solved"]
    return err, st_g


def test_edge_eval_matches_oracle(b200, oracle):
    """K1: residual, Jacobian and robust weights per edge (cost.cc:13-48,78-90)."""
    from lfr_b200 import EDGE_DTYPE
    rng = np.random.default_rng(5)
    n = 20000
    e = np.zeros(n, dtype=EDGE_DTYPE)
    e["flow"] = rng.uniform(-0.5, 0.5, size=(n, 18)).astype(np.float32)
    e["sim"] = rng.uniform(0.5, 1.0, size=n).astype(np.float32)
    kind = rng.integers(1, 3, size=n).astype(np.uint8)
    xs = rng.uniform(-0.8, 0.8, size=(n, 2))          # beyond +-0.5 => clamped branch
    xs[:100] = np.sign(xs[:100]) * 0.5                 # exactly on the clamp boundary
    xd = rng.uniform(-1, 1, size=(n, 2))
    # small residuals so the Tukey inlier branch is exercised too
    e["flow"][: n // 2] *= 0.05
    xd[: n // 2] = xs[: n // 2] + rng.normal(0, 0.02, size=(n // 2, 2))
    rg, jg, rhog = b200.edge_eval(e, kind, xs, xd)
    ro, jo, rhoo = oracle.edge_eval(e, kind, xs, xd)
    np.testing.assert_allclose(rg, ro, rtol=0, atol=4e-16 * 4)
    np.testing.assert_allclose(jg, jo, rtol=0, atol=1e-14)
    np.testing.assert_allclose(rhog[:, :2], rhoo[:, :2], rtol=1e-13, atol=1e-18)


@pytest.mark.parametrize("cfg", ["cfg1", "cfg2", "cfg3", "cfg4"])
def test_solve_matches_oracle(b200, oracle, cfg):
    """BASELINE.json configs[0..3] at full size (cfg4 on one GPU here; its 4-GPU
    sharding is covered by the dist tests)."""
    _, p = get_problem(cfg)
    err, st = _compare(b200, oracle, p)
    print(cfg, "max err %.3e units" % err, "iters", st["total_iterations"], "kernel ms", st["kernel_ms"])


def test_solve_tukey_variant_2(b200, oracle):
    _, p = get_problem("cfg1")
    _compare(b200, oracle, p, tukey_variant=2)


def test_solve_nonzero_start_and_bounds(b200, oracle):
    """Start points outside the box are projected at iteration 0 (A.6)."""
    _, p = get_problem("cfg1")
    rng = np.random.default_rng(3)
    init = rng.uniform(-1.5, 1.5, size=(p.graph.n_nodes, 2))
    pos_g, st_g = b200.solve(p, positions=init)
    pos_o, st_o = oracle.solve(p, oracle.default_options(n_threads=1), positions=init)
    assert np.abs(pos_g - pos_o).max() <= TOL_UNITS
    np.testing.assert_array_equal(st_g["iterations"], st_o["iterations"])


def test_line_search_contraction_path(b200, oracle):
    """Large, inconsistent flows force Armijo contractions (cubic and, on the
    second contraction, quintic interpolation)."""
    from lfr_b200 import synth, build_problem
    ms = synth.generate("cfg1", seed=77)
    rng = np.random.default_rng(11)
    ms.disp1[:] = rng.uniform(-1.2, 1.2, size=ms.disp1.shape).astype(np.float32)
    ms.disp2[:] = rng.uniform(-1.2, 1.2, size=ms.disp2.shape).astype(np.float32)
    p = build_problem(ms)
    from oracle_util import LS_FAST, line_search_mode
    pos_g, st_g = b200.solve(p)
    pos_o, st_o = oracle.solve(p, oracle.default_options(n_threads=1))      # literal polynomial.cc
    assert st_o["total_line_search_steps"] > 0
    assert np.abs(pos_g - pos_o).max() <= TOL_UNITS
    np.testing.assert_array_equal(st_g["iterations"], st_o["iterations"])
    np.testing.assert_array_equal(st_g["termination"], st_o["termination"])
    # the NUMBER of contractions is compared with the formulation the kernel mirrors: in line searches
    # that are doomed to fail (steps shrinking towards 1e-9) Ceres' rank-truncated fit contracts at a
    # different pace than the true interpolant, without changing the outcome (see test_linesearch_modes.py)
    with line_search_mode(oracle, LS_FAST):
        pos_f, st_f = oracle.solve(p, oracle.default_options(n_threads=1))
    assert st_g["total_line_search_steps"] == st_f["total_line_search_steps"]
    assert np.abs(pos_g - pos_f).max() <= TOL_UNITS


def test_duplicate_pairs_take_the_serial_assembly_path(b200, oracle):
    """A pair listed twice duplicates every edge of its matches: the edge/twin
    pairing of the fast assembly does not hold and the kernel must fall back to
    its serial path, with the same answer as the oracle."""
    from lfr_b200 import MatchSet, build_problem, synth
    ms = synth.generate("cfg1", seed=21)
    dup = ms.select_pairs(np.array([0]))
    both = MatchSet.concatenate([ms, dup])
    p = build_problem(both)
    assert p.graph.n_edges == 2 * (ms.n_matches + dup.n_matches)
    _compare(b200, oracle, p)
    # the CTA tier's two-phase matvec (no block-CSR without clean twins)
    pos_g, st_g = b200.solve(p, b200.default_options(linear_solver=2))
    pos_o, st_o = oracle.solve(p, oracle.default_options(n_threads=1))
    assert np.abs(pos_g - pos_o).max() <= TOL_UNITS
    assert np.array_equal(st_g["iterations"], st_o["iterations"])


def test_dense_high_degree_small_component_does_not_fail_the_solve(b200, oracle):
    """ADVICE r1: a small component whose nodes carry thousands of directed out-edges (here: the same
    image pairs listed 45 times, as a densely matched dataset with many pair lists would) needs more
    shared memory per component than one SM has in every staging tier; the schedule must move it to a
    tier that keeps per-edge data in global memory (Cholesky warp kernel, then CTA tier) instead of
    returning LFR_EUNSUPPORTED for the whole dataset."""
    from lfr_b200 import MatchSet, build_problem, synth
    ms = synth.generate("cfg2", scale=0.01, seed=33)
    dense = MatchSet.concatenate([ms] + [ms.select_pairs(np.arange(ms.n_pairs))] * 44)
    p = build_problem(dense)
    deg = np.diff(p.graph.row_ptr.astype(np.int64))
    per_comp = np.array([deg[p.comp_nodes[p.comp_ptr[c]:p.comp_ptr[c + 1]].astype(int)].sum()
                         for c in range(p.n_components)])
    assert per_comp.max() * 176 > 227 * 1024            # staged records + per-edge scratch (176 B / edge) exceed one SM's shared memory
    _compare(b200, oracle, p)


def _compare_dbg(b200, oracle, p, debug_flags, **opts):
    """_compare with lfr_options.debug_flags set on the GPU side only (the oracle ignores them)."""
    pos_g, st_g = b200.solve(p, b200.default_options(debug_flags=debug_flags, **opts))
    pos_o, st_o = oracle.solve(p, oracle.default_options(n_threads=8, **opts))
    assert np.abs(pos_g - pos_o).max() <= TOL_UNITS
    np.testing.assert_array_equal(st_g["termination"], st_o["termination"])
    np.testing.assert_array_equal(st_g["iterations"], st_o["iterations"])
    return pos_g, st_g


@pytest.mark.parametrize("flags,cfg", [("FORCE_SMEM_CHOLESKY", "cfg1"), ("FORCE_SMEM_CHOLESKY", "cfg2"),
                                       ("FORCE_SMEM_CHOLESKY", "cfg3"), ("NO_TILE", "cfg4")])
def test_forced_fallback_tiers_match_oracle(b200, oracle, flags, cfg):
    """The shared-memory Cholesky warp kernel (solve_warp_kernel) is the tier for
    80 < n <= 96 unknowns and the fallback behind the register kernels; lfr_options.debug_flags
    (LFR_DBG_*) route the same scenes through it (cfg4 without the tile tier: v1 for
    32 < n <= 96; cfg2, the flagship scene, with every warp-tier component on it)."""
    from lfr_b200 import capi
    dbg = {"FORCE_SMEM_CHOLESKY": capi.DBG_FORCE_SMEM_CHOLESKY, "NO_TILE": capi.DBG_NO_TILE}[flags]
    _, p = get_problem(cfg)
    _compare_dbg(b200, oracle, p, dbg)


@pytest.mark.parametrize("cfg", ["cfg2", "cfg4", "ring60"])
def test_zero_copy_and_hbm_solves_are_bitwise_identical(b200, oracle, cfg):
    """The same solve with (a) TMA bulk staging from the caller's pinned buffers (zero-copy: edge
    records pulled over PCIe straight into shared memory, results written straight back), (b) the
    same through HBM: identical bits, both equal to the oracle to 1e-4 px.
    ring60 adds the CTA tier: its preparation kernel copies the kept records out of the pinned array."""
    import ctypes as C
    import torch
    from lfr_b200 import capi
    _, p = get_problem(cfg)
    pos_ref, st_ref = _compare_dbg(b200, oracle, p, capi.DBG_NO_ZERO_COPY)
    # pinned caller buffers -> zero-copy
    s, keep = b200.marshal(p)
    e_pin = torch.empty(keep["edges"].nbytes, dtype=torch.uint8).pin_memory()
    e_pin.numpy()[:] = keep["edges"].view(np.uint8).reshape(-1)
    s.edges = e_pin.data_ptr()
    N = p.graph.n_nodes
    pos_pin = torch.zeros(2 * N, dtype=torch.float64).pin_memory()
    st, bufs = b200.make_stats(p.n_components)
    o = b200.default_options()
    rc = b200.lib.lfr_solve(C.byref(s), C.byref(o), C.c_void_p(pos_pin.data_ptr()), C.byref(st))
    b200.check(rc, "lfr_solve")
    assert np.array_equal(pos_pin.numpy().reshape(N, 2), pos_ref)
    assert np.array_equal(bufs["iterations"], st_ref["iterations"])
    assert np.array_equal(bufs["termination"], st_ref["termination"])


def _quartic_cases(rng, n):
    """Quartics in the shapes the line search produces (derivative of a quintic
    interpolant on [1e-3, 0.6] x step) plus adversarial ones: complex pairs whose
    real part lies inside the interval, close root pairs, roots near the 31-cell grid."""
    coef, lohi = [], []
    for k in range(n):
        mode = k % 6
        if mode == 0:      # four real roots, anywhere
            r = rng.uniform(-0.5, 1.5, size=4)
            q = np.poly(r)
        elif mode == 1:    # two real + complex pair with its real part inside the interval
            a, b = rng.uniform(0.05, 0.55), 10.0 ** rng.uniform(-4, 0)
            q = np.real(np.poly([rng.uniform(-0.5, 1.5), rng.uniform(-0.5, 1.5), a + 1j * b, a - 1j * b]))
        elif mode == 2:    # two complex pairs
            a1, b1 = rng.uniform(0.0, 0.6), 10.0 ** rng.uniform(-3, 0)
            a2, b2 = rng.uniform(0.0, 0.6), 10.0 ** rng.uniform(-3, 0)
            q = np.real(np.poly([a1 + 1j * b1, a1 - 1j * b1, a2 + 1j * b2, a2 - 1j * b2]))
        elif mode == 3:    # a close pair (separation 1e-2 .. 1e-5) inside the interval
            c, sep = rng.uniform(0.05, 0.55), 10.0 ** rng.uniform(-5, -2)
            q = np.poly([c - sep / 2, c + sep / 2, rng.uniform(-0.5, 1.5), rng.uniform(-0.5, 1.5)])
        elif mode == 4:    # a root within 1e-9 of a grid point
            g = 1e-3 + (0.6 - 1e-3) * rng.integers(1, 30) / 31.0
            q = np.poly([g * (1 + rng.uniform(-1e-9, 1e-9)), rng.uniform(0, 0.6), rng.uniform(-1, 2), rng.uniform(-1, 2)])
        else:              # random coefficients
            q = rng.normal(size=5)
        q = q * (10.0 ** rng.uniform(-3, 3)) * rng.choice([-1.0, 1.0])
        coef.append(q)
        lohi.append([1e-3, 0.6] if k % 2 == 0 else sorted(rng.uniform(-0.2, 1.2, size=2)))
    return np.ascontiguousarray(coef, dtype=np.float64), np.ascontiguousarray(lohi, dtype=np.float64)


def test_quartic_root_finders_agree(b200, oracle):
    """The line search's Budan-Fourier grid isolation (production) against the
    derivative recursion on the GPU and in the oracle (lfr_ref_polynomial_roots):
    same number of roots, every one a root to working precision (backward error
    <= 1e-12) and at the same place up to the conditioning of root clusters (1e-6);
    a pair of roots closer than 1e-6 (a near-double root, irrelevant to the
    minimisation) may be found by one route and not the other."""
    import ctypes as C
    rng = np.random.default_rng(99)
    n = 6000
    coef, lohi = _quartic_cases(rng, n)
    f = b200.lib.lfr_debug_quartic_roots
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_void_p]
    res = {}
    for use_grid in (0, 1):
        roots = np.zeros((n, 4))
        cnt = np.zeros(n, dtype=np.int32)
        assert f(coef.ctypes.data, lohi.ctypes.data, n, use_grid, roots.ctypes.data, cnt.ctypes.data) == 0
        res[use_grid] = (roots, cnt)
    ro = np.zeros((n, 8))
    co = np.zeros(n, dtype=np.int32)
    for k in range(n):
        co[k] = oracle.lib.lfr_ref_polynomial_roots(coef[k].ctypes.data, 5, float(lohi[k, 0]), float(lohi[k, 1]),
                                                    ro[k].ctypes.data)

    def same(k, ra, na, rb, nb):
        a, b = list(ra[:na]), list(rb[:nb])
        # every returned value is a root to working precision (backward error), whatever the
        # conditioning of a root cluster does to its position
        for r in a:
            mag = np.polyval(np.abs(coef[k]), abs(r))
            if abs(np.polyval(coef[k], r)) > 1e-12 * mag:
                return False
        if na == nb:
            return np.allclose(a, b, rtol=1e-6, atol=1e-9)
        # tolerate a missing near-double pair
        long_, short = (a, b) if na > nb else (b, a)
        if len(long_) - len(short) != 2:
            return False
        for i in range(len(long_) - 1):
            if abs(long_[i + 1] - long_[i]) <= 1e-6 * max(1.0, abs(long_[i])):
                rest = long_[:i] + long_[i + 2:]
                if np.allclose(rest, short, rtol=1e-6, atol=1e-9):
                    return True
        return False

    bad = [k for k in range(n) if not same(k, res[1][0][k], res[1][1][k], ro[k], co[k])]
    assert not bad, (len(bad), bad[:5], [(res[1][0][k][:res[1][1][k]], ro[k][:co[k]]) for k in bad[:3]])
    bad0 = [k for k in range(n) if not same(k, res[0][0][k], res[0][1][k], ro[k], co[k])]
    assert not bad0, (len(bad0), bad0[:5])
    assert (res[1][1] > 0).mean() > 0.4 and (res[1][1] >= 3).sum() > 100   # the cases do exercise multi-root cells


def _ls_cases(rng, n):
    """Line-search states {f0, g0, x1, f1, g1, three, x2, f2, g2, lo, hi}: random ones in Ceres'
    contraction range, and degenerate ones whose interpolant loses its leading coefficients
    exactly (samples of an exact quadratic / cubic with dyadic data -> the generic,
    leading-zero-stripping route of hermite_minimizer)."""
    rows = []
    for k in range(n):
        three = k % 2 == 1
        x2 = 10.0 ** rng.uniform(-3, 0)
        x1 = x2 * (rng.uniform(0.02, 0.6) if three else 1.0)
        if k % 10 < 8:
            f0, g0 = rng.normal(), -abs(rng.normal())
            f1, g1, f2, g2 = rng.normal(size=4) * np.array([1.0, 3.0 / x1, 1.0, 3.0 / x2])
        else:
            # exact low-degree polynomial, dyadic coefficients and abscissae
            x2 = 2.0 ** -int(rng.integers(0, 6))
            x1 = x2 * (0.5 if three else 1.0)
            deg = 2 if k % 10 == 8 else 3
            co = np.concatenate([np.zeros(3 - deg), rng.integers(-4, 5, size=deg + 1).astype(float)])
            if co[-2] >= 0:
                co[-2] = -1.0                      # descent direction at 0
            pl = np.poly1d(co)
            f0, g0 = pl(0.0), pl.deriv()(0.0)
            f1, g1, f2, g2 = pl(x1), pl.deriv()(x1), pl(x2), pl.deriv()(x2)
        rows.append([f0, g0, x1, f1, g1, 1.0 if three else 0.0, x2 if three else 0.0, f2 if three else 0.0,
                     g2 if three else 0.0, 1e-3 * x1, 0.6 * x1])
    return np.ascontiguousarray(rows, dtype=np.float64)


def _ls_reference_poly(row):
    f0, g0, x1, f1, g1, three, x2, f2, g2, lo, hi = row
    pts = [(0.0, f0, g0), (x1, f1, g1)] + ([(x2, f2, g2)] if three else [])
    h = max(p[0] for p in pts)
    deg = 2 * len(pts) - 1
    A, b = [], []
    for (x, f, g) in pts:
        t = x / h
        A.append([t ** k for k in range(deg, -1, -1)])
        b.append(f)
        A.append([k * t ** (k - 1) if k > 0 else 0.0 for k in range(deg, -1, -1)])
        b.append(g * h)
    co = np.linalg.solve(np.array(A), np.array(b))
    return np.poly1d(co), h


def _check_ls(cases, x_test, x_oracle):
    same = np.isclose(x_test, x_oracle, rtol=1e-8, atol=0.0)
    for k in np.nonzero(~same)[0]:
        # a different abscissa is acceptable only where the interpolant takes the same value
        # (two candidates tie to rounding)
        pl, h = _ls_reference_poly(cases[k])
        scale = max(1.0, np.abs(pl.coeffs).max())
        assert abs(pl(x_test[k] / h) - pl(x_oracle[k] / h)) <= 1e-10 * scale, (k, x_test[k], x_oracle[k])
    assert same.mean() >= 0.995, same.mean()
    lo, hi = cases[:, 9], cases[:, 10]
    assert np.all((x_test >= lo) & (x_test <= hi))


def _oracle_ls(oracle, cases, fast):
    from oracle_util import minimize_interpolating
    return minimize_interpolating(oracle, cases, fast=fast)


def test_ls_minimizer_matches_oracle(b200, oracle):
    """The whole step-size selection of the Armijo line search (interpolant, critical
    points, candidate scan) on the GPU, case by case: against the oracle's FAST formulation (which
    the kernel mirrors operation for operation) on every state, and against the LITERAL
    polynomial.cc restatement (Vandermonde full-pivot LU + companion-matrix eigenvalues) on the
    states where Ceres' own fit keeps full numerical rank."""
    import ctypes as C
    from oracle_util import well_conditioned
    cases = _ls_cases(np.random.default_rng(4321), 5000)
    f = b200.lib.lfr_debug_ls_minimizer
    f.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p]
    xg = np.zeros(cases.shape[0])
    assert f(cases.ctypes.data, cases.shape[0], xg.ctypes.data) == 0
    _check_ls(cases, xg, _oracle_ls(oracle, cases, fast=True))
    wc = well_conditioned(cases)
    assert wc.sum() > 1000
    _check_ls(cases[wc], xg[wc], _oracle_ls(oracle, cases[wc], fast=False))


def test_ls_minimizer_on_harvested_states_matches_literal_oracle(b200, oracle):
    """Every interpolation state the line searches of cfg2 and the contraction fixture actually go
    through: the GPU's step equals the literal oracle's wherever Ceres' fit is well conditioned."""
    import ctypes as C
    from oracle_util import harvest_line_search_states, well_conditioned
    f = b200.lib.lfr_debug_ls_minimizer
    f.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p]
    for name, scale in (("cfg2", 1.0), ("cfg4", 0.5), ("ring60", 1.0)):
        _, p = get_problem(name, scale=scale)
        _, _, states = harvest_line_search_states(oracle, p, oracle.default_options(n_threads=8))
        states = np.ascontiguousarray(states[well_conditioned(states)])
        assert states.shape[0] > 10
        xg = np.zeros(states.shape[0])
        assert f(states.ctypes.data, states.shape[0], xg.ctypes.data) == 0
        _check_ls(states, xg, _oracle_ls(oracle, states, fast=False))


def test_cta_pcg_tier_on_large_components(b200, oracle):
    """Components with more than 96 unknowns (ring scene, up to 60 nodes) take the
    CTA tier: matrix-free block-Jacobi PCG to 1e-13 stands in for the exact solve."""
    _, p = get_problem("ring60")
    sizes = np.diff(p.comp_ptr.astype(np.int64))
    assert (sizes > 49).sum() > 50
    pos_g, st_g = b200.solve(p)
    pos_o, st_o = oracle.solve(p, oracle.default_options(n_threads=8))
    assert np.abs(pos_g - pos_o).max() <= TOL_UNITS
    big = sizes > 49
    # the linear solves agree to ~1e-12, so the trajectories coincide
    assert np.array_equal(st_g["iterations"][big], st_o["iterations"][big])
    assert np.array_equal(st_g["termination"], st_o["termination"])


def _per_component_agreement(p, pos_g, st_g, pos_o, st_o):
    err = np.zeros(p.n_components)
    for c in range(p.n_components):
        nodes = p.comp_nodes[p.comp_ptr[c]:p.comp_ptr[c + 1]].astype(int)
        err[c] = np.abs(pos_g[nodes] - pos_o[nodes]).max() if nodes.size else 0.0
    good = (err <= TOL_UNITS) & (st_g["iterations"] == st_o["iterations"]) & (st_g["termination"] == st_o["termination"])
    return good, err


def test_cta_pcg_tier_up_to_400_unknowns(b200, oracle):
    """Ring scene with components of up to ~200 nodes (~400 unknowns): block-Jacobi PCG, refined on
    the true residual to 2e-15, against the oracle's exact factorisation.  EVERY component within
    1e-4 px with identical iteration counts and termination reasons (round 1 needed a 99 % allowance
    at a 1e-13 residual: a few line searches forked on ~1e-12 differences in the step)."""
    _, p = get_problem("ring200")
    sizes = np.diff(p.comp_ptr.astype(np.int64))
    assert sizes.max() > 150
    pos_g, st_g = b200.solve(p)
    pos_o, st_o = oracle.solve(p, oracle.default_options(n_threads=8))
    good, err = _per_component_agreement(p, pos_g, st_g, pos_o, st_o)
    assert good.all(), (int((~good).sum()), err.max())


def test_madrid_topology_components_up_to_1000_nodes_match_oracle(b200, oracle):
    """BASELINE.json configs[4] topology (1000 images on a ring + random partners, cfg5) at 5 % of the
    keypoints: the size cap of solve.cc:586 is reached — components of up to 1000 nodes = 2000
    unknowns, ~100 of them above 500 nodes.  The 24 largest components and every 6th of the others
    are solved by the CTA tier and by the oracle (dense Cholesky: ~8 s per 1000-node component per
    core, which is why this is a subset): every one within 1e-4 px, identical iteration counts.
    (tools/gpu_cta_parity.py checks all 199 components: profiles/r02_cta_parity.json.)"""
    import copy
    import os
    from lfr_b200 import build_problem, synth
    p = build_problem(synth.generate("cfg5", scale=0.05))
    sizes = np.diff(p.comp_ptr.astype(np.int64))
    assert sizes.max() >= 990 and (sizes >= 500).sum() >= 50
    slots = sorted(set(range(24)) | set(range(24, p.n_components, 6)))      # dispatch list is size-descending
    q = copy.copy(p)
    ptr, nodes = [0], []
    for s_ in slots:
        nodes.append(p.comp_nodes[p.comp_ptr[s_]:p.comp_ptr[s_ + 1]])
        ptr.append(ptr[-1] + len(nodes[-1]))
    q.comp_ptr = np.array(ptr, np.uint32)
    q.comp_nodes = np.concatenate(nodes).astype(np.uint32)
    q.comp_order = p.comp_order[slots]
    pos_g, st_g = b200.solve(q)
    pos_o, st_o = oracle.solve(q, oracle.default_options(n_threads=min(len(slots), os.cpu_count() or 8)))
    good, err = _per_component_agreement(q, pos_g, st_g, pos_o, st_o)
    assert good.all(), (int((~good).sum()), err.max())
    assert st_g["total_iterations"] == st_o["total_iterations"] > 100


def test_forced_pcg_matches_cholesky_path(b200, oracle):
    """lfr_options.linear_solver = 2 sends every component through the PCG tier."""
    _, p = get_problem("cfg1")
    pos_g, st_g = b200.solve(p, b200.default_options(linear_solver=2))
    pos_o, st_o = oracle.solve(p, oracle.default_options(n_threads=1))
    assert np.abs(pos_g - pos_o).max() <= TOL_UNITS
    assert np.array_equal(st_g["iterations"], st_o["iterations"])
    from lfr_b200 import synth, build_problem
    p2 = build_problem(synth.generate("cfg2", scale=0.1, seed=3))
    pos_g, st_g = b200.solve(p2, b200.default_options(linear_solver=2))
    pos_o, st_o = oracle.solve(p2, oracle.default_options(n_threads=8))
    assert np.abs(pos_g - pos_o).max() <= TOL_UNITS
    assert np.array_equal(st_g["iterations"], st_o["iterations"])


def test_edge_cases_empty_zero_and_singletons(b200, oracle):
    """Empty graph, SKIP_REFINEMENT-style all-zero grids (compute_match_graph.py:150-152),
    a graph whose components are all single nodes, and roots-only components."""
    from lfr_b200 import MatchSet, build_problem, synth
    ms = synth.generate("cfg1")
    empty = build_problem(ms, banned_images=ms.image_names)
    pos, st = b200.solve(empty)
    assert pos.shape == (0, 2) and st["n_solved"] == 0
    zero = synth.generate("cfg1")
    zero.disp1[:] = 0
    zero.disp2[:] = 0
    p = build_problem(zero)
    pos, st = b200.solve(p)
    pos_o, st_o = oracle.solve(p)
    assert np.all(pos == 0) and np.array_equal(st["iterations"], st_o["iterations"])
    assert np.array_equal(st["termination"], st_o["termination"])
    # every component a singleton: nothing is solved, positions (even non-zero starts) are untouched
    q = build_problem(ms)
    import copy
    single = copy.copy(q)
    n = q.graph.n_nodes
    single.comp = np.arange(n, dtype=np.uint32)
    single.comp_ptr = np.arange(n + 1, dtype=np.uint32)
    single.comp_nodes = np.arange(n, dtype=np.uint32)
    single.comp_order = np.arange(n)
    init = np.random.default_rng(0).uniform(-2, 2, size=(n, 2))
    pos, st = b200.solve(single, positions=init)
    assert np.array_equal(pos, init) and st["n_solved"] == 0 and np.all(st["termination"] == 0)


def test_malformed_edges_are_reported(b200):
    """dst out of range / self edges are caught while the edges are staged on the device."""
    import copy
    _, p = get_problem("cfg1")
    bad = copy.copy(p)
    bad.graph = copy.copy(p.graph)
    e = p.graph.edges.copy()
    e["dst"][5] = p.graph.n_nodes + 7
    bad.graph.edges = e
    with pytest.raises(RuntimeError, match=r"\(-1\)"):
        b200.solve(bad)
    # the library stays usable afterwards
    pos, st = b200.solve(p)
    assert st["n_solved"] > 0


def test_malformed_edges_in_a_cta_tier_component_are_reported(b200):
    """The CTA tier's lists are built on the device (cta_prepare_kernel): a bad destination inside a
    large component raises the same LFR_EINVAL, through HBM and from pinned buffers."""
    import copy
    _, p = get_problem("ring60")
    sizes = np.diff(p.comp_ptr.astype(np.int64))
    c = int(np.argmax(sizes))
    v = int(p.comp_nodes[p.comp_ptr[c]])
    e0 = int(p.graph.row_ptr[v])
    assert p.graph.row_ptr[v + 1] > e0
    for bad_dst in (p.graph.n_nodes + 3, v):   # out of range, self edge
        bad = copy.copy(p)
        bad.graph = copy.copy(p.graph)
        e = p.graph.edges.copy()
        e["dst"][e0] = bad_dst
        bad.graph.edges = e
        with pytest.raises(RuntimeError, match=r"\(-1\)"):
            b200.solve(bad)
    pos, st = b200.solve(p)
    assert st["n_solved"] > 0 and np.isfinite(pos).all()


def test_option_variants(b200, oracle):
    """Non-default options travel through the ABI: iteration cap (NO_CONVERGENCE),
    tight tolerances, a smaller box, other loss widths."""
    _, p = get_problem("cfg1")
    for opts in (dict(max_num_iterations=2), dict(function_tolerance=1e-10, parameter_tolerance=1e-10),
                 dict(bound=0.2), dict(cauchy_a=0.1, tukey_a=0.2), dict(initial_trust_region_radius=1.0),
                 dict(min_relative_decrease=0.6)):
        pos_g, st_g = b200.solve(p, b200.default_options(**opts))
        pos_o, st_o = oracle.solve(p, oracle.default_options(n_threads=2, **opts))
        assert np.abs(pos_g - pos_o).max() <= TOL_UNITS, opts
        np.testing.assert_array_equal(st_g["iterations"], st_o["iterations"], err_msg=str(opts))
        np.testing.assert_array_equal(st_g["termination"], st_o["termination"], err_msg=str(opts))
    _, st = b200.solve(p, b200.default_options(max_num_iterations=2))
    assert (st["termination"] == 5).any()           # LFR_TERM_NO_CONVERGENCE
    pos, _ = b200.solve(p, b200.default_options(bound=0.2))
    assert np.abs(pos).max() <= 0.2


def test_active_bounds_and_clamped_grids(b200, oracle):
    """Flows three times larger than the box: solutions sit on the +-1 bounds and
    many evaluations happen in the clamped region of the interpolator."""
    from lfr_b200 import build_problem, synth
    ms = synth.generate("cfg2", scale=0.05, seed=12)
    ms.disp1 *= 3.0
    ms.disp2 *= 3.0
    p = build_problem(ms)
    err, st = _compare(b200, oracle, p)
    pos, _ = b200.solve(p)
    assert (np.abs(pos) == 1.0).sum() > 10


@pytest.mark.parametrize("seed", [101, 202, 303, 404, 505, 606])
def test_seed_fuzz(b200, oracle, seed):
    """Small random scenes of every family (exhaustive, sequential, ring)."""
    from lfr_b200 import build_problem, synth
    for cfg, scale in (("cfg2", 0.04), ("cfg4", 0.04), ("ring60", 0.3)):
        p = build_problem(synth.generate(cfg, scale=scale, seed=seed))
        pos_g, st_g = b200.solve(p)
        pos_o, st_o = oracle.solve(p, oracle.default_options(n_threads=8))
        sizes = np.diff(p.comp_ptr.astype(np.int64))
        err = np.zeros(p.n_components)
        for c in range(p.n_components):
            nodes = p.comp_nodes[p.comp_ptr[c]:p.comp_ptr[c + 1]].astype(int)
            err[c] = np.abs(pos_g[nodes] - pos_o[nodes]).max()
        good = (err <= TOL_UNITS) & (st_g["iterations"] == st_o["iterations"])
        assert good.all(), (cfg, seed, err.max())      # every tier, every component


@pytest.mark.parametrize("cfg,scale", [("cfg2", 0.3), ("cfg4", 0.25), ("ring60", 1.0)])
def test_multi_device_call_is_bitwise_identical_to_one_device(b200, cfg, scale):
    """lfr_solve_multi (one call, components LPT-packed over the devices, no collective): bitwise the
    result of lfr_solve, with page-locked buffers (zero-copy pulls / write-back) and with pageable ones
    (through HBM, merged on the host).  With one visible GPU the call is exercised with devices = [0]
    (ownership filter, merge and pinned paths); with more, over all of them."""
    import torch
    _, p = get_problem(cfg, scale=scale)
    pos1, st1 = b200.solve(p)
    n_dev = torch.cuda.device_count()
    sets = [[0]] + ([list(range(n_dev))] if n_dev > 1 else []) + ([[1, 0]] if n_dev > 1 else [])
    for devices in sets:
        for pinned in (True, False):
            pos, st = b200.solve_multi(p, devices, pinned=pinned)
            assert np.array_equal(pos, pos1), (devices, pinned)
            for k in ("iterations", "termination", "initial_cost", "final_cost"):
                assert np.array_equal(st[k], st1[k]), (k, devices, pinned)
            assert st["total_iterations"] == st1["total_iterations"] and st["n_solved"] == st1["n_solved"]
            m = st["multi"]
            assert sum(m["n_slots"]) == st1["n_solved"] and m["zero_copy"] == (1 if pinned else 0)
            if len(devices) > 1:
                assert min(m["n_slots"]) > 0 and max(m["n_edges"]) - min(m["n_edges"]) <= max(1, int(0.05 * sum(m["n_edges"])))


def test_solve_launcher_with_gpus_flag(tmp_path):
    """`solve --gpus N` (in-process multi-device call) writes the same SolutionFile bytes as one GPU."""
    import os
    import subprocess
    import torch
    from lfr_b200 import synth, wire
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    m = str(tmp_path / "m.pb")
    wire.write_matching_file(synth.generate("cfg2", scale=0.2), m)
    outs = []
    n = max(1, min(torch.cuda.device_count(), 4))
    for extra in ([], ["--gpus", str(n)]):
        o = str(tmp_path / ("s%d.pb" % len(outs)))
        r = subprocess.run([sys.executable, os.path.join(root, "multi-view-refinement", "build", "solve"),
                            "--matches_file", m, "--output_file", o] + extra, capture_output=True, text=True, cwd=root)
        assert r.returncode == 0, r.stderr
        outs.append(open(o, "rb").read())
    assert outs[0] == outs[1] and len(outs[0]) > 0


def test_plan_resolve_is_deterministic(b200):
    """Row-owned sums, no atomics: re-running the plan is bit-identical."""
    from lfr_b200.capi import Plan
    _, p = get_problem("cfg2")
    plan = Plan(b200, p)
    plan.solve()
    a, st = plan.download()
    plan.solve()
    b, _ = plan.download()
    assert np.array_equal(a, b)
    alg, one = plan.traffic()
    assert alg >= one > 0
    plan.close()
