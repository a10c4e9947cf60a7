"""k_ba_solve (the reduced camera system of LocalBA / BundleAdjustment / GlobalBundleAdjustemnt) past the config-4 size.

The kernel changes regime with n = 6 x active free key frames: panels staged in shared memory up to n = 378 (63 free KFs), read from L2
above that, and from n = 545 on the back substitution has rows >= 512 that its register-held rows do not cover. The dense entry
(Optimizer.solve_dense, the production launch) is checked against a long-double referee (tests/ba_solve_ref.py) and the oracle's LDL^T in
every regime, for bit identity across cluster sizes and stage modes, and for its failure path; LocalBA is checked end to end against the
oracle at 63 .. 129 free key frames."""
import numpy as np
import pytest

from cubemapslam_b200 import synth
from cubemapslam_b200._capi import CslamError

from . import ba_solve_ref as R
from .test_gpu_ba import _compare_ba, rel

pytestmark = pytest.mark.gpu

SIZES = [1, 6, 31, 32, 33, 64, 294, 378, 383, 384, 390, 516, 544, 545, 546, 774, 1200, 1536]
CLUSTERS = [1, 2, 4, 8, 16]
CAPACITY_N = 26112


@pytest.fixture(scope="module")
def opt():
    from cubemapslam_b200.optimizer import Optimizer
    o = Optimizer()
    yield o
    o.close()


def staged_fits(n):
    ldp = ((n + 1 + 8) + 3) & ~3
    return 2 * 32 * ldp * 8 + 8 * n <= 200 * 1024


def bits(x):
    return np.ascontiguousarray(x).view(np.uint64)


def solve_or_unschedulable(opt, Sg, stage, cluster):
    """x, failed; None where the device cannot co-schedule the (non-portable) cluster size, which is a property of the device."""
    try:
        return opt.solve_dense(Sg, stage=stage, cluster=cluster)
    except CslamError as e:
        if cluster > 8 and "cannot be scheduled" in str(e):
            return None
        raise


# ------------------------------------------------------------------------------------------------ accuracy
@pytest.mark.parametrize("fam", ["dense_spd", "ba_shaped", "graded"])
@pytest.mark.parametrize("n", SIZES)
def test_solve_accuracy(oracle, opt, fam, n):
    S = R.FAMILIES[fam](n); g = R.rhs(n)
    x, failed = opt.solve_dense(R.pack(S, g))
    assert not failed
    xs = R.reference_solve(S, g)
    eta = R.backward_error(S, g, x)
    assert eta <= 8 * n * R.U, eta / (n * R.U)
    msg = "%s n=%d eta=%.2e (%.3f n u)" % (fam, n, eta, eta / (n * R.U))
    if fam != "graded":
        k = R.kappa_inf(S)
        fe = R.forward_error(x, xs)
        assert fe <= k * n * R.U, (fe, k)
        xo, ok = oracle.ldlt_solve(S, g)
        assert ok
        # the oracle's x is itself rounded: against it the bound is the same plus the oracle's own distance to x* (triangle inequality;
        # at n = 1 the two solvers may round the single quotient to neighbouring doubles)
        fo = R.forward_error(x, xo)
        assert fo <= k * n * R.U + R.forward_error(xo, xs), (fo, k)
        msg += " fwd=%.2e (%.3g kappa n u) vs oracle %.2e, kappa_inf=%.2e" % (fe, fe / (k * n * R.U), fo, k)
    print(msg)


# ------------------------------------------------------------------------------------------------ bit identity
@pytest.mark.parametrize("n", SIZES)
def test_solve_bits_do_not_depend_on_cluster_or_staging(opt, n):
    """Per element the arithmetic order is fixed: cluster size only deals rows and tiles out differently, staging only changes where the same
    panel values are loaded from. So x is bitwise the same in every launch shape."""
    Sg = R.pack(R.ba_shaped(n), R.rhs(n))
    x0, f0 = opt.solve_dense(Sg, stage=-1, cluster=8)
    assert not f0
    x1, _ = opt.solve_dense(Sg, stage=-1, cluster=8)
    assert np.array_equal(bits(x0), bits(x1))                      # repeatable
    stages = [0, 1] if staged_fits(n) else [0]
    ran = []
    for c in CLUSTERS:
        for s in stages:
            r = solve_or_unschedulable(opt, Sg, s, c)
            if r is None:
                continue
            assert not r[1]
            assert np.array_equal(bits(r[0]), bits(x0)), (c, s)
            ran.append((c, s))
    print("n=%d ran (cluster, stage): %s" % (n, ran))
    assert {c for c, _ in ran} >= {1, 2, 4, 8}


# ------------------------------------------------------------------------------------------------ contract
@pytest.mark.parametrize("n", [33, 378, 384, 546, 1200])
def test_solve_reads_only_the_lower_triangle_and_rhs(opt, n):
    Sg = R.pack(R.dense_spd(n), R.rhs(n))
    P = Sg.copy(); P[:n][np.triu_indices(n, 1)] = np.nan
    x0, _ = opt.solve_dense(Sg)
    x1, failed = opt.solve_dense(P)
    assert not failed and np.array_equal(bits(x0), bits(x1))


def test_solve_ignores_a_stale_arena(opt):
    from cubemapslam_b200.optimizer import Optimizer
    bad = R.pack(R.dense_spd(1200), np.full(1200, np.nan))
    clean = R.pack(R.ba_shaped(700), R.rhs(700))
    opt.solve_dense(bad)
    x1, f1 = opt.solve_dense(clean)
    fresh = Optimizer()
    try:
        x2, f2 = fresh.solve_dense(clean)
    finally:
        fresh.close()
    assert not f1 and not f2 and np.array_equal(bits(x1), bits(x2))


# ------------------------------------------------------------------------------------------------ failure path
@pytest.mark.parametrize("n", [40, 546])
def test_solve_reports_bad_pivots_in_every_launch_shape(opt, n):
    """A zero / non-finite pivot breaks the factorisation in every CTA of the cluster alike and is reported (the LM rejects the trial)."""
    S = R.dense_spd(n); g = R.rhs(n)
    cases = [R.zero_pivot(S, k) for k in (0, 31, 32, 33, n - 1)]
    B = S.copy(); B[33, 33] = np.nan
    cases.append(B)
    stages = [-1, 0, 1] if staged_fits(n) else [-1, 0]
    for c in CLUSTERS:
        for s in stages:
            r = solve_or_unschedulable(opt, R.pack(S, g), s, c)
            if r is None:
                continue
            assert not r[1], (c, s)
            for i, A in enumerate(cases):
                assert opt.solve_dense(R.pack(A, g), stage=s, cluster=c)[1], (c, s, i)


# ------------------------------------------------------------------------------------------------ capacity
def test_solve_capacity_is_reported_before_reading(opt):
    n = CAPACITY_N + 1
    Sg = np.zeros((n + 1, n))             # 5.5 GB of lazily committed zeros: touching it would commit them
    with pytest.raises(CslamError, match=r"error -4: .*n <= 26112"):
        opt.solve_dense(Sg)
    with pytest.raises(CslamError, match="error -2"):
        opt.solve_dense(R.pack(R.dense_spd(384), R.rhs(384)), stage=1)
    assert staged_fits(378) and not staged_fits(384)


# ------------------------------------------------------------------------------------------------ end to end
def _problem(nQ, seed=8):
    """nQ free key frames plus two fixed ones (KF 0 and an lFixedCameras member opposite it on the ring). Not every draw is well posed: with one
    fixed key frame (free monocular scale) or on the seed-7 draw at 129 free KFs, the fp64 oracle run on a reordered edge list drifts from itself
    by up to 5e-6 (relative, points), more than the parity gates allow, so such a problem cannot tell a solver error from rounding. This draw is
    reproducible to ~1e-13, which the parity test checks."""
    nKF = nQ + 2
    p = synth.ba_problem(nKF=nKF, nMP=80 * nKF, kmin=2, kmax=12, faceW=650, seed=seed, radius=2.0)
    p["kf_fixed"][nKF // 2] = 1
    return p


@pytest.mark.parametrize("nQ", [63, 64, 91, 129])
def test_local_ba_parity_past_config4(oracle, opt, nQ):
    p = _problem(nQ)
    assert int((p["kf_fixed"] == 0).sum()) == nQ
    # the problem is well posed: the oracle agrees with itself on a reordered edge list far below the gates
    perm = np.random.default_rng(5).permutation(len(p["eMP"]))
    q = {k: np.ascontiguousarray(p[k][perm]) for k in ("eMP", "eKF", "kpxy", "inv_sigma2")}
    r1 = oracle.local_ba(p["Tcw"], p["kf_fixed"], p["pts"], q["eMP"], q["eKF"], q["kpxy"], q["inv_sigma2"], 650, 650)
    r, g = _compare_ba(oracle, opt, p)
    assert rel(r1["pose64"], r["pose64"]) < 1e-9 and rel(r1["pts64"], r["pts64"]) < 1e-9
    print("nQ=%d n=%d iters=%d pose rel %.2e points rel %.2e" % (nQ, 6 * nQ, r["iters"], rel(g["pose64"], r["pose64"]), rel(g["pts64"], r["pts64"])))


def test_local_ba_with_an_inactive_free_key_frame(oracle, opt):
    """A free key frame without edges is not in the system: n = 6 x 90 while the panel buffers are sized for the 91 candidates."""
    p = _problem(91)
    keep = p["eKF"] != 17
    for k in ("eMP", "eKF", "kpxy", "inv_sigma2"):
        p[k] = np.ascontiguousarray(p[k][keep])
    assert p["kf_fixed"][17] == 0
    _compare_ba(oracle, opt, p)


def test_local_ba_cluster_size_does_not_change_the_result(monkeypatch):
    from cubemapslam_b200.optimizer import Optimizer
    p = _problem(129)

    def run(cluster):
        if cluster is None:
            monkeypatch.delenv("CSLAM_SOLVE_CLUSTER", raising=False)
        else:
            monkeypatch.setenv("CSLAM_SOLVE_CLUSTER", str(cluster))
        o = Optimizer()
        try:
            if cluster and cluster > 8:
                Sg = R.pack(R.dense_spd(6 * 129), R.rhs(6 * 129))
                if solve_or_unschedulable(o, Sg, -1, cluster) is None:
                    return None
            return o.LocalBundleAdjustment(p["Tcw"], p["kf_fixed"], p["pts"], p["eMP"], p["eKF"], p["kpxy"], p["inv_sigma2"], 650, 650)
        finally:
            o.close()

    base = run(None)
    ran = []
    for c in (1, 4, 16):
        g = run(c)
        if g is None:
            continue
        ran.append(c)
        for k in ("pose64", "pts64", "log"):
            assert np.array_equal(bits(g[k]), bits(base[k])), (c, k)
        assert np.array_equal(g["outlier"], base["outlier"]) and g["trials"] == base["trials"], c
    print("LocalBA nQ=129 bitwise equal to cluster 8 at clusters %s" % ran)
    assert 1 in ran and 4 in ran
