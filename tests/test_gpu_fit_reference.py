"""The fit path's kernels against independent references, at the shapes, angles and edges where they
can go wrong without the C oracle noticing (its Jacobian is the kernel's formula):
  a. reproj_jtj (csrc/residual.cu) against oracle/fit_ref.py: complex-step Jacobian, fsum blocks,
     an entry-wise rounding bound;
  b. lm_schur + lm_update (csrc/lm.cu) against a dense solve of the damped arrowhead system, and
     their handling of failed Cholesky factors;
  c. calculate_errors against the oracle's raw sums and a numpy restatement of the distance term;
  d. the starting values (csrc/init.cu, lm.initial_guess) against the generating camera;
  e. the whole fit on noise-free data."""
import ctypes as C
import math

import numpy as np
import pytest

from oracle import fit_ref as fr
from oracle import oracle_c as oc

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

U = fr.U


@pytest.fixture(scope="module")
def cc():
    import cameracalibrations_b200 as m
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    m.context(0)
    return m


@pytest.fixture(scope="module")
def lm(cc):
    from cameracalibrations_b200 import lm
    return lm


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()


def _shared(intr):
    return intr[1], intr[2], intr[3], intr[4]


# ------------------------------------------------------------------ a. reproj_jtj
# (ncorners, nviews, k, aspect, checker_size, planar): every corner count of {1, 4, 31, 32, 33, 64, 65, 280,
# 2048} (lanes without a corner, partial lane sweeps) and every view count of {1, 3, 4, 5, 255, 256, 257, 1031}
# (partial 4-warp blocks, the 256-thread stride of the view reduction) at least once; views cycle through
# fit_ref.THETAS on random axes
JTJ_CASES = [
    (1, 1, 0.0, 1.0, 1.0, True),
    (4, 3, -0.3, 1.1, 0.025, True),
    (31, 4, 0.4, 1.0, 0.025, True),
    (32, 5, 0.0, 1.1, 1.0, True),
    (33, 257, -0.3, 1.0, 1.0, True),
    (64, 256, 0.4, 1.1, 0.025, True),
    (65, 255, 0.0, 1.0, 0.025, True),
    (280, 1031, -0.3, 1.1, 1.0, True),
    (2048, 5, 0.4, 1.0, 1.0, True),
    (280, 16, -0.12, 1.1, 0.025, False),
]


def _jtj_case(nc, nv, k, aspect, cs, planar):
    intr, views, obj, img = fr.case(nc, nv, k=k, aspect=aspect, checker_size=cs, planar=planar, seed=nc * 7 + nv)
    return intr, views, obj, img, fr.blocks(views, _shared(intr), cs, aspect, obj, img)


@pytest.mark.parametrize("nc,nv,k,aspect,cs,planar", JTJ_CASES)
def test_reproj_jtj_vs_reference(cc, nc, nv, k, aspect, cs, planar):
    intr, views, obj, img, ref = _jtj_case(nc, nv, k, aspect, cs, planar)
    pv, sh = cc.reproj_jtj(intr, aspect, _dev(views), _dev(obj), _dev(img))
    pv, sh = pv.cpu().numpy(), sh.cpu().numpy()
    tol_pv, tol_sh = fr.tolerance(ref, "per_view"), fr.tolerance(ref, "shared")
    bad = np.argwhere(np.abs(pv - ref["per_view"]) > tol_pv)
    assert bad.size == 0, [(int(v), int(e), fr.THETAS[v % len(fr.THETAS)], pv[v, e], ref["per_view"][v, e])
                           for v, e in bad[:8]]
    assert np.all(np.abs(sh - ref["shared"]) <= tol_sh), np.abs(sh - ref["shared"]) / tol_sh
    # the 6 x 6 block is exactly symmetric
    A = pv[:, :36].reshape(-1, 6, 6)
    assert np.array_equal(A, A.transpose(0, 2, 1))
    # the host form is the device form behind copies
    pv_h, sh_h = cc.reproj_jtj(intr, aspect, views, obj, img)
    assert np.array_equal(pv_h, pv) and np.array_equal(sh_h, sh)


def test_reproj_jtj_view_blocks_do_not_depend_on_neighbours(cc):
    """Permuting the views permutes the rows of per_view bit for bit."""
    intr, views, obj, img = fr.case(65, 255, k=-0.3, aspect=1.1, checker_size=0.025, seed=4)
    pv, _ = cc.reproj_jtj(intr, 1.1, _dev(views), _dev(obj), _dev(img))
    perm = np.random.default_rng(4).permutation(len(views))
    pvp, _ = cc.reproj_jtj(intr, 1.1, _dev(views[perm]), _dev(obj), _dev(img[perm]))
    assert torch.equal(pvp, pv[torch.from_numpy(perm).cuda()])


# ------------------------------------------------------------------ b. lm_schur + lm_update
def _arrowhead(pv, sh, lam):
    """the damped system (A + lam diag A) x = -g, dense"""
    nv = len(pv)
    n = 6 * nv + 4
    H, g = np.zeros((n, n)), np.zeros(n)
    for v in range(nv):
        s = slice(6 * v, 6 * v + 6)
        H[s, s] = pv[v, :36].reshape(6, 6)
        H[s, 6 * nv:] = pv[v, 36:60].reshape(6, 4)
        H[6 * nv:, s] = pv[v, 36:60].reshape(6, 4).T
        g[s] = pv[v, 60:66]
    H[6 * nv:, 6 * nv:] = sh[:16].reshape(4, 4)
    g[6 * nv:] = sh[16:20]
    H[np.diag_indices(n)] *= 1.0 + lam
    return H, -g


def _kept(nv, mask):
    return np.array(list(range(6 * nv)) + [6 * nv + a for a in range(4) if (mask >> a) & 1], dtype=int)


def _reference_solver(H, b, nv):
    """mask -> solution of the system with the masked shared parameters removed (their entries 0).
    Up to 20 views in mpmath at 40 digits by exact block elimination (at that precision the order of
    elimination cannot matter); above, float64 dense LU with one step of iterative refinement."""
    n = len(b)
    if nv > 20:
        def solve(mask):
            k = _kept(nv, mask)
            Hk, bk = H[np.ix_(k, k)], b[k]
            x = np.linalg.solve(Hk, bk)
            x = x + np.linalg.solve(Hk, bk - Hk @ x)
            out = np.zeros(n)
            out[k] = x
            return out
        return solve
    mpmath = pytest.importorskip("mpmath")
    with mpmath.workdps(40):
        M = lambda a: mpmath.matrix(np.asarray(a).tolist())
        S, s, Ys, zs = M(H[6 * nv:, 6 * nv:]), M(b[6 * nv:]), [], []
        for v in range(nv):
            sv = slice(6 * v, 6 * v + 6)
            Ainv = M(H[sv, sv]) ** -1
            Bv = M(H[sv, 6 * nv:])
            Y, z = Ainv * Bv, Ainv * M(b[sv])
            S -= Bv.T * Y
            s -= Bv.T * z
            Ys.append(Y)
            zs.append(z)

    def solve(mask):
        free = [a for a in range(4) if (mask >> a) & 1]
        with mpmath.workdps(40):
            Sk = mpmath.matrix([[S[i, j] for j in free] for i in free])
            di_k = mpmath.lu_solve(Sk, mpmath.matrix([s[i] for i in free]))
            di = mpmath.matrix(4, 1)
            for i, a in enumerate(free):
                di[a] = di_k[i]
            out = np.zeros(n)
            for v in range(nv):
                out[6 * v:6 * v + 6] = [float(x) for x in zs[v] - Ys[v] * di]
            out[6 * nv:] = [float(x) for x in di]
        return out
    return solve


def _step_case(nv, seed=0):
    intr, views, obj, img = fr.case(48, max(nv, 1), k=-0.12, aspect=1.0, checker_size=1.0,
                                    thetas=(0.3, 1.0, 0.05, 2.0), seed=seed)
    return intr, views[:nv], obj, img[:nv]


@pytest.mark.parametrize("nv", [0, 1, 15, 16, 17, 128, 129, 300])
@pytest.mark.parametrize("lam", [0.0, 1e-3, 1e3])
def test_lm_step_vs_dense_solve(cc, lm, nv, lam):
    """Every free_mask: di and the candidate views within c kappa u of the dense solution (kappa of the
    diagonally scaled system, the one Cholesky's error depends on); masked di exactly 0; delta[4] and
    delta[5] against fsum.  With no views (a rank that holds none) the shared block comes from other
    views: block 0 must still publish di."""
    intr, views, obj, img = _step_case(nv, seed=nv)
    if nv:
        pv, sh = cc.reproj_jtj(intr, 1.0, _dev(views), _dev(obj), _dev(img))
    else:
        i2, v2, o2, m2 = _step_case(3, seed=1)
        pv = torch.empty((0, 66), dtype=torch.float64, device="cuda")
        _, sh = cc.reproj_jtj(i2, 1.0, _dev(v2), _dev(o2), _dev(m2))
    vt = _dev(views.reshape(-1, 6))
    yz, schur = lm.lm_schur(pv, lam)
    assert schur[20].item() == 0.0
    if nv == 0:
        assert torch.all(schur == 0.0)
    pvn, shn = pv.cpu().numpy(), sh.cpu().numpy()
    H, b = _arrowhead(pvn, shn, lam)
    solve = _reference_solver(H, b, nv)
    # kappa of the diagonally scaled system; a masked system is a principal submatrix of it: no larger kappa
    sd = np.sqrt(np.diag(H))
    kappa = np.linalg.cond(H / sd[:, None] / sd[None, :])
    for mask in range(1, 16):
        cand, delta = lm.lm_update(sh, schur, lam, mask, yz, vt)
        d, cand = delta.cpu().numpy(), cand.cpu().numpy()
        x = solve(mask)
        de_ref = x[:6 * nv].reshape(nv, 6)
        assert d[6] == 1.0, (mask, d)
        for a in range(4):
            if not (mask >> a) & 1:
                assert d[a] == 0.0, (mask, d)
        # error in the norm of the diagonal scaling: |D^1/2 (x - x_ref)| <= c kappa_s u |D^1/2 x_ref| (+ rounding
        # of the candidate p + de)
        got = np.concatenate([(cand - views.reshape(-1, 6)).ravel(), d[:4]])
        slack = np.concatenate([2 * U * np.abs(views.reshape(-1)), np.zeros(4)])
        err = np.linalg.norm(sd * (got - x))
        bound = 64 * kappa * U * np.linalg.norm(sd * x) + np.linalg.norm(sd * slack)
        assert err <= bound, (mask, err, bound, kappa)
        rel = 64 * kappa * U + fr.gamma(6 * nv + 1)
        n_de = math.fsum((de_ref ** 2).ravel())
        assert abs(d[4] - n_de) <= 2 * rel * n_de + 1e-300, (d[4], n_de)
        n_p = math.fsum((views.reshape(-1) ** 2))
        assert abs(d[5] - n_p) <= fr.gamma(6 * nv + 1) * n_p


def test_lm_schur_counts_and_zeroes_indefinite_views(cc, lm):
    """Three of 40 views get an indefinite 6 x 6 block (a negative diagonal entry): schur[20] counts them,
    their yz rows are 0 and their Schur shares are exactly 0 -- the sums equal those of a run in which those
    views have A = I, B = 0, g = 0 (a share that is exactly zero), bit for bit."""
    intr, views, obj, img = _step_case(40, seed=3)
    pv, sh = cc.reproj_jtj(intr, 1.0, _dev(views), _dev(obj), _dev(img))
    badv = [3, 17, 38]
    pv_bad, pv_null = pv.clone(), pv.clone()
    for v in badv:
        pv_bad[v, 0] = -abs(pv_bad[v, 0].item()) - 1.0
        pv_null[v] = 0.0
        pv_null[v, 0:36:7] = 1.0
    for lam in (0.0, 1e-3):
        yz, schur = lm.lm_schur(pv_bad, lam)
        yz0, schur0 = lm.lm_schur(pv_null, lam)
        assert schur[20].item() == len(badv) and schur0[20].item() == 0.0
        assert torch.all(yz[badv] == 0.0)
        good = [v for v in range(40) if v not in badv]
        assert torch.equal(yz[good], yz0[good])
        assert torch.equal(schur[:20], schur0[:20])


def test_lm_update_singular_shared_system(cc, lm):
    """C' - S not positive definite: delta[6] == 0, di == 0 and the candidate views are the input views."""
    intr, views, obj, img = _step_case(17, seed=5)
    pv, sh = cc.reproj_jtj(intr, 1.0, _dev(views), _dev(obj), _dev(img))
    yz, schur = lm.lm_schur(pv, 1e-3)
    sh_bad = sh.clone()
    sh_bad[5] = -abs(sh_bad[5].item()) - 1e6            # (crow, crow)
    vt = _dev(views)
    for mask in (0b1111, 0b0010):
        cand, delta = lm.lm_update(sh_bad, schur, 1e-3, mask, yz, vt)
        d = delta.cpu().numpy()
        assert d[6] == 0.0 and np.all(d[:4] == 0.0) and d[4] == 0.0
        assert torch.equal(cand, vt)


# ------------------------------------------------------------------ c. calculate_errors
def _errors_case(n1, n2, nv, S, k, seed):
    rng = np.random.default_rng(seed)
    cs = 0.15
    intr = (1400.0, 1400.0, 540.0, 960.0, k, cs)
    a, b = np.arange(n1 * n2) % n1, np.arange(n1 * n2) // n1           # corner a fastest
    obj = np.stack([a * cs, b * cs, np.zeros(n1 * n2)], 1)
    dist = 3.0 * max(n1, n2) + 20.0
    views = np.concatenate([rng.normal(0, 0.15, (nv, 3)),
                            np.stack([-(n1 - 1) / 2 + rng.normal(0, 1, nv), -(n2 - 1) / 2 + rng.normal(0, 1, nv),
                                      dist + rng.uniform(0, 5, nv)], 1)], 1)
    img = np.empty((nv, n1 * n2, 2))
    for v in range(nv):
        img[v, :, 0], img[v, :, 1] = oc.world2img(oc.chain(intr, views[v, :3], views[v, 3:]), obj)
    img += rng.normal(0, 0.25, img.shape)
    samples = np.stack([rng.uniform(1, 1080, (nv, S)), rng.uniform(1, 1920, (nv, S))], -1)
    return intr, views, obj, img, samples


def _errors_call(cc, intr, views, obj, img, n1, n2, samples, sums=None):
    from cameracalibrations_b200 import _lib
    views, obj, img = (np.ascontiguousarray(x, dtype=np.float64) for x in (views, obj, img))
    ir, ic = np.ascontiguousarray(samples[..., 0]), np.ascontiguousarray(samples[..., 1])
    sums = np.zeros(4) if sums is None else sums
    p = lambda x: C.c_void_p(x.ctypes.data)
    rc = _lib.lib.cc_calculate_errors_f64_host(_lib.context(0).handle, C.byref(_lib.make_intr(*intr)), p(views),
                                               len(views), p(obj), p(img), n1, n2, p(ir), p(ic), samples.shape[1],
                                               p(sums))
    return rc, sums


# boards: 1-wide both ways, a 2 x 2, the example's 7 x 5 and 20 x 14, 544 corners (past the 48 KB default of
# dynamic shared memory), 2133 corners (204 768 B, the largest under the 200 KiB cap); (nviews, samples, k)
# cycle through {1, 3, 5, 9} x {0, 1, 31, 33, 100} x {0, -0.12}
ERR_CASES = [((n1, n2), nv, S, k) for (n1, n2), combos in [
    ((1, 9), [(1, 0, 0.0), (9, 33, -0.12)]),
    ((9, 1), [(3, 1, -0.12), (5, 100, 0.0)]),
    ((2, 2), [(5, 31, 0.0), (1, 100, -0.12)]),
    ((7, 5), [(9, 100, -0.12), (3, 0, 0.0)]),
    ((20, 14), [(3, 33, 0.0), (9, 31, -0.12)]),
    ((32, 17), [(5, 1, -0.12), (1, 33, 0.0)]),
    ((79, 27), [(9, 31, -0.12), (3, 100, 0.0)]),
] for nv, S, k in combos]


@pytest.mark.parametrize("board,nv,S,k", ERR_CASES)
def test_calculate_errors_vs_oracle(cc, board, nv, S, k):
    n1, n2 = board
    intr, views, obj, img, samples = _errors_case(n1, n2, nv, S, k, seed=n1 * 100 + n2 + nv)
    rc, sums = _errors_call(cc, intr, views, obj, img, n1, n2, samples)
    assert rc == 0
    ref = oc.calculate_errors(intr, [(v[:3], v[3:]) for v in views], obj, img, board, samples, raw_sums=True)
    for i in range(3):
        assert abs(sums[i] - ref[i]) <= 1e-9 * abs(ref[i]), (i, sums, ref)
    if n1 > 1 or n2 > 1:
        assert ref[2] > 0.0
    # the inverse term is the round-off of pixel -> world -> pixel: both sides at most (1e-9 px)^2 a sample
    assert ref[3] <= 1e-18 * nv * S and sums[3] <= 1e-18 * nv * S, (sums[3], ref[3])
    # the distance term restated: neighbours (a, b) - (a + 1, b) and (a, b) - (a, b + 1), index a + n1 b
    dist = []
    for v in range(nv):
        ch = oc.chain(intr, views[v, :3], views[v, 3:])
        x, y, z = oc.img2world_soa(ch, img[v, :, 0], img[v, :, 1])
        P = np.stack([x, y, z], -1).reshape(n2, n1, 3)                  # [b, a]
        dist += list((np.linalg.norm(P[:, 1:] - P[:, :-1], axis=-1) - intr[5]).ravel())
        dist += list((np.linalg.norm(P[1:, :] - P[:-1, :], axis=-1) - intr[5]).ravel())
    d_np = math.fsum(np.square(dist))
    assert abs(sums[2] - d_np) <= 1e-9 * d_np
    # per-view calls summed against the batched call
    per = np.sum([_errors_call(cc, intr, views[v:v + 1], obj, img[v:v + 1], n1, n2, samples[v:v + 1])[1]
                  for v in range(nv)], axis=0)
    assert np.all(np.abs(per[:3] - sums[:3]) <= 1e-12 * np.abs(sums[:3]))


def test_calculate_errors_rejects_a_board_past_the_shared_memory_cap(cc):
    """2134 corners (79 x 27 + 1 does not tile, 2 x 1067 does): CC_ERR_INVALID_ARG and sums untouched."""
    from cameracalibrations_b200 import _lib
    intr, views, obj, img, samples = _errors_case(2, 1067, 1, 3, -0.12, seed=1)
    sums = np.full(4, -777.0)
    rc, out = _errors_call(cc, intr, views, obj, img, 2, 1067, samples, sums)
    assert rc == _lib.CC_ERR_INVALID_ARG and np.all(out == -777.0)
    rc, out = _errors_call(cc, intr, views, obj[:2133], img[:, :2133], 3, 711, samples)
    assert rc == 0


# ------------------------------------------------------------------ d. starting values
def _exact_views(nc, nv, aspect, k=0.0, sz=(1081, 1921), seed=0, thetas=None):
    """noise-free views of a planar board, tilted 0.2 to 0.6 rad about random axes (thetas: override)"""
    rng = np.random.default_rng(seed)
    f = 1400.0
    intr = (aspect * f, f, (sz[0] - 1) / 2.0, (sz[1] - 1) / 2.0, k, 1.0)
    obj = fr.board(nc)
    axes = rng.normal(size=(nv, 3))
    axes /= np.linalg.norm(axes, axis=1, keepdims=True)
    th = rng.uniform(0.2, 0.6, nv) if thetas is None else np.asarray(thetas)
    views = np.concatenate([axes * th[:, None],
                            np.stack([rng.normal(0, 1, nv), rng.normal(0, 1, nv), rng.uniform(30, 35, nv)], 1)], 1)
    img = np.empty((nv, nc, 2))
    for v in range(nv):
        img[v, :, 0], img[v, :, 1] = oc.world2img(oc.chain(intr, views[v, :3], views[v, 3:]), obj)
    return intr, views, obj, img, sz


def _close(a, b, rtol):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return np.all(np.abs(a - b) <= rtol * np.maximum(1.0, np.abs(b))), np.max(np.abs(a - b) / np.maximum(1.0, np.abs(b)))


@pytest.mark.parametrize("nc", [4, 5, 31, 33, 280, 2048])
@pytest.mark.parametrize("nv,aspect", [(3, 1.0), (4, 1.25), (5, 1.0), (130, 1.25)])
def test_initial_guess_recovers_the_generating_camera(cc, lm, nc, nv, aspect):
    """Zhang's construction is exact on noise-free views with k = 0 and the principal point at the image
    centre: both the device and the numpy starting values recover f and every pose to 1e-6."""
    intr, views, obj, img, sz = _exact_views(nc, nv, aspect, seed=nc + nv)
    for name, (i0, v0) in (("device", lm.initial_guess_device(obj, img, sz, aspect)),
                           ("host", lm.initial_guess(obj, img, sz, aspect))):
        v0 = v0.cpu().numpy() if torch.is_tensor(v0) else np.asarray(v0)
        ok, e = _close(i0[:4], intr[:4], 1e-6)
        assert ok and i0[4] == 0.0, (name, i0, intr, e)
        ok, e = _close(v0, views, 1e-6)
        assert ok, (name, e)


# ------------------------------------------------------------------ e. the whole fit
def test_fit_recovers_noise_free_camera(cc, lm):
    """k = -0.12, one view at theta = 1e-8, the others tilted; from the device starting values both the
    device-resident loop and the stepwise loop recover the camera to 1e-8 with rms < 1e-9, bit-equal."""
    th = [1e-8] + list(np.random.default_rng(9).uniform(0.2, 0.6, 11))
    intr, views, obj, img, sz = _exact_views(280, 12, 1.0, k=-0.12, seed=9, thetas=th)
    i0, v0 = lm.initial_guess_device(obj, img, sz, 1.0)
    v0 = v0.cpu().numpy()
    a = lm.lm_fit_device(i0, v0, obj, img, max_iter=60, eps=1e-12)
    b = lm.lm_fit(i0, v0, obj, img, max_iter=60, eps=1e-12)
    assert a["iterations"] == b["iterations"] and a["rms"] == b["rms"]
    assert np.array_equal(np.asarray(a["intr"]), np.asarray(b["intr"])) and np.array_equal(a["views"], b["views"])
    assert a["rms"] < 1e-9, a["rms"]
    ok, e = _close(a["intr"], intr[:5], 1e-8)
    assert ok, (a["intr"], e)
    ok, e = _close(a["views"], views, 1e-8)
    assert ok, e
