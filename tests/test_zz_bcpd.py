"""BCPD E-step on the pair kernels (SURVEY section 8(f) row 3) and the ``probreg.bcpd`` surface around it.

Fixtures: tests/golden/bcpd.npz and bcpd_gmat_inv.npz, produced by the UNMODIFIED reference bcpd.py (tests/golden/make_golden_bcpd.py).
CPU tests: the oracle against those fixtures, and the library under the emulation of tests/emu; the gpu-marked tests run the same
bodies on the B200 (first hardware run: round 2, profiles/r2_pytest_runxfail_first.txt).
"""
import numpy as np
import pytest

from conftest import load_golden
from oracle import cpd_oracle as orc
from probreg_b200 import _cabi, bcpd, math_utils

CASES = ["a", "b", "c", "d"]


def _case(g, tag):
    return (g["t_source"], g[str(g[tag + "_target"])], float(g[tag + "_scale"]), g[tag + "_alpha"], g[tag + "_sdiag"],
            float(g[tag + "_sigma2"]), float(g[tag + "_w"]))


# ---- oracle pinned to the reference ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("tag", CASES)
def test_oracle_bcpd_estep_matches_reference(tag):
    g = load_golden("bcpd.npz")
    ts, x, scale, alpha, sdiag, s2, w = _case(g, tag)
    es = orc.bcpd_expectation_step(ts, x, scale, alpha, sdiag, s2, w)
    np.testing.assert_allclose(es.nu_d, g[tag + "_nu_d"], rtol=1e-12, atol=1e-300)
    np.testing.assert_allclose(es.nu, g[tag + "_nu"], rtol=1e-11, atol=1e-300)
    np.testing.assert_allclose(es.px, g[tag + "_px"], rtol=1e-10, atol=1e-14)
    assert es.n_p == pytest.approx(float(g[tag + "_np"]), rel=1e-12)
    # full matrix or its diagonal: the same thing (bcpd.py:61 reads the diagonal only)
    es2 = orc.bcpd_expectation_step(ts, x, scale, alpha, np.diag(sdiag), s2, w)
    assert np.array_equal(es.nu, es2.nu)


# ---- the library ----------------------------------------------------------------------------------------------------------------
def _check_estep_vs_reference(tag):
    g = load_golden("bcpd.npz")
    ts, x, scale, alpha, sdiag, s2, w = _case(g, tag)
    reg = bcpd.CombinedBCPD(g["source"])
    es = reg.expectation_step(ts, x, scale, alpha, np.diag(sdiag), s2, w)
    ref_nu_d, ref_nu, ref_px = g[tag + "_nu_d"], g[tag + "_nu"], g[tag + "_px"]
    # columns the reference zeroes (float64 underflow of the whole column) are zeroed here too
    np.testing.assert_array_equal(es.nu_d == 0, ref_nu_d == 0)
    np.testing.assert_allclose(es.nu_d, ref_nu_d, rtol=2e-5, atol=1e-12)
    np.testing.assert_allclose(es.nu, ref_nu, rtol=5e-5, atol=1e-9)
    np.testing.assert_allclose(es.px, ref_px, rtol=5e-5, atol=5e-5 * np.abs(ref_px).max())
    assert es.n_p == pytest.approx(float(g[tag + "_np"]), rel=1e-6)
    ok = ref_nu > 1e-6
    np.testing.assert_allclose(es.x_hat[ok], g[tag + "_xhat"][ok], atol=5e-5)
    assert es.nu_d.shape == (x.shape[0],) and es.px.shape == ts.shape


def _check_estep_vs_oracle_shapes():
    rng = np.random.default_rng(8)
    for m, n, dim, w in [(1, 1, 3, 0.0), (3, 900, 3, 0.2), (1300, 70, 3, 0.0), (91, 150, 2, 0.1)]:
        src = rng.random((m, dim))
        tgt = rng.random((n, dim)) + 0.03
        alpha = rng.dirichlet(np.ones(m))
        sdiag = rng.uniform(0.0, 0.01, m)
        es = bcpd.CombinedBCPD(src).expectation_step(src, tgt, 1.1, alpha, sdiag, 0.01, w)
        ref = orc.bcpd_expectation_step(src, tgt, 1.1, alpha, sdiag, 0.01, w)
        np.testing.assert_allclose(es.nu_d, ref.nu_d, rtol=2e-5, atol=1e-12)
        np.testing.assert_allclose(es.nu, ref.nu, rtol=5e-5, atol=1e-9)
        np.testing.assert_allclose(es.px, ref.px, rtol=5e-5, atol=5e-5)
    # a source with weight exactly zero contributes nothing; scalar alpha broadcasts (bcpd.py:115: alpha = 1/m)
    src, tgt = rng.random((200, 3)), rng.random((180, 3))
    alpha = np.full(200, 1.0 / 200)
    alpha[7] = 0.0
    es = bcpd.CombinedBCPD(src).expectation_step(src, tgt, 1.0, alpha, np.zeros(200), 0.02, 0.1)
    assert es.nu[7] == 0.0
    es = bcpd.CombinedBCPD(src).expectation_step(src, tgt, 1.0, 1.0 / 200, np.identity(200), 0.02, 0.1)
    ref = orc.bcpd_expectation_step(src, tgt, 1.0, np.full(200, 1.0 / 200), np.ones(200), 0.02, 0.1)
    np.testing.assert_allclose(es.nu, ref.nu, rtol=5e-5, atol=1e-9)
    # the unweighted limit is the CPD E-step: alpha = 1/M, sigma_mm = 0  ->  pt1, p1, px of cpd.py:71-88 with the same w
    h = _cabi.Handle(3)
    h.set_source(src)
    h.set_target(tgt)
    cp = h.estep(src, 0.02, 0.1)
    bp = h.bcpd_estep(src, 1.0, np.full(200, 1.0 / 200), np.zeros(200), 0.02, 0.1)
    # CPD: c = (2 pi s2)^(D/2) w/(1-w) M/N on sum_m K;  BCPD: w/N on (1-w)/M sum_m K / (2 pi s2)^(D/2): the same ratio
    np.testing.assert_allclose(bp[0], cp[0], rtol=1e-9)
    np.testing.assert_allclose(bp[1], cp[1], rtol=1e-9)
    with pytest.raises(_cabi.CpdError):
        h.bcpd_estep(src, 1.0, -np.ones(200), np.zeros(200), 0.02, 0.1)
    with pytest.raises(ValueError):
        h.bcpd_estep(src, 1.0, np.ones(5), np.zeros(200), 0.02, 0.1)


def _check_imq_kernel():
    """inverse_multiquadric_kernel is BIT-identical to the float32 restatement of cc/math_utils.cc:37-39: BCPD inverts this matrix
    (bcpd.py:117, condition ~1e10 in float32), so a last-bit difference would show in the first digits of the registration."""
    g = load_golden("bcpd.npz")
    x = g["reg_source"]
    k = math_utils.inverse_multiquadric_kernel(x, x[:50], 1.0)
    assert k.dtype == np.float32 and k.shape == (x.shape[0], 50)
    assert np.array_equal(k, orc.imq_kernel_f32(x, x[:50], 1.0))
    k2 = math_utils.inverse_multiquadric_kernel(x[:, :2], x[:7, :2], 0.5)
    assert np.array_equal(k2, orc.imq_kernel_f32(x[:, :2], x[:7, :2], 0.5))


def _run_registration(g):
    seen = []
    tfm = bcpd.registration_bcpd(g["reg_source"], g["reg_target"], w=0.05, maxiter=5, tol=-1.0, lmd=2.0,
                                 callbacks=[lambda t: seen.append(t)])
    assert len(seen) == 5
    x = g["reg_source"]
    np.testing.assert_allclose(tfm.transform(x), tfm.rigid_trans.transform(x + tfm.v), atol=0)
    return tfm


def _check_registration_vs_reference(monkeypatch):
    """registration_bcpd against the committed outputs of the UNMODIFIED reference bcpd.py, on any host.  Both M-steps call
    np.linalg.inv on the float32 kernel matrix (condition 1.3e10), whose result differs between LAPACK kernels, CPUs and thread
    counts by far more than the tolerance; so the package is handed the inverse the reference's run used (bcpd_gmat_inv.npz), after
    checking that the matrix it inverts is the oracle's kernel matrix bit for bit and that it takes the inverse the same way.  What
    is compared is then what this package computes itself: five E-steps on the GPU and the M-step around them."""
    g = load_golden("bcpd.npz")
    ref_inv = load_golden("bcpd_gmat_inv.npz")["gmat_inv"]
    initialize = bcpd.CombinedBCPD._initialize

    def with_reference_inverse(self, target):
        out = initialize(self, target)
        assert np.array_equal(self.gmat, orc.imq_kernel_f32(self._source, self._source, 1.0))
        assert self.gmat_inv.dtype == np.float32 and np.array_equal(self.gmat_inv, np.linalg.inv(self.gmat))
        self.gmat_inv = ref_inv.copy()
        return out

    monkeypatch.setattr(bcpd.CombinedBCPD, "_initialize", with_reference_inverse)
    tfm = _run_registration(g)
    np.testing.assert_allclose(tfm.rigid_trans.rot, g["reg_rot"], atol=1e-5)
    np.testing.assert_allclose(tfm.rigid_trans.t, g["reg_t"], atol=1e-5)
    assert tfm.rigid_trans.scale == pytest.approx(float(g["reg_scale"]), rel=1e-5)
    np.testing.assert_allclose(tfm.v, g["reg_v"], atol=1e-5)


@pytest.mark.parametrize("tag", CASES)
def test_bcpd_estep_vs_reference_emulated(emulated, tag):
    _check_estep_vs_reference(tag)


def test_bcpd_estep_shapes_emulated(emulated):
    _check_estep_vs_oracle_shapes()


def test_bcpd_registration_emulated(emulated, monkeypatch):
    _check_imq_kernel()
    _check_registration_vs_reference(monkeypatch)


def test_bcpd_culled_estep_is_bit_exact_emulated(emulated, monkeypatch):
    src, tgt = orc.synthetic_pair(2500)
    ts = orc.apply_rigid(src, orc.rot_z(30.0), np.array([0.1, -0.2, 0.3]))
    rng = np.random.default_rng(4)
    alpha, sdiag = rng.dirichlet(np.ones(2500)), rng.uniform(0, 1e-5, 2500)

    def run(no_cull):
        monkeypatch.setenv("CPD_B200_NO_CULL", "1" if no_cull else "0")
        h = _cabi.Handle(3)
        h.set_source(ts)
        h.set_target(tgt)
        return h.bcpd_estep(ts, 1.0, alpha, sdiag, 5e-5, 0.1)

    a, b = run(False), run(True)
    for x, y in zip(a[:3], b[:3]):
        assert np.array_equal(x, y)


@pytest.mark.gpu
@pytest.mark.timeout(600)
@pytest.mark.parametrize("tag", CASES)
def test_bcpd_estep_vs_reference_gpu(tag):
    _check_estep_vs_reference(tag)


@pytest.mark.gpu
@pytest.mark.timeout(600)
def test_bcpd_estep_shapes_gpu():
    _check_estep_vs_oracle_shapes()


@pytest.mark.gpu
@pytest.mark.timeout(600)
def test_bcpd_registration_gpu(monkeypatch):
    _check_imq_kernel()
    _check_registration_vs_reference(monkeypatch)


def _check_full_size(n, sample):
    """Size-independent properties (sum nu == sum nu_d, sum_m px_m == sum_n nu_d_n x_n) and a column sample against the numpy
    restatement (the constant w / N and the (1 - w) alpha factor of the sample run are matched to the full run's)."""
    src, tgt = orc.synthetic_pair(n)
    rng = np.random.default_rng(1)
    alpha, sdiag = rng.dirichlet(np.ones(n)), rng.uniform(0.0, 1e-3, n)
    h = _cabi.Handle(3)
    h.set_source(src)
    h.set_target(tgt)
    nu_d, nu, px, n_p = h.bcpd_estep(src, 1.0, alpha, sdiag, 2e-3, 0.1)
    assert n_p == pytest.approx(nu_d.sum(), rel=1e-7) and n_p == pytest.approx(nu.sum(), rel=1e-9)
    np.testing.assert_allclose(px.sum(0), (nu_d[:, None] * tgt).sum(0), rtol=1e-6)
    sel = rng.choice(n, sample, replace=False)
    w_s = 0.1 * sample / n
    ref = orc.bcpd_expectation_step(src, tgt[sel], 1.0, alpha * (1.0 - 0.1) / (1.0 - w_s), sdiag, 2e-3, w_s)
    np.testing.assert_allclose(nu_d[sel], ref.nu_d, rtol=5e-5, atol=1e-12)


def test_bcpd_full_size_body_at_emulation_size(emulated):
    _check_full_size(2500, 200)


@pytest.mark.gpu
@pytest.mark.timeout(600)
def test_bcpd_estep_full_size_properties():
    _check_full_size(100000, 400)
