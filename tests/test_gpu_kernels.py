"""GPU parity tests, kernel level: every C-ABI entry point against the oracle / golden vectors of the
reference on the same seeded inputs.  Tolerances: complex128, relative 1e-12 per element (summation
order differs from BLAS; the north-star bar of 1e-10 is on propagated observables, see test_gpu_propagation)."""
import numpy as np
import pytest
import scipy.linalg

from oracle import tdvp_oracle as orc
from tests.golden_io import load_kernels

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    from pytdscf_b200._engine import Engine

    e = Engine(0)
    yield e
    e.close()


@pytest.fixture(scope="module")
def K():
    return load_kernels()


def crand(rng, *shape):
    return (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)) / np.sqrt(2)


def relerr(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def core_of(data, left=False, right=False):
    return orc.SiteCore((0, 1, 2), 1, data, left, right)


# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,N,K_", [(1, 1, 1), (7, 5, 3), (128, 64, 8), (129, 65, 9), (200, 150, 77), (512, 384, 256), (33, 700, 130),
                                    (1100, 1030, 300), (2048, 640, 72), (96, 80, 2100)])
@pytest.mark.parametrize("ta,tb", [(0, 0), (0, 1), (2, 0), (1, 0), (2, 1), (0, 2)])
def test_zgemm(eng, M, N, K_, ta, tb):
    rng = np.random.default_rng(M * 1000 + N * 10 + K_ + ta * 7 + tb)
    A = crand(rng, *((K_, M) if ta else (M, K_)))
    B = crand(rng, *((N, K_) if tb else (K_, N)))
    C0 = crand(rng, M, N)
    opA = {0: A, 1: A.T, 2: A.conj().T}[ta]
    opB = {0: B, 1: B.T, 2: B.conj().T}[tb]
    alpha, beta = 0.7 - 0.2j, -0.3 + 0.5j
    ref = alpha * (opA @ opB) + beta * C0
    Cd = eng.to_device(C0)
    eng.zgemm(eng.to_device(A), eng.to_device(B), ta, tb, alpha, beta, Cd)
    assert relerr(Cd.cpu().numpy(), ref) < 1e-13


HEFF_CASES = {
    "h_343": ("L", "Wf", "R"), "h_333": ("L", "Wd", "R"), "h_143": (None, "W_l1", "R"),
    "h_133": (None, "Wd_l1", "R"), "h_341": ("L", "W_r1", None), "h_331": ("L", "Wd_r1", None),
    "h_311": ("L1", None, None), "h_113": (None, None, "R1"), "h_313": ("L1", None, "R1"),
    "h_111": (None, None, None),
}


@pytest.mark.parametrize("name", sorted(HEFF_CASES))
def test_heff_term_golden(eng, K, name):
    l_, w_, r_ = HEFF_CASES[name]
    L = None if l_ is None else eng.to_device(K[l_])
    R = None if r_ is None else eng.to_device(K[r_])
    core = None if w_ is None else eng.upload_core(K[w_])
    out = eng.heff_apply([(L, core, R, 1.0)], eng.to_device(K["psi"]))
    assert relerr(out.cpu().numpy(), K[name]) < 1e-13


def test_heff_term_sum_and_coef(eng, K):
    terms_np = {"ovlp": (None, None, None), "a": (K["L"], core_of(K["Wf"]), K["R"]), "b": (K["L"], core_of(K["Wd"]), K["R"]),
                "c": (K["L1"], None, None)}
    ref = orc.heff_apply(terms_np, 0.37 - 0.11j, K["psi"])
    dev = [(None, None, None, 0.37 - 0.11j),
           (eng.to_device(K["L"]), eng.upload_core(K["Wf"]), eng.to_device(K["R"]), 1.0),
           (eng.to_device(K["L"]), eng.upload_core(K["Wd"]), eng.to_device(K["R"]), 1.0),
           (eng.to_device(K["L1"]), None, None, 1.0)]
    out = eng.heff_apply(dev, eng.to_device(K["psi"]))
    assert relerr(out.cpu().numpy(), ref) < 1e-13


@pytest.mark.parametrize("Dl,d,Dr,wl,wr", [(37, 5, 29, 3, 4), (64, 10, 64, 6, 6), (130, 4, 131, 9, 2), (1, 8, 4, 1, 3), (4, 2, 1, 3, 1)])
@pytest.mark.parametrize("diag", [False, True])
def test_heff_random_shapes(eng, Dl, d, Dr, wl, wr, diag):
    rng = np.random.default_rng(Dl + 7 * d + 13 * Dr + wl + wr + diag)
    psi = crand(rng, Dl, d, Dr)
    L = crand(rng, Dl, wl, Dl)
    R = crand(rng, Dr, wr, Dr)
    W = crand(rng, wl, d, wr) if diag else crand(rng, wl, d, d, wr)
    ref = orc.heff_term(L, core_of(W), R, psi)
    out = eng.heff_apply([(eng.to_device(L), eng.upload_core(W), eng.to_device(R), 1.0)], eng.to_device(psi))
    assert relerr(out.cpu().numpy(), ref) < 1e-12


def test_keff_golden(eng, K):
    sig = eng.to_device(K["sig"])
    Lk, Rk = eng.to_device(K["Lk"]), eng.to_device(K["Rk"])
    assert relerr(eng.keff_apply([(Lk, Rk, 1.0)], sig).cpu().numpy(), K["k_33"]) < 1e-13
    out = eng.keff_apply([(None, None, 0.5j), (Lk, Rk, 1.0)], sig).cpu().numpy()
    assert relerr(out, 0.5j * K["sig"] + K["k_33"]) < 1e-13
    # one-sided terms exist only with w == 1 ("summed" blocks)
    L1 = K["Lk"][:, :1, :].copy()
    ref = orc.keff_term(L1, None, K["sig"])
    assert relerr(eng.keff_apply([(eng.to_device(L1), None, 1.0)], sig).cpu().numpy(), ref) < 1e-13
    ref = orc.keff_term(None, L1, K["sig"])
    assert relerr(eng.keff_apply([(None, eng.to_device(L1), 1.0)], sig).cpu().numpy(), ref) < 1e-13


ENV_CASES = {
    "e_A32f": ("A", "L", "Wf"), "e_A32d": ("A", "L", "Wd"), "e_A31f": ("A", None, "W_l1"),
    "e_A31d": ("A", None, "Wd_l1"), "e_A11": ("A", None, None),
    "e_B32f": ("B", "R", "Wf"), "e_B32d": ("B", "R", "Wd"), "e_B31f": ("B", None, "W_r1"),
    "e_B31d": ("B", None, "Wd_r1"), "e_B11": ("B", None, None),
}


@pytest.mark.parametrize("name", sorted(ENV_CASES))
def test_env_update_golden(eng, K, name):
    gauge, e_, w_ = ENV_CASES[name]
    A = eng.to_device(K["A"])
    E = None if e_ is None else eng.to_device(K[e_])
    core = None if w_ is None else eng.upload_core(K[w_])
    out = eng.env_update(gauge, A, A, E, core)
    assert out.shape == K[name].shape
    assert relerr(out.cpu().numpy(), K[name]) < 1e-13


def test_env_update_summed_block_and_accumulate(eng, K):
    A = eng.to_device(K["A"])
    L1 = K["L"][:, :1, :].copy()
    ref = orc.env_update_term("A", K["A"], K["A"], L1, None)
    out = eng.env_update("A", A, A, eng.to_device(L1), None)
    assert relerr(out.cpu().numpy(), ref) < 1e-13
    ref2 = ref + orc.env_update_term("A", K["A"], K["A"], None, core_of(K["W_l1"][..., :1].copy()))
    eng.env_update("A", A, A, None, eng.upload_core(K["W_l1"][..., :1].copy()), out=out, accumulate=True)
    assert relerr(out.cpu().numpy(), ref2) < 1e-13
    R1 = K["R"][:, :1, :].copy()
    ref = orc.env_update_term("B", K["A"], K["A"], R1, None)
    out = eng.env_update("B", A, A, eng.to_device(R1), None)
    assert relerr(out.cpu().numpy(), ref) < 1e-13


ENV_SHAPES = [(37, 5, 29, 3, 4), (64, 10, 48, 6, 6), (130, 4, 70, 2, 5)]


@pytest.mark.parametrize("gauge", ["A", "B"])
@pytest.mark.parametrize("Dl,d,Dr,wi,wo,bra_ket,diag",
                         [pytest.param(*s, "same", False, id="-".join(map(str, s))) for s in ENV_SHAPES] +
                         [pytest.param(*s, "independent", diag, id="-".join(map(str, s)) + ("-bra-diag" if diag else "-bra"))
                          for s in ENV_SHAPES for diag in (False, True)])
def test_env_update_random_shapes(eng, gauge, Dl, d, Dr, wi, wo, bra_ket, diag):
    """bra == ket, and independent bra and ket (Simulator.operate, adaptive mode): a swap of the two would show."""
    rng = np.random.default_rng(Dl + 3 * d + 5 * Dr + wi + wo)
    A = crand(rng, Dl, d, Dr)
    shape_W = ((wi, d, wo) if gauge == "A" else (wo, d, wi)) if diag else ((wi, d, d, wo) if gauge == "A" else (wo, d, d, wi))
    if gauge == "A":
        E, W = crand(rng, Dl, wi, Dl), crand(rng, *shape_W)
    else:
        E, W = crand(rng, Dr, wi, Dr), crand(rng, *shape_W)
    bra = A if bra_ket == "same" else crand(rng, Dl, d, Dr)
    ref = orc.env_update_term(gauge, bra, A, E, core_of(W))
    out = eng.env_update(gauge, eng.to_device(bra), eng.to_device(A), eng.to_device(E), eng.upload_core(W))
    assert relerr(out.cpu().numpy(), ref) < 1e-12


# ---------------------------------------------------------------------------------------------
def _check_qr(eng, psi, atol=1e-12, gauges="AB"):
    """Gauge A on psi and gauge B on psi.  Besides the elementwise match with LAPACK: Q^H Q = I and QR = psi to 1e-13
    (~ 450 EPS: Householder orthogonality and backward error are a small multiple of sqrt(rows) EPS up to 37888 rows)."""
    Dl, d, Dr = psi.shape
    if "A" in gauges:
        A, s = orc.shift_qr(psi)
        Ad, sd = eng.qr_shift("A", eng.to_device(psi))
        Ad, sd = Ad.cpu().numpy(), sd.cpu().numpy()
        np.testing.assert_allclose(Ad, A, atol=atol)
        np.testing.assert_allclose(sd, s, atol=atol * max(1.0, np.abs(s).max()))
        Q = Ad.reshape(Dl * d, Dr)
        assert np.abs(Q.conj().T @ Q - np.eye(Dr)).max() <= 1e-13
        assert np.linalg.norm(Q @ sd - psi.reshape(Dl * d, Dr)) <= 1e-13 * np.linalg.norm(psi)
    if "B" in gauges:
        s, B = orc.shift_lq(psi)
        Bd, sd = eng.qr_shift("B", eng.to_device(psi))
        Bd, sd = Bd.cpu().numpy(), sd.cpu().numpy()
        np.testing.assert_allclose(Bd, B, atol=atol)
        np.testing.assert_allclose(sd, s, atol=atol * max(1.0, np.abs(s).max()))
        Q = Bd.reshape(Dl, d * Dr)
        assert np.abs(Q @ Q.conj().T - np.eye(Dl)).max() <= 1e-13
        assert np.linalg.norm(sd @ Q - psi.reshape(Dl, d * Dr)) <= 1e-13 * np.linalg.norm(psi)


def test_qr_shift_golden(eng, K):
    Ad, sd = eng.qr_shift("A", eng.to_device(K["g_psi"]))
    np.testing.assert_allclose(Ad.cpu().numpy(), K["g_A"], atol=1e-13)
    np.testing.assert_allclose(sd.cpu().numpy(), K["g_Asig"], atol=1e-13)
    Bd, sd = eng.qr_shift("B", eng.to_device(K["g_psi"]))
    np.testing.assert_allclose(Bd.cpu().numpy(), K["g_B"], atol=1e-13)
    np.testing.assert_allclose(sd.cpu().numpy(), K["g_Bsig"], atol=1e-13)


def test_qr_shift_zero_padded_matches_lapack_completion(eng, K):
    """Exact zero columns: tau = 0 reflectors, LAPACK's null-space completion (SURVEY hard part)."""
    Ad, sd = eng.qr_shift("A", eng.to_device(K["g_pad"]))
    np.testing.assert_allclose(Ad.cpu().numpy(), K["g_padA"], atol=1e-14)
    np.testing.assert_allclose(sd.cpu().numpy(), K["g_padAsig"], atol=1e-14)
    Bd, sd = eng.qr_shift("B", eng.to_device(K["g_pad"]))
    np.testing.assert_allclose(Bd.cpu().numpy(), K["g_padB"], atol=1e-14)
    np.testing.assert_allclose(sd.cpu().numpy(), K["g_padBsig"], atol=1e-14)


# Tall matricisations (rows, 1, cols) at the QR panel kernels' switch points: k_qr_panel_cluster with 1 CTA (64 rows),
# 2 CTAs (65, 128), 16 CTAs (1024), the last cluster size (4096 = 16 x 256 rows); k_qr_panel above (4097, 8192, 20000),
# its widest grid with shared-memory slabs ("sms": num_sms x 256 rows) and the first size with global-memory slabs.
QR_TALL_ROWS = [64, 65, 128, 1024, 4096, 4097, 8192, 20000, "sms", "sms+1"]
QR_TALL_COLS = [1, 31, 32, 33, 100]


@pytest.mark.parametrize("Dl,d,Dr", [(1, 8, 4), (4, 8, 4), (16, 5, 16), (40, 6, 40), (64, 10, 64), (100, 7, 90), (128, 16, 128)] +
                         [(rows, 1, cols) for rows in QR_TALL_ROWS for cols in QR_TALL_COLS if rows == "sms" or rows == "sms+1" or cols <= rows])
def test_qr_shift_random(eng, Dl, d, Dr):
    if isinstance(Dl, str):
        import torch

        Dl = torch.cuda.get_device_properties(0).multi_processor_count * 256 + (Dl == "sms+1")
    rng = np.random.default_rng(Dl * 100 + d * 10 + Dr)
    psi = crand(rng, Dl, d, Dr)
    if Dl <= Dr * d:
        _check_qr(eng, psi)
    else:   # gauge B factors the same (rows x cols) matrix when given the transposed tensor
        _check_qr(eng, psi, gauges="A")
        _check_qr(eng, np.ascontiguousarray(psi.transpose(2, 1, 0)), gauges="B")


def test_qr_shift_partial_rank(eng):
    """Columns beyond the numerical rank are exactly zero (as after the padded initial sweep)."""
    rng = np.random.default_rng(5)
    psi = np.zeros((12, 5, 40), dtype=complex)
    psi[:, :, :7] = crand(rng, 12, 5, 7)
    A, s = orc.shift_qr(psi)
    Ad, sd = eng.qr_shift("A", eng.to_device(psi))
    np.testing.assert_allclose(Ad.cpu().numpy(), A, atol=1e-12)
    np.testing.assert_allclose(sd.cpu().numpy(), s, atol=1e-12)
    Q = Ad.cpu().numpy().reshape(60, 40)
    np.testing.assert_allclose(Q.conj().T @ Q, np.eye(40), atol=1e-13)


def test_absorb(eng):
    rng = np.random.default_rng(11)
    sig, site = crand(rng, 6, 9), crand(rng, 9, 4, 7)
    np.testing.assert_allclose(eng.absorb("A", eng.to_device(sig), eng.to_device(site)).cpu().numpy(),
                               np.tensordot(sig, site, axes=(1, 0)), atol=1e-13)
    sig2 = crand(rng, 7, 5)
    np.testing.assert_allclose(eng.absorb("B", eng.to_device(sig2), eng.to_device(site)).cpu().numpy(),
                               np.tensordot(site, sig2, axes=(2, 0)), atol=1e-13)


# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tag,kind,mat,cn,hist,scale0", [
    ("sil_cn", "lanczos", "H", True, 0, 1.0), ("sil_free", "lanczos", "H", False, 0, 1.7),
    ("sil_warm", "lanczos", "H", True, 9, 1.0), ("sil_nonherm", "lanczos", "Hd", False, 0, 1.7),
    ("sia_free", "arnoldi", "G", False, 0, 1.7), ("sia_warm", "arnoldi", "G", False, 8, 1.7)])
def test_krylov_golden(eng, K, tag, kind, mat, cn, hist, scale0):
    """Dense operator through the H_eff interface (L = M as a (n,1,n) block, identity core and R)."""
    n = K["kr_H"].shape[0]
    M = {"H": K["kr_H"], "G": K["kr_G"], "Hd": K["kr_H"] + 0.05j * np.diag(np.arange(n))}[mat]
    L = eng.to_device(M.reshape(n, 1, n))
    psi = eng.to_device((K["kr_x0"] * scale0).reshape(n, 1, 1))
    _, n_warm = orc.krylov_warmup(n, hist)
    niter = eng.krylov_expm(kind, -0.05j, 1e-9, n_warm, cn, psi, hterms=[(L, None, None, 1.0)])
    assert niter == int(K[f"kr_{tag}_niter"])
    assert relerr(psi.cpu().numpy().reshape(-1), K[f"kr_{tag}"]) < 1e-12


def test_krylov_exhausted_space(eng):
    """N <= 20: the Krylov space equals the full space -> exact exponential, niter == N."""
    rng = np.random.default_rng(3)
    n = 6
    H = crand(rng, n, n)
    H = (H + H.conj().T) / 2
    x = crand(rng, n)
    x /= np.linalg.norm(x)
    ref, nref = orc.sil_reference(-0.3j, lambda v: H @ v, x, 1e-9)
    psi = eng.to_device(x.reshape(n, 1, 1))
    niter = eng.krylov_expm("lanczos", -0.3j, 1e-9, 0, True, psi, hterms=[(eng.to_device(H.reshape(n, 1, n)), None, None, 1.0)])
    assert niter == nref
    np.testing.assert_allclose(psi.cpu().numpy().reshape(-1), ref, atol=1e-12)
    # (the reference recurrence is NOT exact even when the space is exhausted: its basis is not orthonormal, SURVEY F2)
    assert np.abs(psi.cpu().numpy().reshape(-1) - scipy.linalg.expm(-0.3j * H) @ x).max() < 1e-2


def test_krylov_keff(eng, K):
    D, w = 24, 3
    rng = np.random.default_rng(8)
    L = crand(rng, D, w, D)
    L = (L + L.conj().transpose(2, 1, 0)) / 2
    R = crand(rng, D, w, D)
    R = (R + R.conj().transpose(2, 1, 0)) / 2
    s = crand(rng, D, D)
    s /= np.linalg.norm(s)
    ref, nref = orc.sil_reference(+0.02j, lambda v: orc.keff_term(L, R, v), s, 1e-9)
    sd = eng.to_device(s)
    niter = eng.krylov_expm("lanczos", +0.02j, 1e-9, 0, True, sd, kterms=[(eng.to_device(L), eng.to_device(R), 1.0)])
    assert niter == nref
    assert relerr(sd.cpu().numpy(), ref) < 1e-12


def test_inner_and_overlap(eng):
    rng = np.random.default_rng(21)
    a, b = crand(rng, 5, 3, 7), crand(rng, 5, 3, 7)
    got = eng.inner(eng.to_device(a), eng.to_device(b), True)
    assert abs(got - np.vdot(a, b)) < 1e-12
    got = eng.inner(eng.to_device(a), eng.to_device(b), False)
    assert abs(got - np.sum(a * b)) < 1e-12
    blk = crand(rng, 5, 5)
    for conj in (False, True):
        bra = np.conj(a) if conj else a
        ref = np.einsum("abc,abk->ck", bra, np.einsum("ibk,ai->abk", b, blk))
        out = eng.overlap_site(eng.to_device(a), eng.to_device(b), eng.to_device(blk), conj)
        assert relerr(out.cpu().numpy(), ref) < 1e-13


def test_argument_errors_do_not_crash(eng, K):
    from pytdscf_b200._lib import TdvpError

    L = eng.to_device(K["L"])  # w = 3 with an identity core -> unsupported, as in the reference (gap cores crash there)
    with pytest.raises(TdvpError):
        eng.heff_apply([(L, None, None, 1.0)], eng.to_device(K["psi"]))


def test_lanczos_eigvec(eng):
    """Ground vector of a dense Hermitian operator through the H_eff interface vs the oracle's textbook Lanczos."""
    rng = np.random.default_rng(17)
    n = 60
    H = crand(rng, n, n)
    H = (H + H.conj().T) / 2 + np.diag(np.linspace(-3, 3, n))
    x = crand(rng, n)
    x /= np.linalg.norm(x)
    ref, nref = orc.lanczos_ground_state(lambda v: H @ v, x)
    ref = ref / np.linalg.norm(ref)
    psi = eng.to_device(x.reshape(n, 1, 1))
    niter = eng.lanczos_eigvec(psi, [(eng.to_device(H.reshape(n, 1, n)), None, None, 1.0)])
    got = psi.cpu().numpy().reshape(-1)
    assert abs(niter - nref) <= 1
    assert abs(abs(np.vdot(got, ref)) - 1) < 1e-9
    assert abs(np.linalg.norm(got) - 1) < 1e-13
    assert np.linalg.norm(H @ got - np.vdot(got, H @ got) * got) < 1e-7
    assert abs(np.vdot(got, H @ got).real - np.linalg.eigvalsh(H)[0]) < 1e-9


@pytest.mark.parametrize("tag,kw", [("a", dict(p=1e-7)), ("b", dict(p=1e-3, keepdim=True)),
                                    ("c", dict(p=1e-5, regularize=True, keepdim=True))])
def test_svd_truncate_golden(eng, K, tag, kw):
    """Against the reference's truncate_sigvec on a graded 6x6 matrix (singular values 1 .. 1e-9)."""
    U, S, Vh, rank = eng.svd_truncate(eng.to_device(K["t_sig"]), **kw)
    U, S, Vh = U.cpu().numpy(), S.cpu().numpy(), Vh.cpu().numpy()
    assert U.shape == K[f"t_{tag}_U"].shape and S.shape == K[f"t_{tag}_S"].shape
    np.testing.assert_allclose(S, K[f"t_{tag}_S"], atol=1e-13)
    np.testing.assert_allclose(U @ S @ Vh, K[f"t_{tag}_U"] @ K[f"t_{tag}_S"] @ K[f"t_{tag}_Vh"], atol=1e-12)
    np.testing.assert_allclose(U.conj().T @ U, np.eye(U.shape[1]), atol=1e-13)
    np.testing.assert_allclose(Vh @ Vh.conj().T, np.eye(Vh.shape[0]), atol=1e-13)


@pytest.mark.parametrize("n", [1, 2, 7, 64, 257])
def test_svd_random_and_rank_deficient(eng, n):
    rng = np.random.default_rng(n)
    X = crand(rng, n, n)
    if n > 4:
        X[:, n // 2:] = 0.0  # exact zero columns -> Householder completion path
    U, S, Vh, rank = eng.svd_truncate(eng.to_device(X), p=0.0, keepdim=True)
    U, S, Vh = U.cpu().numpy(), S.cpu().numpy(), Vh.cpu().numpy()
    s_ref = np.linalg.svd(X, compute_uv=False)
    nz = s_ref[s_ref > 1e-12 * s_ref[0]]
    np.testing.assert_allclose(np.diag(S).real[: len(nz)] * np.linalg.norm(nz), nz, rtol=1e-12)
    np.testing.assert_allclose(U.conj().T @ U, np.eye(n), atol=1e-12)
    np.testing.assert_allclose(Vh @ Vh.conj().T, np.eye(n), atol=1e-12)
    np.testing.assert_allclose(U @ (S * np.linalg.norm(nz)) @ Vh, X, atol=1e-12 * max(1.0, s_ref[0]))


def test_pinv(eng, K):
    X = K["t_sig"]
    np.testing.assert_allclose(eng.pinv(eng.to_device(X), 1e-13).cpu().numpy(), np.linalg.pinv(X, rcond=1e-13), rtol=0,
                               atol=1e-6 * np.abs(np.linalg.pinv(X, rcond=1e-13)).max())
    rng = np.random.default_rng(2)
    Y = crand(rng, 40, 40)
    Y[:, 30:] = 0
    ref = np.linalg.pinv(Y, rcond=1e-13)
    np.testing.assert_allclose(eng.pinv(eng.to_device(Y), 1e-13).cpu().numpy(), ref, atol=1e-11 * np.abs(ref).max())


def _graded(rng, n, svals):
    Q1, _ = np.linalg.qr(crand(rng, n, n))
    Q2, _ = np.linalg.qr(crand(rng, n, n))
    return (Q1 * np.asarray(svals)[None, :]) @ Q2.conj().T


def test_svd_and_qr_denormal_directions(eng):
    """Bond matrices of a padded Hartree-product start carry singular values like 1e-13, 1e-18, 1e-157 and exact zeros
    (seen in the site-parallel runs): squares of the smallest are denormal, the factors must stay isometries."""
    rng = np.random.default_rng(11)
    # rows scaled like the bond matrices met in practice: lower-triangular with a 1, 2e-13, 8e-18, 7e-157, 0, 0 diagonal
    L = np.tril(crand(rng, 6, 6)) * np.array([1.0, 2e-13, 8e-18, 7e-157, 0.0, 0.0])[:, None]
    L[1:, 0] *= 1e-14
    U, s, Vh = eng.svd(eng.to_device(L))
    U, Vh = U.cpu().numpy(), Vh.cpu().numpy()
    np.testing.assert_allclose(U.conj().T @ U, np.eye(6), atol=1e-13)
    np.testing.assert_allclose(Vh @ Vh.conj().T, np.eye(6), atol=1e-13)
    np.testing.assert_allclose((U * s[None, :]) @ Vh, L, atol=1e-15)
    np.testing.assert_allclose(s[:3], np.linalg.svd(L, compute_uv=False)[:3], rtol=1e-10)
    # LQ shift of a (6, 4, 6) centre tensor whose rows have those norms
    psi = (crand(rng, 6, 24) * np.array([1.0, 2e-13, 8e-18, 7e-157, 0.0, 0.0])[:, None]).reshape(6, 4, 6)
    B, sig = eng.qr_shift("B", eng.to_device(psi))
    Bm = B.cpu().numpy().reshape(6, 24)
    np.testing.assert_allclose(Bm @ Bm.conj().T, np.eye(6), atol=1e-13)
    np.testing.assert_allclose(np.tensordot(sig.cpu().numpy(), B.cpu().numpy(), axes=(1, 0)), psi, atol=1e-15)
    A, sig = eng.qr_shift("A", eng.to_device(np.ascontiguousarray(psi.transpose(2, 1, 0))))
    Am = A.cpu().numpy().reshape(24, 6)
    np.testing.assert_allclose(Am.conj().T @ Am, np.eye(6), atol=1e-13)


@pytest.mark.parametrize("diag", [False, True])
@pytest.mark.parametrize("l_id,r_id", [(0, 2), (1, 0), (2, 1), (-1, 1), (0, -1)])
def test_heff_identity_channel_shortcut(eng, l_id, r_id, diag):
    """id_channels: the flagged channel of L / R is an exact unit block; the shortcut (copy instead of GEMM slice,
    two-level row GEMMs for the other channels) must equal the full contraction."""
    import dataclasses

    rng = np.random.default_rng(100 + 10 * l_id + r_id + diag)
    Dl, d, Dr, wl, wr = 96, 16, 96, 3, 3          # N = 147456 >= the 2^17 threshold of the shortcut
    psi = crand(rng, Dl, d, Dr)
    L, R = crand(rng, Dl, wl, Dl), crand(rng, Dr, wr, Dr)
    if l_id >= 0:
        L[:, l_id, :] = np.eye(Dl)
    if r_id >= 0:
        R[:, r_id, :] = np.eye(Dr)
    W = crand(rng, wl, d, wr) if diag else crand(rng, wl, d, d, wr)
    ref = orc.heff_term(L, core_of(W), R, psi)
    core = dataclasses.replace(eng.upload_core(W), l_id=l_id, r_id=r_id)
    base = eng.stats()["launches"]
    out = eng.heff_apply([(eng.to_device(L), core, eng.to_device(R), 0.7 - 0.2j)], eng.to_device(psi))
    assert relerr(out.cpu().numpy(), (0.7 - 0.2j) * ref) < 1e-12
    # accumulation into an existing output (second term) goes through the same path
    out2 = eng.heff_apply([(eng.to_device(L), eng.upload_core(W), eng.to_device(R), 1.0), (eng.to_device(L), core, eng.to_device(R), 1.0)],
                          eng.to_device(psi))
    assert relerr(out2.cpu().numpy(), 2 * ref) < 1e-12
    assert eng.stats()["launches"] > base


@pytest.mark.parametrize("l_id,r_id", [(0, 3), (3, 0), (1, 2), (-1, 2), (1, -1)])
def test_keff_identity_channel_shortcut(eng, l_id, r_id):
    rng = np.random.default_rng(200 + 10 * l_id + r_id)
    D, w = 192, 4                                  # D * D * w = 147456
    sig = crand(rng, D, D)
    L, R = crand(rng, D, w, D), crand(rng, D, w, D)
    if l_id >= 0:
        L[:, l_id, :] = np.eye(D)
    if r_id >= 0:
        R[:, r_id, :] = np.eye(D)
    ref = orc.keff_term(L, R, sig)
    out = eng.keff_apply([(eng.to_device(L), eng.to_device(R), 1.0, (l_id, r_id))], eng.to_device(sig))
    assert relerr(out.cpu().numpy(), ref) < 1e-12
    out = eng.keff_apply([(eng.to_device(L), eng.to_device(R), 0.5j), (eng.to_device(L), eng.to_device(R), 1.0, (l_id, r_id))], eng.to_device(sig))
    assert relerr(out.cpu().numpy(), (1 + 0.5j) * ref) < 1e-12
