"""GPU parity tests of the kernel-level entry points (through the C ABI) against NumPy / the oracle.
Tolerances: relative 1e-12 for contractions, 1e-10 for singular values / reconstructions (BASELINE.md §4)."""
import numpy as np
import pytest

import ttn_oracle as o

pytestmark = pytest.mark.gpu


def rnd(rng, shape, cplx):
    a = rng.standard_normal(shape)
    if cplx:
        a = a + 1j * rng.standard_normal(shape)
    return np.asfortranarray(a)


def relerr(a, b):
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


@pytest.mark.parametrize("cplx", [False, True])
@pytest.mark.parametrize("shape", [(1, 1, 1), (5, 3, 7), (64, 64, 16), (130, 70, 33), (200, 300, 129), (257, 129, 64), (20, 20, 1000)])
def test_gemm_shapes(shape, cplx):
    import ttn_b200 as t
    M, N, K = shape
    rng = np.random.default_rng(M * 7 + N * 3 + K)
    A, B = rnd(rng, (M, K), cplx), rnd(rng, (K, N), cplx)
    assert relerr(t.gemm_host(A, B), A @ B) < 1e-13


@pytest.mark.parametrize("cplx", [False, True])
def test_gemm_ops_alpha_beta(cplx):
    import ttn_b200 as t
    rng = np.random.default_rng(5)
    M, N, K = 70, 45, 90
    At, Bt, C0 = rnd(rng, (K, M), cplx), rnd(rng, (N, K), cplx), rnd(rng, (M, N), cplx)
    got = t.gemm_host(At, Bt, transA=True, transB=True, conjA=True, conjB=False, alpha=0.5, beta=-2.0, C0=C0)
    ref = 0.5 * (At.conj().T @ Bt.T) - 2.0 * C0
    assert relerr(got, ref) < 1e-13
    got = t.gemm_host(At, Bt, transA=True, transB=True, conjA=False, conjB=True)
    assert relerr(got, At.T @ Bt.conj().T) < 1e-13


def test_gemm_large_real_hits_big_tile():
    import ttn_b200 as t
    rng = np.random.default_rng(6)
    A, B = rnd(rng, (1500, 700), False), rnd(rng, (700, 1300), False)
    assert relerr(t.gemm_host(A, B), A @ B) < 1e-13
    Ac, Bc = rnd(rng, (900, 300), True), rnd(rng, (300, 1300), True)
    assert relerr(t.gemm_host(Ac, Bc), Ac @ Bc) < 1e-13


@pytest.mark.parametrize("cplx", [False, True])
@pytest.mark.parametrize("shape", [(1, 1), (7, 3), (3, 7), (40, 40), (100, 17), (300, 64), (64, 200), (1024, 96)])
def test_qr(shape, cplx):
    import ttn_b200 as t
    m, n = shape
    rng = np.random.default_rng(m + 13 * n)
    A = rnd(rng, (m, n), cplx)
    Q, R = t.qr_thin(A)
    k = min(m, n)
    assert Q.shape == (m, k) and R.shape == (k, n)
    assert relerr(Q @ R, A) < 1e-13
    assert np.abs(Q.conj().T @ Q - np.eye(k)).max() < 1e-13
    assert np.abs(np.tril(R, -1)).max() == 0.0


def test_qr_rank_deficient():
    import ttn_b200 as t
    rng = np.random.default_rng(3)
    A = rnd(rng, (50, 4), False) @ rnd(rng, (4, 12), False)
    A[:, 5] = 0.0
    Q, R = t.qr_thin(np.asfortranarray(A))
    assert relerr(Q @ R, A) < 1e-13
    assert np.abs(Q.T @ Q - np.eye(12)).max() < 1e-12


@pytest.mark.parametrize("cplx", [False, True])
@pytest.mark.parametrize("shape", [(6, 4), (4, 6), (5, 5), (64, 64), (32, 200), (200, 32), (128, 128), (128, 1024), (300, 180)])
def test_svdtrunc_full(shape, cplx):
    import ttn_b200 as t
    m, n = shape
    rng = np.random.default_rng(m * 3 + n)
    A = rnd(rng, (m, n), cplx)
    U, s, Vt = t.svdtrunc(A)
    sref = np.linalg.svd(A, compute_uv=False)
    assert len(s) == min(m, n)
    assert np.abs(s - sref).max() / sref[0] < 1e-13          # singular values
    assert np.all(np.diff(s) <= 0)
    assert relerr((U * s) @ Vt, A) < 1e-12                   # reconstruction
    assert np.abs(U.conj().T @ U - np.eye(len(s))).max() < 1e-12
    assert np.abs(Vt @ Vt.conj().T - np.eye(len(s))).max() < 1e-10


def test_svdtrunc_rules_and_relative_accuracy():
    # test/test_tdvp.jl:28-44 + Appendix B tail-norm rule; small singular values to high relative accuracy
    import ttn_b200 as t
    rng = np.random.default_rng(11)
    A = rnd(rng, (6, 4), False)
    U, s, Vt = t.svdtrunc(A, max_bond=2)
    assert len(s) == 2 and np.allclose(s, np.linalg.svd(A, compute_uv=False)[:2], rtol=1e-12)
    Q1, _ = np.linalg.qr(rng.standard_normal((40, 5)))
    Q2, _ = np.linalg.qr(rng.standard_normal((30, 5)))
    sv = np.array([1.0, 1e-3, 1e-6, 1e-9, 1e-12])
    B = np.asfortranarray(Q1 @ np.diag(sv) @ Q2.T)
    for te, want in [(1e-4, 2), (1e-7, 3), (0.5, 1), (1e-13, 5)]:
        assert len(t.svdtrunc(B, truncerr=te)[1]) == len(o.svdtrunc(B, truncerr=te)[1]) == want
    s5 = t.svdtrunc(B, max_bond=5)[1]
    assert np.abs(s5[:4] / sv[:4] - 1).max() < 1e-6   # graded spectrum: relative accuracy far below eps*s_max
    U1, s1, Vt1 = t.svdtrunc(B, max_bond=1)
    assert U1.shape == (40, 1) and Vt1.shape == (1, 30)


def test_svdtrunc_rank_deficient_and_zero():
    import ttn_b200 as t
    rng = np.random.default_rng(12)
    A = np.asfortranarray(rnd(rng, (20, 3), False) @ rnd(rng, (3, 16), False))
    U, s, Vt = t.svdtrunc(A)
    assert relerr((U * s) @ Vt, A) < 1e-12
    assert np.all(np.isfinite(U)) and np.all(np.isfinite(Vt))
    Z = np.zeros((5, 4), order="F")
    U, s, Vt = t.svdtrunc(Z)
    assert np.all(s == 0) and np.all(np.isfinite(U)) and np.all(np.isfinite(Vt))


@pytest.mark.parametrize("cplx", [False, True])
@pytest.mark.parametrize("sym", [False, True])
@pytest.mark.parametrize("dims", [(1, 1, 1, 1, 4), (3, 3, 8, 8, 4), (5, 5, 17, 9, 4), (2, 4, 33, 20, 2), (5, 5, 64, 64, 4)])
def test_matvec2_vs_oracle(dims, sym, cplx):
    # K_matfree of src/solvers/dmrg.jl:239-244
    import ttn_b200 as t
    wl, wr, cl, cr, nn = dims
    rng = np.random.default_rng(sum(dims))
    G, H = rnd(rng, (wl, cl, cl), cplx), rnd(rng, (wr, cr, cr), cplx)
    Am, V = rnd(rng, (wl, nn, nn, wr), cplx), rnd(rng, (cl, nn, cr), cplx)
    Y = t.matvec2(G, Am, H, V, symmetrize=sym)
    assert relerr(Y, o.dmrg_matvec2(G, Am, V, H, symmetrize=sym)) < 1e-13


@pytest.mark.parametrize("cplx", [False, True])
def test_env_updates_vs_oracle(cplx):
    # update_G! / update_H! of src/solvers/dmrg.jl:27-35
    import ttn_b200 as t
    rng = np.random.default_rng(21)
    n, wl, wr, rl, rr = 2, 3, 4, 7, 5
    x, A = rnd(rng, (n, rl, rr), cplx), rnd(rng, (n, n, wl, wr), cplx)
    G, H = rnd(rng, (wl, rl, rl), cplx), rnd(rng, (wr, rr, rr), cplx)
    assert relerr(t.env_left(G, x, A), o.dmrg_update_G(x, A, G)) < 1e-13
    assert relerr(t.env_right(H, x, A), o.dmrg_update_H(x, A, H)) < 1e-13
    n, wl, wr, rl, rr = 3, 5, 5, 40, 33
    x, A = rnd(rng, (n, rl, rr), cplx), rnd(rng, (n, n, wl, wr), cplx)
    G, H = rnd(rng, (wl, rl, rl), cplx), rnd(rng, (wr, rr, rr), cplx)
    assert relerr(t.env_left(G, x, A), o.dmrg_update_G(x, A, G)) < 1e-13
    assert relerr(t.env_right(H, x, A), o.dmrg_update_H(x, A, H)) < 1e-13


@pytest.mark.gpu
@pytest.mark.parametrize("nranks", [1, 2, 4])
@pytest.mark.parametrize("cplx", [False, True])
def test_sharded_matvec_slices_vs_oracle(nranks, cplx):
    """cfg4 sharding (SURVEY.md section 8(e)): every rank's slice Y[:, :, c_p] against K_matfree (dmrg.jl:239-244); the ranks
    are emulated one after the other on the single test GPU (unbound operators write only their own slice)."""
    import ttn_b200 as t
    rng = np.random.default_rng(5)
    w_l, w_r, chi_l, chi_r, nn = 3, 5, 24, 30, 4

    def rnd(*s):
        a = rng.standard_normal(s)
        return a + 1j * rng.standard_normal(s) if cplx else a
    G, H, Am, V = rnd(w_l, chi_l, chi_l), rnd(w_r, chi_r, chi_r), rnd(w_l, nn, nn, w_r), rnd(chi_l, nn, chi_r)
    Yref = o.dmrg_matvec2(G, Am, V, H, symmetrize=False)
    parts = []
    for r in range(nranks):
        op = t.ShardedMatvec(G, Am, H, rank=r, nranks=nranks)
        assert (op.c0, op.cp) == t.shard_range(chi_r, r, nranks)
        parts.append(op.local_slice(V))
        op.free()
    Y = t.assemble_slices(parts, axis=2)
    assert relerr(Y, Yref) < 1e-13


@pytest.mark.gpu
def test_sharded_eigsolve_single_rank_matches_dense():
    """Lanczos on the sharded operator (nranks = 1) against eigvalsh of the dense K (dmrg.jl:49-54, 245)."""
    import ttn_b200 as t
    rng = np.random.default_rng(6)
    w, chi, nn = 3, 6, 4
    G = rng.standard_normal((w, chi, chi)); G = G + np.transpose(G, (0, 2, 1))
    H = rng.standard_normal((w, chi, chi)); H = H + np.transpose(H, (0, 2, 1))
    Am = rng.standard_normal((w, nn, nn, w)); Am = Am + np.transpose(Am, (0, 2, 1, 3))
    from ttn_oracle import dmrg as odmrg
    K, dims = odmrg.K_full(G, H, Am)
    K = 0.5 * (K + K.T)
    # symmetric pieces make the single application symmetric up to the G/H/Amid transposes used above
    op = t.ShardedMatvec(G, Am, H)
    th, x, mv = op.eigsolve(rng.standard_normal((chi, nn, chi)), krylovdim=40, maxiter=20, tol=1e-12)
    op.free()
    ev = np.linalg.eigvalsh(K)
    assert abs(th - ev[0]) < 1e-9 * max(1.0, abs(ev[0]))


@pytest.mark.gpu
@pytest.mark.parametrize("bad", [np.nan, np.inf])
@pytest.mark.parametrize("shape", [(20, 30), (100, 100), (400, 500), (700, 660)])
def test_svdtrunc_non_finite_input_raises(shape, bad):
    """One NaN or inf entry is reported as a non-finite singular value, not returned as a result.  The shapes reach each Jacobi
    engine: one SM (n < 32), the 8-CTA cluster, the cross-CTA block path and the Gram-block path, whose rotation guards skip
    a pair unless both squared column norms are positive (false for NaN)."""
    import ttn_b200 as t
    rng = np.random.default_rng(shape[0] + shape[1])
    A = rnd(rng, shape, False)
    A[shape[0] // 3, shape[1] // 2] = bad
    with pytest.raises(RuntimeError, match="non-finite singular value"):
        t.svdtrunc(A)


@pytest.mark.gpu
@pytest.mark.parametrize("cond", [1e2, 1e6, 1e12])
@pytest.mark.parametrize("shape", [(1024, 128), (128, 1024), (300, 64), (96, 96)])
def test_svdtrunc_across_condition_numbers(shape, cond):
    """`_svdtrunc` (tt_cross_interpolation.jl:149-166) on prescribed spectra: the CholeskyQR2 preconditioner is taken for
    well-conditioned tall/wide inputs and must hand over to Householder QR as the conditioning degrades; singular values to
    1e-12 of sigma_1 (gesdd's absolute accuracy), reconstruction to 1e-12."""
    import ttn_b200 as t
    rng = np.random.default_rng(int(np.log10(cond)) + shape[0])
    m, n = shape
    k = min(m, n)
    U, _ = np.linalg.qr(rng.standard_normal((m, k)))
    V, _ = np.linalg.qr(rng.standard_normal((n, k)))
    s = np.logspace(0, -np.log10(cond), k)
    A = np.asfortranarray((U * s) @ V.T)
    Ug, sg, Vtg = t.svdtrunc(A)
    assert np.abs(sg - s).max() < 1e-12
    assert relerr((Ug * sg) @ Vtg, A) < 1e-12
    assert np.abs(Ug.T @ Ug - np.eye(k)).max() < 1e-11


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(1024, 1024), (1100, 1030), (700, 660)])
def test_svdtrunc_large_gram_block_path(shape):
    """Bond matrices of DMRG size take the Gram-block Jacobi on the DMMA pipe (jacobi_gram.cu, two pair groups on two
    streams) after the Householder preconditioning: singular values and reconstruction against LAPACK."""
    import ttn_b200 as t
    rng = np.random.default_rng(shape[1])
    m, n = shape
    k = min(m, n)
    U, _ = np.linalg.qr(rng.standard_normal((m, k)))
    V, _ = np.linalg.qr(rng.standard_normal((n, k)))
    s = np.logspace(0, -8, k)
    A = np.asfortranarray((U * s) @ V.T)
    Ug, sg, Vtg = t.svdtrunc(A)
    assert np.abs(sg - s).max() < 1e-11
    assert relerr((Ug * sg) @ Vtg, A) < 1e-11
    assert np.abs(Ug.T @ Ug - np.eye(k)).max() < 1e-10


@pytest.mark.gpu
@pytest.mark.parametrize("cond", [3.0, 1e3, 1e9])
@pytest.mark.parametrize("shape,cplx", [((1024, 128), True), ((128, 1024), True), ((1024, 256), False), ((256, 1024), False)])
def test_svdtrunc_two_panel_cholqr(shape, cplx, cond):
    """Column counts whose k x k Cholesky does not fit one SM (ComplexF64 k = 128, the cfg5 bond; Float64 k = 256) take the
    two-panel CholeskyQR2 (cholqr.cu) for well-conditioned inputs and Householder QR otherwise: same accuracy either way."""
    import ttn_b200 as t
    rng = np.random.default_rng(shape[0] + int(cond))
    m, n = shape
    k = min(m, n)
    g = lambda a, b: rng.standard_normal((a, b)) + (1j * rng.standard_normal((a, b)) if cplx else 0.0)
    U, _ = np.linalg.qr(g(m, k))
    V, _ = np.linalg.qr(g(n, k))
    s = np.logspace(0, -np.log10(cond), k)
    A = np.asfortranarray((U * s) @ V.conj().T)
    Ug, sg, Vtg = t.svdtrunc(A)
    assert np.abs(sg - s).max() < 1e-12
    assert relerr((Ug * sg) @ Vtg, A) < 1e-12
    assert np.abs(Ug.conj().T @ Ug - np.eye(k)).max() < 1e-11


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(128, 128), (96, 200), (256, 192), (700, 660)])
def test_svdtrunc_degenerate_multiplets(shape):
    """Exactly degenerate singular values (multiplets, as symmetric DMRG states produce): the Jacobi rotations inside a
    multiplet have large angles however small the inner product is, so the "all rotations were second order" shortcut of the
    cluster / Gram-block kernels must not fire on them; U stays orthonormal to 1e-11 and the reconstruction exact."""
    import ttn_b200 as t
    rng = np.random.default_rng(shape[0] * 7 + shape[1])
    m, n = shape
    k = min(m, n)
    U, _ = np.linalg.qr(rng.standard_normal((m, k)))
    V, _ = np.linalg.qr(rng.standard_normal((n, k)))
    s = np.repeat(np.logspace(0, -6, (k + 3) // 4), 4)[:k]
    A = np.asfortranarray((U * s) @ V.T)
    Ug, sg, Vtg = t.svdtrunc(A)
    assert np.abs(sg - s).max() < 1e-12
    assert relerr((Ug * sg) @ Vtg, A) < 1e-12
    assert np.abs(Ug.T @ Ug - np.eye(k)).max() < 1e-11


@pytest.mark.gpu
@pytest.mark.parametrize("cplx", [False, True])
@pytest.mark.parametrize("shape", [(1500, 700), (2100, 530), (600, 600), (5000, 96)])
def test_qr_tall_single_matrix_smem_panels(shape, cplx):
    """Householder QR of tall single matrices (the shared-memory sub-panel kernel of qr.cu: sub-panels of 8 / 4 / 2 columns
    depending on the panel height and element size, then the unblocked kernel once fewer than 512 rows remain)."""
    import ttn_b200 as t
    rng = np.random.default_rng(shape[0] + shape[1])
    m, n = shape
    A = rng.standard_normal((m, n)) + (1j * rng.standard_normal((m, n)) if cplx else 0.0)
    A = np.asfortranarray(A * np.logspace(0, -6, n)[None, :])            # graded columns
    Q, R = t.qr_thin(A)
    k = min(m, n)
    assert np.abs(np.tril(R, -1)).max() == 0.0
    assert relerr(Q @ R, A) < 1e-13
    assert np.abs(Q.conj().T @ Q - np.eye(k)).max() < 1e-12


@pytest.mark.parametrize("transB", [False, True])
@pytest.mark.parametrize("shape", [(1536, 1280, 16), (1536, 1280, 96), (2048, 1152, 1040), (1280, 1536, 48)])
def test_gemm_tma_staged_big_tile(shape, transB):
    """The TMA-staged big-tile kernel (cp.async.bulk + mbarrier, csrc/gemm.cu::gemm_bulk_kernel) is taken for Float64 full-tile
    problems with unit-stride tile rows (both B layouts: k-fastest and n-fastest); same result as the LDGSTS kernel and NumPy,
    with alpha / beta."""
    import ttn_b200 as t
    M, N, K = shape
    rng = np.random.default_rng(M + N + K + transB)
    A = rnd(rng, (M, K), False)
    B = rnd(rng, (N, K) if transB else (K, N), False)
    C0 = rnd(rng, (M, N), False)
    ref = 0.75 * (A @ (B.T if transB else B)) - 0.5 * C0
    assert t.get_option("gemm_bulk") == 1.0
    got = t.gemm_host(A, B, transB=transB, alpha=0.75, beta=-0.5, C0=C0)
    assert relerr(got, ref) < 1e-13
    t.set_option("gemm_bulk", 0)
    try:
        plain = t.gemm_host(A, B, transB=transB, alpha=0.75, beta=-0.5, C0=C0)
    finally:
        t.set_option("gemm_bulk", 1)
    assert relerr(plain, ref) < 1e-13
    assert relerr(got, plain) < 1e-14


@pytest.mark.parametrize("cplx", [False, True])
@pytest.mark.parametrize("shape", [(1024, 20, 20), (777, 10, 32), (4096, 32, 7), (256, 1, 1)])
def test_gemm_thin_right_multiplication(shape, cplx):
    """The streaming kernel for thin right-multiplications (csrc/gemm.cu::gemm_thin_kernel; the middle contraction T2 = T1 . W of
    the effective operators, dmrg.jl:239-244, with K = w n^2 <= 32) against NumPy and against the DMMA tile path, with alpha / beta,
    both B layouts and conj(B)."""
    import ttn_b200 as t
    M, N, K = shape
    rng = np.random.default_rng(M + 3 * N + 7 * K + cplx)
    A = rnd(rng, (M, K), cplx)
    C0 = rnd(rng, (M, N), cplx)
    assert t.get_option("gemm_thin") == 1.0
    for transB, conjB in [(False, False), (True, False), (True, True)]:
        B = rnd(rng, (N, K) if transB else (K, N), cplx)
        Bm = B.T if transB else B
        ref = 1.25 * (A @ (Bm.conj() if conjB else Bm)) + 0.5 * C0
        got = t.gemm_host(A, B, transB=transB, conjB=conjB, alpha=1.25, beta=0.5, C0=C0)
        assert relerr(got, ref) < 1e-14
        t.set_option("gemm_thin", 0)
        try:
            tiles = t.gemm_host(A, B, transB=transB, conjB=conjB, alpha=1.25, beta=0.5, C0=C0)
        finally:
            t.set_option("gemm_thin", 1)
        assert relerr(got, tiles) < 1e-14
    assert relerr(t.gemm_host(A, rnd(rng, (K, N), cplx) * 0 + 1.0), A.sum(axis=1, keepdims=True) * np.ones((1, N))) < 1e-14
