"""GPU tests of the small Hermitian eigensolver behind the Gram path of tt_compress! (csrc/heig.cu) through the C ABI
(`ttn_heig_host`): eigenvalues 1e-13 |G|, residual |G U - U L| 1e-13 |G|, orthonormality 5e-12 (the accuracy the rank-cap path
needs: reconstructions 1e-10, BASELINE.md §4); clustered / degenerate / decaying spectra must either meet the same bar or raise
the fall-back flag."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def wishart(rng, n, q, cplx):
    th = rng.standard_normal((n, q)) + (1j * rng.standard_normal((n, q)) if cplx else 0)
    return th @ th.conj().T


def check(G, nev, lam, U, tol_orth=5e-12):
    w = np.linalg.eigvalsh(G)[::-1]
    nrm = max(abs(w[0]), 1e-300)
    assert np.max(np.abs(lam - w[:nev])) / nrm < 1e-13
    assert np.linalg.norm(U.conj().T @ U - np.eye(nev)) < tol_orth
    assert np.linalg.norm(G @ U - U * lam) / nrm < 1e-13 * max(4, G.shape[0]) ** 0.5 * 4


@pytest.mark.parametrize("cplx", [False, True])
@pytest.mark.parametrize("n,nev", [(128, 64), (128, 128), (64, 64), (64, 17), (96, 40), (33, 33), (16, 8), (5, 3), (2, 2), (2, 1), (1, 1)])
def test_heig_single(n, nev, cplx):
    import ttn_b200 as t
    rng = np.random.default_rng(1000 * n + nev + cplx)
    G = wishart(rng, n, 4 * n + 3, cplx)
    lam, U, flag = t.heig_top(G, nev)
    assert flag == 0
    check(G, nev, lam, U)


def test_heig_real_176():
    import ttn_b200 as t
    rng = np.random.default_rng(7)
    G = wishart(rng, 176, 700, False)
    lam, U, flag = t.heig_top(G, 90)
    assert flag == 0
    check(G, 90, lam, U)


@pytest.mark.parametrize("cplx", [False, True])
def test_heig_batched(cplx):
    import ttn_b200 as t
    rng = np.random.default_rng(11 + cplx)
    for n, nev, b in ((128, 64, 160), (64, 64, 300), (24, 10, 7)):
        G = np.stack([wishart(rng, n, 3 * n, cplx) for _ in range(b)])
        lam, U, flags = t.heig_top(G, nev)
        assert not flags.any()
        for k in range(b):
            check(G[k], nev, lam[k], U[k])


def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


# Launch switches of heig_top, by batch size against the SM count: multisection M = 32 (batch <= sm/16), M = 8 (<= sm/4),
# then one CTA per matrix with M = 4 (nev <= 64) or M = 2 (nev > 64); back-transformation over many CTAs (batch <= sm/8) or
# one CTA per matrix.  The four batches below reach every pair of them.
BATCHES = {"sm/16": lambda sm: sm // 16, "sm/8": lambda sm: sm // 8, "sm/4": lambda sm: sm // 4, "sm/4+1": lambda sm: sm // 4 + 1}
# n: the three register tridiagonalisations (Float64 n <= 32 / 64 / 128), the shared-memory one (ComplexF64, Float64 > 128),
# back-transformation rows per lane NR = 4 / 8 / 16 / 22;  nev: one vector chunk, chunk boundary (64 / 65), all
SHAPES = [(cplx, n, nev) for cplx, ns in ((False, (32, 33, 64, 65, 128, 129, 176)), (True, (32, 33, 64, 65, 128)))
          for n in ns for nev in sorted({1, 64, 65, n}) if nev <= n]


@pytest.mark.parametrize("batch", list(BATCHES))
@pytest.mark.parametrize("cplx,n,nev", SHAPES)
def test_heig_batched_launch_branches(cplx, n, nev, batch):
    """every matrix of a batch on each side of the launch switches, against NumPy"""
    import ttn_b200 as t
    b = BATCHES[batch](sm_count())
    rng = np.random.default_rng(100000 * cplx + 1000 * n + nev)
    G = np.stack([wishart(rng, n, 3 * n, cplx) for _ in range(b)])
    lam, U, flags = t.heig_top(G, nev)
    assert not flags.any()
    for k in range(b):
        check(G[k], nev, lam[k], U[k])


def with_spectrum(rng, w, cplx):
    n = len(w)
    Q, _ = np.linalg.qr(rng.standard_normal((n, n)) + (1j * rng.standard_normal((n, n)) if cplx else 0))
    G = (Q * w) @ Q.conj().T
    return (G + G.conj().T) / 2


@pytest.mark.parametrize("cplx", [False, True])
def test_heig_clusters_across_vector_chunks(cplx):
    """The twisted-vector kernel works in chunks of at most 64 vectors (halved when shared memory is short: 32 at real
    n = 176) and re-orthogonalises clusters after the last chunk.  Close pairs (gap 1e-8) at indices 31/32, 63/64 and 95/96
    straddle the chunk boundaries; a pair straddling the nev cut; a cluster of 8 is served; a cluster of 9 raises flag 1."""
    import ttn_b200 as t
    n = 128 if cplx else 176
    rng = np.random.default_rng(50 + cplx)
    base = np.linspace(2.0, 1.0, n)            # descending, spacing far above the cluster tolerance

    def spectrum(groups):
        w = base.copy()
        for i0, size in groups:
            w[i0:i0 + size] = w[i0] - 1e-8 * np.arange(size)
        return w

    for nev, groups in ((n, [(31, 2), (63, 2), (95, 2)]), (64, [(63, 2)]), (n, [(60, 8)]), (40, [(36, 8)])):
        G = with_spectrum(rng, spectrum(groups), cplx)
        lam, U, flag = t.heig_top(G, nev)
        assert flag == 0, (nev, groups)
        check(G, nev, lam, U)
    for nev in (n, 69):
        G = with_spectrum(rng, spectrum([(60, 9)]), cplx)
        _, _, flag = t.heig_top(G, nev)
        assert flag & 1, nev


def test_heig_clusters_and_fallback_flags():
    import ttn_b200 as t
    rng = np.random.default_rng(3)
    n = 64
    Q, _ = np.linalg.qr(rng.standard_normal((n, n)))
    # close pairs inside the kept set are re-orthogonalised
    for gap in (1e-5, 1e-8):
        w = np.r_[np.linspace(1, 2, n - 2), 2.5, 2.5 + gap]
        G = (Q * w) @ Q.T
        lam, U, flag = t.heig_top(G, 32)
        assert flag == 0
        check(G, 32, lam, U)
    # exactly degenerate pair in the kept set / decaying spectrum: either accurate or flagged for the Jacobi path
    for w in (np.r_[np.linspace(1, 2, n - 2), 2.5, 2.5], 10.0 ** -np.arange(n, dtype=float)):
        G = (Q * w) @ Q.T
        lam, U, flag = t.heig_top(G, 32)
        if flag == 0:
            check(G, 32, lam, U)
    # a zero matrix has no basis to vouch for: it must be handed to the Jacobi path
    _, _, flag = t.heig_top(np.zeros((n, n)), 32)
    assert flag & 16
    # a multiplet outside the kept set does not matter
    w = np.r_[np.ones(10), np.linspace(2, 3, n - 10)]
    G = (Q * w) @ Q.T
    lam, U, flag = t.heig_top(G, 40)
    assert flag == 0
    check(G, 40, lam, U)
