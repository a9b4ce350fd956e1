"""GPU tests of the Gram path of tt_compress! (`tt_compress_gram`, csrc/tt.cu) and of the fused `apply_compress` at the
shapes and batch sizes where its kernels change: the benchmark's cfg5 call (ComplexF64, d = 30, rank 64, MPO rank 4, chunks
of 296 vectors), batches on both sides of every launch switch of the Gram GEMM and of the eigensolver (csrc/heig.cu),
sweeps that mix Gram steps with classic steps, two sweeps, a batch in which one train declines, and inputs whose Gram
matrices sit near the under- and overflow range.

Every test that expects the fast path also checks that it served the call: `gram_calls` went up by the number of calls,
`gram_fallbacks` did not move and `gram_last_flags` is 0.  A Gram path that declined everything would still return right
answers (from the QR + Jacobi path), so without that check a broken fast path passes.

Results are held to the oracle (`ttn_oracle.tt_compress`) within `max(40 sens, 10 eps sum_steps sigma_1 / sigma_r)`:
`sens` is the oracle's own response to a 1e-16 relative perturbation of its input (truncating a flat spectrum is ill
conditioned), the second term is the Gram path's error bound, eps sigma_1 / sigma_r per bond step.  Trains that are not
sent to the oracle are compared with the same vector computed at another batch size, on the device: the distance is the
norm of the first core of the right-orthogonalised difference, which resolves rounding level."""
import math

import numpy as np
import pytest

import ttn_oracle as o

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps


def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def counters(t):
    return int(t.get_option("gram_calls")), int(t.get_option("gram_fallbacks"))


def assert_served(t, before, ncalls):
    """the Gram path served the last `ncalls` calls: counted, not redone by the Jacobi path, no flag raised"""
    calls, fb = counters(t)
    assert calls == before[0] + ncalls, (calls, before)
    assert fb == before[1], (fb, before)
    assert int(t.get_option("gram_last_flags")) == 0


def assert_declined(t, before, ncalls, flag):
    """each of the last `ncalls` calls took the Gram path, raised `flag` and was redone by the Jacobi path"""
    calls, fb = counters(t)
    assert calls == before[0] + ncalls, (calls, before)
    assert fb == before[1] + ncalls, (fb, before)
    assert int(t.get_option("gram_last_flags")) & flag


def oracle(y, max_bond, sweeps=1, seed=0):
    """the oracle's tt_compress of the host train `y` -> (result, per-step singular values, tolerance of a comparison)"""
    sig = []
    ref = o.tt_compress(o.copy_tt(y), max_bond, sweeps=sweeps, sigma_out=sig)
    pert = o.copy_tt(y)
    rng = np.random.default_rng(seed)
    for k in range(pert.N):
        pert.ttv_vec[k] = pert.ttv_vec[k] * (1 + 1e-16 * rng.standard_normal(pert.ttv_vec[k].shape))
    sens = o.rel_distance(o.tt_compress(pert, max_bond, sweeps=sweeps), ref)
    tol = max(40 * sens, 10 * EPS * sum(s[0] / s[-1] for s in sig))
    return ref, sig, tol


def assert_matches(y, ref, tol, what=""):
    assert list(y.ttv_rks) == list(ref.ttv_rks), (what, y.ttv_rks, ref.ttv_rks)
    dist = o.rel_distance(y, ref)
    print(f"  {what}: oracle distance {dist:.2e}, tolerance {tol:.2e}")
    assert dist < tol, (what, dist, tol)
    return dist


def assert_sigma(sig, sig_ref, what=""):
    """the singular values of train 0 at every bond step, to 1e-10 sigma_1 of the step"""
    assert len(sig) == len(sig_ref), (what, len(sig), len(sig_ref))
    for st, (a, c) in enumerate(zip(sig, sig_ref)):
        assert len(a) == len(c), (what, st, len(a), len(c))
        assert np.abs(np.asarray(a) - np.asarray(c)).max() <= 1e-10 * c[0], (what, st)


def dev_distances(t, a, b):
    """||a_i - b_i|| / ||b_i|| for every train of two batched device trains of the same shape"""
    diff = t.orthogonalize(t.sub(a, b), 1)
    return np.atleast_1d(t.norm(diff)) / np.atleast_1d(t.norm(b))


def heig_max_n(cplx):
    """largest Gram matrix the eigensolver serves (csrc/heig.cu)"""
    return 128 if cplx else 176


# ---------------------------------------------------------------------------------------------------------------------
# A.1 cfg5 at the benchmark's batch size
# ---------------------------------------------------------------------------------------------------------------------
def test_cfg5_fused_at_benchmark_batch_vs_oracle():
    """`apply_compress(A, x, 64)` on 296 cfg5 vectors (the benchmark's chunk): the fast path serves it, trains 0, 1, 147 and
    295 match the oracle (ranks, TT distance, truncation error to 1e-11 of ||Ax||), the sigma of train 0 matches at all 58
    steps, and every train matches the same vector rounded in a batch of 8 (other launch branches of the eigensolver)."""
    import bench
    import ttn_b200 as t
    nb, chunk, d = 296, 8, bench.D5
    rks, _ = bench.cfg5_ranks()
    A = bench.make_mpo(o)
    xs = [o.TTvector(d, bench.make_vector(100 + b), (2,) * d, list(rks), [0] * d) for b in range(nb)]
    Ad = t.DeviceTTO.upload(A)
    xd = t.DeviceTT.upload(xs)
    c0 = counters(t)
    yd, sig = t.apply_compress(Ad, xd, bench.MAXB5, return_sigma=True)
    assert_served(t, c0, 1)
    ys = yd.download()
    yd.free(); xd.free()
    tols = []
    for b in (0, 1, 147, 295):
        ax = o.apply(A, xs[b])
        ref, sig_ref, tol = oracle(ax, bench.MAXB5, seed=b)
        if b == 0:
            assert len(sig_ref) == 2 * (d - 1)
            assert_sigma(sig, sig_ref, "cfg5 train 0")
        tols.append(tol)
        assert_matches(ys[b], ref, tol, f"cfg5 train {b}")
        # truncation error ||y - Ax|| of the device result and of the oracle's, from inner products (no cancellation: the
        # error is 0.8 ||Ax|| here)
        nax2 = np.real(o.dot(ax, ax))

        def err(y):
            return math.sqrt(max(np.real(o.dot(y, y)) + nax2 - 2 * np.real(o.dot(ax, y)), 0.0))
        gap = abs(err(ys[b]) - err(ref)) / math.sqrt(nax2)
        print(f"  cfg5 train {b}: truncation-error difference {gap:.2e}")
        assert gap < 1e-11, (b, gap)
    # every train against the same vector in a batch of 8 (other launch branches of the Gram GEMM and of the eigensolver);
    # both are within `tol` of the exact rounding
    worst = 0.0
    for s in range(0, nb, chunk):
        c1 = counters(t)
        y8 = t.apply_compress(Ad, t.DeviceTT.upload(xs[s:s + chunk]), bench.MAXB5)
        assert_served(t, c1, 1)
        assert y8.ttv_rks == ys[s].ttv_rks
        y296 = t.DeviceTT.upload(ys[s:s + chunk])
        dist = dev_distances(t, y296, y8)
        worst = max(worst, float(dist.max()))
        y8.free(); y296.free()
    print(f"  cfg5 batch 296 vs batch 8: worst distance {worst:.2e}, tolerance {2 * max(tols):.2e}")
    assert worst < 2 * max(tols)


# ---------------------------------------------------------------------------------------------------------------------
# A.2 batch sweep of the fused and the two-call path
# ---------------------------------------------------------------------------------------------------------------------
def small_problem(cplx, nvec, d=12, r=64, W=2, seed=0):
    rng = np.random.default_rng(seed + 1000 * cplx)
    dt = np.complex128 if cplx else np.float64
    A = o.rand_tto((2,) * d, W, rng=rng, dtype=dt)
    xs = [o.rand_tt((2,) * d, r, rng=rng, dtype=dt, normalise=True) for _ in range(nvec)]
    return A, xs


def test_batch_sweep_over_launch_switches():
    """Complex d = 12, rank 64, MPO rank 2, max_bond 64 (Gram matrices 128 x 128, q >= 128 so the split-K Gram GEMM can
    split): batches 1, sm/16, sm/16 + 1, sm/8, sm/8 + 1, sm/4, sm/4 + 1 and 2 sm cross every launch switch of the Gram GEMM
    split, the multisection (M = 32 / 8 / 4 / 2) and the back-transformation.  Fused and two-call paths are served by the
    fast path; the first and last train of each batch match the oracle; every train matches its batch-of-1 result."""
    import ttn_b200 as t
    sm = sm_count()
    batches = sorted({1, sm // 16, sm // 16 + 1, sm // 8, sm // 8 + 1, sm // 4, sm // 4 + 1, 2 * sm})
    mb = 64
    A, xs = small_problem(True, max(batches))
    Ad = t.DeviceTTO.upload(A)
    # batch-of-1 results of every vector (fused)
    c0 = counters(t)
    ones = [t.apply_compress(Ad, t.DeviceTT.upload(x), mb).download() for x in xs]
    assert_served(t, c0, len(xs))
    refs = {}
    tol_max = 0.0
    for b in sorted({0} | {B - 1 for B in batches}):
        refs[b] = oracle(o.apply(A, xs[b]), mb, seed=b)
        tol_max = max(tol_max, refs[b][2])
    for b in refs:
        assert_matches(ones[b], refs[b][0], refs[b][2], f"batch 1, vector {b}")
    for B in batches:
        xd = t.DeviceTT.upload(xs[:B] if B > 1 else xs[0])
        c1 = counters(t)
        yf = t.apply_compress(Ad, xd, mb)
        assert_served(t, c1, 1)
        c1 = counters(t)
        y2 = t.tt_compress_(t.apply(Ad, xd), mb)
        assert_served(t, c1, 1)
        one = t.DeviceTT.upload(ones[:B] if B > 1 else ones[0])
        for name, y in (("fused", yf), ("two calls", y2)):
            host = y.download()
            host = host if B > 1 else [host]
            for b in (0, B - 1):
                assert_matches(host[b], refs[b][0], refs[b][2], f"{name}, batch {B}, train {b}")
            dist = dev_distances(t, y, one)
            print(f"  {name}, batch {B}: worst distance to batch-of-1 {dist.max():.2e}, tolerance {2 * tol_max:.2e}")
            assert dist.max() < 2 * tol_max, (name, B, dist.max())
            y.free()
        one.free(); xd.free()


# ---------------------------------------------------------------------------------------------------------------------
# A.3 one train of a batch declines
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("bad", ["rank_deficient", "zero"])
@pytest.mark.parametrize("call", ["apply_compress", "tt_compress_"])
def test_one_flagged_train_redoes_the_batch(bad, call):
    """A batch of 296 in which only train 200 declines: rank-deficient (its padding rows are zero, so the kept spectrum
    holds zeros: flag 8) or all zeros (flag 16).  The call is counted as one fall-back; every train matches what the fast
    path gives for it in a batch where train 200 is a regular vector, the flagged train and a sample of the others match
    the oracle, and the sigma of train 0 matches the oracle at every step.
    max_bond is 48, not 64: at 64 two bonds keep the full rank 64 of a square 128 x 128 Theta, whose smallest singular value
    is that of a random square matrix, and a few trains of the pool come within 2x of the sigma_r < 1e-5 sigma_1 bound the
    fast path declines at.  At 48 the smallest kept ratio over the pool is 1.8e-4, so train 200 is the only one to decline."""
    import ttn_b200 as t
    nb, pos, mb, flag = 296, 200, 48, 8 if bad == "rank_deficient" else 16
    A, xs = small_problem(True, nb, seed=3)
    good = list(xs)
    x = o.copy_tt(xs[pos])
    for k in range(x.N):
        if bad == "zero":
            x.ttv_vec[k][:] = 0
        else:
            x.ttv_vec[k][:, 4:, :] = 0
            x.ttv_vec[k][:, :, 4:] = 0
    xs[pos] = x
    Ad = t.DeviceTTO.upload(A)

    def run(vecs):
        xd = t.DeviceTT.upload(vecs)
        if call == "apply_compress":
            return t.apply_compress(Ad, xd, mb, return_sigma=True)
        return t.tt_compress_(t.apply(Ad, xd), mb, return_sigma=True)

    c0 = counters(t)
    yg, _ = run(good)
    assert_served(t, c0, 1)
    c0 = counters(t)
    yd, sig = run(xs)
    assert_declined(t, c0, 1, flag)
    ys = yd.download()
    for y in ys:
        assert all(np.isfinite(c).all() for c in y.ttv_vec)
    # the fall-back result of every train against the fast-path result of the same train (train 200 differs)
    dist = dev_distances(t, yd, yg)
    ax = o.apply(A, xs[pos])
    ref = o.tt_compress(o.copy_tt(ax), mb)
    assert ys[pos].ttv_rks == ref.ttv_rks
    if bad == "zero":
        assert o.norm_stable(ys[pos]) == 0.0
    else:
        # A x has rank 8 < 48: nothing is truncated and both results are A x to rounding
        assert o.rel_distance(ys[pos], ref) < 1e-12 and o.rel_distance(ys[pos], ax) < 1e-12
    tol_max = 0.0
    for b in (0, pos - 1, pos + 1, nb - 1):
        ref_b, sig_ref, tol = oracle(o.apply(A, xs[b]), mb, seed=b)
        tol_max = max(tol, tol_max)
        assert_matches(ys[b], ref_b, tol, f"{call}, {bad}, train {b}")
        if b == 0:
            assert_sigma(sig, sig_ref, f"{call}, {bad}")
    others = np.delete(dist, pos)
    print(f"  {call}, {bad}: worst distance Jacobi path vs Gram path {others.max():.2e}, tolerance {2 * tol_max:.2e}")
    assert others.max() < 2 * tol_max


# ---------------------------------------------------------------------------------------------------------------------
# A.4 sweeps that mix Gram steps with classic steps
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cplx,mb", [(True, 80), (False, 100)])
def test_mixed_gram_and_classic_steps(cplx, mb):
    """d = 16, rank 128 cut to `mb`: the bonds between two rank-`mb`/128 sites have a Gram matrix of order 2 mb (160 > 128
    complex, 200 > 176 real), which the eigensolver does not serve, so they take the classic step inside the Gram sweep.
    The call is still served by the fast path; result and sigma over all 2 (d - 1) steps match the oracle."""
    import ttn_b200 as t
    dt = np.complex128 if cplx else np.float64
    rng = np.random.default_rng(40 + cplx)
    xs = [o.rand_tt((2,) * 16, 128, rng=rng, dtype=dt, normalise=True) for _ in range(3)]
    c0 = counters(t)
    yd, sig = t.tt_compress_(t.DeviceTT.upload(xs), mb, return_sigma=True)
    assert_served(t, c0, 1)
    ys = yd.download()
    for b in (0, 2):
        ref, sig_ref, tol = oracle(xs[b], mb, seed=b)
        assert max(min(2 * ref.ttv_rks[k], 2 * ref.ttv_rks[k + 2]) for k in range(15)) > heig_max_n(cplx)
        assert_matches(ys[b], ref, tol, f"mixed, train {b}")
        if b == 0:
            assert len(sig_ref) == 30
            assert_sigma(sig, sig_ref, "mixed")


# ---------------------------------------------------------------------------------------------------------------------
# A.5 two sweeps
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("call", ["apply_compress", "tt_compress_"])
@pytest.mark.parametrize("cplx", [False, True])
def test_two_sweeps(cplx, call):
    """sweeps = 2 through the Gram path (sigma rows of the second sweep, the column norms handed from each L->R step to the
    R->L step of the same bond in both sweeps): result and sigma over all 4 (d - 1) steps match the oracle."""
    import ttn_b200 as t
    mb, d = 40, 12
    A, xs = small_problem(cplx, 3, d=d, seed=5)
    Ad = t.DeviceTTO.upload(A)
    xd = t.DeviceTT.upload(xs)
    c0 = counters(t)
    if call == "apply_compress":
        yd, sig = t.apply_compress(Ad, xd, mb, sweeps=2, return_sigma=True)
    else:
        yd, sig = t.tt_compress_(t.apply(Ad, xd), mb, sweeps=2, return_sigma=True)
    assert_served(t, c0, 1)
    ys = yd.download()
    for b in (0, 2):
        ref, sig_ref, tol = oracle(o.apply(A, xs[b]), mb, sweeps=2, seed=b)
        assert_matches(ys[b], ref, tol, f"two sweeps, train {b}")
        if b == 0:
            assert len(sig_ref) == 4 * (d - 1)
            assert_sigma(sig, sig_ref, "two sweeps")


# ---------------------------------------------------------------------------------------------------------------------
# A.6 Gram matrices near the under- and overflow range
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("c", [1e-150, 1e-100, 1e100, 1e150])
@pytest.mark.parametrize("call", ["apply_compress", "tt_compress_"])
@pytest.mark.parametrize("cplx", [False, True])
def test_scale_edges(cplx, call, c):
    """c x with Theta Theta^H near the under- or overflow range: the result is finite and is c times the result for x to
    1e-10 (compared after dividing one core by c, so that the comparison cannot overflow).  Declining is allowed; the
    QR + Jacobi path that then computes the result is also run on its own (Gram path off), at every scale."""
    import ttn_b200 as t
    mb, nb = 12, 4
    A, xs = small_problem(cplx, nb, d=10, r=16, seed=7)
    xc = []
    for x in xs:
        y = o.copy_tt(x)
        y.ttv_vec[0] = y.ttv_vec[0] * c
        xc.append(y)
    Ad = t.DeviceTTO.upload(A)

    def run(vecs):
        xd = t.DeviceTT.upload(vecs)
        if call == "apply_compress":
            return t.apply_compress(Ad, xd, mb).download()
        return t.tt_compress_(t.apply(Ad, xd), mb).download()

    c0 = counters(t)
    y1 = run(xs)
    assert_served(t, c0, 1)
    c0 = counters(t)
    yc = run(xc)
    print(f"  scale {c:g}: {'declined' if counters(t)[1] > c0[1] else 'served'}")
    t.set_option("gram_compress", 0)
    try:
        yj = run(xc)
    finally:
        t.set_option("gram_compress", 1)
    for y in (yc, yj):
        for b in range(nb):
            assert all(np.isfinite(v).all() for v in y[b].ttv_vec), b
            assert y[b].ttv_rks == y1[b].ttv_rks
            y[b].ttv_vec[0] = y[b].ttv_vec[0] / c
            dist = o.rel_distance(y[b], y1[b])
            assert dist < 1e-10, (b, dist)
