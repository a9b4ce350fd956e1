"""How the C ABI takes a handle, through ctypes: a train from `ttn_ttv_upload_async` may go to every entry point at once, an
in-place entry point after `ttn_ttv_download_async` leaves the downloaded values intact, and malformed input is refused before
anything is launched."""
import ctypes as C

import numpy as np
import pytest

import ttn_oracle as o

pytestmark = pytest.mark.gpu

EARG, EDIM = 2, 1
F64, C128 = 0, 1
vp = C.c_void_p


def _lib():
    import ttn_b200  # noqa: F401
    from ttn_b200 import _lib as L
    return L.lib()


def _check(st):
    from ttn_b200 import _lib as L
    L.check(st)


class Pinned:
    """The cores of a train (or of `batch` identically shaped trains) in page-locked host memory, batch axis last."""

    def __init__(self, dims, rks, dtype, batch, rng):
        import torch
        self.dims, self.rks, self.dtype, self.batch = tuple(dims), list(rks), np.dtype(dtype), batch
        self.keep, self.cores = [], []
        w = 2 if self.dtype == np.complex128 else 1
        for k, n in enumerate(dims):
            shp = (n, rks[k], rks[k + 1], batch)
            buf = torch.empty(w * int(np.prod(shp)), dtype=torch.float64).pin_memory()
            a = buf.numpy().view(self.dtype).reshape(shp, order="F")
            a[...] = rng.standard_normal(shp) if w == 1 else rng.standard_normal(shp) + 1j * rng.standard_normal(shp)
            self.keep.append(buf)
            self.cores.append(a)

    @classmethod
    def of(cls, x, rng):
        return cls(x.ttv_dims, x.ttv_rks, x.ttv_vec[0].dtype, 1, rng)

    def upload(self, asynchronous):
        lib = _lib()
        d = len(self.dims)
        ptrs = (vp * d)(*[a.ctypes.data for a in self.cores])
        i64 = lambda v: (C.c_int64 * len(v))(*v)  # noqa: E731
        h = vp()
        fn = lib.ttn_ttv_upload_async if asynchronous else lib.ttn_ttv_upload
        _check(fn(F64 if self.dtype == np.float64 else C128, d, i64(self.dims), i64(self.rks), i64([0] * d), ptrs, self.batch,
                  C.byref(h)))
        return h


def _nan_cores(h):
    """NaN-filled host arrays shaped like the cores of the train behind `h` (from its metadata alone)"""
    lib = _lib()
    code, d, batch = C.c_int(), C.c_int(), C.c_int()
    _check(lib.ttn_ttv_info(h, C.byref(code), C.byref(d), C.byref(batch)))
    code, d, batch = code.value, d.value, batch.value
    dims, rks = (C.c_int64 * d)(), (C.c_int64 * (d + 1))()
    _check(lib.ttn_ttv_dims(h, dims))
    _check(lib.ttn_ttv_ranks(h, rks))
    return [np.full((dims[k], rks[k], rks[k + 1], batch), np.nan, dtype=np.float64 if code == F64 else np.complex128, order="F")
            for k in range(d)]


def _cores(h):
    """device -> host copy of every core of the train behind `h` (synchronous)"""
    out = _nan_cores(h)
    _check(_lib().ttn_ttv_download(h, (vp * len(out))(*[a.ctypes.data for a in out])))
    return out


def _take(h):
    """the cores of a result handle, which is freed"""
    c = _cores(h)
    _check(_lib().ttn_ttv_free(h))
    return c


def _params(**kw):
    from ttn_b200.api import _params as p
    return p(**kw)


def _tdvp_params(steps):
    from ttn_b200._lib import TdvpParams
    p = TdvpParams()
    _check(_lib().ttn_tdvp_params_default(C.byref(p)))
    p.steps = C.cast(steps, C.POINTER(C.c_double))
    p.n_steps = len(steps)
    p.krylovdim = 12
    return p


def _tto(A):
    """a raw operator handle that the caller frees (the uploading wrapper gives up ownership)"""
    import ttn_b200 as t
    w = t.DeviceTTO.upload(A)
    h, w._h = w._h, None
    return h


D = 6


def _solver_cases(A, S):
    """(name, run(up) -> list of arrays): every solver entry point, its trains made by `up(name)`"""
    lib = _lib()

    def lin(fn, **kw):
        def run(up):
            p, keep = _params(**kw)
            out, res = vp(), C.c_double()
            _check(fn(A, up("b"), up("x0"), C.byref(p), C.byref(out), C.byref(res)))
            return _take(out) + [np.array([res.value])]
        return run

    def eig(fn, hist, **kw):
        def run(up):
            p, keep = _params(**kw)
            out, E, rh, nE = vp(), (C.c_double * 64)(), (C.c_int64 * 64)(), C.c_int()
            args = (E, rh, 64, C.byref(nE)) if hist else (E, 64, C.byref(nE))
            _check(fn(A, up("x0"), C.byref(p), C.byref(out), *args))
            return _take(out) + [np.array(E[:nE.value]), np.array(rh[:nE.value])]
        return run

    def gen(up):
        p, keep = _params(sweep_schedule=[2], rmax_schedule=[4])
        out, E, nE = vp(), (C.c_double * 64)(), C.c_int()
        _check(lib.ttn_als_gen_eigsolv(A, S, up("x0"), C.byref(p), C.byref(out), E, 64, C.byref(nE)))
        return _take(out) + [np.array(E[:nE.value])]

    def sharded(up):
        p, keep = _params(N=2, sweep_schedule=[2], rmax_schedule=[4], linsolv_tol=1e-8, symmetrize=1)
        sc = vp()
        _check(lib.ttn_shard_ctx_create(F64, 4096, 0, 1, C.byref(sc)))
        out, E, rh, nE = vp(), (C.c_double * 64)(), (C.c_int64 * 64)(), C.c_int()
        try:
            _check(lib.ttn_dmrg_eigsolve_sharded(A, up("x0"), C.byref(p), sc, C.byref(out), E, rh, 64, C.byref(nE)))
        finally:
            _check(lib.ttn_shard_ctx_free(sc))
        return _take(out) + [np.array(E[:nE.value])]

    def tdvp(up):
        out, steps = vp(), (C.c_double * 2)(0.05, 0.05)
        _check(lib.ttn_tdvp(A, up("x0"), C.byref(_tdvp_params(steps)), C.byref(out)))   # real state, real time: complex promotion
        return _take(out)

    sched = dict(sweep_schedule=[2], rmax_schedule=[4])
    return [
        ("als_linsolve", lin(lib.ttn_als_linsolve, sweep_count=2)),
        ("mals_linsolve", lin(lib.ttn_mals_linsolve, rmax=4)),
        ("dmrg_linsolve", lin(lib.ttn_dmrg_linsolve, N=2, it_solver=1, linsolv_tol=1e-8, **sched)),
        ("als_eigsolve", eig(lib.ttn_als_eigsolve, False, **sched)),
        ("als_gen_eigsolv", gen),
        ("mals_eigsolve", eig(lib.ttn_mals_eigsolve, True, **sched)),
        ("dmrg_eigsolve", eig(lib.ttn_dmrg_eigsolve, True, N=2, linsolv_tol=1e-8, symmetrize=1, **sched)),
        ("dmrg_eigsolve_sharded", sharded),
        ("tdvp", tdvp),
    ]


def _train_cases(A):
    """(name, run(up) -> list of arrays): every other entry point that reads or replaces the cores of a train"""
    lib = _lib()

    def res(fn, *args):
        def run(up):
            out = vp()
            _check(fn(*[up(a) if isinstance(a, str) else a for a in args], C.byref(out)))
            return _take(out)
        return run

    def inplace(fn, *args):
        def run(up):
            h = up("x")
            _check(fn(h, *args))
            return _cores(h)
        return run

    def dot(up):
        out = (C.c_double * 2)()
        _check(lib.ttn_dot(up("x"), up("b"), out))
        return [np.array(out[:])]

    def norm(up):
        out = (C.c_double * 1)()
        _check(lib.ttn_norm(up("x"), out))
        return [np.array(out[:])]

    def bond_truncate(up):
        h, out = up("x"), vp()
        _check(lib.ttn_bond_truncate(h, 3, 2, 0.0, C.byref(out)))
        return _cores(h) + _take(out)

    def download(up):
        return _cores(up("x"))

    def download_async(up):
        h = up("x")
        dst = _nan_cores(h)
        _check(lib.ttn_ttv_download_async(h, (vp * len(dst))(*[a.ctypes.data for a in dst])))
        _check(lib.ttn_copy_synchronize())
        return dst

    return [
        ("dot", dot), ("norm", norm),
        ("add", res(lib.ttn_add, "x", "b")),
        ("scale", res(lib.ttn_scale, "x", 2.5, 0.0)),
        ("orthogonalize", res(lib.ttn_orthogonalize, "x", 3)),
        ("ttv_copy", res(lib.ttn_ttv_copy, "x")),
        ("ttv_complex", res(lib.ttn_ttv_complex, "x")),
        ("apply", res(lib.ttn_apply, A, "x")),
        ("apply_compress", res(lib.ttn_apply_compress, A, "x", 3, 0.0, 1, None, 0)),
        ("compress", inplace(lib.ttn_compress, 3, 0.0, 1, None, 0)),
        ("bond_truncate", bond_truncate),
        ("swap_sites", inplace(lib.ttn_swap_sites, 2, 1, 64, 0.0)),
        ("merge_sites_diag", inplace(lib.ttn_merge_sites_diag, 2)),
        ("split_site", inplace(lib.ttn_split_site, 1, 2, 1, 64, 0.0)),
        ("download", download), ("download_async", download_async),
    ]


def _handles(hosts, asynchronous, made):
    def up(name):
        h = hosts[name].upload(asynchronous)
        made.append(h)
        return h
    return up


def test_async_upload_read_at_once_large():
    """A 272 MB batch of trains read by ttn_dot / ttn_norm right after ttn_ttv_upload_async, before any synchronous upload of the
    same values (only other values of the same shape came first, so the kernels are loaded and the reused blocks hold other
    numbers): the results are those of the synchronously uploaded copy."""
    lib = _lib()
    rng = np.random.default_rng(2024)
    shape = ((2,) * 4, [1, 64, 64, 64, 1], np.float64, 2048)
    dot, nrm = (C.c_double * (2 * shape[3]))(), (C.c_double * shape[3])()
    # other values of the same shape first: the kernels are loaded and the block cache holds blocks of this size
    w = Pinned(*shape, rng).upload(asynchronous=False)
    _check(lib.ttn_dot(w, w, dot))
    _check(lib.ttn_norm(w, nrm))
    _check(lib.ttn_ttv_free(w))
    x = Pinned(*shape, rng)
    assert sum(a.nbytes for a in x.cores) >= 256 << 20
    h = x.upload(asynchronous=True)
    _check(lib.ttn_dot(h, h, dot))
    _check(lib.ttn_norm(h, nrm))
    got = [np.array(dot[:]), np.array(nrm[:])]
    _check(lib.ttn_ttv_free(h))
    h = x.upload(asynchronous=False)
    _check(lib.ttn_dot(h, h, dot))
    _check(lib.ttn_norm(h, nrm))
    ref = [np.array(dot[:]), np.array(nrm[:])]
    _check(lib.ttn_ttv_free(h))
    assert np.array_equal(got[0], ref[0])
    assert np.array_equal(got[1], ref[1])
    assert np.all(ref[1] > 0)


def test_async_upload_every_entry_point():
    """Every entry point that takes a ttn_ttv, given handles straight from ttn_ttv_upload_async (no wait of any kind), returns
    bit for bit what it returns for synchronously uploaded copies of the same trains."""
    rng = np.random.default_rng(7)
    A = o.tto_add(o.laplace_dd(D), o.tto_scale(3.0, o.id_tto(D)))
    Ah, Sh = _tto(A), _tto(o.id_tto(D))
    hosts = {
        "x": Pinned.of(o.rand_tt((2,) * D, 4, rng=rng, normalise=True), rng),
        "b": Pinned.of(o.rand_tt((2,) * D, 2, rng=rng, normalise=True), rng),
        "x0": Pinned.of(o.rand_tt((2,) * D, 4, rng=rng, normalise=True), rng),
    }
    split_hosts = {"x": Pinned.of(o.rand_tt((4,) + (2,) * (D - 1), 4, rng=rng, normalise=True), rng)}
    cases = _train_cases(Ah) + _solver_cases(Ah, Sh)
    assert len(cases) == 25
    for name, run in cases:
        hs = split_hosts if name == "split_site" else hosts
        results = []
        for asynchronous in (True, False):
            made = []
            try:
                results.append(run(_handles(hs, asynchronous, made)))
            finally:
                for h in made:
                    _check(_lib().ttn_ttv_free(h))
        got, ref = results
        assert len(got) == len(ref), name
        for g, r in zip(got, ref):
            assert g.shape == r.shape and np.array_equal(g, r), name
    for h in (Ah, Sh):
        _check(_lib().ttn_tto_free(h))


@pytest.mark.parametrize("op", ["compress", "bond_truncate", "swap_sites", "merge_sites_diag", "split_site"])
def test_inplace_after_download_async_keeps_downloaded_values(op):
    """ttn_ttv_download_async(x), then an in-place entry point on x, then ttn_copy_synchronize: the host arrays hold the cores x had
    before the in-place call, although that call replaced them and handed the old buffers back to the block cache."""
    import torch
    lib = _lib()
    rng = np.random.default_rng(11)
    dims = (4,) * 6
    x = Pinned(dims, [1, 4, 16, 64, 16, 4, 1], np.float64, 1, rng)
    h = x.upload(asynchronous=False)
    try:
        before = _cores(h)
        dst = []
        for a in before:
            buf = torch.empty(a.size, dtype=torch.float64).pin_memory()
            x.keep.append(buf)
            dst.append(buf.numpy().reshape(a.shape, order="F"))
            dst[-1][...] = np.nan
        _check(lib.ttn_ttv_download_async(h, (vp * len(dst))(*[a.ctypes.data for a in dst])))
        if op == "compress":
            _check(lib.ttn_compress(h, 2, 0.0, 1, None, 0))
        elif op == "bond_truncate":
            _check(lib.ttn_bond_truncate(h, 3, 2, 0.0, None))
        elif op == "swap_sites":
            _check(lib.ttn_swap_sites(h, 3, 1, 8, 0.0))
        elif op == "merge_sites_diag":
            _check(lib.ttn_merge_sites_diag(h, 3))
        else:
            _check(lib.ttn_split_site(h, 3, 2, 1, 8, 0.0))
        # fresh allocations on the compute stream that may reuse the released blocks
        fresh = [Pinned(dims, [1, 4, 16, 64, 16, 4, 1], np.float64, 1, rng).upload(asynchronous=False) for _ in range(2)]
        _check(lib.ttn_copy_synchronize())
        for s in fresh:
            _check(lib.ttn_ttv_free(s))
        for a, b in zip(dst, before):
            assert np.array_equal(a, b), op
    finally:
        _check(lib.ttn_ttv_free(h))


def test_unknown_dtype_is_refused_before_any_launch():
    """Every entry point that takes a dtype code refuses an unknown one with TTN_EARG and launches nothing."""
    lib = _lib()
    bad = 7
    host = np.zeros(4096, dtype=np.complex128)   # large enough for any of the tiny shapes below, read as ComplexF64
    hp = host.ctypes.data
    dev = vp()
    _check(lib.ttn_dev_alloc(host.nbytes, C.byref(dev)))
    i64 = lambda v: (C.c_int64 * len(v))(*v)  # noqa: E731
    dims, rks, cores = i64([2, 2]), i64([1, 2, 1]), (vp * 2)(hp, hp)
    lam, flags, r = (C.c_double * 16)(), (C.c_int * 4)(), C.c_int()
    out = vp()
    calls = {
        "ttv_upload": lambda: lib.ttn_ttv_upload(bad, 2, dims, rks, None, cores, 1, C.byref(out)),
        "ttv_upload_async": lambda: lib.ttn_ttv_upload_async(bad, 2, dims, rks, None, cores, 1, C.byref(out)),
        "tto_upload": lambda: lib.ttn_tto_upload(bad, 2, dims, rks, cores, C.byref(out)),
        "gemm": lambda: lib.ttn_gemm(bad, 2, 2, 2, dev, 1, 2, 0, dev, 1, 2, 0, dev, 1, 2, 1.0, 0.0, 1, 0, 0, 0),
        "matvec2_host": lambda: lib.ttn_matvec2_host(bad, 1, 1, 2, 2, 2, hp, hp, hp, hp, hp, 0),
        "matvec2_create": lambda: lib.ttn_matvec2_create(bad, 1, 1, 2, 2, 2, hp, hp, hp, C.byref(out)),
        "shard_matvec_create": lambda: lib.ttn_shard_matvec_create(bad, 1, 1, 2, 2, 2, hp, hp, hp, 0, 1, C.byref(out)),
        "shard_ctx_create": lambda: lib.ttn_shard_ctx_create(bad, 64, 0, 1, C.byref(out)),
        "env_left_host": lambda: lib.ttn_env_left_host(bad, 2, 1, 1, 2, 2, hp, hp, hp, hp),
        "env_right_host": lambda: lib.ttn_env_right_host(bad, 2, 1, 1, 2, 2, hp, hp, hp, hp),
        "svdtrunc_host": lambda: lib.ttn_svdtrunc_host(bad, 4, 4, hp, 4, 0.0, hp, lam, hp, C.byref(r)),
        "heig_host": lambda: lib.ttn_heig_host(bad, 4, 2, 1, hp, lam, hp, flags),
        "qr_host": lambda: lib.ttn_qr_host(bad, 4, 4, hp, hp, hp),
    }
    try:
        _check(lib.ttn_synchronize())
        for name, call in calls.items():
            n0 = lib.ttn_launch_count()
            assert call() == EARG, name
            assert lib.ttn_launch_count() == n0, name
    finally:
        _check(lib.ttn_dev_free(dev))


@pytest.mark.parametrize("zero", ["dim", "rank"])
def test_tto_upload_rejects_empty_cores(zero):
    lib = _lib()
    host = np.zeros(64)
    cores = (vp * 2)(host.ctypes.data, host.ctypes.data)
    dims = (C.c_int64 * 2)(*([0, 2] if zero == "dim" else [2, 2]))
    rks = (C.c_int64 * 3)(*([1, 2, 1] if zero == "dim" else [1, 0, 1]))
    out = vp()
    assert lib.ttn_tto_upload(F64, 2, dims, rks, cores, C.byref(out)) == EDIM


@pytest.mark.parametrize("side", ["left", "right"])
def test_tdvp_rejects_an_operator_with_boundary_rank_above_one(side):
    """The boundary environments of a sweep are 1 x 1 x 1: ttn_tdvp refuses an operator whose first or last rank is 2 with
    TTN_EDIM, like the other solvers, instead of reading that environment as 1 x 2 x 1."""
    lib = _lib()
    rng = np.random.default_rng(13)
    dims, rks = [2, 2, 2], ([2, 2, 2, 1] if side == "left" else [1, 2, 2, 2])
    host = [rng.standard_normal(n * n * rks[k] * rks[k + 1]) for k, n in enumerate(dims)]
    i64 = lambda v: (C.c_int64 * len(v))(*v)  # noqa: E731
    H = vp()
    _check(lib.ttn_tto_upload(F64, 3, i64(dims), i64(rks), (vp * 3)(*[a.ctypes.data for a in host]), C.byref(H)))
    x = Pinned((2,) * 3, [1, 2, 2, 1], np.float64, 1, rng).upload(asynchronous=False)
    steps = (C.c_double * 1)(0.05)
    p = _tdvp_params(steps)
    p.imaginary_time = 1
    out = vp()
    try:
        assert lib.ttn_tdvp(H, x, C.byref(p), C.byref(out)) == EDIM
        assert not out.value
    finally:
        _check(lib.ttn_ttv_free(x))
        _check(lib.ttn_tto_free(H))


def test_sharded_dmrg_rejects_a_context_of_another_dtype():
    """A Float64 shard context with a ComplexF64 train and operator is TTN_EDIM, not a silent unsharded run."""
    lib = _lib()
    rng = np.random.default_rng(3)
    Ar = _tto(o.tto_add(o.laplace_dd(4), o.tto_scale(3.0, o.id_tto(4))))
    Ah = vp()
    _check(lib.ttn_tto_complex(Ar, C.byref(Ah)))
    x = Pinned((2,) * 4, [1, 2, 4, 2, 1], np.complex128, 1, rng).upload(asynchronous=False)
    sc = vp()
    _check(lib.ttn_shard_ctx_create(F64, 4096, 0, 1, C.byref(sc)))
    try:
        p, keep = _params(N=2, sweep_schedule=[2], rmax_schedule=[4])
        out, E, rh, nE = vp(), (C.c_double * 64)(), (C.c_int64 * 64)(), C.c_int()
        assert lib.ttn_dmrg_eigsolve_sharded(Ah, x, C.byref(p), sc, C.byref(out), E, rh, 64, C.byref(nE)) == EDIM
        assert not out.value
    finally:
        _check(lib.ttn_shard_ctx_free(sc))
        _check(lib.ttn_ttv_free(x))
        _check(lib.ttn_tto_free(Ah))
        _check(lib.ttn_tto_free(Ar))


def test_null_output_pointers_are_refused():
    lib = _lib()
    rng = np.random.default_rng(5)
    x = Pinned((2,) * 3, [1, 2, 2, 1], np.float64, 1, rng).upload(asynchronous=False)
    try:
        for fn in (lib.ttn_ttv_ranks, lib.ttn_ttv_dims, lib.ttn_ttv_ot, lib.ttn_ttv_download):
            assert fn(x, None) == EARG, fn.__name__
        assert lib.ttn_profile_read(None, None) == EARG
    finally:
        _check(lib.ttn_ttv_free(x))
