"""Host-side mirror of the reference's operator API for the hot path (same names, argument meaning and
error behaviour as TensorTrainNumerics.jl; Julia's `f!` is spelled `f_`).

Every function here is a thin marshalling layer over the C ABI (include/ttn_b200.h): host TT cores are
uploaded, the whole operation (a full sweep, a full solver run) executes on the GPU inside libttn_b200.so,
and the result is downloaded.  `DeviceTT` / `DeviceTTO` keep trains resident in HBM between calls.
Nothing in this module computes on the CPU and nothing imports the oracle.

Reference API mirrored (file:line under the reference repo):
  TTvector / TToperator            src/tt_tools.jl:23-29, 48-54
  A * x  (apply)                   src/tt_operations.jl:101-111
  dot, norm, +, scalar *           src/tt_operations.jl:239-250, 465-470, 10-35, 256-266
  orthogonalize(x; i)              src/tt_tools.jl:511-543
  tt_compress!(x, max_bond; ...)   src/tt_tools.jl:772-789   (+ _tt_bond_truncate! :743-770)
  als_linsolve / als_eigsolve      src/solvers/als.jl:161-225, 251-321
  mals_linsolve / mals_eigsolve    src/solvers/mals.jl:240-309, 335-425
  dmrg_linsolve / dmrg_eigsolve    src/solvers/dmrg.jl:385-473, 501-578
  tdvp / tdvp2                     src/solvers/tdvp.jl:154-203, 303-357
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np

from . import _lib
from ._lib import TTN_F64, TTN_C128, SolverParams, TdvpParams, check

__all__ = [
    "TTvector", "TToperator", "DeviceTT", "DeviceTTO", "apply", "dot", "norm", "add", "add_", "scale", "sub", "euclidean_distance",
    "euclidean_distance_normalized",
    "orthogonalize", "tt_compress_", "tt_bond_truncate_", "als_linsolve", "als_eigsolve", "als_gen_eigsolv", "mals_linsolve",
    "mals_eigsolve", "dmrg_linsolve", "dmrg_eigsolve", "tdvp", "tdvp2", "matvec2", "env_left", "env_right",
    "shard_range", "shard_batch", "assemble_slices", "ShardedMatvec", "ShardContext", "apply_compress", "increase_ranks", "rand_orthogonal", "r_and_d_to_rks", "svdtrunc", "heig_top", "set_option", "get_option", "copy_synchronize", "qr_thin", "gemm_host", "launch_count", "reset_launch_count", "synchronize", "library_path", "profile", "profile_read", "stream_handle",
    "KERNEL_FAMILIES",
]


def library_path():
    return _lib.LIB_PATH


def launch_count() -> int:
    return int(_lib.lib().ttn_launch_count())


def reset_launch_count():
    _lib.lib().ttn_reset_launch_count()


def synchronize():
    check(_lib.lib().ttn_synchronize())


KERNEL_FAMILIES = ("gemm", "copy", "apply", "qr_panel", "qr_apply", "jacobi", "reduce", "gather")


def profile(enable: bool):
    """switch the per-kernel-family CUDA-event timing on/off (clears previous records)"""
    check(_lib.lib().ttn_profile(int(bool(enable))))


def profile_read():
    """{family: (total_ms, launches)} accumulated since profile(True)"""
    ms, cnt = (C.c_double * 8)(), (C.c_longlong * 8)()
    check(_lib.lib().ttn_profile_read(ms, cnt))
    return {KERNEL_FAMILIES[i]: (float(ms[i]), int(cnt[i])) for i in range(8)}


def copy_synchronize() -> None:
    """waits for the asynchronous host <-> device copies (`upload_batched(..., asynchronous=True)`, `download_into(..., asynchronous=True)`)"""
    check(_lib.lib().ttn_copy_synchronize())


def set_option(key: str, value) -> None:
    """run-time switch of the library (`ttn_set_option`): gram_compress, gram_jacobi_min, gemm_bulk, gemm_thin, reset_flops"""
    check(_lib.lib().ttn_set_option(key.encode(), float(value)))


def get_option(key: str) -> float:
    v = C.c_double()
    check(_lib.lib().ttn_get_option(key.encode(), C.byref(v)))
    return float(v.value)


def stream_handle() -> int:
    """cudaStream_t the library launches on (for torch.cuda.ExternalStream / event timing)"""
    return int(_lib.lib().ttn_stream() or 0)


# ------------------------------------------------------------------------------------------------------
# host containers (same field names as the reference structs)
# ------------------------------------------------------------------------------------------------------
class TTvector:
    """src/tt_tools.jl:23-29.  ttv_vec[k] is an (n_k, r_{k-1}, r_k) array."""

    def __init__(self, N, ttv_vec, ttv_dims, ttv_rks, ttv_ot=None):
        self.N = int(N)
        self.ttv_vec = list(ttv_vec)
        self.ttv_dims = tuple(int(n) for n in ttv_dims)
        self.ttv_rks = [int(r) for r in ttv_rks]
        self.ttv_ot = [0] * self.N if ttv_ot is None else [int(o) for o in ttv_ot]

    @property
    def dtype(self):
        return self.ttv_vec[0].dtype


class TToperator:
    """src/tt_tools.jl:48-54.  tto_vec[k] is an (n_k, n_k, R_{k-1}, R_k) array."""

    def __init__(self, N, tto_vec, tto_dims, tto_rks, tto_ot=None):
        self.N = int(N)
        self.tto_vec = list(tto_vec)
        self.tto_dims = tuple(int(n) for n in tto_dims)
        self.tto_rks = [int(r) for r in tto_rks]
        self.tto_ot = [0] * self.N if tto_ot is None else [int(o) for o in tto_ot]

    @property
    def dtype(self):
        return self.tto_vec[0].dtype


def _dtype_code(dt):
    dt = np.dtype(dt)
    if dt == np.float64:
        return TTN_F64
    if dt == np.complex128:
        return TTN_C128
    raise TypeError(f"only Float64 / ComplexF64 are supported on the device path, got {dt}")


def _np_dtype(code):
    return np.float64 if code == TTN_F64 else np.complex128


def _i64(seq):
    return (C.c_int64 * len(seq))(*[int(v) for v in seq])


# ------------------------------------------------------------------------------------------------------
# device-resident handles
# ------------------------------------------------------------------------------------------------------
class DeviceTT:
    """A TTvector (or a batch of identically-shaped TTvectors) resident in HBM behind a `ttn_ttv` handle."""

    def __init__(self, handle):
        self._h = C.c_void_p(handle) if not isinstance(handle, C.c_void_p) else handle

    @classmethod
    def upload(cls, x):
        """`x` is a TTvector-like object (fields N, ttv_vec, ttv_dims, ttv_rks, ttv_ot) or a list of them with
        identical dims/ranks (uploaded as one batch)."""
        lib = _lib.lib()
        xs = list(x) if isinstance(x, (list, tuple)) else [x]
        x0 = xs[0]
        d = x0.N
        dt = np.result_type(*[c.dtype for t in xs for c in t.ttv_vec])
        code = _dtype_code(dt)
        for t in xs[1:]:
            if tuple(t.ttv_dims) != tuple(x0.ttv_dims) or list(t.ttv_rks) != list(x0.ttv_rks):
                raise AssertionError("Incompatible dimensions")
        keep, ptrs = [], (C.c_void_p * d)()
        for k in range(d):
            shp = (x0.ttv_dims[k], x0.ttv_rks[k], x0.ttv_rks[k + 1])
            if len(xs) == 1:
                a = np.asfortranarray(x0.ttv_vec[k], dtype=dt)
                if a.shape != shp:
                    raise AssertionError("Incompatible dimensions")
            else:
                a = np.empty(shp + (len(xs),), dtype=dt, order="F")
                for b, t in enumerate(xs):
                    a[..., b] = t.ttv_vec[k]
            keep.append(a)
            ptrs[k] = a.ctypes.data
        out = C.c_void_p()
        check(lib.ttn_ttv_upload(code, d, _i64(x0.ttv_dims), _i64(x0.ttv_rks), _i64(x0.ttv_ot), ptrs, len(xs),
                                 C.byref(out)))
        return cls(out)

    @classmethod
    def upload_batched(cls, cores, dims, rks, ot=None, asynchronous=False):
        """A batch of identically shaped trains given as ONE array per site, `cores[k]` of shape (n_k, r_k, r_{k+1}, batch),
        Fortran-contiguous (e.g. views of pinned host memory): no host-side repacking, one H2D copy per site.
        `asynchronous=True` (pinned memory only): the copies run on the library's copy stream and overlap the compute stream."""
        d = len(cores)
        dt = np.result_type(*[c.dtype for c in cores])
        code = _dtype_code(dt)
        batch = cores[0].shape[3]
        ptrs = (C.c_void_p * d)()
        for k, c in enumerate(cores):
            if c.shape != (dims[k], rks[k], rks[k + 1], batch) or not c.flags["F_CONTIGUOUS"] or c.dtype != dt:
                raise AssertionError("Incompatible dimensions")
            ptrs[k] = c.ctypes.data
        out = C.c_void_p()
        fn = _lib.lib().ttn_ttv_upload_async if asynchronous else _lib.lib().ttn_ttv_upload
        check(fn(code, d, _i64(dims), _i64(rks), _i64(ot if ot is not None else [0] * d), ptrs, batch, C.byref(out)))
        return cls(out)

    def download_into(self, arrays, asynchronous=False):
        """device -> host into caller-provided Fortran-contiguous arrays (one per site, with the trailing batch axis when
        batch > 1); the counterpart of `upload_batched` for pinned result buffers.  `asynchronous=True`: the copies run on the
        copy stream, the arrays are valid after `copy_synchronize()`."""
        code, d, batch = self._info()
        dims, rks = self.ttv_dims, self.ttv_rks
        ptrs = (C.c_void_p * d)()
        for k in range(d):
            shp = (dims[k], rks[k], rks[k + 1]) + ((batch,) if batch > 1 else ())
            a = arrays[k]
            if tuple(a.shape) != shp or not a.flags["F_CONTIGUOUS"] or a.dtype != _np_dtype(code):
                raise AssertionError("Incompatible dimensions")
            ptrs[k] = a.ctypes.data
        check((_lib.lib().ttn_ttv_download_async if asynchronous else _lib.lib().ttn_ttv_download)(self._h, ptrs))
        return arrays

    # -- metadata ---------------------------------------------------------------------------------------
    def _info(self):
        dt, d, b = C.c_int(), C.c_int(), C.c_int()
        check(_lib.lib().ttn_ttv_info(self._h, C.byref(dt), C.byref(d), C.byref(b)))
        return dt.value, d.value, b.value

    @property
    def N(self):
        return self._info()[1]

    @property
    def batch(self):
        return self._info()[2]

    @property
    def dtype(self):
        return np.dtype(_np_dtype(self._info()[0]))

    def _vec(self, fn, n):
        buf = (C.c_int64 * n)()
        check(fn(self._h, buf))
        return [int(v) for v in buf]

    @property
    def ttv_rks(self):
        return self._vec(_lib.lib().ttn_ttv_ranks, self.N + 1)

    @property
    def ttv_dims(self):
        return tuple(self._vec(_lib.lib().ttn_ttv_dims, self.N))

    @property
    def ttv_ot(self):
        return self._vec(_lib.lib().ttn_ttv_ot, self.N)

    # -- data -------------------------------------------------------------------------------------------
    def download(self):
        """Returns a TTvector (batch == 1) or a list of TTvectors."""
        code, d, batch = self._info()
        dims, rks, ot = self.ttv_dims, self.ttv_rks, self.ttv_ot
        arrs, ptrs = [], (C.c_void_p * d)()
        for k in range(d):
            shp = (dims[k], rks[k], rks[k + 1]) + ((batch,) if batch > 1 else ())
            a = np.empty(shp, dtype=_np_dtype(code), order="F")
            arrs.append(a)
            ptrs[k] = a.ctypes.data
        check(_lib.lib().ttn_ttv_download(self._h, ptrs))
        if batch == 1:
            return TTvector(d, arrs, dims, rks, ot)
        return [TTvector(d, [np.asfortranarray(a[..., b]) for a in arrs], dims, rks, ot) for b in range(batch)]

    def copy(self):
        out = C.c_void_p()
        check(_lib.lib().ttn_ttv_copy(self._h, C.byref(out)))
        return DeviceTT(out)

    def complex(self):
        out = C.c_void_p()
        check(_lib.lib().ttn_ttv_complex(self._h, C.byref(out)))
        return DeviceTT(out)

    def free(self):
        if self._h is not None and self._h.value:
            _lib.load().ttn_ttv_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class DeviceTTO:
    """A TToperator resident in HBM behind a `ttn_tto` handle."""

    def __init__(self, handle, dtype_code, N):
        self._h = handle
        self._code = dtype_code
        self.N = N

    @classmethod
    def upload(cls, A):
        lib = _lib.lib()
        d = A.N
        dt = np.result_type(*[c.dtype for c in A.tto_vec])
        code = _dtype_code(dt)
        keep, ptrs = [], (C.c_void_p * d)()
        for k in range(d):
            a = np.asfortranarray(A.tto_vec[k], dtype=dt)
            if a.shape != (A.tto_dims[k], A.tto_dims[k], A.tto_rks[k], A.tto_rks[k + 1]):
                raise AssertionError("Incompatible dimensions")
            keep.append(a)
            ptrs[k] = a.ctypes.data
        out = C.c_void_p()
        check(lib.ttn_tto_upload(code, d, _i64(A.tto_dims), _i64(A.tto_rks), ptrs, C.byref(out)))
        return cls(out, code, d)

    @property
    def dtype(self):
        return np.dtype(_np_dtype(self._code))

    def complex(self):
        out = C.c_void_p()
        check(_lib.lib().ttn_tto_complex(self._h, C.byref(out)))
        return DeviceTTO(out, TTN_C128, self.N)

    @property
    def tto_rks(self):
        buf = (C.c_int64 * (self.N + 1))()
        check(_lib.lib().ttn_tto_ranks(self._h, buf))
        return [int(v) for v in buf]

    @property
    def tto_dims(self):
        buf = (C.c_int64 * self.N)()
        check(_lib.lib().ttn_tto_dims(self._h, buf))
        return tuple(int(v) for v in buf)

    def download(self):
        """device -> host TToperator (cores (n_k, n_k, R_{k-1}, R_k), Fortran order, as src/tt_tools.jl:48-54 stores them)"""
        dims, rks = self.tto_dims, self.tto_rks
        cores = [np.zeros((dims[k], dims[k], rks[k], rks[k + 1]), dtype=self.dtype, order="F") for k in range(self.N)]
        ptrs = (C.c_void_p * self.N)(*[c.ctypes.data for c in cores])
        check(_lib.lib().ttn_tto_download(self._h, ptrs))
        return TToperator(self.N, cores, dims, rks)

    def free(self):
        if self._h is not None and self._h.value:
            _lib.load().ttn_tto_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def _dev(x):
    """(DeviceTT, was_host)"""
    if isinstance(x, DeviceTT):
        return x, False
    return DeviceTT.upload(x), True


def _devo(A, want_dtype=None):
    if isinstance(A, DeviceTTO):
        d = A
    else:
        d = DeviceTTO.upload(A)
    if want_dtype is not None and np.dtype(want_dtype) == np.complex128 and d.dtype != np.complex128:
        d = d.complex()
    return d


def _match(*devs):
    """promote a set of DeviceTT to a common element type (Julia would promote_type)."""
    if any(v.dtype == np.complex128 for v in devs):
        return [v if v.dtype == np.complex128 else v.complex() for v in devs]
    return list(devs)


def _ret(dev, host):
    return dev.download() if host else dev


# ------------------------------------------------------------------------------------------------------
# TT algebra
# ------------------------------------------------------------------------------------------------------
def apply(A, x):
    """`A * x`, src/tt_operations.jl:101-111."""
    xd, host = _dev(x)
    Ad = _devo(A, xd.dtype)
    if Ad.dtype == np.complex128 and xd.dtype != np.complex128:
        xd = xd.complex()
    out = C.c_void_p()
    check(_lib.lib().ttn_apply(Ad._h, xd._h, C.byref(out)))
    return _ret(DeviceTT(out), host)


def dot(a, b):
    """src/tt_operations.jl:239-250 (conjugates the first argument)."""
    ad, _ = _dev(a)
    bd, _ = _dev(b)
    ad, bd = _match(ad, bd)
    batch = ad.batch
    buf = (C.c_double * (2 * batch))()
    check(_lib.lib().ttn_dot(ad._h, bd._h, buf))
    vals = np.array(buf[:]).reshape(batch, 2)
    res = vals[:, 0] + 1j * vals[:, 1] if ad.dtype == np.complex128 else vals[:, 0].copy()
    return res[0] if batch == 1 else res


def norm(a):
    """src/tt_operations.jl:465-470."""
    ad, _ = _dev(a)
    batch = ad.batch
    buf = (C.c_double * batch)()
    check(_lib.lib().ttn_norm(ad._h, buf))
    return float(buf[0]) if batch == 1 else np.array(buf[:])


def add(x, y):
    """`x + y`, src/tt_operations.jl:10-35."""
    xd, host = _dev(x)
    yd, _ = _dev(y)
    xd, yd = _match(xd, yd)
    out = C.c_void_p()
    check(_lib.lib().ttn_add(xd._h, yd._h, C.byref(out)))
    return _ret(DeviceTT(out), host)


def scale(a, x):
    """`a * x`, src/tt_operations.jl:256-266."""
    xd, host = _dev(x)
    a = complex(a)
    if a.imag != 0.0 and xd.dtype != np.complex128:
        xd = xd.complex()
    out = C.c_void_p()
    check(_lib.lib().ttn_scale(xd._h, a.real, a.imag, C.byref(out)))
    return _ret(DeviceTT(out), host)


def sub(x, y):
    """`x - y` = (-1.0 * y) + x, src/tt_operations.jl:280-282."""
    xd, host = _dev(x)
    yd, _ = _dev(y)
    return _ret(add(scale(-1.0, yd), xd), host)


def add_(x, y):
    """`add!(x, y)`, src/tt_operations.jl:36-66: x <- x + y in place (host TTvector fields overwritten, `ttv_ot` zeroed);
    a DeviceTT cannot change identity, so the sum is returned for it."""
    z = add(x, y)
    if isinstance(x, DeviceTT):
        return z
    x.ttv_vec, x.ttv_rks, x.ttv_ot = z.ttv_vec, z.ttv_rks, [0] * x.N
    return x


def euclidean_distance(a, b):
    """src/tt_operations.jl:452-455: sqrt(max(<a,a> - 2 Re<b,a> + <b,b>, 0)) from three transfer-matrix chains."""
    ad, _ = _dev(a)
    bd, _ = _dev(b)
    assert tuple(ad.ttv_dims) == tuple(bd.ttv_dims), "TT dimensions must match"
    return math.sqrt(max(float(np.real(dot(ad, ad) - 2.0 * np.real(dot(bd, ad)) + dot(bd, bd))), 0.0))


def euclidean_distance_normalized(a, b):
    """src/tt_operations.jl:457-460: sqrt(1 + <a,a>/<b,b> - 2 Re<b,a>/<b,b>)."""
    ad, _ = _dev(a)
    bd, _ = _dev(b)
    assert tuple(ad.ttv_dims) == tuple(bd.ttv_dims), "TT dimensions must match"
    bb = dot(bd, bd)
    v = 1.0 + dot(ad, ad) / bb - 2.0 * np.real(dot(bd, ad)) / bb
    return float(np.sqrt(np.real(v))) if np.real(v) >= 0 else float("nan")


# ------------------------------------------------------------------------------------------------------
# canonicalisation / rounding
# ------------------------------------------------------------------------------------------------------
def orthogonalize(x, i: int = 1):
    """src/tt_tools.jl:511-543 (pure; centre `i` is 1-based)."""
    xd, host = _dev(x)
    out = C.c_void_p()
    check(_lib.lib().ttn_orthogonalize(xd._h, int(i), C.byref(out)))
    return _ret(DeviceTT(out), host)


def apply_compress(A, x, max_bond: int, truncerr: float = 0.0, sweeps: int = 1, return_sigma: bool = False):
    """`tt_compress!(A * x, max_bond; truncerr, sweeps)` as ONE call (`ttn_apply_compress`): src/tt_operations.jl:101-111 fused
    into the first pass of src/tt_tools.jl:772-789 — for truncerr == 0 the product cores never reach HBM.  Same result as
    `tt_compress_(apply(A, x), max_bond, ...)`."""
    lib = _lib.lib()
    xd, host = _dev(x)
    Ad = _devo(A, xd.dtype)
    if Ad.dtype == np.complex128 and xd.dtype != np.complex128:
        xd = xd.complex()
    sig, stride, nsteps = None, 0, 0
    if return_sigma:
        stride = int(min(int(max_bond), 4096))      # retained singular values per bond step never exceed max_bond
        nsteps = 2 * (xd.N - 1) * max(int(sweeps), 0)
        sig = (C.c_double * max(1, stride * nsteps))()
    out = C.c_void_p()
    check(lib.ttn_apply_compress(Ad._h, xd._h, int(max_bond), float(truncerr), int(sweeps), sig, int(stride), C.byref(out)))
    yd = DeviceTT(out)
    res = yd.download() if host else yd
    if return_sigma:
        s = np.array(sig[:]).reshape(nsteps, stride) if nsteps else np.zeros((0, stride))
        return res, [row[row > 0] for row in s]
    return res


def tt_compress_(x, max_bond: int, truncerr: float = 0.0, sweeps: int = 1, verbose: bool = False, return_sigma: bool = False):
    """`tt_compress!(ψ, max_bond; truncerr, sweeps, verbose)`, src/tt_tools.jl:772-789: mutates and returns `x`.
    With `return_sigma=True` also returns the retained singular values of every bond step."""
    lib = _lib.lib()
    xd, host = _dev(x)
    sig, stride, nsteps = None, 0, 0
    if return_sigma:
        rks = xd.ttv_rks
        dims = xd.ttv_dims
        stride = int(max(min(dims[k] * rks[k], dims[k + 1] * rks[k + 2]) for k in range(xd.N - 1))) if xd.N > 1 else 1
        nsteps = 2 * (xd.N - 1) * max(int(sweeps), 0)
        sig = (C.c_double * max(1, stride * nsteps))()
    check(lib.ttn_compress(xd._h, int(max_bond), float(truncerr), int(sweeps), sig, int(stride)))
    if host:
        y = xd.download()
        # the same object and the same `ttv_vec` / `ttv_rks` lists are mutated (tt_tools.jl:754-767 writes element-wise, which
        # is what lets the QTTvector wrapper of qtt_tools.jl:783-786 share them); `ttv_ot` untouched (test_tt_tools.jl:514)
        if isinstance(x.ttv_vec, list) and isinstance(x.ttv_rks, list):
            x.ttv_vec[:] = y.ttv_vec
            x.ttv_rks[:] = y.ttv_rks
        else:
            x.ttv_vec, x.ttv_rks = y.ttv_vec, y.ttv_rks
        res = x
    else:
        res = xd
    if return_sigma:
        s = np.array(sig[:]).reshape(nsteps, stride) if nsteps else np.zeros((0, stride))
        return res, [row[row > 0] for row in s]
    return res


def tt_bond_truncate_(x, k: int, max_bond: int | None = None, truncerr: float = 0.0):
    """`_tt_bond_truncate!(ψ, k; max_bond, truncerr)`, src/tt_tools.jl:743-770: mutates `x` and returns
    `orthogonalize(ψ; i=k)` as the reference does."""
    xd, host = _dev(x)
    out = C.c_void_p()
    mb = (1 << 62) if max_bond is None else int(max_bond)
    check(_lib.lib().ttn_bond_truncate(xd._h, int(k), mb, float(truncerr), C.byref(out)))
    y = DeviceTT(out)
    if host:
        z = xd.download()
        x.ttv_vec, x.ttv_rks = z.ttv_vec, z.ttv_rks
        return y.download()
    return y


# ------------------------------------------------------------------------------------------------------
# solvers
# ------------------------------------------------------------------------------------------------------
def _params(**kw):
    p = SolverParams()
    check(_lib.lib().ttn_solver_params_default(C.byref(p)))
    keep = []
    for name in ("sweep_schedule", "rmax_schedule"):
        v = kw.pop(name, None)
        if v is not None:
            arr = _i64(list(v))
            keep.append(arr)
            setattr(p, name, C.cast(arr, C.POINTER(C.c_int64)))
            setattr(p, "n_" + name, len(v))
    for k, v in kw.items():
        if v is not None:
            setattr(p, k, v)
    return p, keep


def _isqrt_prod(dims):
    pr = 1
    for n in dims:
        pr *= int(n)
    return math.isqrt(pr)


def _solve_lin(fn, A, b, x0, p):
    xd, host = _dev(x0)
    bd, _ = _dev(b)
    xd, bd = _match(xd, bd)
    Ad = _devo(A, xd.dtype)
    if Ad.dtype == np.complex128 and xd.dtype != np.complex128:
        xd, bd = xd.complex(), bd.complex()
    out, res = C.c_void_p(), C.c_double()
    check(fn(Ad._h, bd._h, xd._h, C.byref(p), C.byref(out), C.byref(res)))
    return DeviceTT(out), host, res.value


def als_linsolve(A, b, tt_start, sweep_count=2, it_solver=False, r_itsolver=5000, return_info=False,
                 linsolv_maxiter=200, krylovdim=30):
    """src/solvers/als.jl:161-225 (`sweep_count` counts half sweeps, als.jl:198-222)."""
    p, keep = _params(sweep_count=int(sweep_count), linsolv_maxiter=int(linsolv_maxiter), krylovdim=int(krylovdim),
                      it_solver=int(bool(it_solver)))
    x, host, res = _solve_lin(_lib.lib().ttn_als_linsolve, A, b, tt_start, p)
    x = _ret(x, host)
    return (x, {"residual": res}) if return_info else x


def r_and_d_to_rks(rks, dims, rmax=1024):
    """src/tt_tools.jl:407-425 (library host code, `ttn_r_and_d_to_rks`)."""
    d = len(dims)
    out = (C.c_int64 * (d + 1))()
    check(_lib.load().ttn_r_and_d_to_rks(_i64(rks), _i64(dims), d, int(rmax), out))
    return [int(v) for v in out]


def rand_orthogonal(n, m, rng=None, dtype=np.float64):
    """src/tt_tools.jl:80-84: the leading n x m block of the Q factor of a uniform random square matrix (NumPy RNG, so the
    stream differs from Julia's; the distribution is the same)."""
    rng = np.random.default_rng() if rng is None else rng
    N = max(n, m)
    a = rng.random((N, N))
    if np.dtype(dtype) == np.complex128:
        a = a + 1j * rng.random((N, N))
    q, _ = np.linalg.qr(a)
    return q[:n, :m]


def increase_ranks(x, max_bond, rks=None, noise=0.0, rng=None):
    """src/tt_tools.jl:443-489: pad every core to the ranks `r_and_d_to_rks(rks, dims; rmax = max_bond)`; with `noise != 0` the new
    block of a core whose left / right / both ranks grew is `noise` x a slice of a random orthogonal matrix (the three branches of
    `increase_ranks_noise`, tt_tools.jl:443-460).  Host function on TTvector (a DeviceTT is downloaded first)."""
    x = x.download() if isinstance(x, DeviceTT) else x
    d = x.N
    if not max_bond > max(x.ttv_rks):
        raise AssertionError("New bond dimension too low")
    if rks is None:
        rks = [1] + [int(max_bond)] * (d - 1) + [1]
    rks = r_and_d_to_rks(rks, x.ttv_dims, rmax=max_bond)
    T = np.result_type(*[c.dtype for c in x.ttv_vec])
    out, ot = [], [0] * d
    for i in range(d):
        c = x.ttv_vec[i]
        n, a, b = c.shape
        rkm, rk = rks[i], rks[i + 1]
        v = np.zeros((n, rkm, rk), dtype=T, order="F")
        v[:, :a, :b] = c
        if noise != 0.0:
            if rkm == a and rk > b:
                Q = rand_orthogonal(n * rkm, rk - b, rng, T)
                v[:, :, b:] = noise * Q.reshape((n, rkm, rk - b), order="F")
            elif rk == b and rkm > a:
                Q = rand_orthogonal(rkm - a, n * rk, rng, T)
                v[:, a:, :] = noise * Q.reshape((n, rkm - a, rk), order="F")
            elif rk > b and rkm > a:
                Q = rand_orthogonal((rkm - a) * n, rk - b, rng, T)
                v[:, a:, b:] = noise * Q.reshape((n, rkm - a, rk - b), order="F")
        out.append(v)
    return TTvector(d, out, x.ttv_dims, rks, ot)


def als_eigsolve(A, tt_start, sweep_schedule=(2,), rmax_schedule=None, noise_schedule=None, it_solver=False,
                 itslv_thresh=1024, maxiter=200, linsolv_tol=1e-8, krylovdim=30, rng=None):
    """src/solvers/als.jl:251-321 → (E, tt_opt).  With a non-zero `noise_schedule` the rank increases between the stages of the
    schedule (als.jl:289-291) are done on the host by `increase_ranks(...; noise)` with the NumPy generator `rng` — the one step of
    the solver that draws random numbers — and every stage's sweeps run on the device."""
    if noise_schedule is not None and any(float(v) != 0.0 for v in noise_schedule):
        sched = [int(v) for v in sweep_schedule]
        if rmax_schedule is None or not (len(rmax_schedule) == len(sched) == len(noise_schedule)):
            raise AssertionError("Sweep schedule error")
        kw = dict(it_solver=it_solver, itslv_thresh=itslv_thresh, maxiter=maxiter, linsolv_tol=linsolv_tol, krylovdim=krylovdim)
        host = not isinstance(tt_start, DeviceTT)
        x, Es = tt_start, []
        for j, ns in enumerate(sched):
            if j > 0:       # als.jl:289-291: increase_ranks + orthogonalize + init_H (the last two open every device call)
                x = increase_ranks(x, int(rmax_schedule[j]), noise=float(noise_schedule[j]), rng=rng)
            # stage j runs the sweeps sched[j-1] .. sched[j] - 1 of the reference's counter (the first stage starts at 1)
            nsw = ns - (sched[j - 1] if j > 0 else 1)
            if nsw > 0:
                E, x = als_eigsolve(A, x, sweep_schedule=(nsw + 1,), rmax_schedule=(max(x.ttv_rks),), **kw)
                Es.append(E)
        if host and isinstance(x, DeviceTT):
            x = x.download()
        return (np.concatenate(Es) if Es else np.zeros(0)), x
    xd, host = _dev(tt_start)
    if rmax_schedule is None:
        rmax_schedule = [max(xd.ttv_rks)]
    if len(rmax_schedule) != len(sweep_schedule):
        raise AssertionError("Sweep schedule error")
    Ad = _devo(A, xd.dtype)
    if Ad.dtype == np.complex128 and xd.dtype != np.complex128:
        xd = xd.complex()
    p, keep = _params(sweep_schedule=sweep_schedule, rmax_schedule=rmax_schedule, linsolv_maxiter=int(maxiter),
                      linsolv_tol=float(linsolv_tol), krylovdim=int(krylovdim))
    cap = 2 * xd.N * (int(sweep_schedule[-1]) + 1) + 8
    E, nE, out = (C.c_double * cap)(), C.c_int(), C.c_void_p()
    check(_lib.lib().ttn_als_eigsolve(Ad._h, xd._h, C.byref(p), C.byref(out), E, cap, C.byref(nE)))
    return np.array(E[:nE.value]), _ret(DeviceTT(out), host)


def als_gen_eigsolv(A, S, tt_start, sweep_schedule=(2,), rmax_schedule=None, tol=1e-10, it_solver=False, itslv_thresh=2500,
                    maxiter=500, linsolv_tol=1e-12, krylovdim=40):
    """`als_gen_eigsolv(A, S, tt_start; sweep_schedule, rmax_schedule, …)`, src/solvers/als.jl:344-440 → (E, tt_opt): lowest
    pair of A x = λ S x (S Hermitian positive definite).  The local pencil is solved densely on the device as the reference's
    `K_eiggenmin` does (als.jl:89-102; its `lobpcg` branch works on the same dense matrices), so `it_solver` / `itslv_thresh`
    only select between two routes to the same eigenpair and are accepted for signature compatibility."""
    xd, host = _dev(tt_start)
    if rmax_schedule is None:
        rmax_schedule = [max(xd.ttv_rks)]
    if len(rmax_schedule) != len(sweep_schedule):
        raise AssertionError("Sweep schedule error")
    Ad = _devo(A, xd.dtype)
    Sd = _devo(S, Ad.dtype)
    if Sd.dtype == np.complex128 and Ad.dtype != np.complex128:
        Ad = Ad.complex()
    if Ad.dtype == np.complex128 and xd.dtype != np.complex128:
        xd = xd.complex()
    p, keep = _params(sweep_schedule=sweep_schedule, rmax_schedule=rmax_schedule, linsolv_maxiter=int(maxiter),
                      linsolv_tol=float(linsolv_tol), krylovdim=int(krylovdim))
    cap = 2 * xd.N * (int(sweep_schedule[-1]) + 1) + 8
    E, nE, out = (C.c_double * cap)(), C.c_int(), C.c_void_p()
    check(_lib.lib().ttn_als_gen_eigsolv(Ad._h, Sd._h, xd._h, C.byref(p), C.byref(out), E, cap, C.byref(nE)))
    return np.array(E[:nE.value]), _ret(DeviceTT(out), host)


def mals_linsolve(A, b, tt_start, tol=1e-12, rmax=None, return_info=False, linsolv_maxiter=200, krylovdim=30):
    """src/solvers/mals.jl:240-309 (exactly one forward and one backward sweep)."""
    dims = tt_start.ttv_dims
    if rmax is None:
        rmax = int(round(math.sqrt(float(np.prod([float(n) for n in dims])))))
    p, keep = _params(tol=float(tol), rmax=int(rmax), linsolv_maxiter=int(linsolv_maxiter), krylovdim=int(krylovdim))
    x, host, res = _solve_lin(_lib.lib().ttn_mals_linsolve, A, b, tt_start, p)
    x = _ret(x, host)
    return (x, {"residual": res}) if return_info else x


def _eig_with_hist(fn, A, tt_start, p, cap, shard_ctx=None):
    xd, host = _dev(tt_start)
    Ad = _devo(A, xd.dtype)
    if Ad.dtype == np.complex128 and xd.dtype != np.complex128:
        xd = xd.complex()
    E, rh, nE, out = (C.c_double * cap)(), (C.c_int64 * cap)(), C.c_int(), C.c_void_p()
    if shard_ctx is None:
        check(fn(Ad._h, xd._h, C.byref(p), C.byref(out), E, rh, cap, C.byref(nE)))
    else:
        check(fn(Ad._h, xd._h, C.byref(p), shard_ctx.h, C.byref(out), E, rh, cap, C.byref(nE)))
    return np.array(E[:nE.value]), _ret(DeviceTT(out), host), [int(v) for v in rh[:nE.value]]


class ShardContext:
    """Exchange buffers of the sharded Lanczos matvec inside a multi-GPU DMRG sweep (`ttn_shard_ctx_*`): one per rank, created once
    per solve with `max_elems >= chi_max^2 * n^N`; `exchange` all-gathers a bytes object over the ranks
    (e.g. torch.distributed.all_gather_object) so that every rank can map its peers' buffers (CUDA IPC over NVLink)."""

    def __init__(self, dtype, max_elems, rank, nranks, exchange):
        lib = _lib.lib()
        self.h = C.c_void_p()
        self.rank, self.nranks = int(rank), int(nranks)
        check(lib.ttn_shard_ctx_create(_dtype_code(dtype), int(max_elems), self.rank, self.nranks, C.byref(self.h)))
        if self.nranks > 1:
            buf = (C.c_char * 384)()
            check(lib.ttn_shard_ctx_handles(self.h, buf))
            allb = exchange(bytes(buf))
            assert len(allb) == self.nranks and all(len(b) == 384 for b in allb)
            joined = (C.c_char * (384 * self.nranks)).from_buffer_copy(b"".join(allb))
            check(lib.ttn_shard_ctx_bind(self.h, joined))

    def free(self):
        if self.h:
            check(_lib.lib().ttn_shard_ctx_free(self.h))
            self.h = C.c_void_p()


def mals_eigsolve(A, tt_start, tol=1e-12, sweep_schedule=(2,), rmax_schedule=None, it_solver=False, linsolv_maxiter=200,
                  linsolv_tol=None, itslv_thresh=256, krylovdim=30):
    """src/solvers/mals.jl:335-425 → (E, tt_opt, r_hist)."""
    if rmax_schedule is None:
        rmax_schedule = [int(round(math.sqrt(float(np.prod([float(n) for n in tt_start.ttv_dims])))))]
    if len(rmax_schedule) != len(sweep_schedule):
        raise AssertionError("Sweep schedule error")
    if linsolv_tol is None:
        linsolv_tol = max(math.sqrt(tol), 1e-8)
    p, keep = _params(tol=float(tol), sweep_schedule=sweep_schedule, rmax_schedule=rmax_schedule,
                      linsolv_maxiter=int(linsolv_maxiter), linsolv_tol=float(linsolv_tol), krylovdim=int(krylovdim))
    cap = 2 * tt_start.N * (int(sweep_schedule[-1]) + 1) + 8
    return _eig_with_hist(_lib.lib().ttn_mals_eigsolve, A, tt_start, p, cap)


def dmrg_linsolve(A, b, tt_start, sweep_count=2, N=2, tol=1e-12, sweep_schedule=(2,), rmax_schedule=None, it_solver=True,
                  linsolv_maxiter=200, linsolv_tol=None, itslv_thresh=256, return_info=False, krylovdim=30, symmetrize=True):
    """src/solvers/dmrg.jl:385-473 (`sweep_count` is accepted and ignored, as in the reference :386)."""
    if rmax_schedule is None:
        rmax_schedule = [_isqrt_prod(tt_start.ttv_dims)]
    if linsolv_tol is None:
        linsolv_tol = max(math.sqrt(tol), 1e-8)
    p, keep = _params(N=int(N), tol=float(tol), sweep_schedule=sweep_schedule, rmax_schedule=rmax_schedule,
                      linsolv_maxiter=int(linsolv_maxiter), linsolv_tol=float(linsolv_tol), krylovdim=int(krylovdim),
                      symmetrize=int(bool(symmetrize)), it_solver=int(bool(it_solver)), itslv_thresh=int(itslv_thresh))
    x, host, res = _solve_lin(_lib.lib().ttn_dmrg_linsolve, A, b, tt_start, p)
    x = _ret(x, host)
    return (x, {"residual": res}) if return_info else x


def dmrg_eigsolve(A, tt_start, N=2, tol=1e-12, sweep_schedule=(2,), rmax_schedule=None, it_solver=False,
                  linsolv_maxiter=200, linsolv_tol=None, itslv_thresh=256, krylovdim=30, symmetrize=True, shard=None):
    """src/solvers/dmrg.jl:501-578 → (E, tt_opt, r_hist).  `shard`: a bound `ShardContext` — every rank of a one-node job calls this
    with identical arguments; the sweep runs replicated and the Lanczos matvec of every bond step is sharded over the ranks."""
    if rmax_schedule is None:
        rmax_schedule = [_isqrt_prod(tt_start.ttv_dims)]
    if len(rmax_schedule) != len(sweep_schedule):
        raise AssertionError("Sweep schedule error")
    if linsolv_tol is None:
        linsolv_tol = max(math.sqrt(tol), 1e-8)
    p, keep = _params(N=int(N), tol=float(tol), sweep_schedule=sweep_schedule, rmax_schedule=rmax_schedule,
                      linsolv_maxiter=int(linsolv_maxiter), linsolv_tol=float(linsolv_tol), krylovdim=int(krylovdim),
                      symmetrize=int(bool(symmetrize)))
    cap = 2 * tt_start.N * (int(sweep_schedule[-1]) + 1) + 8
    if shard is not None and shard.nranks > 1:
        return _eig_with_hist(_lib.lib().ttn_dmrg_eigsolve_sharded, A, tt_start, p, cap, shard_ctx=shard)
    return _eig_with_hist(_lib.lib().ttn_dmrg_eigsolve, A, tt_start, p, cap)


def _tdvp(two_site, H, u0, steps, normalize, sweeps, imaginary_time, max_bond, truncerr, krylovdim, tol, maxiter):
    lib = _lib.lib()
    ud, host = _dev(u0)
    Hd = _devo(H, ud.dtype)
    if Hd.dtype == np.complex128 and ud.dtype != np.complex128:
        ud = ud.complex()
    p = TdvpParams()
    check(lib.ttn_tdvp_params_default(C.byref(p)))
    st = (C.c_double * len(steps))(*[float(s) for s in steps])
    p.two_site = int(two_site)
    p.steps = C.cast(st, C.POINTER(C.c_double))
    p.n_steps = len(steps)
    p.normalize, p.sweeps, p.imaginary_time = int(bool(normalize)), int(sweeps), int(bool(imaginary_time))
    p.max_bond = (1 << 62) if max_bond is None else int(max_bond)
    p.truncerr = float(truncerr)
    p.krylovdim, p.krylov_tol, p.krylov_maxiter = int(krylovdim), float(tol), int(maxiter)
    out = C.c_void_p()
    check(lib.ttn_tdvp(Hd._h, ud._h, C.byref(p), C.byref(out)))
    return _ret(DeviceTT(out), host)


def tdvp(H, u0, steps, normalize=True, sweeps=1, imaginary_time=False, krylovdim=30, tol=1e-12, maxiter=100):
    """src/solvers/tdvp.jl:154-203."""
    return _tdvp(0, H, u0, steps, normalize, sweeps, imaginary_time, None, 0.0, krylovdim, tol, maxiter)


def tdvp2(H, u0, steps, normalize=True, sweeps=1, max_bond=None, truncerr=0.0, imaginary_time=False, krylovdim=30,
          tol=1e-12, maxiter=100):
    """src/solvers/tdvp.jl:303-357."""
    return _tdvp(1, H, u0, steps, normalize, sweeps, imaginary_time, max_bond, truncerr, krylovdim, tol, maxiter)


# ------------------------------------------------------------------------------------------------------
# kernel-level entry points (tests / benchmarks), host arrays in the reference layouts
# ------------------------------------------------------------------------------------------------------
def _f(a, dt):
    return np.asfortranarray(a, dtype=dt)


def matvec2(G, Amid, H, V, symmetrize=False):
    """K_matfree of src/solvers/dmrg.jl:239-244 on host arrays: G (w_l,chi_l,chi_l), Amid (w_l,nn,nn,w_r),
    H (w_r,chi_r,chi_r), V (chi_l,nn,chi_r)."""
    dt = np.result_type(G.dtype, Amid.dtype, H.dtype, V.dtype)
    code = _dtype_code(dt)
    G, Amid, H, V = _f(G, dt), _f(Amid, dt), _f(H, dt), _f(V, dt)
    Y = np.empty(V.shape, dtype=dt, order="F")
    check(_lib.lib().ttn_matvec2_host(code, G.shape[0], H.shape[0], G.shape[1], H.shape[1], Amid.shape[1], G.ctypes.data,
                                      Amid.ctypes.data, H.ctypes.data, V.ctypes.data, Y.ctypes.data, int(bool(symmetrize))))
    return Y


# ------------------------------------------------------------------------------------------------------
# multi-GPU partitioning (host logic; SURVEY.md section 8(e))
# ------------------------------------------------------------------------------------------------------
def shard_range(chi: int, rank: int, nranks: int):
    """Contiguous slice (c0, cp) of a bond index of size `chi` owned by `rank` — the same rule as the library's
    ttn_shard_range (the first chi % nranks ranks own one extra index).  Pure host arithmetic (no GPU needed)."""
    if not (chi >= 1 and nranks >= 1 and 0 <= rank < nranks):
        raise AssertionError("shard_range: bad arguments")
    base, rem = divmod(chi, nranks)
    return rank * base + min(rank, rem), base + (1 if rank < rem else 0)


def shard_batch(total: int, rank: int, nranks: int):
    """Slice (first, count) of a batch of `total` independent TT problems owned by `rank` (cfg5: no collective)."""
    return shard_range(total, rank, nranks) if total >= 1 else (0, 0)


def assemble_slices(slices, axis=-1):
    """Inverse of the partition: concatenates the per-rank slices (in rank order) along the sharded axis."""
    return np.concatenate(list(slices), axis=axis)


class ShardedMatvec:
    """Two-site effective operator of src/solvers/dmrg.jl:239-244 sharded over `nranks` GPUs on the bra index of the right
    environment (one process per GPU).  `exchange` is a callable that all-gathers a bytes object over the ranks
    (e.g. torch.distributed.all_gather_object); without it (or nranks == 1) only the local slice is produced."""

    def __init__(self, G, Amid, H, rank=0, nranks=1, exchange=None):
        dt = np.result_type(G.dtype, Amid.dtype, H.dtype)
        self.dtype, self.code = dt, _dtype_code(dt)
        G, Amid, H = _f(G, dt), _f(Amid, dt), _f(H, dt)
        self.shape = (G.shape[1], Amid.shape[1], H.shape[1])
        self.rank, self.nranks = rank, nranks
        self.h = C.c_void_p()
        check(_lib.lib().ttn_shard_matvec_create(self.code, G.shape[0], H.shape[0], G.shape[1], H.shape[1], Amid.shape[1],
                                                 G.ctypes.data, Amid.ctypes.data, H.ctypes.data, rank, nranks, C.byref(self.h)))
        c0, cp = C.c_int(), C.c_int()
        check(_lib.lib().ttn_shard_matvec_slice(self.h, C.byref(c0), C.byref(cp)))
        self.c0, self.cp = c0.value, cp.value
        assert (self.c0, self.cp) == shard_range(self.shape[2], rank, nranks)
        if exchange is not None and nranks > 1:
            mine = C.create_string_buffer(192)
            check(_lib.lib().ttn_shard_matvec_handles(self.h, mine))
            allh = exchange(bytes(mine.raw))
            assert len(allh) == nranks and all(len(b) == 192 for b in allh)
            buf = C.create_string_buffer(b"".join(allh), 192 * nranks)
            check(_lib.lib().ttn_shard_matvec_bind(self.h, buf))

    @property
    def nbytes(self):
        return int(np.prod(self.shape)) * np.dtype(self.dtype).itemsize

    def apply_dev(self, V_dev):
        """device pointer in → device pointer of the library-owned result vector (complete on every bound rank)"""
        out = C.c_void_p()
        check(_lib.lib().ttn_shard_matvec_apply(self.h, V_dev, C.byref(out)))
        return out

    def apply(self, V):
        """host vector in → host copy of this rank's result buffer (complete if peers are bound, else only the local slice
        Y[:, :, c0:c0+cp] is meaningful)"""
        V = _f(V, self.dtype)
        dV = C.c_void_p()
        check(_lib.lib().ttn_dev_alloc(V.nbytes, C.byref(dV)))
        try:
            check(_lib.lib().ttn_h2d(dV, V.ctypes.data, V.nbytes))
            dY = self.apply_dev(dV)
            Y = np.empty(self.shape, dtype=self.dtype, order="F")
            check(_lib.lib().ttn_d2h(Y.ctypes.data, dY, Y.nbytes))
        finally:
            check(_lib.lib().ttn_dev_free(dV))
        return Y

    def local_slice(self, V):
        return self.apply(V)[:, :, self.c0:self.c0 + self.cp]

    def eigsolve(self, x0, krylovdim=8, maxiter=1, tol=1e-10):
        """lowest eigenpair (KrylovKit.eigsolve(..., :SR) stand-in, dmrg.jl:245) → (theta, x, matvecs)"""
        x = _f(x0, self.dtype).copy(order="F")
        dx = C.c_void_p()
        check(_lib.lib().ttn_dev_alloc(x.nbytes, C.byref(dx)))
        try:
            check(_lib.lib().ttn_h2d(dx, x.ctypes.data, x.nbytes))
            th, mv = C.c_double(), C.c_int()
            check(_lib.lib().ttn_shard_eigsolve(self.h, dx, krylovdim, maxiter, tol, C.byref(th), C.byref(mv)))
            check(_lib.lib().ttn_d2h(x.ctypes.data, dx, x.nbytes))
        finally:
            check(_lib.lib().ttn_dev_free(dx))
        return th.value, x, mv.value

    def error(self):
        e = C.c_int()
        check(_lib.lib().ttn_shard_matvec_error(self.h, C.byref(e)))
        return e.value

    def free(self):
        if self.h:
            check(_lib.lib().ttn_shard_matvec_free(self.h))
            self.h = C.c_void_p()


def env_left(G, x, A):
    """update_G! of src/solvers/dmrg.jl:32-35: G (w_l,r_l,r_l), x (n,r_l,r_r), A (n,n,w_l,w_r) → (w_r,r_r,r_r)."""
    dt = np.result_type(G.dtype, x.dtype, A.dtype)
    G, x, A = _f(G, dt), _f(x, dt), _f(A, dt)
    n, rl, rr = x.shape
    wl, wr = A.shape[2], A.shape[3]
    out = np.empty((wr, rr, rr), dtype=dt, order="F")
    check(_lib.lib().ttn_env_left_host(_dtype_code(dt), n, wl, wr, rl, rr, G.ctypes.data, x.ctypes.data, A.ctypes.data,
                                       out.ctypes.data))
    return out


def env_right(H, x, A):
    """update_H! of src/solvers/dmrg.jl:27-30: H (w_r,r_r,r_r), x (n,r_l,r_r), A (n,n,w_l,w_r) → (w_l,r_l,r_l)."""
    dt = np.result_type(H.dtype, x.dtype, A.dtype)
    H, x, A = _f(H, dt), _f(x, dt), _f(A, dt)
    n, rl, rr = x.shape
    wl, wr = A.shape[2], A.shape[3]
    out = np.empty((wl, rl, rl), dtype=dt, order="F")
    check(_lib.lib().ttn_env_right_host(_dtype_code(dt), n, wl, wr, rl, rr, H.ctypes.data, x.ctypes.data, A.ctypes.data,
                                        out.ctypes.data))
    return out


def svdtrunc(A, max_bond=None, truncerr=0.0):
    """`_svdtrunc(A; max_bond, truncerr)` (the tail-norm method, src/tt_cross_interpolation.jl:149-166)
    → (U, s, Vt)."""
    dt = A.dtype
    A = _f(A, dt)
    m, n = A.shape
    k = min(m, n)
    U = np.empty((m, k), dtype=dt, order="F")
    Vt = np.empty((k * n,), dtype=dt)
    s = (C.c_double * k)()
    r = C.c_int()
    mb = (1 << 62) if max_bond is None else int(max_bond)
    check(_lib.lib().ttn_svdtrunc_host(_dtype_code(dt), m, n, A.ctypes.data, mb, float(truncerr), U.ctypes.data, s,
                                       Vt.ctypes.data, C.byref(r)))
    r = r.value
    return (np.asfortranarray(U.reshape(-1, order="F")[: m * r].reshape(m, r, order="F")), np.array(s[:r]),
            Vt[: r * n].reshape(r, n, order="F"))


def heig_top(G, nev):
    """Top `nev` eigenpairs (descending) of a batch of Hermitian PSD matrices `G` (batch, n, n) or (n, n) — test hook of
    csrc/heig.cu (the Gram-path SVD engine of `tt_compress!`).  → (lam (batch, nev), U (batch, n, nev), flags (batch,))."""
    G = np.asarray(G)
    single = G.ndim == 2
    if single:
        G = G[None]
    dt = np.complex128 if np.iscomplexobj(G) else np.float64
    b, n, _ = G.shape
    Gf = np.ascontiguousarray(np.transpose(G, (0, 2, 1)).astype(dt))      # each matrix column-major
    lam = np.empty((b, nev), dtype=np.float64)
    U = np.empty((b, nev, n), dtype=dt)                                    # column-major n x nev per matrix
    flags = np.zeros((b,), dtype=np.int32)
    check(_lib.lib().ttn_heig_host(_dtype_code(dt), n, int(nev), b, Gf.ctypes.data,
                                   lam.ctypes.data_as(C.POINTER(C.c_double)), U.ctypes.data,
                                   flags.ctypes.data_as(C.POINTER(C.c_int))))
    U = np.transpose(U, (0, 2, 1))
    return (lam[0], U[0], flags[0]) if single else (lam, U, flags)


def qr_thin(A):
    """thin Householder QR (LAPACK conventions) of a host matrix → (Q, R)."""
    dt = A.dtype
    A = _f(A, dt)
    m, n = A.shape
    k = min(m, n)
    Q = np.empty((m, k), dtype=dt, order="F")
    R = np.empty((k, n), dtype=dt, order="F")
    check(_lib.lib().ttn_qr_host(_dtype_code(dt), m, n, A.ctypes.data, Q.ctypes.data, R.ctypes.data))
    return Q, R


def gemm_host(A, B, conjA=False, conjB=False, transA=False, transB=False, alpha=1.0, beta=0.0, C0=None):
    """C = alpha·op(A)·op(B) + beta·C0 through the DMMA GEMM (device round trip; test helper)."""
    lib = _lib.lib()
    dt = np.result_type(A.dtype, B.dtype)
    code = _dtype_code(dt)
    A, B = _f(A, dt), _f(B, dt)
    M = A.shape[1] if transA else A.shape[0]
    K = A.shape[0] if transA else A.shape[1]
    N = B.shape[0] if transB else B.shape[1]
    Cm = np.zeros((M, N), dtype=dt, order="F") if C0 is None else _f(C0, dt).copy(order="F")
    es = np.dtype(dt).itemsize
    ptrs = []
    for arr in (A, B, Cm):
        p = C.c_void_p()
        check(lib.ttn_dev_alloc(max(arr.nbytes, es), C.byref(p)))
        check(lib.ttn_h2d(p, arr.ctypes.data, arr.nbytes))
        ptrs.append(p)
    sAm, sAk = (A.shape[0], 1) if transA else (1, A.shape[0])
    sBk, sBn = (B.shape[0], 1) if transB else (1, B.shape[0])
    check(lib.ttn_gemm(code, M, N, K, ptrs[0], sAm, sAk, int(conjA), ptrs[1], sBk, sBn, int(conjB), ptrs[2], 1, M,
                       float(alpha), float(beta), 1, 0, 0, 0))
    check(lib.ttn_synchronize())
    check(lib.ttn_d2h(Cm.ctypes.data, ptrs[2], Cm.nbytes))
    for p in ptrs:
        check(lib.ttn_dev_free(p))
    return Cm
