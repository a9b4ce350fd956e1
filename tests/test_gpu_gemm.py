"""Every single-GPU kernel of csrc/gemm.cu against an extended-precision reference, at the layouts the library issues.

Each case calls `ttn_gemm` directly on device buffers.  Every operand is scattered into a NaN-filled buffer with a guard
region before and after it, by its own element strides and batch stride; padding between columns and between batches
stays NaN.  The tile kernels zero-fill out-of-range elements without reading them and the bulk and thin kernels read only in
range, so a NaN in the result means that a kernel read an element it must not read.  C lives in a guarded buffer of the same
kind: everything outside the M x N x batch window must come back bit-for-bit unchanged, everything inside it finite and within
the worst-case rounding bound of `alpha*op(A_b)*op(B_b) + beta*C0_b` computed in long double, element by element.  With
beta = 0 the window starts as NaN (BLAS convention: C is overwritten, not scaled).

`expected_kernel` restates the dispatch of `gemm()` (csrc/gemm.cu, with `try_thin` and `try_bulk`), and each case checks,
through the CUDA profiler, that the instance it was written for is the one that ran, and how many launches it took.  The
table reaches all 22 instances that run on one GPU; the 12 fused all-gather epilogue instances need two or more GPUs and are
covered by tests/test_gpu_multi.py.  `test_compiled_gemm_kernel_inventory` (no GPU) holds the compiled set to these 34, so a
GEMM kernel added later fails until this table covers it.
"""
from __future__ import annotations

import ctypes as C
import os
import re
import shutil
import subprocess
from dataclasses import dataclass

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.path.join(ROOT, "tensortrainnumerics.jl_b200", "libttn_b200.so")

U = 2.0 ** -53            # unit roundoff of float64
MAX_GRID_Z = 65535        # CUDA grid.z limit: the tile kernels put the batch there
B200_SMS = 148


def _gk(T, bm, bn, wm, wn, amaj, bmaj, ns):
    return f"gemm_kernel<{T},{bm},{bn},{wm},{wn},{int(amaj)},{int(bmaj)},{ns}>"


_MAJORS = [(a, b) for a in (True, False) for b in (True, False)]
SINGLE_GPU_INSTANCES = frozenset(
    [f"gemm_thin_kernel<double,{kt},2>" for kt in (8, 16, 24)] + ["gemm_thin_kernel<double,32,1>"]
    + [f"gemm_thin_kernel<double2,{kt},1>" for kt in (8, 16, 24, 32)]
    + [f"gemm_bulk_kernel<double,128,64,32,32,{b}>" for b in (0, 1)]
    + [_gk("double", 128, 64, 32, 32, a, b, 3) for a, b in _MAJORS]
    + [_gk("double", 64, 64, 32, 16, a, b, 4) for a, b in _MAJORS]
    + [_gk("double2", 64, 64, 32, 16, a, b, 2) for a, b in _MAJORS])
EPILOGUE_INSTANCES = frozenset(
    [_gk("double2", 64, 64, 32, 16, a, b, 4) for a, b in _MAJORS]
    + [_gk("double2", 64, 128, 32, 32, a, b, 4) for a, b in _MAJORS]
    + [_gk("double", 128, 128, 64, 32, a, b, 4) for a, b in _MAJORS])

_KERNEL_NAME = re.compile(r"\b(gemm_(?:thin_|bulk_)?kernel)\s*<([^<>]*)>")


def canonical(name):
    """`void ttn::(anonymous namespace)::gemm_kernel<double, (int)64, ..., (bool)1, true, ...>(ttn::GemmArgs)` →
    `gemm_kernel<double,64,...,1,1,...>`; None for a name that is not a GEMM kernel."""
    m = _KERNEL_NAME.search(name)
    if m is None:
        return None
    args = [re.sub(r"\((?:unsigned )?(?:int|bool|long)\)", "", a).strip() for a in m.group(2).split(",")]
    args = [{"true": "1", "false": "0"}.get(a, a) for a in args]
    return f"{m.group(1)}<{','.join(args)}>"


# ----------------------------------------------------------------------------------------------------------------------
# the case table
# ----------------------------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Case:
    id: str
    cplx: bool
    M: int
    N: int
    K: int
    batch: int
    A: tuple            # (sAm, sAk, bA, off): element strides of A (M x K), batch stride, elements past the front guard
    B: tuple            # (sBk, sBn, bB, off)
    C: tuple            # (sCm, sCn, bC, off)
    conjA: bool = False
    conjB: bool = False
    alpha: float = 1.0
    beta: float = 0.0
    not_kernel: str | None = None   # a fast path this case must decline (its kernel name prefix)


def _dense(rows, cols, fast, pad, bpad, bcast):
    """(s_row, s_col, s_batch) of a rows x cols operand stored `fast`-index-first with leading dimension (extent + pad) and
    `bpad` elements between batches (0 batch stride when broadcast)."""
    if fast == "row":
        sr, sc, ext = 1, rows + pad, (rows + pad) * cols
    else:
        sr, sc, ext = cols + pad, 1, (cols + pad) * rows
    return sr, sc, 0 if bcast else ext + bpad


def case(id, cplx, M, N, K, batch=1, a="m", b="k", c="m", pad=(3, 2, 5), bpad=(7, 5, 6), bcast="", off=(0, 0, 0),
         A=None, B=None, C=None, **kw):
    """A case with dense operands: `a` = "m" stores A m-fastest (column-major M x K), "k" k-fastest; `b` = "k" stores B
    k-fastest (column-major K x N), "n" n-fastest; `c` = "m" stores C column-major, "n" row-major.  `pad` pads the leading
    dimensions, `bpad` the batch strides, `bcast` names the operands shared by the whole batch ("A", "B").  A, B, C given
    as full (s_row, s_col, s_batch, off) tuples override the dense layout."""
    if A is None:
        A = _dense(M, K, "row" if a == "m" else "col", pad[0], bpad[0], "A" in bcast) + (off[0],)
    if B is None:
        B = _dense(K, N, "row" if b == "k" else "col", pad[1], bpad[1], "B" in bcast) + (off[1],)
    if C is None:
        C = _dense(M, N, "row" if c == "m" else "col", pad[2], bpad[2], False) + (off[2],)
    return Case(id, cplx, M, N, K, batch, A, B, C, **kw)


def _dot_transfer(id, cplx, n, ral, rbl, rbr, **kw):
    # tt.cu tt_dot, first GEMM of a site: T[z,alpha,b] = sum_beta M[alpha,beta] B[z,beta,b]; the batch is the physical index z,
    # which interleaves with the rows of B and C (batch stride 1), so a stray write lands in a neighbour
    return case(id, cplx, ral, rbr, rbl, n, A=(1, ral, 0, 0), B=(n, n * rbl, 1, 0), C=(n, n * ral, 1, 0), **kw)


def _dot_partner(id, cplx, trains, n, ral, rar, rbr, **kw):
    # tt.cu tt_dot, second GEMM: M'[a,b] = sum_(z,alpha) conj(A[(z,alpha),a]) T[(z,alpha),b]: k-fastest, conjugated A
    return case(id, cplx, rar, rbr, n * ral, trains, A=(n * ral, 1, n * ral * rar, 0), B=(1, n * ral, n * ral * rbr, 0),
                C=(1, rar, rar * rbr, 0), conjA=True, **kw)


def _merge(id, cplx, n1, rl, r, n2, rr, **kw):
    # tt.cu tt_bond_truncate, two-site merge: Theta[(s1,alpha),(s2,beta)] = sum_gamma A[s1,alpha,gamma] B[s2,gamma,beta], batch s2
    p = n1 * rl
    return case(id, cplx, p, rr, r, n2, A=(1, p, 0, 0), B=(n2, n2 * r, 1, 0), C=(1, p * n2, p, 0), **kw)


def _localop_mid(id, cplx, cl, wl, nn, wr, nb, **kw):
    # localop.cu, middle contraction T2[a,(b,z),(f,j)] = T1[a,(y,e),(f,j)] W'[(y,e),(b,z)]: one W for the whole batch
    return case(id, cplx, cl, nn * wr, wl * nn, nb, A=(1, cl, cl * wl * nn, 0), B=(1, wl * nn, 0, 0),
                C=(1, cl, cl * nn * wr, 0), **kw)


CASES = [
    # --- Float64 64 x 64 tile (4 stages): four majors with partial tiles in M and N, K % 16 != 0, padded leading dims ---
    case("f64s_mk", False, 65, 63, 17, 3, a="m", b="k", alpha=0.75, beta=-0.5),
    case("f64s_mn", False, 65, 63, 17, 3, a="m", b="n", alpha=-2.0),
    case("f64s_kk", False, 63, 65, 17, 3, a="k", b="k", beta=1.0),
    case("f64s_kn", False, 63, 65, 33, 2, a="k", b="n", alpha=0.75, beta=1.0),
    # edges: M, N, K in {1, tile - 1, tile, tile + 1} (tile 64 x 64 x 16), N = 1, K = 0
    case("f64s_1x1x1", False, 1, 1, 1, 2),
    case("f64s_63x64x15", False, 63, 64, 15, 2, a="k", b="n", beta=-0.5),
    case("f64s_64x65x16", False, 64, 65, 16, 2, b="n", alpha=-2.0),
    case("f64s_65x1x64", False, 65, 1, 64, 3, a="k", alpha=0.75),
    case("f64s_1x65x65", False, 1, 65, 65, 2, b="n"),
    case("f64s_n1_m100", False, 100, 1, 20, 1, beta=1.0),
    case("f64s_k0_beta0", False, 70, 50, 0, 2),
    case("f64s_k0_beta", False, 70, 50, 0, 2, alpha=-2.0, beta=-0.5),
    case("f64s_m0_noop", False, 0, 50, 7, 2),
    # broadcast operands with batch > 1 (tile kernels)
    case("f64s_bcastA", False, 90, 70, 40, 4, bcast="A", beta=-0.5),
    case("f64s_bcastB", False, 100, 40, 20, 3, bcast="B", alpha=0.75),
    # --- Float64 128 x 64 tile, 3 LDGSTS stages: big by batch (ceil(M/128)·ceil(N/128)·batch >= 3/4 of the SMs), bulk declines
    case("f64b_mk", False, 200, 200, 33, 30, a="m", b="k", alpha=0.75, beta=-0.5),
    case("f64b_mn", False, 200, 200, 33, 30, a="m", b="n"),
    case("f64b_kk", False, 200, 200, 33, 30, a="k", b="k", alpha=-2.0, beta=1.0),
    case("f64b_kn", False, 200, 200, 33, 30, a="k", b="n", beta=-0.5),
    case("f64b_127x129x15", False, 127, 129, 15, 56, a="k", b="k"),
    case("f64b_129x127x17", False, 129, 127, 17, 56, b="n", alpha=0.75, beta=1.0),
    case("f64b_128x128x16_kfastA", False, 128, 128, 16, 120, a="k", b="n"),
    # --- Float64 bulk (TMA) big tile: full tiles, unit-stride tile rows, 16-byte aligned (even) strides and pointers ---
    case("f64t_bk", False, 128, 128, 32, 120, b="k", pad=(2, 2, 3), bpad=(4, 2, 1), alpha=0.75, beta=-0.5),
    case("f64t_bn", False, 128, 128, 32, 120, b="n", pad=(2, 4, 3), bpad=(4, 2, 1)),
    case("f64t_256x128x16", False, 256, 128, 16, 56, b="n", pad=(0, 0, 0), bpad=(0, 0, 0), alpha=-2.0, beta=1.0),
    # ... and the same shapes when the bulk kernel must decline: the 3-stage tile serves them
    case("f64t_decl_ptr_off1", False, 128, 128, 32, 120, b="k", pad=(2, 2, 3), bpad=(4, 2, 1), off=(1, 0, 0), beta=-0.5,
         not_kernel="gemm_bulk"),
    case("f64t_decl_odd_bstride", False, 128, 128, 32, 120, b="n", pad=(2, 4, 3), bpad=(1, 2, 1), alpha=0.75,
         not_kernel="gemm_bulk"),
    case("f64t_decl_m192", False, 192, 128, 32, 56, b="k", pad=(2, 2, 3), bpad=(4, 2, 1), not_kernel="gemm_bulk"),
    case("f64t_decl_conjA", False, 128, 128, 32, 120, b="n", pad=(2, 4, 3), bpad=(4, 2, 1), conjA=True, beta=1.0,
         not_kernel="gemm_bulk"),
    # --- thin right-multiplication, Float64 (N, K <= 32, M >= 256, one B for the batch) ---
    case("f64thin_k8", False, 777, 20, 8, 3, bcast="B", alpha=0.75, beta=1.0),
    case("f64thin_256x1x1", False, 256, 1, 1, 2, bcast="B"),
    case("f64thin_k0_beta0", False, 300, 5, 0, 2, bcast="B"),
    case("f64thin_k0_beta", False, 300, 5, 0, 1, bcast="B", beta=-0.5),
    case("f64thin_k16", False, 1000, 32, 16, 2, b="n", bcast="B", alpha=-2.0),
    case("f64thin_k9", False, 513, 7, 9, 3, bcast="B", beta=-0.5),
    case("f64thin_k24", False, 513, 12, 24, 4, b="n", bcast="B"),
    case("f64thin_k17", False, 600, 31, 17, 1, bcast="B", beta=1.0),
    case("f64thin_k32", False, 256, 32, 32, 2, bcast="B", alpha=0.75, beta=-0.5),
    case("f64thin_k25", False, 1025, 3, 25, 2, b="n", bcast="B"),
    _localop_mid("f64thin_localop", False, 300, 5, 4, 5, 6, alpha=0.75),
    # thin declines: sCm != 1, bB != 0, K = 33, M = 255
    case("f64thin_decl_sCm", False, 300, 20, 20, 2, c="n", bcast="B", not_kernel="gemm_thin"),
    case("f64thin_decl_bB", False, 300, 20, 20, 3, beta=1.0, not_kernel="gemm_thin"),
    case("f64thin_decl_k33", False, 300, 20, 33, 2, bcast="B", not_kernel="gemm_thin"),
    case("f64thin_decl_m255", False, 255, 20, 20, 2, bcast="B", alpha=-2.0, not_kernel="gemm_thin"),
    # --- ComplexF64 64 x 64 tile (2 stages): four majors x conj flags, partial tiles, K % 16 != 0 ---
    case("c128_mk", True, 65, 63, 17, 3, a="m", b="k", alpha=0.75, beta=-0.5),
    case("c128_mn_conjB", True, 65, 63, 17, 3, a="m", b="n", conjB=True, alpha=-2.0),
    case("c128_kk_conjA", True, 63, 65, 17, 3, a="k", b="k", conjA=True, beta=1.0),
    case("c128_kn_conjAB", True, 63, 65, 33, 2, a="k", b="n", conjA=True, conjB=True),
    case("c128_mk_conjAB", True, 65, 64, 15, 2, a="m", b="k", conjA=True, conjB=True, beta=-0.5),
    case("c128_kn", True, 64, 1, 16, 2, a="k", b="n", alpha=0.75),
    case("c128_1x1x1", True, 1, 1, 1, 2, conjB=True),
    case("c128_k0_beta0", True, 40, 30, 0, 2),
    case("c128_k0_beta", True, 40, 30, 0, 2, alpha=0.75, beta=-0.5),
    case("c128_big_by_batch", True, 100, 130, 20, 60, b="n", beta=1.0),
    case("c128_bcastA", True, 70, 66, 18, 3, bcast="A", conjA=True),
    # --- thin right-multiplication, ComplexF64 ---
    case("c128thin_k8", True, 300, 20, 8, 3, bcast="B", conjB=True, alpha=0.75, beta=1.0),
    case("c128thin_k16", True, 256, 32, 16, 2, b="n", bcast="B", beta=-0.5),
    case("c128thin_k24", True, 777, 9, 20, 3, b="n", bcast="B", conjB=True, alpha=-2.0),
    case("c128thin_k32", True, 513, 1, 32, 2, bcast="B"),
    _localop_mid("c128thin_localop", True, 300, 5, 4, 5, 4, beta=1.0),
    # thin declines: conj(A), bB != 0
    case("c128thin_decl_conjA", True, 300, 20, 20, 2, bcast="B", conjA=True, not_kernel="gemm_thin"),
    # --- call sites of the library, with one batch dimension ---
    _dot_transfer("f64_dot_transfer", False, 4, 65, 33, 70, alpha=1.0),
    _dot_transfer("c128_dot_transfer", True, 4, 65, 33, 70),
    _dot_partner("f64_dot_partner", False, 3, 4, 17, 65, 70),
    _dot_partner("c128_dot_partner", True, 3, 4, 17, 65, 70),
    _merge("f64_merge", False, 4, 33, 20, 4, 45),
    _merge("c128_merge_thin_decl_bB", True, 2, 132, 20, 4, 20, not_kernel="gemm_thin"),
]


# ----------------------------------------------------------------------------------------------------------------------
# dispatch mirror (gemm() at csrc/gemm.cu, with try_thin / try_bulk; gemm_bulk = gemm_thin = 1, one GPU)
# ----------------------------------------------------------------------------------------------------------------------
def expected_kernel(c: Case, sm_count: int, addr_A: int, addr_B: int):
    """(instance, launches) that `ttn_gemm` must run for case `c` whose A / B start at device addresses addr_A / addr_B."""
    if c.M <= 0 or c.N <= 0 or c.batch <= 0:
        return None, 0
    T = "double2" if c.cplx else "double"
    sAm, sAk, bA, _ = c.A
    sBk, sBn, bB, _ = c.B
    sCm, _, _, _ = c.C
    bigm, bign = (64 if c.cplx else 128), 128
    ctas_big = -(-c.M // bigm) * -(-c.N // bign) * c.batch
    big = c.M >= bigm * 3 // 4 and c.N >= bign * 3 // 4 and ctas_big >= sm_count * 3 // 4
    if (c.N <= 32 and c.K <= 32 and c.M >= 256 and not c.conjA and sAm == 1 and sCm == 1 and bB == 0
            and c.batch <= MAX_GRID_Z):
        kt = 8 if c.K <= 8 else 16 if c.K <= 16 else 24 if c.K <= 24 else 32
        rows = 1 if c.cplx or kt == 32 else 2
        return f"gemm_thin_kernel<{T},{kt},{rows}>", 1
    amaj, bmaj = abs(sAm) <= abs(sAk), abs(sBn) < abs(sBk)
    launches = -(-c.batch // MAX_GRID_Z)
    if c.cplx:
        return _gk("double2", 64, 64, 32, 16, amaj, bmaj, 2), launches
    if not big:
        return _gk("double", 64, 64, 32, 16, amaj, bmaj, 4), launches
    al = lambda v: v % 2 == 0            # 16 bytes = 2 doubles
    if (not c.conjA and not c.conjB and c.M % 128 == 0 and c.N % 64 == 0 and c.K % 16 == 0 and c.K >= 16
            and c.batch <= MAX_GRID_Z and sAm == 1 and al(sAk) and al(bA) and addr_A % 16 == 0 and al(bB)
            and addr_B % 16 == 0):
        if sBn == 1 and al(sBk):
            return "gemm_bulk_kernel<double,128,64,32,32,1>", 1
        if sBk == 1 and al(sBn):
            return "gemm_bulk_kernel<double,128,64,32,32,0>", 1
    return _gk("double", 128, 64, 32, 32, amaj, bmaj, 3), launches


# ----------------------------------------------------------------------------------------------------------------------
# guarded operands
# ----------------------------------------------------------------------------------------------------------------------
def _guard(s_row, s_col):
    # a multiple of 64 elements, so that the alignment of an operand is set by its `off` alone
    return -(-max(1024, 128 * max(s_row, s_col)) // 64) * 64


class Guarded:
    """A rows x cols x nb operand scattered at origin + i*s_row + j*s_col + b*s_batch into a NaN-filled buffer; the guards
    before and after it hold at least 1024 elements and at least one 128-row / 128-column tile extent of the operand."""

    def __init__(self, rows, cols, nb, s_row, s_col, s_batch, off, dtype):
        assert min(s_row, s_col, s_batch) >= 0
        guard = _guard(s_row, s_col)
        span = 0 if rows * cols * nb == 0 else (rows - 1) * s_row + (cols - 1) * s_col + (nb - 1) * s_batch + 1
        self.origin = guard + off
        self.buf = np.full(self.origin + span + guard, complex(np.nan, np.nan) if dtype == np.complex128 else np.nan,
                           dtype=dtype)
        self.idx = (self.origin + np.arange(nb)[:, None, None] * s_batch + np.arange(rows)[None, :, None] * s_row
                    + np.arange(cols)[None, None, :] * s_col)
        assert np.unique(self.idx).size == self.idx.size, "operand layout overlaps itself"
        self.dev = None

    def upload(self, lib, check):
        p = C.c_void_p()
        check(lib.ttn_dev_alloc(self.buf.nbytes, C.byref(p)))
        self.dev = p
        check(lib.ttn_h2d(p, self.buf.ctypes.data, self.buf.nbytes))

    @property
    def addr(self):
        return self.dev.value + self.origin * self.buf.itemsize

    def download(self, lib, check):
        out = np.empty_like(self.buf)
        check(lib.ttn_d2h(out.ctypes.data, self.dev, out.nbytes))
        return out

    def free(self, lib, check):
        if self.dev is not None:
            check(lib.ttn_dev_free(self.dev))
            self.dev = None


def _rand(rng, shape, cplx):
    a = rng.standard_normal(shape)
    return a + 1j * rng.standard_normal(shape) if cplx else a


def _profiled_gemm_names(lib, check, fn):
    """Runs fn() under the CUDA profiler, synchronises the library's stream inside the capture, and returns the raw names
    of the GEMM kernels that ran, in launch order."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        check(lib.ttn_synchronize())
    evs = [e for e in prof.events() if e.device_type == DeviceType.CUDA and "gemm_" in e.name]
    return [e.name for e in sorted(evs, key=lambda e: e.time_range.start)]


SEEN = {}          # case id -> canonical instances launched (filled by test_gemm_case)
RAW_NAMES = []     # one raw profiler name per instance, to show what the normaliser was fitted to


def run_case(c: Case, seed: int, seen=None):
    """Runs one case through `ttn_gemm` and checks guards, numerics and the instance that ran; returns the launched names."""
    import torch
    from ttn_b200 import _lib
    lib, check = _lib.lib(), _lib.check
    sm_count = torch.cuda.get_device_properties(0).multi_processor_count
    dt = np.complex128 if c.cplx else np.float64
    rng = np.random.default_rng(seed)
    nbA = c.batch if c.A[2] else 1
    nbB = c.batch if c.B[2] else 1
    Al, Bl = _rand(rng, (nbA, c.M, c.K), c.cplx), _rand(rng, (nbB, c.K, c.N), c.cplx)
    C0 = _rand(rng, (c.batch, c.M, c.N), c.cplx) if c.beta != 0.0 else None
    gA = Guarded(c.M, c.K, nbA, c.A[0], c.A[1], c.A[2], c.A[3], dt)
    gB = Guarded(c.K, c.N, nbB, c.B[0], c.B[1], c.B[2], c.B[3], dt)
    gC = Guarded(c.M, c.N, c.batch, c.C[0], c.C[1], c.C[2], c.C[3], dt)
    gA.buf[gA.idx] = Al
    gB.buf[gB.idx] = Bl
    if C0 is not None:
        gC.buf[gC.idx] = C0
    try:
        for g in (gA, gB, gC):
            g.upload(lib, check)
        want, n_launch = expected_kernel(c, sm_count, gA.addr, gB.addr)
        lib.ttn_reset_launch_count()
        code = _lib.TTN_C128 if c.cplx else _lib.TTN_F64
        raw = _profiled_gemm_names(lib, check, lambda: check(lib.ttn_gemm(
            code, c.M, c.N, c.K, C.c_void_p(gA.addr), c.A[0], c.A[1], int(c.conjA), C.c_void_p(gB.addr), c.B[0], c.B[1],
            int(c.conjB), C.c_void_p(gC.addr), c.C[0], c.C[1], float(c.alpha), float(c.beta), c.batch, c.A[2], c.B[2],
            c.C[2])))
        launches = lib.ttn_launch_count()
        got = gC.download(lib, check)
    finally:
        for g in (gA, gB, gC):
            g.free(lib, check)
    names = [canonical(n) or n for n in raw]
    if seen is not None:
        seen[c.id] = set(names)
    for n in raw:
        if canonical(n) not in {canonical(r) for r in RAW_NAMES}:
            RAW_NAMES.append(n)

    # which kernel ran, and how often
    assert names == [want] * n_launch, f"expected {n_launch} x {want}, the profiler saw {raw}"
    assert launches == n_launch
    if c.not_kernel is not None:
        assert not any(n.startswith(c.not_kernel) for n in names), names

    # nothing outside the M x N x batch window was written
    outside = np.ones(got.size, dtype=bool)
    outside[gC.idx.ravel()] = False
    es = got.itemsize
    changed = np.flatnonzero(np.any(got.view(np.uint8).reshape(-1, es)[outside]
                                    != gC.buf.view(np.uint8).reshape(-1, es)[outside], axis=1))
    assert changed.size == 0, f"{changed.size} elements outside the C window were written (first at buffer offset " \
                              f"{np.flatnonzero(outside)[changed[0]] - gC.origin} from C)"

    # the window: finite and within the worst-case rounding bound of every summation order
    out = got[gC.idx]
    assert np.all(np.isfinite(out)), f"{np.count_nonzero(~np.isfinite(out))} non-finite results (first at batch, m, n = " \
                                     f"{tuple(int(v[0]) for v in np.nonzero(~np.isfinite(out)))})"
    ld = np.clongdouble if c.cplx else np.longdouble
    opA, opB = (np.conj(Al) if c.conjA else Al), (np.conj(Bl) if c.conjB else Bl)
    ref = np.broadcast_to(np.matmul(opA.astype(ld), opB.astype(ld)), out.shape) * ld(c.alpha)
    scale = abs(c.alpha) * np.matmul(np.abs(Al), np.abs(Bl))
    if C0 is not None:
        ref = ref + ld(c.beta) * C0.astype(ld)
        scale = scale + abs(c.beta) * np.abs(C0)
    bound = ((4 if c.cplx else 2) * c.K + 4) * U * np.broadcast_to(scale, out.shape)
    err = np.abs(out.astype(ld) - ref)
    bad = err > bound
    if np.any(bad):
        i = np.unravel_index(np.argmax(np.where(bad, err / np.maximum(bound, 1e-300), 0)), out.shape)
        pytest.fail(f"{np.count_nonzero(bad)} of {out.size} elements outside the rounding bound; worst at (batch, m, n) = "
                    f"{tuple(int(v) for v in i)}: got {out[i]}, reference {complex(ref[i]) if c.cplx else float(ref[i])}, "
                    f"bound {bound[i]:.3e}")
    return names


def _assert_default_switches():
    import ttn_b200 as t
    assert t.get_option("gemm_bulk") == 1.0 and t.get_option("gemm_thin") == 1.0, "the dispatch mirror assumes the defaults"


# ----------------------------------------------------------------------------------------------------------------------
# tests
# ----------------------------------------------------------------------------------------------------------------------
def _flops(c):
    return (8 if c.cplx else 2) * c.M * c.N * c.K * c.batch


def test_case_table_reaches_every_single_gpu_instance():
    """The table itself (no GPU; B200 SM count, allocations 256-byte aligned as cudaMalloc returns them): every single-GPU
    instance is the expected kernel of some case with batch > 1, every `gemm_kernel` instance of some case with partial
    tiles in M and N and K % 16 != 0 (the bulk kernel requires full tiles), and the long-double reference stays cheap."""
    by_kernel = {}
    for c in CASES:
        es = 16 if c.cplx else 8
        addr = lambda op: (_guard(op[0], op[1]) + op[3]) * es
        k, _ = expected_kernel(c, B200_SMS, addr(c.A), addr(c.B))
        by_kernel.setdefault(k, []).append(c)
    assert set(by_kernel) - {None} == SINGLE_GPU_INSTANCES, sorted(SINGLE_GPU_INSTANCES ^ (set(by_kernel) - {None}))
    for k, cs in by_kernel.items():
        if k is None:
            continue
        assert any(c.batch > 1 for c in cs), k
        if k.startswith("gemm_kernel<"):
            bm, bn = (int(v) for v in k.split("<")[1].split(",")[1:3])
            assert any(c.M % bm and c.N % bn and c.K % 16 and c.batch > 1 for c in cs), k
    assert sum(_flops(c) for c in CASES) < 2e9
    assert len({c.id for c in CASES}) == len(CASES)


@pytest.mark.gpu
@pytest.mark.parametrize("c", CASES, ids=[c.id for c in CASES])
def test_gemm_case(c):
    _assert_default_switches()
    run_case(c, seed=sum(map(ord, c.id)), seen=SEEN)


@pytest.mark.gpu
def test_gemm_table_launched_every_instance():
    """Across the whole table the profiler saw exactly the 22 single-GPU instances (runs after the table in file order)."""
    if set(SEEN) != {c.id for c in CASES}:
        pytest.skip("the case table did not run in full in this session")
    seen = set().union(*SEEN.values())
    print(f"\ngemm kernel coverage: {len(seen & SINGLE_GPU_INSTANCES)}/{len(SINGLE_GPU_INSTANCES)} single-GPU instances")
    for n in RAW_NAMES:
        print("  profiler name:", n)
    assert seen == SINGLE_GPU_INSTANCES, sorted(seen ^ SINGLE_GPU_INSTANCES)


@pytest.mark.gpu
@pytest.mark.parametrize("cplx,shape", [(False, (2, 3, 4)), (True, (3, 2, 5))], ids=["f64", "c128"])
def test_gemm_batch_past_grid_limit(cplx, shape):
    """`ttn_gemm` with 65537 products in the batch, more than grid.z holds: two launches of the 64 x 64 tile, every product
    and the guards checked."""
    _assert_default_switches()
    M, N, K = shape
    c = case(f"batch65537_{'c128' if cplx else 'f64'}", cplx, M, N, K, MAX_GRID_Z + 2, a="k", b="n", alpha=0.75, beta=-0.5)
    names = run_case(c, seed=65537 + cplx)
    assert len(names) == 2 and names[0] == _gk("double2" if cplx else "double", 64, 64, 32, 16, False, True,
                                               2 if cplx else 4)


@pytest.mark.gpu
@pytest.mark.parametrize("cplx", [False, True], ids=["f64", "c128"])
def test_dot_norm_batch_past_grid_limit(cplx):
    """`dot` / `norm` of 16385 batched trains (d = 3, n = 4, ranks 1-3-3-1).  The first transfer GEMM of each site runs with
    batch1 = n = 4 and batch2 = trains, so `gemm()` splits it at 65535 // 4 = 16383 trains: trains 16383 and 16384 land in a
    second launch.  Every train against a dense contraction, to 1e-13 of ‖x‖·‖y‖."""
    import ttn_b200 as t
    from ttn_b200 import _lib
    lib = _lib.lib()
    _assert_default_switches()
    trains, dims, rks = 16385, (4, 4, 4), (1, 3, 3, 1)
    rng = np.random.default_rng(16385 + cplx)
    mk = lambda: [np.asfortranarray(_rand(rng, (dims[k], rks[k], rks[k + 1], trains), cplx)) for k in range(3)]
    xc, yc = mk(), mk()
    x, y = t.DeviceTT.upload_batched(xc, dims, rks), t.DeviceTT.upload_batched(yc, dims, rks)
    full = lambda cs: np.einsum("iab,jacb,kcb->bijk", cs[0][:, 0], cs[1], cs[2][:, :, 0])
    X, Y = full(xc), full(yc)
    ref_dot = np.einsum("bijk,bijk->b", X.conj(), Y)
    nx, ny = np.sqrt(np.einsum("bijk,bijk->b", X.conj(), X).real), np.sqrt(np.einsum("bijk,bijk->b", Y.conj(), Y).real)

    got = {}
    raw = _profiled_gemm_names(lib, _lib.check, lambda: got.setdefault("dot", t.dot(x, y)))
    T, ns = ("double2", 2) if cplx else ("double", 4)
    first, second = _gk(T, 64, 64, 32, 16, True, False, ns), _gk(T, 64, 64, 32, 16, False, False, ns)
    names = [canonical(n) for n in raw]
    assert names.count(first) == 2 * 3 and names.count(second) == 3 and len(names) == 9, raw
    d = np.asarray(got["dot"])
    assert d.shape == (trains,)
    err = np.abs(d - ref_dot) / (nx * ny)
    assert err.max() < 1e-13, (int(err.argmax()), float(err.max()))
    nrm = np.asarray(t.norm(x))
    errn = np.abs(nrm - nx) / nx
    assert errn.max() < 1e-13, (int(errn.argmax()), float(errn.max()))


def _cuda_tool(name):
    exe = shutil.which(name)
    if exe is None:
        cand = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", name)
        exe = cand if os.path.exists(cand) else None
    return exe


def test_compiled_gemm_kernel_inventory():
    """The GEMM kernels compiled into libttn_b200.so are exactly the 22 single-GPU instances this file's case table covers
    plus the 12 fused all-gather epilogue instances (two or more GPUs, tests/test_gpu_multi.py).  No GPU needed."""
    if not os.path.exists(LIB_PATH):
        pytest.skip("libttn_b200.so is not built")
    cuobjdump, cufilt = _cuda_tool("cuobjdump"), _cuda_tool("cu++filt")
    if cuobjdump is None or cufilt is None:
        pytest.skip("cuobjdump / cu++filt not found")
    elf = subprocess.run([cuobjdump, "-elf", LIB_PATH], capture_output=True, text=True, check=True).stdout
    mangled = sorted(set(re.findall(r"_ZN3ttn\w*gemm_\w*kernel\w*", elf)))
    demangled = subprocess.run([cufilt], input="\n".join(mangled), capture_output=True, text=True, check=True).stdout
    kernels = {canonical(line) for line in demangled.splitlines()
               if re.fullmatch(r"void ttn::.*::gemm_\w*kernel<[^<>]*>\(ttn::GemmArgs\)", line.strip())}
    assert kernels == SINGLE_GPU_INSTANCES | EPILOGUE_INSTANCES, sorted(kernels ^ (SINGLE_GPU_INSTANCES | EPILOGUE_INSTANCES))
    assert len(kernels) == 34
