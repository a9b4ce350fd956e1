// Strided-batched FP64 / ComplexF64 GEMM on the sm_100a FP64 tensor pipe (SASS: DMMA.8x8x4).
//
// This is kernel family F1/F2/F3 of SURVEY.md §2.1: every contraction on the reference's hot path —
// the effective-operator matvec L·W·X·R (src/solvers/dmrg.jl:239-244, als.jl:78, mals.jl:193-198,
// tdvp.jl:30,34,206-207), the environment updates (dmrg.jl:27-35, als.jl:23-55, mals.jl:10-13,
// tdvp.jl:37-43), the two-site merge (tt_tools.jl:749) and the bond absorbs (als.jl:116,132,
// dmrg.jl:318,334) — is issued as one or more calls of this kernel.  Operands are addressed through
// explicit element strides plus two batch dimensions, so the (s,l,r)/(l,s,r) permutes that the reference
// performs with `permutedims` (tt_tools.jl:746-747, dmrg.jl:39, tdvp.jl:54-55) are folded into the loads.
//
// Design (B200): 256-thread CTAs, BK=16 k-slabs streamed by a 4-stage cp.async (LDGSTS) pipeline into padded shared
// memory (pitch ≡ 4 mod 16 doubles → the m8n8k4 fragment loads are bank-conflict free), each warp owns a
// WM x WN accumulator block held in registers and issues mma.sync.m8n8k4.f64.  ComplexF64 runs as four
// real DMMA products on split re/im fragments.  sm_100a has no f64 kind for tcgen05.mma, so DMMA via
// mma.sync is the FP64 tensor path on this chip (larger f64 shapes decompose to 8x8x4 in SASS).
#include "ttn_internal.h"
#include "dmma.h"
#include "tma.h"

namespace ttn {

namespace {

constexpr int BK = 16;
constexpr int NT = 256;
constexpr int NSTAGE = 4;       // cp.async pipeline depth (k-slabs in flight)

template <class T> struct Pad { static constexpr int v = 4; };
template <> struct Pad<zc> { static constexpr int v = 2; };

// tiles with at most 64 KB of accumulators whose pipeline fits in ~110 KB of shared memory are compiled for two CTAs per SM
// (<= 128 registers per thread): 16 resident warps hide the DMMA / shared-memory latency that 8 warps leave exposed
template <class T, int BM, int BN, int NS>
struct MinBlocks {
  static constexpr size_t smem = sizeof(T) * NS * BK * (BM + BN + 2 * Pad<T>::v);
  static constexpr int v = (sizeof(T) * BM * BN <= 65536 && smem <= 112 * 1024) ? 2 : 1;
};

template <class T, int BM, int BN, int WM, int WN, bool AMAJ, bool BMAJ, int NS = NSTAGE>
__global__ void __launch_bounds__(NT, MinBlocks<T, BM, BN, NS>::v) gemm_kernel(const GemmArgs g) {
  constexpr int PAD = Pad<T>::v;
  constexpr int PA = BM + PAD, PB = BN + PAD;
  constexpr int EA = BM * BK / NT, EB = BN * BK / NT;
  constexpr int MT = WM / 8, NTL = WN / 8;
  constexpr int WARPS_M = BM / WM;
  constexpr int STAGE = BK * (PA + PB);              // elements per pipeline stage
  static_assert((BM / WM) * (BN / WN) == NT / 32, "warp layout must cover the CTA tile");
  static_assert(BM * BK % NT == 0 && BN * BK % NT == 0, "tile loads must divide evenly");

  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* Sm = reinterpret_cast<T*>(smem_raw);            // [NS][ A: [BK][PA] | B: [BK][PB] ]

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int g8 = lane >> 2, t4 = lane & 3;
  const int wm0 = (warp % WARPS_M) * WM, wn0 = (warp / WARPS_M) * WN;
  const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
  const int b = blockIdx.z, b1 = b % g.batch1, b2 = b / g.batch1;

  const T* __restrict__ A = reinterpret_cast<const T*>(g.A) + b1 * g.bA1 + b2 * g.bA2;
  const T* __restrict__ B = reinterpret_cast<const T*>(g.B) + b1 * g.bB1 + b2 * g.bB2;
  T* __restrict__ C = reinterpret_cast<T*>(g.C) + b1 * g.bC1 + b2 * g.bC2;

  Acc<T> acc[MT][NTL];
#pragma unroll
  for (int i = 0; i < MT; ++i)
#pragma unroll
    for (int j = 0; j < NTL; ++j) acc[i][j].zero();

  const int nkt = (g.K + BK - 1) / BK;

  // per-thread element coordinates inside a k-slab are fixed; only the k offset advances
  int am[EA], ak[EA], bn[EB], bk[EB];
  int64_t aoff[EA], boff[EB];
  bool aok[EA], bok[EB];
#pragma unroll
  for (int r = 0; r < EA; ++r) {
    const int idx = tid + r * NT;
    am[r] = AMAJ ? (idx % BM) : (idx / BK);
    ak[r] = AMAJ ? (idx / BM) : (idx % BK);
    aok[r] = m0 + am[r] < g.M;
    aoff[r] = (int64_t)(m0 + am[r]) * g.sAm + (int64_t)ak[r] * g.sAk;
  }
#pragma unroll
  for (int r = 0; r < EB; ++r) {
    const int idx = tid + r * NT;
    bn[r] = BMAJ ? (idx % BN) : (idx / BK);
    bk[r] = BMAJ ? (idx / BN) : (idx % BK);
    bok[r] = n0 + bn[r] < g.N;
    boff[r] = (int64_t)bk[r] * g.sBk + (int64_t)(n0 + bn[r]) * g.sBn;
  }
  auto issue = [&](int kt) {
    if (kt < nkt) {
      T* as = Sm + (size_t)(kt % NS) * STAGE;
      T* bs = as + BK * PA;
      const int k0 = kt * BK;
#pragma unroll
      for (int r = 0; r < EA; ++r) {
        const bool ok = aok[r] && k0 + ak[r] < g.K;
        cp_async_elem<T>(as + ak[r] * PA + am[r], ok ? A + aoff[r] + (int64_t)k0 * g.sAk : A, ok);
      }
#pragma unroll
      for (int r = 0; r < EB; ++r) {
        const bool ok = bok[r] && k0 + bk[r] < g.K;
        cp_async_elem<T>(bs + bk[r] * PB + bn[r], ok ? B + boff[r] + (int64_t)k0 * g.sBk : B, ok);
      }
    }
    cp_async_commit();     // one group per slab, empty past the end, so that wait_group counts stay uniform
  };

#pragma unroll
  for (int s = 0; s < NS - 1; ++s) issue(s);

  const bool cja = g.conjA, cjb = g.conjB;
  for (int kt = 0; kt < nkt; ++kt) {
    cp_async_wait<NS - 2>();      // slab kt has landed (for this thread's copies) ...
    __syncthreads();                  // ... and for everyone; slab kt-1 is no longer being read
    issue(kt + NS - 1);           // refills the buffer of slab kt-1
    const T* as = Sm + (size_t)(kt % NS) * STAGE;
    const T* bs = as + BK * PA;
#pragma unroll
    for (int kk = 0; kk < BK; kk += 4) {
      T af[MT], bf[NTL];
#pragma unroll
      for (int i = 0; i < MT; ++i) {
        const T v = as[(kk + t4) * PA + wm0 + i * 8 + g8];
        af[i] = (is_cplx<T>::value && cja) ? t_conj(v) : v;
      }
#pragma unroll
      for (int j = 0; j < NTL; ++j) {
        const T v = bs[(kk + t4) * PB + wn0 + j * 8 + g8];
        bf[j] = (is_cplx<T>::value && cjb) ? t_conj(v) : v;
      }
#pragma unroll
      for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < NTL; ++j) acc[i][j].mma(af[i], bf[j]);
    }
  }
  cp_async_wait<0>();

  // epilogue: C = alpha*acc + beta*C, written straight from the DMMA accumulator layout
  const bool has_beta = (g.beta != 0.0);
#pragma unroll
  for (int i = 0; i < MT; ++i) {
    const int row = m0 + wm0 + i * 8 + g8;
    if (row >= g.M) continue;
#pragma unroll
    for (int j = 0; j < NTL; ++j) {
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int col = n0 + wn0 + j * 8 + 2 * t4 + e;
        if (col < g.N) {
          T* p = C + (int64_t)row * g.sCm + (int64_t)col * g.sCn;
          T v = t_scale(acc[i][j].get(e), g.alpha);
          if (has_beta) v = t_add(v, t_scale(*p, g.beta));
          *p = v;
          // compute -> all-gather fusion: the same element goes straight to the peers' buffers over NVLink (P2P stores)
          for (int q = 0; q < g.npeer; ++q)
            (reinterpret_cast<T*>(g.Cpeer[q]) + b1 * g.bC1 + b2 * g.bC2)[(int64_t)row * g.sCm + (int64_t)col * g.sCn] = v;
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// TMA-staged variant of the big tile (north star: "DMMA tiles staged through TMA and shared memory").  Operands whose tile
// rows are contiguous in global memory (A: m fastest; B: n fastest or k fastest) are moved by the copy engine: warp 0 issues
// one bulk asynchronous copy per tile row (cp.async.bulk, SASS UBLKCP) into the same padded shared-memory rows the DMMA
// fragment loads expect, all copies of a k-slab complete on that stage's mbarrier (expect_tx = bytes of the slab), and the
// other seven warps never touch an address computation for them.  B with k fastest has tile rows of only 128 bytes: issuing
// 128 bulk copies per slab measured 2x SLOWER than LDGSTS (12.5 vs 24.9 TFLOP/s on the cfg4 matvec), so that operand keeps the
// per-element LDGSTS staging of gemm_kernel while A still comes through the copy engine.
// Requirements (checked by the host dispatcher): unit stride along the tile rows, full tiles, 16-byte aligned rows.
// ---------------------------------------------------------------------------------------------------------------------
template <class T, int BM, int BN, int WM, int WN, bool BMAJ>
__global__ void __launch_bounds__(NT, MinBlocks<T, BM, BN, NSTAGE>::v) gemm_bulk_kernel(const GemmArgs g) {
  constexpr int PAD = Pad<T>::v;
  constexpr int PA = BM + PAD, PB = BN + PAD;
  constexpr int EB = BN * BK / NT;
  constexpr int MT = WM / 8, NTL = WN / 8;
  constexpr int WARPS_M = BM / WM;
  constexpr int STAGE = BK * (PA + PB);
  // bytes the copy engine delivers per k-slab: the A rows, and the B rows when B is n-fastest (k-fastest B has 128-byte tile
  // rows — measured 2x slower as 128 bulk copies per slab — and is staged by LDGSTS like in gemm_kernel)
  constexpr uint32_t STAGE_BYTES = (uint32_t)(sizeof(T) * (BM * BK + (BMAJ ? BN * BK : 0)));
  static_assert((BM / WM) * (BN / WN) == NT / 32, "warp layout must cover the CTA tile");

  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* Sm = reinterpret_cast<T*>(smem_raw);
  __shared__ __align__(8) uint64_t full[NSTAGE];

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int g8 = lane >> 2, t4 = lane & 3;
  const int wm0 = (warp % WARPS_M) * WM, wn0 = (warp / WARPS_M) * WN;
  const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
  const int b = blockIdx.z, b1 = b % g.batch1, b2 = b / g.batch1;
  const T* __restrict__ A = reinterpret_cast<const T*>(g.A) + b1 * g.bA1 + b2 * g.bA2;
  const T* __restrict__ B = reinterpret_cast<const T*>(g.B) + b1 * g.bB1 + b2 * g.bB2;
  T* __restrict__ C = reinterpret_cast<T*>(g.C) + b1 * g.bC1 + b2 * g.bC2;

  Acc<T> acc[MT][NTL];
#pragma unroll
  for (int i = 0; i < MT; ++i)
#pragma unroll
    for (int j = 0; j < NTL; ++j) acc[i][j].zero();
  const int nkt = g.K / BK;

  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < NSTAGE; ++s) mbar_init(&full[s], 1);
    mbar_fence_init();
  }
  __syncthreads();

  // k-fastest B: per-thread element coordinates of the LDGSTS staging (as in gemm_kernel, !BMAJ)
  int bn[EB], bk[EB];
  int64_t boff[EB];
#pragma unroll
  for (int r = 0; r < EB; ++r) {
    const int idx = tid + r * NT;
    bn[r] = idx / BK;
    bk[r] = idx % BK;
    boff[r] = (int64_t)bk[r] * g.sBk + (int64_t)(n0 + bn[r]) * g.sBn;
  }
  auto issue = [&](int kt) {
    if (kt < nkt) {
      const int s = kt % NSTAGE;
      T* as = Sm + (size_t)s * STAGE;
      T* bs = as + BK * PA;
      const int k0 = kt * BK;
      if (warp == 0) {
        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");   // generic-proxy reads of the slot before the async writes
        if (lane == 0) mbar_arrive_expect_tx(&full[s], STAGE_BYTES);
        __syncwarp();
        for (int r = lane; r < BK; r += 32)
          bulk_copy_g2s(as + r * PA, A + m0 + (int64_t)(k0 + r) * g.sAk, (uint32_t)(sizeof(T) * BM), &full[s]);
        if (BMAJ)
          for (int r = lane; r < BK; r += 32)
            bulk_copy_g2s(bs + r * PB, B + (int64_t)(k0 + r) * g.sBk + n0, (uint32_t)(sizeof(T) * BN), &full[s]);
      }
      if (!BMAJ) {
#pragma unroll
        for (int r = 0; r < EB; ++r) cp_async_elem<T>(bs + bk[r] * PB + bn[r], B + boff[r] + (int64_t)k0 * g.sBk, true);
      }
    }
    if (!BMAJ) cp_async_commit();   // one group per slab (empty past the end): wait_group counts stay uniform
  };
#pragma unroll
  for (int s = 0; s < NSTAGE - 1; ++s) issue(s);

  for (int kt = 0; kt < nkt; ++kt) {
    if (!BMAJ) cp_async_wait<NSTAGE - 2>();                         // this thread's LDGSTS of slab kt
    mbar_wait(&full[kt % NSTAGE], (uint32_t)((kt / NSTAGE) & 1));   // the copy engine's rows of slab kt
    __syncthreads();                                                // slab kt-1 is no longer being read by anyone
    issue(kt + NSTAGE - 1);
    const T* as = Sm + (size_t)(kt % NSTAGE) * STAGE;
    const T* bs = as + BK * PA;
#pragma unroll
    for (int kk = 0; kk < BK; kk += 4) {
      T af[MT], bf[NTL];
#pragma unroll
      for (int i = 0; i < MT; ++i) af[i] = as[(kk + t4) * PA + wm0 + i * 8 + g8];
#pragma unroll
      for (int j = 0; j < NTL; ++j)
        bf[j] = bs[(kk + t4) * PB + wn0 + j * 8 + g8];
#pragma unroll
      for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < NTL; ++j) acc[i][j].mma(af[i], bf[j]);
    }
  }

  if (!BMAJ) cp_async_wait<0>();
  const bool has_beta = (g.beta != 0.0);
#pragma unroll
  for (int i = 0; i < MT; ++i) {
    const int row = m0 + wm0 + i * 8 + g8;
#pragma unroll
    for (int j = 0; j < NTL; ++j) {
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int col = n0 + wn0 + j * 8 + 2 * t4 + e;
        T* p = C + (int64_t)row * g.sCm + (int64_t)col * g.sCn;
        T v = t_scale(acc[i][j].get(e), g.alpha);
        if (has_beta) v = t_add(v, t_scale(*p, g.beta));
        *p = v;
      }
    }
  }
}

template <class T, int BM, int BN, int WM, int WN, bool BMAJ>
void launch_bulk(const GemmArgs& g) {
  constexpr int PAD = Pad<T>::v;
  const size_t smem = sizeof(T) * NSTAGE * BK * ((BM + PAD) + (BN + PAD));
  auto kern = gemm_bulk_kernel<T, BM, BN, WM, WN, BMAJ>;
  static int attr_dev = -1;
  if (attr_dev != ctx().device) {
    TTN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_dev = ctx().device;
  }
  dim3 grid(g.M / BM, g.N / BN, (unsigned)(g.batch1 * g.batch2));
  kern<<<grid, NT, smem, ctx().stream>>>(g);
  TTN_CHECK_LAUNCH();
  ctx().launches++;
}

// true when the TMA-staged big-tile kernel can serve g (and then launches it)
template <class T, int BM, int BN, int WM, int WN>
bool try_bulk(const GemmArgs& g) {
  if (!ctx().gemm_bulk || g.npeer != 0 || g.conjA || g.conjB) return false;
  if (g.M % BM || g.N % BN || g.K % BK || g.K < BK) return false;
  if ((int64_t)g.batch1 * g.batch2 > 65535 || g.N / BN > 65535) return false;
  const int64_t ev = 16 / (int64_t)sizeof(T);                 // elements per 16 bytes
  auto al = [&](int64_t v) { return v % ev == 0; };
  if (g.sAm != 1 || !al(g.sAk) || !al(g.bA1) || !al(g.bA2) || (reinterpret_cast<uintptr_t>(g.A) & 15)) return false;
  if (!al(g.bB1) || !al(g.bB2) || (reinterpret_cast<uintptr_t>(g.B) & 15)) return false;
  if (g.sBn == 1 && al(g.sBk)) { launch_bulk<T, BM, BN, WM, WN, true>(g); return true; }
  if (g.sBk == 1 && al(g.sBn)) { launch_bulk<T, BM, BN, WM, WN, false>(g); return true; }
  return false;
}

template <class T, int BM, int BN, int WM, int WN, bool AMAJ, bool BMAJ, int NS = NSTAGE>
void launch_cfg(const GemmArgs& g) {
  constexpr int PAD = Pad<T>::v;
  const size_t smem = sizeof(T) * NS * BK * ((BM + PAD) + (BN + PAD));
  auto kern = gemm_kernel<T, BM, BN, WM, WN, AMAJ, BMAJ, NS>;
  static int attr_dev = -1;   // function attributes are per device (ttn_init may re-bind)
  if (attr_dev != ctx().device) {
    TTN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_dev = ctx().device;
  }
  // grid.z is limited to 65535: split the outer batch dimension if needed
  const int64_t max_b2 = std::max<int64_t>(1, 65535 / g.batch1);
  ttn_assert(g.batch1 <= 65535, 2, "gemm: inner batch dimension too large");
  ttn_assert(g.npeer == 0 || g.batch2 <= max_b2, 2, "gemm: peer epilogue needs a single launch");
  for (int64_t s = 0; s < g.batch2; s += max_b2) {
    GemmArgs h = g;
    const int64_t nb2 = std::min<int64_t>(max_b2, g.batch2 - s);
    h.batch2 = (int)nb2;
    const size_t es = sizeof(T);
    h.A = reinterpret_cast<const char*>(g.A) + es * s * g.bA2;
    h.B = reinterpret_cast<const char*>(g.B) + es * s * g.bB2;
    h.C = reinterpret_cast<char*>(g.C) + es * s * g.bC2;
    dim3 grid((g.M + BM - 1) / BM, (g.N + BN - 1) / BN, (unsigned)(g.batch1 * nb2));
    ttn_assert(grid.y <= 65535, 2, "gemm: N too large for grid.y");
    kern<<<grid, NT, smem, ctx().stream>>>(h);
    TTN_CHECK_LAUNCH();
    ctx().launches++;
  }
}

template <class T, int BM, int BN, int WM, int WN, int NS = NSTAGE>
void launch_major(const GemmArgs& g) {
  const bool amaj = std::llabs(g.sAm) <= std::llabs(g.sAk);   // m is the faster index of A in memory
  const bool bmaj = std::llabs(g.sBn) < std::llabs(g.sBk);    // n is the faster index of B in memory
  if (amaj && bmaj) launch_cfg<T, BM, BN, WM, WN, true, true, NS>(g);
  else if (amaj && !bmaj) launch_cfg<T, BM, BN, WM, WN, true, false, NS>(g);
  else if (!amaj && bmaj) launch_cfg<T, BM, BN, WM, WN, false, true, NS>(g);
  else launch_cfg<T, BM, BN, WM, WN, false, false, NS>(g);
}

// ---------------------------------------------------------------------------------------------------------------------
// Thin right-multiplication  C_b (M x N) = alpha A_b (M x K) W (K x N) + beta C_b  with N, K <= 32 and one W for the whole batch:
// the middle contraction of the three-GEMM effective operator (T2 = T1 . W, K = w n^2 = 20 at cfg4) and of the environment
// updates.  It is a streaming operation (2 x 8 bytes moved per 2 K flop): a DMMA tile would idle on 20 of its 64 columns, so each
// thread keeps one row of A_b in registers (loads coalesced along M), W sits in shared memory (broadcast reads) and the row of C
// goes back coalesced.  Bound: HBM bandwidth.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int THIN_MAX = 32;
// KT = compile-time bound on K (registers), ROWS = rows of A per thread (every W value read from shared memory is used ROWS times)
template <class T, int KT, int ROWS>
__global__ void __launch_bounds__(256) gemm_thin_kernel(const GemmArgs g) {
  __shared__ __align__(16) T Ws[THIN_MAX * KT];
  const int K = g.K, N = g.N;
  const T* __restrict__ Bp = reinterpret_cast<const T*>(g.B);
  for (int idx = threadIdx.x; idx < KT * N; idx += blockDim.x) {
    const int k = idx % KT, n = idx / KT;
    T w = t_zero<T>();
    if (k < K) {
      w = Bp[k * g.sBk + n * g.sBn];
      if (g.conjB) w = t_conj(w);
    }
    Ws[n * KT + k] = w;                      // zero padding up to KT: the inner loop needs no bound checks
  }
  __syncthreads();
  const int m0 = blockIdx.x * (256 * ROWS) + threadIdx.x;
  const int b = blockIdx.y, b1 = b % g.batch1, b2 = b / g.batch1;
  const T* __restrict__ A = reinterpret_cast<const T*>(g.A) + b1 * g.bA1 + b2 * g.bA2;
  T* __restrict__ C = reinterpret_cast<T*>(g.C) + b1 * g.bC1 + b2 * g.bC2;
  T x[ROWS][KT];
#pragma unroll
  for (int r = 0; r < ROWS; ++r) {
    const int m = m0 + 256 * r;
#pragma unroll
    for (int k = 0; k < KT; ++k) x[r][k] = (k < K && m < g.M) ? A[m + k * g.sAk] : t_zero<T>();
  }
  for (int n = 0; n < N; ++n) {
    T acc[ROWS][2];
#pragma unroll
    for (int r = 0; r < ROWS; ++r) acc[r][0] = acc[r][1] = t_zero<T>();
    const T* w = Ws + n * KT;
#pragma unroll
    for (int k = 0; k < KT; k += 2) {
      const T w0 = w[k], w1 = w[k + 1];      // 16-byte aligned pair: one LDS.128 for Float64
#pragma unroll
      for (int r = 0; r < ROWS; ++r) { t_fma(acc[r][0], x[r][k], w0); t_fma(acc[r][1], x[r][k + 1], w1); }
    }
#pragma unroll
    for (int r = 0; r < ROWS; ++r) {
      const int m = m0 + 256 * r;
      if (m >= g.M) continue;
      T v = t_scale(t_add(acc[r][0], acc[r][1]), g.alpha);
      if (g.beta != 0.0) v = t_add(v, t_scale(C[m + n * g.sCn], g.beta));
      C[m + n * g.sCn] = v;
    }
  }
}

template <class T, int KT, int ROWS>
void launch_thin(const GemmArgs& g) {
  dim3 grid((g.M + 256 * ROWS - 1) / (256 * ROWS), (unsigned)((int64_t)g.batch1 * g.batch2));
  gemm_thin_kernel<T, KT, ROWS><<<grid, 256, 0, ctx().stream>>>(g);
  TTN_CHECK_LAUNCH();
  ctx().launches++;
}

template <class T>
bool try_thin(const GemmArgs& g) {
  if (g.N > THIN_MAX || g.K > THIN_MAX || g.M < 256 || g.npeer != 0 || g.conjA) return false;
  if (g.sAm != 1 || g.sCm != 1 || g.bB1 != 0 || g.bB2 != 0) return false;
  if ((int64_t)g.batch1 * g.batch2 > 65535) return false;
  constexpr int R = is_cplx<T>::value ? 1 : 2;      // register budget: ROWS * KT values of T per thread
  if (g.K <= 8) launch_thin<T, 8, R>(g);
  else if (g.K <= 16) launch_thin<T, 16, R>(g);
  else if (g.K <= 24) launch_thin<T, 24, R>(g);
  else launch_thin<T, 32, 1>(g);
  return true;
}

}  // namespace

template <class T>
void gemm(const GemmArgs& g) {
  if (g.M <= 0 || g.N <= 0 || g.batch1 <= 0 || g.batch2 <= 0) return;
  ProfScope prof_scope_(KF_GEMM);
  constexpr bool cplx = is_cplx<T>::value;
  ctx().flops_gemm += gemm_flops(g, cplx);
  // a "big" product fills 3/4 of a 128 x 128 (Float64) / 64 x 128 (ComplexF64) tile and, with such tiles, 3/4 of the SMs
  constexpr int BIGM = cplx ? 64 : 128, BIGN = 128;
  const int64_t ctas_big = (int64_t)((g.M + BIGM - 1) / BIGM) * ((g.N + BIGN - 1) / BIGN) * g.batch1 * g.batch2;
  const bool big = g.M >= (BIGM * 3) / 4 && g.N >= (BIGN * 3) / 4 && ctas_big >= (int64_t)(ctx().sm_count * 3) / 4;
  if (ctx().gemm_thin && try_thin<T>(g)) return;
  if (g.npeer != 0) {
    // fused all-gather epilogue (two or more GPUs): four-stage tiles, one CTA per SM on the big ones
    if (!big) launch_major<T, 64, 64, 32, 16>(g);
    else if constexpr (cplx) launch_major<zc, 64, 128, 32, 32>(g);
    else launch_major<double, 128, 128, 64, 32>(g);
  } else if constexpr (cplx) {
    // 64 x 64 tile, two pipeline stages: 68 KB of shared memory and 32 K registers per CTA, so that one such CTA fits on an SM next
    // to a CTA of the (latency-bound, 132 KB) ComplexF64 tridiagonalisation kernel of another stream
    launch_major<zc, 64, 64, 32, 16, 2>(g);
  } else if (big) {
    // 128 x 64 tile at two CTAs per SM: TMA-staged when the operands allow it, else three LDGSTS stages
    if (!try_bulk<double, 128, 64, 32, 32>(g)) launch_major<double, 128, 64, 32, 32, 3>(g);
  } else {
    launch_major<double, 64, 64, 32, 16>(g);
  }
}

template void gemm<double>(const GemmArgs&);
template void gemm<zc>(const GemmArgs&);

double gemm_flops(const GemmArgs& g, bool cplx) {
  return (cplx ? 8.0 : 2.0) * (double)g.M * (double)g.N * (double)g.K * (double)g.batch1 * (double)g.batch2;
}

}  // namespace ttn
