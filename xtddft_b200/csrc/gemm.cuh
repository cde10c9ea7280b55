// FP64 tensor-core GEMM for the sigma path: DMMA (mma.sync m8n8k4 f64 -> SASS DMMA.8x8x4, the only FP64
// MMA shape sm_100a executes natively; tcgen05 has no f64 kind) fed by a TMA (cp.async.bulk.tensor) +
// mbarrier multi-stage pipeline with one producer warp and eight consumer warps per CTA.
//
//   C[zb] (+)= alpha * sum_{s < nouter} opA(A[qa(zb)+s]) * opB(B[qb(zb)+s])^T
//
// Operands are 3-level strided views (q-slice, row, contiguous column).  Each operand is either
// K-contiguous (the contraction index is the contiguous one: "row-major M x K") or K-strided (the
// contraction index is the row index: "row-major K x M").  The second contraction level (q) lets one launch
// accumulate over e.g. all auxiliary functions P of a density-fitting block:  sum_P sum_b U[P,i,b] L[P,a,b].
//
// Tile 128x128x16 doubles, 6 stages of 32 KB, warp tile 64x32 (8x4 DMMA tiles, 64 accumulator doubles per
// thread).  Shared-memory tiles are written by TMA with the 128-byte swizzle; fragment loads undo it.
// Measured ceiling on B200 for this instruction mix: 37.1 TFLOP/s (profiles/fp64_peaks_r01.json).
#pragma once
#include "common.cuh"

namespace xtd {

constexpr int BM = 128, BN = 128, BK = 16;
constexpr int STAGES = 6;
constexpr int CONSUMER_WARPS = 8;
constexpr int GEMM_THREADS = (CONSUMER_WARPS + 1) * 32;
constexpr int TILE_BYTES_A = BM * BK * 8;   // 16 KB
constexpr int TILE_BYTES_B = BN * BK * 8;   // 16 KB
constexpr int STAGE_BYTES = TILE_BYTES_A + TILE_BYTES_B;
constexpr int GEMM_SMEM = STAGES * STAGE_BYTES + 1024 /*alignment slack*/ + 2 * STAGES * 8;

struct MatView {
  const double* base = nullptr;  // tensor base (16-byte aligned)
  long ld = 0;                   // row stride (elements, even)
  long sq = 0;                   // q-slice stride (elements, even); ignored when nq == 1
  int row0 = 0, col0 = 0;        // view offset inside a slice
  int rows = 0, cols = 0;        // view extent
  int q0 = 0, nq = 1;            // slice range
};

struct GemmDesc {
  MatView A, B;
  bool a_kc = true, b_kc = true;   // operand is K-contiguous?
  int M = 0, N = 0, K = 0;
  int nouter = 1;                  // second-level contraction steps (q advances by one per step)
  int batches = 1;                 // independent outputs (grid.z)
  int z_div = 1;                   // batch zb -> (hi, lo) = (zb / z_div, zb % z_div)
  int a_hi = 0, a_lo = 0;          // qa(zb) = A.q0 + hi*a_hi + lo*a_lo
  int b_hi = 0, b_lo = 0;
  double* C = nullptr;
  long ldc = 0;
  long c_batch_stride = 0;
  double alpha = 1.0;
  bool accumulate = false;         // C += instead of C =
  int splits = 0;                  // split of the (nouter x ktiles) iteration space; 0 = choose
  // optional two-level output rows: row m lives at (m / c_row_div) * c_row_hi + (m % c_row_div) * c_row_lo
  // (elements; both even) instead of m * ldc.  c_row_div == 0: plain rows.
  int c_row_div = 0;
  long c_row_hi = 0, c_row_lo = 0;
};

struct GemmKernelParams {
  int M, N, K, nouter;
  int a_row0, a_k0, b_row0, b_k0;
  int z_div, a_q0, a_hi, a_lo, b_q0, b_hi, b_lo;
  int splits;
  double* C;
  long ldc, c_batch_stride, c_split_stride;
  double alpha;
  int accumulate;
  int c_row_div;
  long c_row_hi, c_row_lo;
  int m_tail_cfg, n_tail_cfg;      // warp layout of the last (partial) tile row / column: 0 = the main 128 x 128 layout
};

__host__ __device__ __forceinline__ long c_row_offset(int m, long ldc, int div, long hi, long lo) {
  return div ? (long)(m / div) * hi + (long)(m % div) * lo : (long)m * ldc;
}

// ------------------------------------------------------------------------------------------------------
// PTX helpers
// ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t addr, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(addr), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  while (!mbar_try_wait(addr, parity)) {
  }
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, int c0, int c1, int c2, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}
__device__ __forceinline__ double lds_f64(uint32_t addr) {
  double v;
  asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
  return v;
}

// byte offset of element (r = M/N index within the 128-wide tile, k = 0..15) inside a swizzled stage tile
template <bool KC>
__device__ __forceinline__ uint32_t frag_off(int r, int k) {
  if (KC) {  // one TMA box [128 rows][16 k]: row pitch 128 B, 16-byte chunks XOR (row & 7)
    return (uint32_t)(r * 128 + ((((k >> 1) ^ (r & 7)) & 7) << 4) + ((k & 1) << 3));
  } else {   // eight TMA boxes [16 k rows][16 m]: box (r>>4) of 2 KB, row pitch 128 B, chunk XOR (k & 7)
    int rl = r & 15;
    return (uint32_t)((r >> 4) * 2048 + k * 128 + ((((rl >> 1) ^ (k & 7)) & 7) << 4) + ((rl & 1) << 3));
  }
}

// ------------------------------------------------------------------------------------------------------
// the kernel
// ------------------------------------------------------------------------------------------------------
// IT x JT DMMA tiles per warp (warp tile 8 IT x 8 JT), WM warps along M and 8 / WM along N.  The main layout <8, 4, 2>
// covers the 128 x 128 CTA tile; the others cover a partial last tile with all eight warps instead of leaving most of them
// multiplying zero padding:  <4,4,4> 128 x 64 and <2,4,8> 128 x 32 for a short N tail,  <8,2,1> 64 x 128 and <2,2,1> 16 x 128
// for a short M tail.  TMA still fetches full boxes (rows past the view are zero-filled, no traffic); the CTAs of partial
// tiles sit in the same grid as the full ones and fill the gaps of the last wave.
template <bool A_KC, bool B_KC, int IT, int JT, int WM>
__device__ __forceinline__ void dmma_consume(const GemmKernelParams& p, uint8_t* smem, uint64_t* full, uint64_t* empty, int warp, int lane,
                                             int tile_m, int tile_n, int zb, int sp, long it0, long it1) {
  const int g = lane >> 2, t = lane & 3;
  const int wm = (warp % WM) * (8 * IT), wn = (warp / WM) * (8 * JT);
  // K-strided operand tiles: fragment address = one lane-dependent register + a compile-time constant per (i, kk); the
  // swizzle XOR is split into its lane bits and its (i, kk) bits by hand (left to the compiler these variants spilled):
  //   frag_off<false>(r, k) = (r>>4)*2048 + k*128 + ((((r&15)>>1) ^ (k&7)) << 4) + ((r&1) << 3),   r = w + 8 i + g,  k = 4 kk + t
  //     = [(w>>4)*2048 + t*128 + (((g>>1)^t) << 4) + ((g&1)<<3)]  +  (i>>1)*2048 + kk*512 + (((i&1)^(kk&1)) << 6)
  // (warp tiles start on multiples of 16 rows in every layout).  K-contiguous tiles keep frag_off<true>.
  const uint32_t a_lane = (uint32_t)((wm >> 4) * 2048 + t * 128 + ((((g >> 1) ^ t) & 3) << 4) + ((g & 1) << 3));
  const uint32_t b_lane = (uint32_t)((wn >> 4) * 2048 + t * 128 + ((((g >> 1) ^ t) & 3) << 4) + ((g & 1) << 3));
  double acc[IT][JT][2];
#pragma unroll
  for (int i = 0; i < IT; ++i)
#pragma unroll
    for (int j = 0; j < JT; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

  const uint32_t smem_base = smem_u32(smem);
  for (long it = it0; it < it1; ++it) {
    const long rel = it - it0;
    const int s = (int)(rel % STAGES);
    const uint32_t ph = (uint32_t)((rel / STAGES) & 1);
    mbar_wait(&full[s], ph);
    const uint32_t sa = smem_base + s * STAGE_BYTES;
    const uint32_t sb = sa + TILE_BYTES_A;
#pragma unroll
    for (int kk = 0; kk < BK / 4; ++kk) {
      double a[IT], b[JT];
#pragma unroll
      for (int i = 0; i < IT; ++i)
        a[i] = A_KC ? lds_f64(sa + frag_off<true>(wm + i * 8 + g, kk * 4 + t))
                    : lds_f64(sa + a_lane + ((i >> 1) * 2048 + kk * 512 + (((i & 1) ^ (kk & 1)) << 6)));
#pragma unroll
      for (int j = 0; j < JT; ++j)
        b[j] = B_KC ? lds_f64(sb + frag_off<true>(wn + j * 8 + g, kk * 4 + t))
                    : lds_f64(sb + b_lane + ((j >> 1) * 2048 + kk * 512 + (((j & 1) ^ (kk & 1)) << 6)));
#pragma unroll
      for (int i = 0; i < IT; ++i)
#pragma unroll
        for (int j = 0; j < JT; ++j) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty[s]);
  }

  // ===================== epilogue: registers -> global (16-byte stores) =====================
  double* C = p.C + (long)zb * p.c_batch_stride + (long)sp * p.c_split_stride;
  const int m_base = tile_m * BM + wm, n_base = tile_n * BN + wn;
#pragma unroll
  for (int i = 0; i < IT; ++i) {
    const int m = m_base + i * 8 + g;
    if (m >= p.M) continue;
    double* crow = C + c_row_offset(m, p.ldc, p.c_row_div, p.c_row_hi, p.c_row_lo);
#pragma unroll
    for (int j = 0; j < JT; ++j) {
      const int n = n_base + j * 8 + 2 * t;
      if (n >= p.N) continue;
      double v0 = p.alpha * acc[i][j][0], v1 = p.alpha * acc[i][j][1];
      if (n + 1 < p.N) {
        double2* dst = reinterpret_cast<double2*>(crow + n);
        if (p.accumulate) {
          double2 old = *dst;
          v0 += old.x;
          v1 += old.y;
        }
        *dst = make_double2(v0, v1);
      } else {
        if (p.accumulate) v0 += crow[n];
        crow[n] = v0;
      }
    }
  }
}

template <bool A_KC, bool B_KC, bool TAILS>
__global__ void __launch_bounds__(GEMM_THREADS, 1)   // 9 warps are allocated as 12 (granularity 4): 168 registers per thread
dgemm_dmma_tma_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                      const GemmKernelParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* full = (uint64_t*)(smem + STAGES * STAGE_BYTES);
  uint64_t* empty = full + STAGES;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tile_m = blockIdx.x, tile_n = blockIdx.y;
  const int zb = blockIdx.z / p.splits, sp = blockIdx.z - zb * p.splits;
  const int ktiles = (p.K + BK - 1) / BK;
  const long total = (long)p.nouter * ktiles;
  const long it0 = total * sp / p.splits, it1 = total * (sp + 1) / p.splits;
  const int hi = zb / p.z_div, lo = zb - hi * p.z_div;
  const int qa = p.a_q0 + hi * p.a_hi + lo * p.a_lo;
  const int qb = p.b_q0 + hi * p.b_hi + lo * p.b_lo;

  if (threadIdx.x == CONSUMER_WARPS * 32) {   // the producer lane: fetch both tensor maps while the barriers are set up
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmB)) : "memory");
  }
  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], CONSUMER_WARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();

  if (warp == CONSUMER_WARPS) {
    // ===================== TMA producer (one elected lane) =====================
    if (lane == 0) {
      for (long it = it0; it < it1; ++it) {
        const long rel = it - it0;
        const int s = (int)(rel % STAGES);
        const uint32_t ph = (uint32_t)((rel / STAGES) & 1);
        mbar_wait(&empty[s], ph ^ 1u);
        mbar_expect_tx(&full[s], STAGE_BYTES);
        const int so = (int)(it / ktiles);
        const int k = (int)(it - (long)so * ktiles) * BK;
        uint8_t* sa = smem + s * STAGE_BYTES;
        uint8_t* sb = sa + TILE_BYTES_A;
        if (A_KC) {
          tma_load_3d(sa, &tmA, p.a_k0 + k, p.a_row0 + tile_m * BM, qa + so, &full[s]);
        } else {
#pragma unroll
          for (int b = 0; b < BM / 16; ++b)
            tma_load_3d(sa + b * 2048, &tmA, p.a_row0 + tile_m * BM + b * 16, p.a_k0 + k, qa + so, &full[s]);
        }
        if (B_KC) {
          tma_load_3d(sb, &tmB, p.b_k0 + k, p.b_row0 + tile_n * BN, qb + so, &full[s]);
        } else {
#pragma unroll
          for (int b = 0; b < BN / 16; ++b)
            tma_load_3d(sb + b * 2048, &tmB, p.b_row0 + tile_n * BN + b * 16, p.b_k0 + k, qb + so, &full[s]);
        }
      }
    }
    return;
  }

  // ===================== DMMA consumers: warp layout by tile position =====================
  if (!TAILS) {   // no short last tile in this launch: the main layout only
    dmma_consume<A_KC, B_KC, 8, 4, 2>(p, smem, full, empty, warp, lane, tile_m, tile_n, zb, sp, it0, it1);
    return;
  }
  const int mcfg = (tile_m == (int)gridDim.x - 1) ? p.m_tail_cfg : 0;
  const int ncfg = (tile_n == (int)gridDim.y - 1) ? p.n_tail_cfg : 0;
  if (mcfg == 3) dmma_consume<A_KC, B_KC, 8, 2, 1>(p, smem, full, empty, warp, lane, tile_m, tile_n, zb, sp, it0, it1);
  else if (mcfg == 4) dmma_consume<A_KC, B_KC, 2, 2, 1>(p, smem, full, empty, warp, lane, tile_m, tile_n, zb, sp, it0, it1);
  else if (ncfg == 1) dmma_consume<A_KC, B_KC, 4, 4, 4>(p, smem, full, empty, warp, lane, tile_m, tile_n, zb, sp, it0, it1);
  else if (ncfg == 2) dmma_consume<A_KC, B_KC, 2, 4, 8>(p, smem, full, empty, warp, lane, tile_m, tile_n, zb, sp, it0, it1);
  else dmma_consume<A_KC, B_KC, 8, 4, 2>(p, smem, full, empty, warp, lane, tile_m, tile_n, zb, sp, it0, it1);
}

// ------------------------------------------------------------------------------------------------------
// naive checker kernel (one thread per output element).  Debug / validation only: selected with
// XTD_GEMM=naive; never used on the measured path.
// ------------------------------------------------------------------------------------------------------
struct NaiveParams {
  const double *A, *B;
  long lda, sqa, ldb, sqb;
  int a_kc, b_kc;
  int a_row0, a_col0, b_row0, b_col0;
  GemmKernelParams g;
};
__global__ void dgemm_naive_kernel(const NaiveParams q) {
  const GemmKernelParams& p = q.g;
  int n = blockIdx.x * blockDim.x + threadIdx.x;
  int m = blockIdx.y * blockDim.y + threadIdx.y;
  int zb = blockIdx.z;
  if (m >= p.M || n >= p.N) return;
  int hi = zb / p.z_div, lo = zb - hi * p.z_div;
  long qa = p.a_q0 + hi * p.a_hi + lo * p.a_lo, qb = p.b_q0 + hi * p.b_hi + lo * p.b_lo;
  double acc = 0.0;
  for (int s = 0; s < p.nouter; ++s) {
    const double* A = q.A + (qa + s) * q.sqa;
    const double* B = q.B + (qb + s) * q.sqb;
    for (int k = 0; k < p.K; ++k) {
      double a = q.a_kc ? A[(long)(q.a_row0 + m) * q.lda + q.a_col0 + k] : A[(long)(q.a_row0 + k) * q.lda + q.a_col0 + m];
      double b = q.b_kc ? B[(long)(q.b_row0 + n) * q.ldb + q.b_col0 + k] : B[(long)(q.b_row0 + k) * q.ldb + q.b_col0 + n];
      acc = fma(a, b, acc);
    }
  }
  double* c = p.C + (long)zb * p.c_batch_stride + c_row_offset(m, p.ldc, p.c_row_div, p.c_row_hi, p.c_row_lo) + n;
  *c = p.alpha * acc + (p.accumulate ? *c : 0.0);
}

// C (+)= sum_s partial[s]   (deterministic split-K reduction)
__global__ void reduce_splits_kernel(double* __restrict__ C, long ldc, long c_batch_stride, const double* __restrict__ part,
                                     long ldp, long p_batch_stride, long p_split_stride, int splits, int M, int N,
                                     int accumulate, int row_div, long row_hi, long row_lo) {
  const int zb = blockIdx.y;
  const long total = (long)M * N;
  for (long e = (long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long)gridDim.x * blockDim.x) {
    const long m = e / N;
    const int n = (int)(e - m * N);
    const double* src = part + (long)zb * p_batch_stride + m * ldp + n;
    double acc = 0.0;
    for (int s = 0; s < splits; ++s) acc += src[(long)s * p_split_stride];
    double* dst = C + (long)zb * c_batch_stride + c_row_offset((int)m, ldc, row_div, row_hi, row_lo) + n;
    *dst = acc + (accumulate ? *dst : 0.0);
  }
}

// ------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

struct GemmContext {
  PFN_encodeTiled encode = nullptr;
  int num_sms = 148;
  bool naive = false;        // XTD_GEMM=naive
  double* split_ws = nullptr;  // workspace for split-K partials
  size_t split_ws_bytes = 0;
  // statistics
  double flops = 0.0;        // executed useful flops (2*M*N*K*nouter*batches)
  unsigned long long launches = 0;
};

inline int gemm_context_init(GemmContext& ctx) {
  if (!ctx.encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    XTD_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    XTD_REQUIRE(fn != nullptr && qres == cudaDriverEntryPointSuccess, XTD_ERR_CUDA, "cuTensorMapEncodeTiled not available");
    ctx.encode = (PFN_encodeTiled)fn;
  }
  int dev = 0;
  XTD_CUDA(cudaGetDevice(&dev));
  XTD_CUDA(cudaDeviceGetAttribute(&ctx.num_sms, cudaDevAttrMultiProcessorCount, dev));
  const char* e = getenv("XTD_GEMM");
  ctx.naive = (e && e[0] == 'n');
  return XTD_OK;
}

template <bool A_KC, bool B_KC, bool TAILS>
inline int launch_kernel(dim3 grd, cudaStream_t stream, const CUtensorMap& ma, const CUtensorMap& mb, const GemmKernelParams& kp) {
  static bool attr_set[64] = {false};      // the opt-in is per device
  int dev = 0;
  XTD_CUDA(cudaGetDevice(&dev));
  if (!attr_set[dev & 63]) {
    XTD_CUDA(cudaFuncSetAttribute(dgemm_dmma_tma_kernel<A_KC, B_KC, TAILS>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM));
    attr_set[dev & 63] = true;
  }
  dgemm_dmma_tma_kernel<A_KC, B_KC, TAILS><<<grd, GEMM_THREADS, GEMM_SMEM, stream>>>(ma, mb, kp);
  XTD_COUNT_LAUNCH();
  XTD_CUDA(cudaGetLastError());
  return XTD_OK;
}

// Tensor map of a view, clipped at the view's end in every dimension so out-of-view reads are zero-filled.
inline int make_tensor_map(const GemmContext& ctx, const MatView& v, bool kc, CUtensorMap* out) {
  XTD_REQUIRE(((uintptr_t)v.base & 15) == 0, XTD_ERR_ALIGN, "tensor base %p not 16-byte aligned", (const void*)v.base);
  XTD_REQUIRE(v.ld % 2 == 0 && v.ld > 0, XTD_ERR_ALIGN, "leading dimension %ld must be even", v.ld);
  // measured on B200: a TMA box whose innermost start coordinate is odd (8-byte aligned fp64) raises
  // "illegal instruction"; contiguous-dimension view offsets must be even (16-byte aligned)
  XTD_REQUIRE(v.col0 % 2 == 0, XTD_ERR_ALIGN, "contiguous-dimension view offset %d must be even", v.col0);
  XTD_REQUIRE(v.nq == 1 || (v.sq % 2 == 0 && v.sq > 0), XTD_ERR_ALIGN, "slice stride %ld must be even", v.sq);
  cuuint64_t dims[3] = {(cuuint64_t)(v.col0 + v.cols), (cuuint64_t)(v.row0 + v.rows), (cuuint64_t)(v.q0 + v.nq)};
  long sq = (v.nq == 1 && v.sq == 0) ? v.ld * (long)dims[1] : v.sq;
  if (sq <= 0) sq = v.ld * (long)dims[1];
  cuuint64_t strides[2] = {(cuuint64_t)v.ld * 8ull, (cuuint64_t)sq * 8ull};
  cuuint32_t box[3] = {16u, kc ? 128u : 16u, 1u};
  cuuint32_t estr[3] = {1u, 1u, 1u};
  CUresult r = ctx.encode(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, (void*)v.base, dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  XTD_REQUIRE(r == CUDA_SUCCESS, XTD_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d): dims %llu %llu %llu ld %ld sq %ld", (int)r,
              (unsigned long long)dims[0], (unsigned long long)dims[1], (unsigned long long)dims[2], v.ld, sq);
  return XTD_OK;
}

inline int gemm(GemmContext& ctx, const GemmDesc& d, cudaStream_t stream) {
  if (d.M <= 0 || d.N <= 0 || d.batches <= 0) return XTD_OK;
  XTD_REQUIRE(d.C != nullptr, XTD_ERR_ARG, "gemm: null C");
  if (d.K <= 0 || d.nouter <= 0) {
    // empty contraction: C = 0 unless accumulating
    if (!d.accumulate)
      for (int z = 0; z < d.batches; ++z)
        XTD_CUDA(cudaMemset2DAsync(d.C + (long)z * d.c_batch_stride, d.ldc * 8, 0, (size_t)d.N * 8, d.M, stream));
    return XTD_OK;
  }
  // views must describe the same logical operands the kernel will read
  XTD_REQUIRE((d.a_kc ? d.A.rows : d.A.cols) == d.M && (d.a_kc ? d.A.cols : d.A.rows) == d.K, XTD_ERR_ARG,
              "gemm: A view %dx%d inconsistent with M=%d K=%d", d.A.rows, d.A.cols, d.M, d.K);
  XTD_REQUIRE((d.b_kc ? d.B.rows : d.B.cols) == d.N && (d.b_kc ? d.B.cols : d.B.rows) == d.K, XTD_ERR_ARG,
              "gemm: B view %dx%d inconsistent with N=%d K=%d", d.B.rows, d.B.cols, d.N, d.K);
  GemmKernelParams p;
  p.M = d.M; p.N = d.N; p.K = d.K; p.nouter = d.nouter;
  p.a_row0 = d.a_kc ? d.A.row0 : d.A.col0;   // M-offset
  p.a_k0 = d.a_kc ? d.A.col0 : d.A.row0;     // K-offset
  p.b_row0 = d.b_kc ? d.B.row0 : d.B.col0;
  p.b_k0 = d.b_kc ? d.B.col0 : d.B.row0;
  p.z_div = d.z_div < 1 ? 1 : d.z_div;
  p.a_q0 = d.A.q0; p.a_hi = d.a_hi; p.a_lo = d.a_lo;
  p.b_q0 = d.B.q0; p.b_hi = d.b_hi; p.b_lo = d.b_lo;
  p.C = d.C; p.ldc = d.ldc; p.c_batch_stride = d.c_batch_stride; p.c_split_stride = 0;
  p.alpha = d.alpha; p.accumulate = d.accumulate ? 1 : 0; p.splits = 1;
  p.c_row_div = d.c_row_div; p.c_row_hi = d.c_row_hi; p.c_row_lo = d.c_row_lo;
  p.m_tail_cfg = 0; p.n_tail_cfg = 0;
  XTD_REQUIRE(d.c_row_div == 0 || (d.c_row_hi % 2 == 0 && d.c_row_lo % 2 == 0), XTD_ERR_ALIGN, "gemm: split row strides must be even");
  ctx.flops += 2.0 * d.M * d.N * (double)d.K * d.nouter * d.batches;

  if (ctx.naive) {
    NaiveParams q;
    q.A = d.A.base; q.B = d.B.base; q.lda = d.A.ld; q.ldb = d.B.ld; q.sqa = d.A.sq; q.sqb = d.B.sq;
    q.a_kc = d.a_kc; q.b_kc = d.b_kc;
    q.a_row0 = d.A.row0; q.a_col0 = d.A.col0; q.b_row0 = d.B.row0; q.b_col0 = d.B.col0;
    q.g = p;
    dim3 blk(32, 8), grd((unsigned)cdiv(d.N, 32), (unsigned)cdiv(d.M, 8), d.batches);
    dgemm_naive_kernel<<<grd, blk, 0, stream>>>(q);
    XTD_COUNT_LAUNCH(); ctx.launches++;
    XTD_CUDA(cudaGetLastError());
    return XTD_OK;
  }

  const int tm = (int)cdiv(d.M, BM), tn = (int)cdiv(d.N, BN);
  XTD_REQUIRE(tn <= 65535, XTD_ERR_ARG, "gemm: N too large for grid.y");
  const long ktiles = cdiv(d.K, BK);
  const long total_it = ktiles * d.nouter;
  int splits = d.splits;
  if (splits <= 0) {
    // Choose the split of the (nouter x ktiles) iteration space that minimises
    //   waves(tiles*s) * (iterations per unit + fixed per-unit overhead)
    // i.e. trade wave quantisation on 148 SMs against pipeline fill / epilogue / partial-sum traffic.
    const long tiles = (long)tm * tn * d.batches;
    const double ovh = 4.0;
    long max_s = total_it / 64;      // (a split costs a second launch for the reduction: not worth it below ~64 iterations per unit)
    if (max_s > 64) max_s = 64;
    if (max_s > 65535 / d.batches) max_s = 65535 / d.batches;
    if (max_s < 1) max_s = 1;
    double best_cost = 1e300;
    splits = 1;
    for (long s = 1; s <= max_s; ++s) {
      const long units = tiles * s;
      const long waves = cdiv(units, ctx.num_sms);
      const double cost = (double)waves * ((double)total_it / (double)s + ovh + (s > 1 ? 1.0 : 0.0));
      if (cost < best_cost * 0.98) {  // prefer fewer splits unless clearly better
        best_cost = cost;
        splits = (int)s;
      }
    }
  }
  if (splits > total_it) splits = (int)total_it;
  // the split partials need workspace; fall back to fewer splits if it does not fit
  long part_ld = pad_ld(d.N);
  long part_batch = (long)d.M * part_ld;
  if (splits > 1) {
    size_t need = (size_t)splits * d.batches * part_batch * 8;
    if (need > ctx.split_ws_bytes) {
      long fit = (long)(ctx.split_ws_bytes / ((size_t)d.batches * part_batch * 8));
      splits = fit >= 2 ? (int)fit : 1;
    }
  }
  XTD_REQUIRE((long)d.batches * splits <= 65535, XTD_ERR_ARG, "gemm: batches*splits %ld exceeds grid.z", (long)d.batches * splits);
  p.splits = splits;
  GemmKernelParams kp = p;
  if (splits > 1) {
    kp.C = ctx.split_ws;
    kp.ldc = part_ld;
    kp.c_split_stride = part_batch;
    kp.c_batch_stride = part_batch * splits;
    kp.accumulate = 0;
    kp.alpha = d.alpha;
    kp.c_row_div = 0;
  }
  CUtensorMap ma, mb;
  XTD_TRY(make_tensor_map(ctx, d.A, d.a_kc, &ma));
  XTD_TRY(make_tensor_map(ctx, d.B, d.b_kc, &mb));
  XTD_REQUIRE(((uintptr_t)kp.C & 15) == 0 && kp.ldc % 2 == 0 && kp.c_batch_stride % 2 == 0, XTD_ERR_ALIGN,
              "gemm: C must be 16-byte aligned with even ldc");
  // A short last tile in M or N (<= 64 of 128) gets a warp layout that covers only its live part (dmma_consume).
  const int m_tail = d.M % BM, n_tail = d.N % BN;
  if (m_tail > 0 && m_tail <= 64) kp.m_tail_cfg = m_tail <= 16 ? 4 : 3;
  if (n_tail > 0 && n_tail <= 64) kp.n_tail_cfg = n_tail <= 32 ? 2 : 1;
  const dim3 grd(tm, tn, (unsigned)(d.batches * splits));
  const bool tails = kp.m_tail_cfg || kp.n_tail_cfg;
#define XTD_LAUNCH(AK, BK_)                                                        \
  do {                                                                             \
    if (tails) XTD_TRY((launch_kernel<AK, BK_, true>(grd, stream, ma, mb, kp)));   \
    else XTD_TRY((launch_kernel<AK, BK_, false>(grd, stream, ma, mb, kp)));        \
  } while (0)
  if (d.a_kc && d.b_kc) XTD_LAUNCH(true, true);
  else if (d.a_kc && !d.b_kc) XTD_LAUNCH(true, false);
  else if (!d.a_kc && d.b_kc) XTD_LAUNCH(false, true);
  else XTD_LAUNCH(false, false);
#undef XTD_LAUNCH
  ctx.launches++;
  if (splits > 1) {
    long nblk = cdiv((long)d.M * d.N, 256);
    dim3 rg((unsigned)(nblk > 4096 ? 4096 : nblk), d.batches);
    reduce_splits_kernel<<<rg, 256, 0, stream>>>(d.C, d.ldc, d.c_batch_stride, ctx.split_ws, part_ld, part_batch * splits,
                                                 part_batch, splits, d.M, d.N, d.accumulate ? 1 : 0, d.c_row_div, d.c_row_hi,
                                                 d.c_row_lo);
    XTD_COUNT_LAUNCH(); ctx.launches++;
    XTD_CUDA(cudaGetLastError());
  }
  return XTD_OK;
}

}  // namespace xtd
