// The joint's optional pre-projections (rnnt/joint.py:8-12, 26-30: audio_ln / text_ln, used by the non-"convjs" configs)
// as a tcgen05 prologue GEMM inside the library, with their backward:
//   forward   y[M,N]  = x[M,K] . W[N,K]^T + bias[N]            (M = B*T or B*(U+1), K = features, N = hidden)
//   d-input   dx[M,K] = dy[M,N] . W[N,K]
//   d-weight  dW[N,K] = dy[M,N]^T . x[M,K]     db[N] = column sums of dy
// One generic kernel, D[m,n] = sum_k A(m,k) B(n,k) with each operand either K-major (row-major [rows][k]) or MN-major
// (row-major [k][rows]), so all three contractions read the SAME fp16 copies of x, W and dy through different TMA
// views -- no transposed copies.  Operands are rounded to fp16 (RN, one elementwise pass; the joint GEMM rounds
// tanh(enc + pred) to fp16 right afterwards anyway), accumulation is fp32 in TMEM.
//
// Persistent single-CTA tiles of 128 x 128 (cta_group::1): warp 0 TMA loader (4-stage ring of 16 KB + 16 KB), warp 1
// tcgen05.mma issuer with two ping-pong accumulators, warps 2-5 epilogue (thread = output row; bias, fp32 stores, or
// vector reductions when the contraction is split over CTAs).  These GEMMs are ~1 % of the step (27 GFLOP each at the
// bench shape), so the kernel favours generality (any M, N; K % 8 == 0) over the last 20 % of tensor-pipe rate.
#include <algorithm>

#include "kernels.h"
#include "tc_kernel.cuh"

namespace rb {
namespace {

constexpr int kLinStages = 4;
constexpr int kLinTile = 128;
constexpr int kLinBytes = kLinTile * kBK * 2;        // 16 KB per operand tile (128 rows x 64 k, fp16)
constexpr int kLinThreads = 192;
constexpr int kLinTmemCols = 256;                    // two 128-column fp32 accumulators

struct LinSmem {
  static constexpr int a_ring = 0;
  static constexpr int b_ring = a_ring + kLinStages * kLinBytes;
  static constexpr int bars = b_ring + kLinStages * kLinBytes;
  static constexpr int total = bars + 256;
};
struct LinBars {
  uint64_t full[kLinStages], empty[kLinStages], tmem_full[2], tmem_empty[2];
  uint32_t tmem_slot;
};
static_assert(sizeof(LinBars) <= LinSmem::total - LinSmem::bars, "barrier block overflows its region");

struct LinArgs {
  int M, N, K;             // D is M x N, contraction length K
  float* out;              // [M][ldo] fp32
  long long ldo;
  const float* bias;       // [N] added in the epilogue (may be nullptr)
  int ksplit;              // > 1: the contraction is split over CTAs and partial tiles are added with red.global
  long long* out_fx;       // deterministic split: 64-bit fixed-point accumulation instead (may be nullptr)
};

template <bool A_MN, bool B_MN>
__global__ void __launch_bounds__(kLinThreads, 1)
linear_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, LinArgs p) {
  extern __shared__ uint8_t smem_raw[];
  const AlignedSmem smem = aligned_smem(smem_raw);
  const uint32_t a_ring = smem.addr + LinSmem::a_ring, b_ring = smem.addr + LinSmem::b_ring;
  LinBars* bars = reinterpret_cast<LinBars*>(smem.ptr + LinSmem::bars);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const int tm = (p.M + kLinTile - 1) / kLinTile, tn = (p.N + kLinTile - 1) / kLinTile;
  const int nkc_all = (p.K + kBK - 1) / kBK;
  const int nitems = tm * tn * p.ksplit;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < kLinStages; ++s) { mbar_init(smem_u32(&bars->full[s]), 1); mbar_init(smem_u32(&bars->empty[s]), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(smem_u32(&bars->tmem_full[a]), 1); mbar_init(smem_u32(&bars->tmem_empty[a]), 4); }
    mbar_fence_init();
  }
  const uint32_t tmem_base = tmem_setup<false>(warp, &bars->tmem_slot, kLinTmemCols);

  // item -> (m tile, n tile, k range); consecutive items share the B tile column (n fastest would thrash A instead)
  auto decode = [&](int item, int& m0, int& n0, int& kc0, int& kc1) {
    const int ks = item % p.ksplit;
    const int t = item / p.ksplit;
    m0 = (t % tm) * kLinTile;
    n0 = (t / tm) * kLinTile;
    kc0 = static_cast<int>(static_cast<long long>(nkc_all) * ks / p.ksplit);
    kc1 = static_cast<int>(static_cast<long long>(nkc_all) * (ks + 1) / p.ksplit);
  };

  if (warp == 0) {
    if (lane == 0) {
      uint32_t it = 0;
      for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
        int m0, n0, kc0, kc1;
        decode(item, m0, n0, kc0, kc1);
        for (int kc = kc0; kc < kc1; ++kc, ++it) {
          const uint32_t s = it % kLinStages, ph = (it / kLinStages) & 1;
          const uint32_t full = smem_u32(&bars->full[s]);
          mbar_wait(smem_u32(&bars->empty[s]), ph ^ 1);
          mbar_expect_tx(full, 2 * kLinBytes);
          if (A_MN) {          // [k][m] storage: two boxes of 64 (m) x 64 (k rows)
            tma_load_2d(a_ring + s * kLinBytes, &tmA, full, m0, kc * kBK);
            tma_load_2d(a_ring + s * kLinBytes + 8192, &tmA, full, m0 + 64, kc * kBK);
          } else {             // [m][k] storage: one box of 64 (k) x 128 (m rows)
            tma_load_2d(a_ring + s * kLinBytes, &tmA, full, kc * kBK, m0);
          }
          if (B_MN) {
            tma_load_2d(b_ring + s * kLinBytes, &tmB, full, n0, kc * kBK);
            tma_load_2d(b_ring + s * kLinBytes + 8192, &tmB, full, n0 + 64, kc * kBK);
          } else {
            tma_load_2d(b_ring + s * kLinBytes, &tmB, full, kc * kBK, n0);
          }
        }
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = make_idesc(kLinTile, kLinTile, A_MN ? 1 : 0, B_MN ? 1 : 0, kFmtF16, kFmtF16);
    uint32_t it = 0, ic = 0;
    for (int item = blockIdx.x; item < nitems; item += gridDim.x, ++ic) {
      int m0, n0, kc0, kc1;
      decode(item, m0, n0, kc0, kc1);
      const uint32_t acc = ic & 1;
      mbar_wait(smem_u32(&bars->tmem_empty[acc]), ((ic >> 1) & 1) ^ 1);
      tc_fence_after();
      for (int kc = kc0; kc < kc1; ++kc, ++it) {
        const uint32_t s = it % kLinStages, ph = (it / kLinStages) & 1;
        mbar_wait(smem_u32(&bars->full[s]), ph);
        tc_fence_after();
        if (lane == 0) {
          mma_kchunk<false, A_MN, B_MN>(tmem_base + acc * kLinTile, a_ring + s * kLinBytes, b_ring + s * kLinBytes, idesc,
                                        kc > kc0);
          umma_commit(smem_u32(&bars->empty[s]));
        }
        __syncwarp();
      }
      if (lane == 0) umma_commit(smem_u32(&bars->tmem_full[acc]));   // (an empty k range never happens: ksplit <= number of k chunks)
      __syncwarp();
    }
  } else {
    const int lane_grp = warp & 3;
    const int row = lane_grp * 32 + lane;
    uint32_t ic = 0;
    for (int item = blockIdx.x; item < nitems; item += gridDim.x, ++ic) {
      int m0, n0, kc0, kc1;
      decode(item, m0, n0, kc0, kc1);
      const uint32_t acc = ic & 1;
      mbar_wait(smem_u32(&bars->tmem_full[acc]), (ic >> 1) & 1);
      tc_fence_after();
      const int m = m0 + row;
#pragma unroll 1
      for (int c32 = 0; c32 < kLinTile / 32; ++c32) {
        const int col0 = n0 + c32 * 32;
        if (col0 >= p.N) break;                  // uniform
        float v[32];
        tmem_ld32(tmem_lane_addr(tmem_base, lane_grp, acc * kLinTile + c32 * 32), v);
        tmem_ld_wait();
        if (m < p.M) {
          if (p.out_fx) {
            long long* dst = p.out_fx + static_cast<long long>(m) * p.N + col0;
#pragma unroll
            for (int e = 0; e < 32; ++e)
              if (col0 + e < p.N) fx_add(dst + e, v[e]);
            continue;
          }
          float* dst = p.out + static_cast<long long>(m) * p.ldo + col0;
          const bool vec = (p.ldo & 3) == 0 && col0 + 32 <= p.N;
          if (p.bias && kc0 == 0) {
#pragma unroll
            for (int e = 0; e < 32; ++e) v[e] += (col0 + e < p.N) ? __ldg(p.bias + col0 + e) : 0.f;
          }
          if (p.ksplit > 1) {
            if (vec) {
#pragma unroll
              for (int q = 0; q < 8; ++q) red_add_v4(dst + 4 * q, v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
            } else {
#pragma unroll
              for (int e = 0; e < 32; ++e)
                if (col0 + e < p.N) atomicAdd(dst + e, v[e]);
            }
          } else if (vec) {
#pragma unroll
            for (int q = 0; q < 8; ++q)
              reinterpret_cast<float4*>(dst)[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
          } else {
#pragma unroll
            for (int e = 0; e < 32; ++e)
              if (col0 + e < p.N) dst[e] = v[e];
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&bars->tmem_empty[acc]));
    }
  }

  tmem_teardown<false>(warp, tmem_base, kLinTmemCols);
}

__global__ void f32_to_f16_kernel(const float* __restrict__ src, __half* __restrict__ dst, long long n) {
  const long long n4 = n >> 2;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(src) + i);
    uint2 o;
    o.x = pack_f16x2(v.x, v.y);
    o.y = pack_f16x2(v.z, v.w);
    reinterpret_cast<uint2*>(dst)[i] = o;
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) dst[(n4 << 2) + threadIdx.x] = __float2half_rn(src[(n4 << 2) + threadIdx.x]);
}

// db[n] = sum_m dy[m][n]: block = 32 columns x 8 row lanes, rows strided over blockIdx.y; fixed-point or fp32 atomics
__global__ void colsum_kernel(const float* __restrict__ dy, int M, int N, float* __restrict__ db, long long* db_fx) {
  __shared__ float red[8][33];
  const int n = blockIdx.x * 32 + threadIdx.x;
  float acc = 0.f;
  if (n < N)
    for (int m = blockIdx.y * 8 + threadIdx.y; m < M; m += gridDim.y * 8) acc += dy[static_cast<long long>(m) * N + n];
  red[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0 && n < N) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += red[i][threadIdx.x];
    if (db_fx) fx_add(db_fx + n, t); else atomicAdd(db + n, t);
  }
}

__global__ void fx_to_f32_kernel(const long long* __restrict__ fx, float* __restrict__ out, long long n) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x)
    out[i] = static_cast<float>(static_cast<double>(fx[i]) * kFxInv);
}

int to_f16(const float* src, __half* dst, long long n, cudaStream_t stream) {
  const int grid = static_cast<int>(std::min<long long>((n / 4 + 255) / 256 + 1, 148 * 8));
  f32_to_f16_kernel<<<grid, 256, 0, stream>>>(src, dst, n);
  RB_CUDA_CHECK(cudaGetLastError());
  return 0;
}

template <bool A_MN, bool B_MN>
int launch_linear(const __half* A, const __half* Bm, const LinArgs& args, cudaStream_t stream) {
  // tensor maps: K-major operand [rows][K] -> box (64 k, 128 rows); MN-major operand [K][rows] -> box (64 rows, 64 k)
  CUtensorMap tmA, tmB;
  int rc;
  if (A_MN) rc = make_tmap_2d(&tmA, A, 2, args.M, args.K, static_cast<uint64_t>(args.M) * 2, 64, 64);
  else rc = make_tmap_2d(&tmA, A, 2, args.K, args.M, static_cast<uint64_t>(args.K) * 2, 64, 128);
  if (rc) return rc;
  if (B_MN) rc = make_tmap_2d(&tmB, Bm, 2, args.N, args.K, static_cast<uint64_t>(args.N) * 2, 64, 64);
  else rc = make_tmap_2d(&tmB, Bm, 2, args.K, args.N, static_cast<uint64_t>(args.K) * 2, 64, 128);
  if (rc) return rc;
  const size_t smem = LinSmem::total + kSmemAlign;
  RB_CUDA_CHECK(cudaFuncSetAttribute(linear_gemm_kernel<A_MN, B_MN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const long long items = static_cast<long long>((args.M + kLinTile - 1) / kLinTile) * ((args.N + kLinTile - 1) / kLinTile) * args.ksplit;
  const int grid = static_cast<int>(std::max<long long>(1, std::min<long long>(items, device_sm_count())));
  linear_gemm_kernel<A_MN, B_MN><<<grid, kLinThreads, smem, stream>>>(tmA, tmB, args);
  RB_CUDA_CHECK(cudaGetLastError());
  return 0;
}

inline size_t al(size_t x) { return (x + 255) & ~static_cast<size_t>(255); }

}  // namespace

size_t linear_workspace_bytes(long long M, int K, int N, bool backward, bool deterministic) {
  size_t b = al(static_cast<size_t>(M) * K * 2) + al(static_cast<size_t>(N) * K * 2);
  if (backward) {
    b += al(static_cast<size_t>(M) * N * 2);
    if (deterministic) b += al((static_cast<size_t>(N) * K + N) * 8);
  }
  return b;
}

int launch_linear_fwd(const float* x, const float* W, const float* bias, long long M, int K, int N, float* y,
                      void* workspace, cudaStream_t stream) {
  ProfScope prof_(kProfOther, stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  __half* x16 = reinterpret_cast<__half*>(ws);
  __half* w16 = reinterpret_cast<__half*>(ws + al(static_cast<size_t>(M) * K * 2));
  int rc = to_f16(x, x16, M * K, stream);
  if (rc) return rc;
  rc = to_f16(W, w16, static_cast<long long>(N) * K, stream);
  if (rc) return rc;
  LinArgs a{};
  a.M = static_cast<int>(M); a.N = N; a.K = K; a.out = y; a.ldo = N; a.bias = bias; a.ksplit = 1; a.out_fx = nullptr;
  return launch_linear<false, false>(x16, w16, a, stream);       // y = x . W^T : both operands K-major
}

int launch_linear_bwd(const float* x, const float* W, const float* dy, long long M, int K, int N, float* dx, float* dW,
                      float* db, bool deterministic, void* workspace, cudaStream_t stream) {
  ProfScope prof_(kProfOther, stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  size_t off = 0;
  __half* x16 = reinterpret_cast<__half*>(ws + off); off += al(static_cast<size_t>(M) * K * 2);
  __half* w16 = reinterpret_cast<__half*>(ws + off); off += al(static_cast<size_t>(N) * K * 2);
  __half* dy16 = reinterpret_cast<__half*>(ws + off); off += al(static_cast<size_t>(M) * N * 2);
  long long* fx = deterministic ? reinterpret_cast<long long*>(ws + off) : nullptr;
  int rc = to_f16(dy, dy16, M * N, stream);
  if (rc) return rc;
  if (dx) {         // dx[M,K] = dy[M,N] . W[N,K]: A = dy (K-major over N), B(k', n) = W[n][k'] = MN-major view of W
    rc = to_f16(W, w16, static_cast<long long>(N) * K, stream);
    if (rc) return rc;
    LinArgs a{};
    a.M = static_cast<int>(M); a.N = K; a.K = N; a.out = dx; a.ldo = K; a.bias = nullptr; a.ksplit = 1; a.out_fx = nullptr;
    rc = launch_linear<false, true>(dy16, w16, a, stream);
    if (rc) return rc;
  }
  if (dW) {         // dW[N,K] = dy^T . x: A(n, m) = dy[m][n], B(k', m) = x[m][k']: both MN-major, contraction over M
    rc = to_f16(x, x16, M * K, stream);
    if (rc) return rc;
    LinArgs a{};
    a.M = N; a.N = K; a.K = static_cast<int>(M); a.out = dW; a.ldo = K; a.bias = nullptr;
    const long long tiles = static_cast<long long>((N + kLinTile - 1) / kLinTile) * ((K + kLinTile - 1) / kLinTile);
    const long long nkc = (M + kBK - 1) / kBK;
    a.ksplit = static_cast<int>(std::max<long long>(1, std::min<long long>(device_sm_count() / std::max<long long>(1, tiles), nkc)));
    a.out_fx = nullptr;
    if (a.ksplit > 1) {
      if (deterministic) {
        a.out_fx = fx;
        RB_CUDA_CHECK(cudaMemsetAsync(fx, 0, static_cast<size_t>(N) * K * 8, stream));
      } else {
        RB_CUDA_CHECK(cudaMemsetAsync(dW, 0, static_cast<size_t>(N) * K * 4, stream));
      }
    }
    rc = launch_linear<true, true>(dy16, x16, a, stream);
    if (rc) return rc;
    if (a.out_fx) {
      fx_to_f32_kernel<<<148 * 4, 256, 0, stream>>>(fx, dW, static_cast<long long>(N) * K);
      RB_CUDA_CHECK(cudaGetLastError());
    }
  }
  if (db) {
    long long* fxb = deterministic ? fx + static_cast<size_t>(N) * K : nullptr;
    if (fxb) RB_CUDA_CHECK(cudaMemsetAsync(fxb, 0, static_cast<size_t>(N) * 8, stream));
    else RB_CUDA_CHECK(cudaMemsetAsync(db, 0, static_cast<size_t>(N) * 4, stream));
    const int gy = static_cast<int>(std::max<long long>(1, std::min<long long>((M + 63) / 64, 64)));
    colsum_kernel<<<dim3((N + 31) / 32, gy), dim3(32, 8), 0, stream>>>(dy, static_cast<int>(M), N, db, fxb);
    RB_CUDA_CHECK(cudaGetLastError());
    if (fxb) {
      fx_to_f32_kernel<<<1, 256, 0, stream>>>(fxb, db, N);
      RB_CUDA_CHECK(cudaGetLastError());
    }
  }
  return 0;
}

}  // namespace rb
