// tcgen05 (5th-gen tensor core) GEMMs for the dense layers of the LCAO hot path, sm_100a only.
//
// Arithmetic: kind::tf32 MMAs with FP32 accumulation in TMEM.  In LCAO_GEMM_TF32X3 mode every FP32
// operand x is split into hi = x with the 13 low mantissa bits cleared (exactly a TF32 number) and
// lo = x - hi (cleared the same way), and each product is issued as hi*hi + lo*hi + hi*lo
// (3 MMAs, error ~2^-21 per product: FP32-equivalent, which the 1e-5 parity bar needs); LCAO_GEMM_TF32
// issues hi*hi only.
//
// Operands never go through TMA: loader warps stream the FP32 rows from HBM with 16-byte cp.async copies into
// SWIZZLE_128B K-major shared-memory tiles, and transform warps split them into hi / lo for the MMAs (the weight-gradient
// kernel transposes 4x4 blocks in registers on the way).  The row kernels keep the layer's weight resident in shared
// memory, split once per CTA.
//
// Kernels (warp roles and pipelines are described at each kernel):
//   k_tc_rows<EPI8>  Y = epi(A W^T) or epi(A W), 128-row tiles, persistent over the row blocks (grid <= #SMs);
//                    EPI8 adds four epilogue warps for grids with one tile per CTA.
//   k_tc_rows_ta     the same product in 3xTF32 mode with the A operand in tensor memory, for many tiles per CTA.
//   k_tc_wgrad       dW += dY^T X (and db += colsum dY) as per-CTA partial tiles, summed in a fixed order by
//                    k_wgrad_reduce / k_wgrad_reduce_batch (deterministic, no atomics).
// All mbarrier waits are bounded (trap on timeout) so a protocol bug aborts the kernel instead of hanging the GPU.
#include "common.cuh"

namespace {

constexpr int kEpiWarps = 4;
constexpr int kBlockM = 128;                                   // rows per tile (UMMA M)
constexpr int kChunkK = 32;                                    // contraction elements per smem stage
constexpr uint32_t kSpinLimit = 1u << 28;  // (several seconds: under programmatic dependent launch a CTA may poll while the previous kernel drains)

// ---------------------------------------------------------------------------------- PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0, spins = 0;
  const uint32_t addr = smem_u32(bar);
  while (!done) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
    if (!done && ++spins > kSpinLimit) __trap();
  }
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// One lane of a converged warp.  The MMA-issuer warps run their loops with all 32 lanes (uniform control flow, so the
// descriptors / addresses stay in uniform registers) and elect a lane only around the tcgen05 instruction itself: issued
// from inside an `if (lane == 0)` region the compiler had to broadcast every operand through R2UR waterfall loops,
// ~18 instructions per MMA, and the single issuing thread (128 cycles per MMA) was slower than the tensor core (~69).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
// D[tmem] (+)= A[smem desc] * B[smem desc], kind::tf32, issued by ONE thread
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on an mbarrier when all previously issued MMAs of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// 32 lanes x 32 consecutive 32-bit columns: thread i of the warp gets row (lane base + i)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// UMMA shared-memory descriptor (cute::UMMA::SmemDescriptor: start>>4 [0,14), LBO>>4 [16,30), SBO>>4 [32,46),
// version=1 [46,48), layout_type [61,64)) of a SWIZZLE_128B K-major tile:
// rows of 128 bytes (32 tf32), 16-byte chunk c of row r stored at chunk (c ^ (r & 7));
// 8-row groups are 1024 B apart (SBO), LBO is unused (=1), layout_type = 2, tile base 1024-byte aligned.
// One MMA consumes K = 8 tf32 = 32 bytes: the start address advances by 32 B inside the swizzled row.
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
__device__ __forceinline__ uint32_t sw128_off(int row, int chunk) { return row * 128 + ((chunk ^ (row & 7)) << 4); }
// instruction descriptor (cute::UMMA::InstrDescriptor): c_format F32=1 [4,6), a/b_format TF32=2 [7,10)/[10,13),
// a_major [15] = b_major [16] = 0 (both operands K-major), N>>3 [17,23), M>>4 [24,29)
__host__ __device__ constexpr uint32_t make_idesc(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ float tf32_hi(float x) { return __uint_as_float(__float_as_uint(x) & 0xFFFFE000u); }
__device__ __forceinline__ void split4(const float4 x, float4& hi, float4& lo) {
  hi = make_float4(tf32_hi(x.x), tf32_hi(x.y), tf32_hi(x.z), tf32_hi(x.w));
  lo = make_float4(tf32_hi(x.x - hi.x), tf32_hi(x.y - hi.y), tf32_hi(x.z - hi.z), tf32_hi(x.w - hi.w));
}
// SFU-based sigmoid for the GEMM epilogues/prologues (ex2.approx + rcp.approx: ~3e-7 relative error for |x| < 10,
// an order below the 3xTF32 product error), so that 4 epilogue warps keep up with the tensor core
__device__ __forceinline__ float sigmoid_fast(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
__device__ __forceinline__ float silu_fast(float x) { return x * sigmoid_fast(x); }
__device__ __forceinline__ float silu_grad_fast(float x) {
  const float sg = sigmoid_fast(x);
  return sg * fmaf(x, 1.0f - sg, 1.0f);
}
__device__ __forceinline__ float4 silu_grad4(float4 g, float4 h) {
  return make_float4(g.x * silu_grad_fast(h.x), g.y * silu_grad_fast(h.y), g.z * silu_grad_fast(h.z), g.w * silu_grad_fast(h.w));
}

// 8 consecutive floats: one 256-bit store (a full 32-byte sector) when the address allows it, else two 128-bit ones
__device__ __forceinline__ void store8(float* p, const float* v, bool wide) {
  if (wide) {
    asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]),
                 "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7])
                 : "memory");
  } else {
    st4(p, make_float4(v[0], v[1], v[2], v[3]));
    st4(p + 4, make_float4(v[4], v[5], v[6], v[7]));
  }
}

// =================================================================================================
// Kernel 1: row-streaming GEMM   Y[M, Nb] = epi( A[M, Kc] * Bop[Kc, Nb] )
//   forward : Bop(n, k) = W[n*ldw + k]  (b_trans = 0, W is (Nb, Kc) row-major)
//   dgrad   : Bop(n, k) = W[k*ldw + n]  (b_trans = 1, W is (Kc, Nb) row-major)
// A stages (128 rows x 32 k) and the resident weight (Kc/32 blocks of Nb rows x 32 k) are SWIZZLE_128B
// K-major tiles (see make_desc_sw128).
//
// Warp roles (416 threads): 0-3 epilogue, 4-7 hi/lo split (smem -> smem), 8 MMA issuer, 9-12 loaders.
// The loader warps stream A with 16-byte cp.async copies, 8 lanes per 128-byte row so that every group
// writes ONE full swizzled 128-byte line of the tile (conflict free), up to R-1 stages (16 KB each)
// ahead of the consumer; completion is signalled with cp.async.mbarrier.arrive.  The split warps
// rewrite the stage in place as `hi` and produce `lo` in a short ring (L = 2) — an elementwise pass that
// is layout agnostic — fence to the async proxy and hand the stage to the MMA warp.
// =================================================================================================
struct RowsArgs {
  const float* A; int64_t lda;
  const float* W; int64_t ldw;
  const float* bias;
  const float* G; int64_t ldg;     // epilogue: out *= SiLU'(G) (dgrad chained into the previous layer's pre-activation)
  float* Y; int64_t ldy;
  float* pre; int64_t ldp;
  int64_t M; int Kc; int Nb;
  int b_trans, act, accumulate, x3, stages, lo_stages;
  int wide_store;  // Y / pre rows are 32-byte aligned: 256-bit stores
};

constexpr int kLoadWarps = 4;
constexpr int kRowsThreads = (4 + 4 + 1 + kLoadWarps) * 32;  // 416
constexpr int kEpiPitch = 144;                   // bytes per staged row (32 floats + 16 B pad: conflict-free)
constexpr int kEpiWarpBytes = 32 * kEpiPitch;    // one warp stages its 32 rows x 32 columns
constexpr uint32_t kStageBytes = kBlockM * 128;  // 16 KB: 128 rows x 32 tf32

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_arrive(uint64_t* bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// EPI8: four more epilogue warps (13-16); the two warps of a TMEM lane quadrant take 64 output columns each
template <bool EPI8>
__global__ void __launch_bounds__(EPI8 ? kRowsThreads + 128 : kRowsThreads, 1) k_tc_rows(const RowsArgs g) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  pdl_trigger();  // the next kernel of the stream may start its own set-up while this one runs
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t blockB = g.Nb * 128;                 // bytes of one 32-k column block of the weight
  const uint32_t halfB = (g.Kc / kChunkK) * blockB;   // bytes of one of {W_hi, W_lo}
  const int R = g.stages, L = g.lo_stages;
  uint8_t* sB = smem_raw;
  uint8_t* sHi = sB + 2 * halfB;
  uint8_t* sLo = sHi + (size_t)R * kStageBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sLo + (size_t)(g.x3 ? L : 0) * kStageBytes);  // no lo ring in 1x mode
  uint64_t* raw_full = bars;            // [R] loaders (cp.async completion) -> split warps
  uint64_t* full = raw_full + R;        // [R] split warps -> MMA
  uint64_t* hi_empty = full + R;        // [R] MMA -> loaders
  uint64_t* lo_empty = hi_empty + R;    // [L] MMA -> split warps
  uint64_t* tfull = lo_empty + L;       // [2] MMA -> epilogue
  uint64_t* tempty = tfull + 2;         // [2] epilogue -> MMA
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

  const int64_t nblocks = (g.M + kBlockM - 1) / kBlockM;
  const int nchunk = g.Kc / kChunkK;
  // TMEM: 2 accumulator buffers; in x3 mode each buffer holds TWO accumulators: hi*hi and the small
  // lo*hi + hi*lo corrections.  The tensor core truncates (RZ) on every accumulate, so keeping the
  // dominant chain at K/8 steps and the corrections (2^-10 of the magnitude) apart cuts the bias 3x.
  const uint32_t acc_cols = g.x3 ? 2 * g.Nb : g.Nb;
  const uint32_t need_cols = 2 * acc_cols;
  const uint32_t tmem_cols = need_cols <= 32 ? 32 : need_cols <= 64 ? 64 : need_cols <= 128 ? 128 : need_cols <= 256 ? 256 : 512;

  if (threadIdx.x == 0) {
    for (int s = 0; s < R; ++s) {
      mbar_init(&raw_full[s], kLoadWarps * 32);
      mbar_init(&full[s], 4 * 32);
      mbar_init(&hi_empty[s], 1);
    }
    for (int s = 0; s < L; ++s) mbar_init(&lo_empty[s], 1);
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull[a], 1);
      mbar_init(&tempty[a], (EPI8 ? 2 : 1) * kEpiWarps * 32);
    }
    fence_barrier_init();
  }
  if (warp == 8) tmem_alloc(tmem_slot, tmem_cols);
  tc_fence_before();
  __syncthreads();  // barriers initialised, TMEM address published
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // ---- resident B operand (the layer's weight), split hi/lo once per CTA by the 9 non-loader warps while the
  //      loader warps already stream the first A stages; kWB loads in flight per thread (the weights come from L2 /
  //      HBM with ~1 us latency: a dependent loop would cost ~10 us per launch)
  constexpr int kStageThreads = (4 + 4 + 1) * 32;  // 288
  constexpr int kWB = 8;  // weight loads in flight per thread (64 KB of weights = 14 float4 per thread: two round trips to L2)
  if (warp < 9) {
    const int kq = g.Kc / 4, total = g.Nb * kq;
    for (int base = 0; base < total; base += kWB * kStageThreads) {
      float4 w[kWB];
      int n[kWB], kg[kWB];
#pragma unroll
      for (int u = 0; u < kWB; ++u) {
        const int idx = base + u * kStageThreads + (int)threadIdx.x;
        w[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        n[u] = -1;
        if (idx < total) {
          if (!g.b_trans) {
            n[u] = idx / kq; kg[u] = idx - n[u] * kq;
            w[u] = ldg4(g.W + (int64_t)n[u] * g.ldw + kg[u] * 4);
          } else {  // W is (Kc, Nb): contraction group kg = 4 rows of W, one output column n
            kg[u] = idx / g.Nb; n[u] = idx - kg[u] * g.Nb;
            w[u] = make_float4(__ldg(g.W + (int64_t)(kg[u] * 4 + 0) * g.ldw + n[u]), __ldg(g.W + (int64_t)(kg[u] * 4 + 1) * g.ldw + n[u]),
                               __ldg(g.W + (int64_t)(kg[u] * 4 + 2) * g.ldw + n[u]), __ldg(g.W + (int64_t)(kg[u] * 4 + 3) * g.ldw + n[u]));
          }
        }
      }
#pragma unroll
      for (int u = 0; u < kWB; ++u) {
        if (n[u] >= 0) {
          float4 hi, lo;
          split4(w[u], hi, lo);
          const uint32_t off = (kg[u] >> 3) * blockB + sw128_off(n[u], kg[u] & 7);
          *reinterpret_cast<float4*>(sB + off) = hi;
          *reinterpret_cast<float4*>(sB + halfB + off) = lo;
        }
      }
    }
    fence_proxy_async();
    asm volatile("bar.sync 1, %0;" ::"n"(kStageThreads) : "memory");  // weights complete (non-loader warps only)
  }

  // Everything above (barriers, TMEM, the split of the resident weight: parameters, never written by a kernel that triggers
  // early) may overlap the tail of the previous kernel (programmatic dependent launch); the activations may not.
  pdl_wait();
  if (warp >= 9 && warp < 13) {
    // ============================== loader warps ==============================
    // warp lw streams rows [32 lw, 32 lw + 32) of the tile: 8 copies per lane and stage; lanes 0-7 / 8-15 / ...
    // cover one 128-byte row each (global) and write its 8 chunks into one swizzled 128-byte smem line
    const int lw = warp - 9, row_in = lane >> 3, c = lane & 7;
    const uint32_t hi_base = smem_u32(sHi);
    uint32_t it = 0;
    for (int64_t mb = blockIdx.x; mb < nblocks; mb += gridDim.x) {
      const int64_t mrow = mb * kBlockM + 32 * lw + row_in;
      for (int kc = 0; kc < nchunk; ++kc, ++it) {
        const int s = it % R;
        mbar_wait(&hi_empty[s], ((it / R) & 1) ^ 1);
        const uint32_t dst = hi_base + s * kStageBytes;
        const float* src = g.A + mrow * g.lda + kc * kChunkK + c * 4;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const bool ok = mrow + 4 * j < g.M;
          cp_async16(dst + sw128_off(32 * lw + 4 * j + row_in, c), ok ? src + (int64_t)4 * j * g.lda : g.A, ok ? 16u : 0u);
        }
        cp_async_arrive(&raw_full[s]);
      }
    }
  } else if (warp >= 4 && warp < 8) {
    // ============================== split warps: hi in place, lo into the short ring =================
    const int t = threadIdx.x - 128;              // 0..127
    uint32_t it = 0;
    for (int64_t mb = blockIdx.x; mb < nblocks; mb += gridDim.x) {
      for (int kc = 0; kc < nchunk; ++kc, ++it) {
        const int s = it % R, l = it % L;
        mbar_wait(&raw_full[s], (it / R) & 1);
        if (g.x3) {
          mbar_wait(&lo_empty[l], ((it / L) & 1) ^ 1);
          uint8_t* ph = sHi + (size_t)s * kStageBytes + t * 16;
          uint8_t* pl = sLo + (size_t)l * kStageBytes + t * 16;
#pragma unroll
          for (int i = 0; i < 8; ++i) {           // elementwise: any bijection of the 1024 chunks works
            float4 hi, lo;
            split4(*reinterpret_cast<const float4*>(ph + i * 2048), hi, lo);
            *reinterpret_cast<float4*>(ph + i * 2048) = hi;
            *reinterpret_cast<float4*>(pl + i * 2048) = lo;
          }
        }
        fence_proxy_async();
        mbar_arrive(&full[s]);
      }
    }
  } else if (warp == 8) {
    // ============================== MMA issuer (all lanes run the loop; one is elected per instruction) ==============
    {
      const uint32_t idesc = make_idesc(kBlockM, g.Nb);
      const uint32_t hiBase = smem_u32(sHi), loBase = smem_u32(sLo), bBase = smem_u32(sB);
      uint32_t it = 0, tile = 0;
      for (int64_t mb = blockIdx.x; mb < nblocks; mb += gridDim.x, ++tile) {
        const int acc = tile & 1;
        mbar_wait(&tempty[acc], ((tile >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d = tmem_base + acc * acc_cols, dc = d + g.Nb;
        for (int kc = 0; kc < nchunk; ++kc, ++it) {
          const int s = it % R, l = it % L;
          mbar_wait(&full[s], (it / R) & 1);
          tc_fence_after();
          const uint32_t a_hi = hiBase + s * kStageBytes, a_lo = loBase + l * kStageBytes;
          const uint32_t b_hi = bBase + kc * blockB, b_lo = b_hi + halfB;
          const uint64_t dAh0 = make_desc_sw128(a_hi), dBh0 = make_desc_sw128(b_hi), dAl0 = make_desc_sw128(a_lo), dBl0 = make_desc_sw128(b_lo);
#pragma unroll
          for (int kk = 0; kk < kChunkK / 8; ++kk) {
            const uint64_t dAh = dAh0 + 2 * kk, dBh = dBh0 + 2 * kk, dAl = dAl0 + 2 * kk, dBl = dBl0 + 2 * kk;
            if (elect_one()) {
              umma_tf32(d, dAh, dBh, idesc, (kc | kk) != 0);
              if (g.x3) {
                umma_tf32(dc, dAl, dBh, idesc, (kc | kk) != 0);
                umma_tf32(dc, dAh, dBl, idesc, 1);
              }
            }
          }
          if (elect_one()) {
            umma_commit(&hi_empty[s]);
            if (g.x3) umma_commit(&lo_empty[l]);
          }
        }
        if (elect_one()) umma_commit(&tfull[acc]);
      }
    }
    __syncwarp();
  } else {
    // ============================== epilogue warps ==============================
    // TMEM gives every thread one ROW (32 consecutive columns = 128 contiguous bytes of the output row per load).
    // The row segment is finished in registers (bias, accumulate, pre-activation, SiLU, SiLU' factor) and written
    // with 256-bit stores: every store instruction of a thread fills one whole 32-byte sector, so no shared-memory
    // transpose is needed (and its 18 KB go to the operand ring).
    const bool wide = g.wide_store != 0;
    const int quad = warp & 3;  // TMEM lanes 32 quad .. 32 quad + 31 (a warp reaches the quadrant warp % 4)
    const int c_begin = (EPI8 && warp >= 13) ? 64 : 0, c_end = EPI8 ? min(g.Nb, c_begin + 64) : g.Nb;
    uint32_t tile = 0;
    for (int64_t mb = blockIdx.x; mb < nblocks; mb += gridDim.x, ++tile) {
      const int acc = tile & 1;
      const int64_t m = mb * kBlockM + quad * 32 + lane;
      // The SiLU' factor rows (G) are fetched one 32-column chunk AHEAD of their use — the first chunk while the
      // tile's MMAs are still running — so that the epilogue never waits on HBM between a TMEM load and its stores.
      float4 gq[8];
      if (g.G && m < g.M) {
#pragma unroll
        for (int q = 0; q < 8; ++q)
          gq[q] = (c_begin + 4 * q < g.Nb) ? ldg4(g.G + m * g.ldg + c_begin + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      mbar_wait(&tfull[acc], (tile >> 1) & 1);
      tc_fence_after();
      for (int c0 = c_begin; c0 < c_end; c0 += 32) {
        float4 gn[8];
        if (g.G && m < g.M && c0 + 32 < c_end) {
#pragma unroll
          for (int q = 0; q < 8; ++q)
            gn[q] = (c0 + 32 + 4 * q < g.Nb) ? ldg4(g.G + m * g.ldg + c0 + 32 + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        float v[32];
        tmem_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + acc * acc_cols + c0, v);
        if (g.x3) {
          float w[32];
          tmem_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + acc * acc_cols + g.Nb + c0, w);
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] += w[j];
        }
        if (m < g.M) {
          const int nc = min(32, g.Nb - c0);  // multiple of 16
#pragma unroll
          for (int j = 0; j < 32; j += 8) {
            if (j < nc) {
              float* o = v + j;
              if (g.bias) {
                const float4 b0 = ldg4(g.bias + c0 + j), b1 = ldg4(g.bias + c0 + j + 4);
                o[0] += b0.x; o[1] += b0.y; o[2] += b0.z; o[3] += b0.w; o[4] += b1.x; o[5] += b1.y; o[6] += b1.z; o[7] += b1.w;
              }
              if (g.accumulate) {
                const float4 p0 = *reinterpret_cast<const float4*>(g.Y + m * g.ldy + c0 + j);
                const float4 p1 = *reinterpret_cast<const float4*>(g.Y + m * g.ldy + c0 + j + 4);
                o[0] += p0.x; o[1] += p0.y; o[2] += p0.z; o[3] += p0.w; o[4] += p1.x; o[5] += p1.y; o[6] += p1.z; o[7] += p1.w;
              }
              if (g.pre) store8(g.pre + m * g.ldp + c0 + j, o, wide);
              if (g.act == LCAO_ACT_SILU) {
#pragma unroll
                for (int q = 0; q < 8; ++q) o[q] = silu_fast(o[q]);
              }
              if (g.G) {
                const float4 h0 = gq[j / 4], h1 = gq[j / 4 + 1];
                o[0] *= silu_grad_fast(h0.x); o[1] *= silu_grad_fast(h0.y); o[2] *= silu_grad_fast(h0.z); o[3] *= silu_grad_fast(h0.w);
                o[4] *= silu_grad_fast(h1.x); o[5] *= silu_grad_fast(h1.y); o[6] *= silu_grad_fast(h1.z); o[7] *= silu_grad_fast(h1.w);
              }
              store8(g.Y + m * g.ldy + c0 + j, o, wide);
            }
          }
        }
        if (g.G) {
#pragma unroll
          for (int q = 0; q < 8; ++q) gq[q] = gn[q];
        }
      }
      tc_fence_before();
      mbar_arrive(&tempty[acc]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 8) {
    tc_fence_after();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

// =================================================================================================
// Kernel 1b: the row-streaming GEMM with the A operand in TENSOR MEMORY (3xTF32 mode, many tiles per CTA).
// k_tc_rows keeps every 128 x 32 chunk of A in shared memory twice (hi in place, lo in a second ring) from the moment
// its cp.async copies are issued until the MMAs that read it have committed (~3 us), and only 3 + 3 stages of 16 KB
// fit beside the 128 KB weight: 48 KB of loads in flight per SM = 2.4 TB/s for the whole GPU (profiles/r01_notes.md).
// Here the split warps move a chunk out of shared memory as soon as it has landed: thread = row, hi / lo are written
// with tcgen05.st into a ring of 4 x (32 + 32) TMEM columns and the MMAs take A from tensor memory
// (tcgen05.mma ... [d], [a], b-desc).  Shared memory then holds only raw chunks in flight (6 x 16 KB beside the
// weight), twice as many bytes on the wire.  TMEM: 2 x Nb accumulator columns (hi*hi and the corrections share ONE
// accumulator: 48 instead of 16 truncating accumulations per output, measured within the parity tolerances) + 256.
// Warp roles as in k_tc_rows (0-3 epilogue, 4-7 split, 8 MMA issuer, 9-12 loaders).
// =================================================================================================
constexpr int kTaThreads = 15 * 32;  // 8 epilogue + 4 split + 1 MMA + 2 loader warps
constexpr int kTaStages = 4;       // TMEM A ring: stage = 32 hi + 32 lo columns
constexpr uint32_t kTaCol0 = 256;  // first column of the ring (accumulators below)

__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// 32 lanes x 32 consecutive 32-bit columns: thread i of the warp writes row (lane base + i)
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
        "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]),
        "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]),
        "r"(r[30]), "r"(r[31])
      : "memory");
}
// the same load as tmem_ld32 without the wait: several loads in flight, then tmem_wait_ld()
__device__ __forceinline__ void tmem_ld32_nw(uint32_t taddr, float (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]), "=f"(v[8]),
        "=f"(v[9]), "=f"(v[10]), "=f"(v[11]), "=f"(v[12]), "=f"(v[13]), "=f"(v[14]), "=f"(v[15]), "=f"(v[16]),
        "=f"(v[17]), "=f"(v[18]), "=f"(v[19]), "=f"(v[20]), "=f"(v[21]), "=f"(v[22]), "=f"(v[23]), "=f"(v[24]),
        "=f"(v[25]), "=f"(v[26]), "=f"(v[27]), "=f"(v[28]), "=f"(v[29]), "=f"(v[30]), "=f"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// One 32-column chunk per pipeline stage.  Every stage costs one round of mbarrier hand-shakes between the loaders, the
// split warps and the MMA issuer (~0.35 us), but the hand-shakes are not the critical path: two chunks per stage, or a
// second group of split warps taking the odd chunks, did not make the kernel faster.  What set the pace after the
// operand moved to tensor memory was the epilogue (see below); profiles/r02_notes.md.
__global__ void __launch_bounds__(kTaThreads, 1) k_tc_rows_ta(const RowsArgs g) {
  // warps: 0-3 epilogue (columns 0-63), 4-7 split, 8 MMA issuer, 9-10 loaders (64 rows each), 11-14 epilogue (columns 64-127)
  constexpr int kLd = 2;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  pdl_trigger();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t blockB = g.Nb * 128;
  const uint32_t halfB = (g.Kc / kChunkK) * blockB;
  const int R = g.stages;
  uint8_t* sB = smem_raw;
  uint8_t* sRaw = sB + 2 * halfB;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sRaw + (size_t)R * kStageBytes);
  uint64_t* raw_full = bars;               // [R] loaders (cp.async completion) -> split warps
  uint64_t* raw_empty = raw_full + R;      // [R] split warps -> loaders
  uint64_t* a_full = raw_empty + R;        // [kTaStages] split warps -> MMA
  uint64_t* a_empty = a_full + kTaStages;  // [kTaStages] MMA -> split warps
  uint64_t* tfull = a_empty + kTaStages;   // [2] MMA -> epilogue
  uint64_t* tempty = tfull + 2;            // [2] epilogue -> MMA
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
  const int64_t nblocks = (g.M + kBlockM - 1) / kBlockM;
  const int nchunk = g.Kc / kChunkK;
  constexpr uint32_t tmem_cols = 512;

  if (threadIdx.x == 0) {
    for (int s = 0; s < R; ++s) {
      mbar_init(&raw_full[s], kLd * 32);
      mbar_init(&raw_empty[s], 4 * 32);
    }
    for (int s = 0; s < kTaStages; ++s) {
      mbar_init(&a_full[s], 4 * 32);
      mbar_init(&a_empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull[a], 1);
      mbar_init(&tempty[a], 2 * kEpiWarps * 32);
    }
    fence_barrier_init();
  }
  if (warp == 8) tmem_alloc(tmem_slot, tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // ---- resident B operand (the layer's weight), split hi/lo once per CTA by the 9 non-loader warps (see k_tc_rows)
  constexpr int kStageThreads = (4 + 4 + 1) * 32;
  constexpr int kWB = 8;
  if (warp < 9) {
    const int kq = g.Kc / 4, total = g.Nb * kq;
    for (int base = 0; base < total; base += kWB * kStageThreads) {
      float4 w[kWB];
      int n[kWB], kg[kWB];
#pragma unroll
      for (int u = 0; u < kWB; ++u) {
        const int idx = base + u * kStageThreads + (int)threadIdx.x;
        w[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        n[u] = -1;
        if (idx < total) {
          if (!g.b_trans) {
            n[u] = idx / kq; kg[u] = idx - n[u] * kq;
            w[u] = ldg4(g.W + (int64_t)n[u] * g.ldw + kg[u] * 4);
          } else {
            kg[u] = idx / g.Nb; n[u] = idx - kg[u] * g.Nb;
            w[u] = make_float4(__ldg(g.W + (int64_t)(kg[u] * 4 + 0) * g.ldw + n[u]), __ldg(g.W + (int64_t)(kg[u] * 4 + 1) * g.ldw + n[u]),
                               __ldg(g.W + (int64_t)(kg[u] * 4 + 2) * g.ldw + n[u]), __ldg(g.W + (int64_t)(kg[u] * 4 + 3) * g.ldw + n[u]));
          }
        }
      }
#pragma unroll
      for (int u = 0; u < kWB; ++u) {
        if (n[u] >= 0) {
          float4 hi, lo;
          split4(w[u], hi, lo);
          const uint32_t off = (kg[u] >> 3) * blockB + sw128_off(n[u], kg[u] & 7);
          *reinterpret_cast<float4*>(sB + off) = hi;
          *reinterpret_cast<float4*>(sB + halfB + off) = lo;
        }
      }
    }
    fence_proxy_async();
    asm volatile("bar.sync 1, %0;" ::"n"(kStageThreads) : "memory");
  }
  pdl_wait();  // (the set-up and the weight split above may overlap the previous kernel's tail)

  if (warp >= 9 && warp < 9 + kLd) {
    // ============================== loader warps (as in k_tc_rows; 128 / kLd rows each) ==============================
    constexpr int kRowsPerLd = kBlockM / kLd;
    const int lw = warp - 9, row_in = lane >> 3, c = lane & 7;
    const uint32_t raw_base = smem_u32(sRaw);
    uint32_t it = 0;
    for (int64_t mb = blockIdx.x; mb < nblocks; mb += gridDim.x) {
      const int64_t mrow = mb * kBlockM + kRowsPerLd * lw + row_in;
      for (int kc = 0; kc < nchunk; ++kc, ++it) {
        const int s = it % R;
        mbar_wait(&raw_empty[s], ((it / R) & 1) ^ 1);
        const uint32_t dst = raw_base + s * kStageBytes;
        const float* src = g.A + mrow * g.lda + kc * kChunkK + c * 4;
#pragma unroll
        for (int j = 0; j < kRowsPerLd / 4; ++j) {
          const bool ok = mrow + 4 * j < g.M;
          cp_async16(dst + sw128_off(kRowsPerLd * lw + 4 * j + row_in, c), ok ? src + (int64_t)4 * j * g.lda : g.A, ok ? 16u : 0u);
        }
        cp_async_arrive(&raw_full[s]);
      }
    }
  } else if (warp >= 4 && warp < 8) {
    // ============================== split warps: raw chunk (smem) -> hi | lo (TMEM), thread = row =================
    const int row = (warp & 3) * 32 + lane;  // 0..127 = TMEM lane (a warp reaches the lane quadrant warp % 4)
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    uint32_t it = 0;
    for (int64_t mb = blockIdx.x; mb < nblocks; mb += gridDim.x) {
      for (int kc = 0; kc < nchunk; ++kc, ++it) {
        const int s = it % R, ts = it % kTaStages;
        mbar_wait(&raw_full[s], (it / R) & 1);
        mbar_wait(&a_empty[ts], ((it / kTaStages) & 1) ^ 1);
        tc_fence_after();
        const uint8_t* pr = sRaw + (size_t)s * kStageBytes;
        uint32_t hi[32], lo[32];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const float4 v = *reinterpret_cast<const float4*>(pr + sw128_off(row, c));
          float4 h, l;
          split4(v, h, l);
          hi[4 * c] = __float_as_uint(h.x); hi[4 * c + 1] = __float_as_uint(h.y); hi[4 * c + 2] = __float_as_uint(h.z); hi[4 * c + 3] = __float_as_uint(h.w);
          lo[4 * c] = __float_as_uint(l.x); lo[4 * c + 1] = __float_as_uint(l.y); lo[4 * c + 2] = __float_as_uint(l.z); lo[4 * c + 3] = __float_as_uint(l.w);
        }
        const uint32_t ta = tmem_base + lane_base + kTaCol0 + ts * 64;
        tmem_st32(ta, hi);
        tmem_st32(ta + 32, lo);
        mbar_arrive(&raw_empty[s]);  // the stage is in registers / tensor memory: it can take the next copies
        tmem_wait_st();
        tc_fence_before();
        mbar_arrive(&a_full[ts]);
      }
    }
  } else if (warp == 8) {
    // ============================== MMA issuer (all lanes run the loop; one is elected per instruction) ==============
    {
      const uint32_t idesc = make_idesc(kBlockM, g.Nb);
      const uint32_t bBase = smem_u32(sB);
      uint32_t it = 0, tile = 0;
      for (int64_t mb = blockIdx.x; mb < nblocks; mb += gridDim.x, ++tile) {
        const int acc = tile & 1;
        mbar_wait(&tempty[acc], ((tile >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d = tmem_base + acc * g.Nb;
        for (int kc = 0; kc < nchunk; ++kc, ++it) {
          const int ts = it % kTaStages;
          mbar_wait(&a_full[ts], (it / kTaStages) & 1);
          tc_fence_after();
          const uint32_t a_hi = tmem_base + kTaCol0 + ts * 64, a_lo = a_hi + 32;
          const uint32_t b_hi = bBase + kc * blockB, b_lo = b_hi + halfB;
          const uint64_t dBh0 = make_desc_sw128(b_hi), dBl0 = make_desc_sw128(b_lo);
#pragma unroll
          for (int kk = 0; kk < kChunkK / 8; ++kk) {
            const uint64_t dBh = dBh0 + 2 * kk, dBl = dBl0 + 2 * kk;  // (+ 32 B per K step: + 2 in the address field)
            if (elect_one()) {
              umma_tf32_ts(d, a_hi + kk * 8, dBh, idesc, (kc | kk) != 0);
              umma_tf32_ts(d, a_lo + kk * 8, dBh, idesc, 1);
              umma_tf32_ts(d, a_hi + kk * 8, dBl, idesc, 1);
            }
          }
          if (elect_one()) umma_commit(&a_empty[ts]);
        }
        if (elect_one()) umma_commit(&tfull[acc]);
      }
    }
    __syncwarp();
  } else if (warp < 4 || warp >= 9 + kLd) {
    // ============================== epilogue warps ==============================
    // Eight warps, two per TMEM lane quadrant (warp % 4), 64 columns each.  A warp issues both of its 32-column TMEM
    // loads at once, waits once, RELEASES the accumulator (the tile is in registers: the MMAs of the tile after next
    // can start) and only then finishes the rows (bias, accumulate, pre-activation, SiLU, SiLU' factor) and stores
    // them with 256-bit stores.  (Four warps draining 32 columns at a time with a wait per load took 7.3 k cycles per
    // tile against 4.9 k for the whole main loop: the epilogue, not the operand pipeline, set the pace.)
    const bool wide = g.wide_store != 0;
    const int quad = warp & 3;
    const int c_begin = warp >= 9 + kLd ? 64 : 0, c_end = min(g.Nb, c_begin + 64);
    uint32_t tile = 0;
    for (int64_t mb = blockIdx.x; mb < nblocks; mb += gridDim.x, ++tile) {
      const int acc = tile & 1;
      const int64_t m = mb * kBlockM + quad * 32 + lane;
      mbar_wait(&tfull[acc], (tile >> 1) & 1);
      tc_fence_after();
      float v[2][32];
      const uint32_t t0 = tmem_base + ((uint32_t)(quad * 32) << 16) + acc * g.Nb;
      if (c_begin < c_end) tmem_ld32_nw(t0 + c_begin, v[0]);
      if (c_begin + 32 < c_end) tmem_ld32_nw(t0 + c_begin + 32, v[1]);
      tmem_wait_ld();
      tc_fence_before();
      mbar_arrive(&tempty[acc]);
      if (m < g.M) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int c0 = c_begin + 32 * h;
          if (c0 < c_end) {
            const int nc = min(32, c_end - c0);  // multiple of 16
#pragma unroll
            for (int j = 0; j < 32; j += 8) {
              if (j < nc) {
                float* o = v[h] + j;
                if (g.bias) {
                  const float4 b0 = ldg4(g.bias + c0 + j), b1 = ldg4(g.bias + c0 + j + 4);
                  o[0] += b0.x; o[1] += b0.y; o[2] += b0.z; o[3] += b0.w; o[4] += b1.x; o[5] += b1.y; o[6] += b1.z; o[7] += b1.w;
                }
                if (g.accumulate) {
                  const float4 p0 = *reinterpret_cast<const float4*>(g.Y + m * g.ldy + c0 + j);
                  const float4 p1 = *reinterpret_cast<const float4*>(g.Y + m * g.ldy + c0 + j + 4);
                  o[0] += p0.x; o[1] += p0.y; o[2] += p0.z; o[3] += p0.w; o[4] += p1.x; o[5] += p1.y; o[6] += p1.z; o[7] += p1.w;
                }
                if (g.pre) store8(g.pre + m * g.ldp + c0 + j, o, wide);
                if (g.act == LCAO_ACT_SILU) {
#pragma unroll
                  for (int q = 0; q < 8; ++q) o[q] = silu_fast(o[q]);
                }
                if (g.G) {
                  const float4 h0 = ldg4(g.G + m * g.ldg + c0 + j), h1 = ldg4(g.G + m * g.ldg + c0 + j + 4);
                  o[0] *= silu_grad_fast(h0.x); o[1] *= silu_grad_fast(h0.y); o[2] *= silu_grad_fast(h0.z); o[3] *= silu_grad_fast(h0.w);
                  o[4] *= silu_grad_fast(h1.x); o[5] *= silu_grad_fast(h1.y); o[6] *= silu_grad_fast(h1.z); o[7] *= silu_grad_fast(h1.w);
                }
                store8(g.Y + m * g.ldy + c0 + j, o, wide);
              }
            }
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 8) {
    tc_fence_after();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

// =================================================================================================
// Kernel 2: weight gradient   dW[128, Kx] += sum_m dY[m, 0:128]^T X[m, 0:Kx] ,  db += colsum(dY)
// Both operands stream and the contraction runs over the rows m, so the row-major HBM tiles have to be
// TRANSPOSED into K-major operand tiles.  Pipeline (416 threads):
//   loaders (warps 9-12): cp.async 32-row chunks of dY and X into a raw row-major ring (16-byte pieces
//       XOR-swizzled by (row/4) so the transposing reads below are conflict free), 2-3 chunks ahead;
//   transform (warps 4-7): 4x4 register transposes raw -> SWIZZLE_128B K-major {A,B} x {hi,lo} tiles;
//   MMA (warp 8): short TMEM chains (8 chunks = 256 rows; the tensor core truncates on accumulate);
//   epilogue (warps 0-3): drain each chain into round-to-nearest FP32 registers, red.global.add at the end.
// =================================================================================================
struct WgradArgs {
  const float* dY; int64_t ldy;
  const float* X; int64_t ldx;
  float* dW; int64_t ldw;
  float* db;
  float* part;     // per-CTA partial sums: [grid][Kx][128] then [grid][128] column sums (deterministic two-stage reduction)
  int64_t M; int Kx; int x3, raw_stages, op_stages;
};

__global__ void __launch_bounds__(kRowsThreads, 1) k_tc_wgrad(const WgradArgs g) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rawA = kChunkK * 512, rawB = kChunkK * g.Kx * 4;     // raw chunk bytes (dY: 128 cols, X: Kx cols)
  const uint32_t opA = 128 * 128, opB = g.Kx * 128;                   // operand tile bytes (rows x 32 k)
  const uint32_t op_stage = (g.x3 ? 2 : 1) * (opA + opB);
  const int Rr = g.raw_stages, S = g.op_stages;
  uint8_t* sOp = smem_raw;                                            // 1024-aligned tiles first
  uint8_t* sRaw = sOp + (size_t)S * op_stage;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sRaw + (size_t)Rr * (rawA + rawB));
  uint64_t* raw_full = bars;             // [Rr] loaders -> transform
  uint64_t* raw_empty = raw_full + Rr;   // [Rr] transform -> loaders
  uint64_t* op_full = raw_empty + Rr;    // [S]  transform -> MMA
  uint64_t* op_empty = op_full + S;      // [S]  MMA -> transform
  uint64_t* tfull = op_empty + S;        // [2]
  uint64_t* tempty = tfull + 2;          // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
  constexpr int kFlush = 8;
  const uint32_t acc_cols = g.x3 ? 2 * g.Kx : g.Kx;
  const uint32_t need_cols = 2 * acc_cols;
  const uint32_t tmem_cols = need_cols <= 32 ? 32 : need_cols <= 64 ? 64 : need_cols <= 128 ? 128 : need_cols <= 256 ? 256 : 512;

  // contiguous row range of this CTA, in units of 32 rows
  const int64_t nchunks = (g.M + kChunkK - 1) / kChunkK;
  const int64_t per = (nchunks + gridDim.x - 1) / gridDim.x;
  const int64_t c_beg = min(nchunks, (int64_t)blockIdx.x * per), c_end = min(nchunks, c_beg + per);

  if (threadIdx.x == 0) {
    for (int s = 0; s < Rr; ++s) {
      mbar_init(&raw_full[s], kLoadWarps * 32);
      mbar_init(&raw_empty[s], 4 * 32);
    }
    for (int s = 0; s < S; ++s) {
      mbar_init(&op_full[s], 4 * 32);
      mbar_init(&op_empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull[a], 1);
      mbar_init(&tempty[a], kEpiWarps * 32);
    }
    fence_barrier_init();
  }
  if (warp == 8) tmem_alloc(tmem_slot, tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_trigger();
  pdl_wait();  // (set-up above overlaps the previous kernel's tail)
  if (c_beg >= c_end) {  // more CTAs than row chunks: nothing to do but to zero this CTA's partial slot
    for (int i = threadIdx.x; i < g.Kx * 128; i += kRowsThreads) g.part[(size_t)blockIdx.x * g.Kx * 128 + i] = 0.f;
    if (g.db && threadIdx.x < 128) g.part[(size_t)gridDim.x * g.Kx * 128 + (size_t)blockIdx.x * 128 + threadIdx.x] = 0.f;
    __syncthreads();
    if (warp == 8) tmem_dealloc(tmem_base, tmem_cols);
    return;
  }

  if (warp >= 9) {
    // ============================== loader warps ==============================
    // raw tile: row r (0..31) at r*pitch, 16-byte piece q stored at piece (q ^ (r >> 2)); lanes 0-7 of an
    // instruction copy 8 consecutive pieces of one row = one full 128-byte line on both sides.
    const int lw = warp - 9, r_in = lane >> 3, pl = lane & 7;
    const uint32_t raw_base = smem_u32(sRaw);
    const int pgB = g.Kx / 32;  // 128-byte piece groups per X row
    uint32_t it = 0;
    for (int64_t c = c_beg; c < c_end; ++c, ++it) {
      const int s = it % Rr;
      mbar_wait(&raw_empty[s], ((it / Rr) & 1) ^ 1);
      const uint32_t dA = raw_base + s * (rawA + rawB), dB = dA + rawA;
      const int64_t m0 = c * kChunkK;
#pragma unroll
      for (int j = 0; j < 8; ++j) {   // dY: 32 rows x 4 piece groups; this warp: rows 8 lw .. 8 lw + 7
        const int r = 8 * lw + (j & 1) * 4 + r_in, pg = j >> 1;
        const bool ok = m0 + r < g.M;
        cp_async16(dA + r * 512 + (((pg * 8 + pl) ^ (r >> 2)) << 4), ok ? g.dY + (m0 + r) * g.ldy + (pg * 8 + pl) * 4 : g.dY,
                   ok ? 16u : 0u);
      }
      for (int j = 0; j < 2 * pgB; ++j) {
        const int r = 8 * lw + (j & 1) * 4 + r_in, pg = j >> 1;
        const bool ok = m0 + r < g.M;
        cp_async16(dB + r * (g.Kx * 4) + (((pg * 8 + pl) ^ (r >> 2)) << 4), ok ? g.X + (m0 + r) * g.ldx + (pg * 8 + pl) * 4 : g.X,
                   ok ? 16u : 0u);
      }
      cp_async_arrive(&raw_full[s]);
    }
  } else if (warp >= 4 && warp < 8) {
    // ============================== transform warps ==============================
    const int t = threadIdx.x - 128;             // 0..127
    const int kg = t & 7, g0 = t >> 3;           // 4-row group of the chunk, first 4-column group
    const int ngB = g.Kx / 4;
    float4 colsum[2] = {make_float4(0.f, 0.f, 0.f, 0.f), make_float4(0.f, 0.f, 0.f, 0.f)};
    uint32_t it = 0;
    for (int64_t c = c_beg; c < c_end; ++c, ++it) {
      const int r = it % Rr, s = it % S;
      mbar_wait(&raw_full[r], (it / Rr) & 1);
      mbar_wait(&op_empty[s], ((it / S) & 1) ^ 1);
      const uint8_t* rA = sRaw + (size_t)r * (rawA + rawB);
      const uint8_t* rB = rA + rawA;
      uint8_t* oA = sOp + (size_t)s * op_stage;
      uint8_t* oB = oA + (g.x3 ? 2 : 1) * opA;
#pragma unroll
      for (int i = 0; i < 2; ++i) {              // A operand rows = dY columns: 32 column groups, 2 per thread
        const int ng = g0 + 16 * i;
        float4 v[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) v[q] = *reinterpret_cast<const float4*>(rA + (4 * kg + q) * 512 + ((ng ^ kg) << 4));
#pragma unroll
        for (int q = 0; q < 4; ++q)
          colsum[i] = make_float4(colsum[i].x + v[q].x, colsum[i].y + v[q].y, colsum[i].z + v[q].z, colsum[i].w + v[q].w);
        const float4 col[4] = {make_float4(v[0].x, v[1].x, v[2].x, v[3].x), make_float4(v[0].y, v[1].y, v[2].y, v[3].y),
                               make_float4(v[0].z, v[1].z, v[2].z, v[3].z), make_float4(v[0].w, v[1].w, v[2].w, v[3].w)};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float4 hi, lo;
          split4(col[j], hi, lo);
          const uint32_t off = sw128_off(4 * ng + j, kg);
          *reinterpret_cast<float4*>(oA + off) = hi;
          if (g.x3) *reinterpret_cast<float4*>(oA + opA + off) = lo;
        }
      }
      for (int ng = g0; ng < ngB; ng += 16) {    // B operand rows = X columns
        float4 v[4];
#pragma unroll
        for (int q = 0; q < 4; ++q)
          v[q] = *reinterpret_cast<const float4*>(rB + (4 * kg + q) * (g.Kx * 4) + ((ng ^ kg) << 4));
        const float4 col[4] = {make_float4(v[0].x, v[1].x, v[2].x, v[3].x), make_float4(v[0].y, v[1].y, v[2].y, v[3].y),
                               make_float4(v[0].z, v[1].z, v[2].z, v[3].z), make_float4(v[0].w, v[1].w, v[2].w, v[3].w)};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float4 hi, lo;
          split4(col[j], hi, lo);
          const uint32_t off = sw128_off(4 * ng + j, kg);
          *reinterpret_cast<float4*>(oB + off) = hi;
          if (g.x3) *reinterpret_cast<float4*>(oB + opB + off) = lo;
        }
      }
      fence_proxy_async();
      mbar_arrive(&op_full[s]);
      mbar_arrive(&raw_empty[r]);
    }
    if (g.db) {  // the 8 row-group threads (kg = lane & 7) of a column group are adjacent lanes
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        float4 c = colsum[i];
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) {
          c.x += __shfl_xor_sync(0xffffffffu, c.x, o); c.y += __shfl_xor_sync(0xffffffffu, c.y, o);
          c.z += __shfl_xor_sync(0xffffffffu, c.z, o); c.w += __shfl_xor_sync(0xffffffffu, c.w, o);
        }
        if (kg == 0)
          *reinterpret_cast<float4*>(g.part + (size_t)gridDim.x * g.Kx * 128 + (size_t)blockIdx.x * 128 + (g0 + 16 * i) * 4) = c;
      }
    }
  } else if (warp == 8) {
    // ============================== MMA issuer (all lanes run the loop; one is elected per instruction) ==============
    {
      const uint32_t idesc = make_idesc(kBlockM, g.Kx);
      const uint32_t base = smem_u32(sOp);
      uint32_t it = 0, fl = 0;
      for (int64_t c = c_beg; c < c_end; ++fl) {
        const int acc = fl & 1;
        mbar_wait(&tempty[acc], ((fl >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d = tmem_base + acc * acc_cols, dc = d + g.Kx;
        const int64_t c_stop = min(c_end, c + kFlush);
        for (int first = 1; c < c_stop; ++c, ++it) {
          const int s = it % S;
          mbar_wait(&op_full[s], (it / S) & 1);
          tc_fence_after();
          const uint32_t a_hi = base + s * op_stage, a_lo = a_hi + opA, b_hi = a_hi + (g.x3 ? 2 : 1) * opA, b_lo = b_hi + opB;
          // (a K step of 8 tf32 = 32 B inside the swizzled row: + 2 in the descriptor's 16-byte address field)
          const uint64_t dAh0 = make_desc_sw128(a_hi), dBh0 = make_desc_sw128(b_hi), dAl0 = make_desc_sw128(a_lo), dBl0 = make_desc_sw128(b_lo);
#pragma unroll
          for (int kk = 0; kk < kChunkK / 8; ++kk) {
            const uint64_t dAh = dAh0 + 2 * kk, dBh = dBh0 + 2 * kk, dAl = dAl0 + 2 * kk, dBl = dBl0 + 2 * kk;
            if (elect_one()) {
              umma_tf32(d, dAh, dBh, idesc, !first);
              if (g.x3) {
                umma_tf32(dc, dAl, dBh, idesc, !first);
                umma_tf32(dc, dAh, dBl, idesc, 1);
              }
            }
            first = 0;
          }
          if (elect_one()) umma_commit(&op_empty[s]);
        }
        if (elect_one()) umma_commit(&tfull[acc]);
      }
    }
    __syncwarp();
  } else {
    // ============================== epilogue warps: drain TMEM chains into registers, then dW += ==============
    constexpr int kMaxCols = 128;
    float sum[kMaxCols];
#pragma unroll
    for (int j = 0; j < kMaxCols; ++j) sum[j] = 0.f;
    const int64_t n_flush = (c_end - c_beg + kFlush - 1) / kFlush;
    for (int64_t fl = 0; fl < n_flush; ++fl) {
      const int acc = fl & 1;
      mbar_wait(&tfull[acc], (fl >> 1) & 1);
      tc_fence_after();
      const uint32_t t0 = tmem_base + ((uint32_t)(warp * 32) << 16) + acc * acc_cols;
#pragma unroll
      for (int c0 = 0; c0 < kMaxCols; c0 += 32) {
        if (c0 < g.Kx) {
          float v[32];
          tmem_ld32(t0 + c0, v);
#pragma unroll
          for (int j = 0; j < 32; ++j) sum[c0 + j] += v[j];
          if (g.x3) {
            tmem_ld32(t0 + g.Kx + c0, v);
#pragma unroll
            for (int j = 0; j < 32; ++j) sum[c0 + j] += v[j];
          }
        }
      }
      tc_fence_before();
      mbar_arrive(&tempty[acc]);
    }
    const int n = warp * 32 + lane;
    float* pp = g.part + (size_t)blockIdx.x * g.Kx * 128 + n;   // [cta][j][n]: coalesced over the 128 rows n
#pragma unroll
    for (int j = 0; j < kMaxCols; ++j)
      if (j < g.Kx) pp[(size_t)j * 128] = sum[j];
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 8) {
    tc_fence_after();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

// stage 2 of the weight gradient: dW[n, j] += sum_cta part[cta][j][n] ; db[n] += sum_cta part_db[cta][n].
// CTA = one column j (or the bias row), 8 thread rows split the CTA range, fixed-order tree over the 8 partial sums.
__global__ void __launch_bounds__(1024) k_wgrad_reduce(const float* __restrict__ part, int ncta, int Kx, float* __restrict__ dW,
                                                       int64_t ldw, float* __restrict__ db) {
  __shared__ float s_p[8][128];
  pdl_trigger();
  pdl_wait();
  const int j = blockIdx.x, n = threadIdx.x & 127, ty = threadIdx.x >> 7;
  const bool bias_row = j >= Kx;
  const float* src = bias_row ? part + (size_t)ncta * Kx * 128 + n : part + (size_t)j * 128 + n;
  const size_t stride = bias_row ? 128 : (size_t)Kx * 128;
  float acc = 0.f;
  for (int c = ty; c < ncta; c += 8) acc += src[(size_t)c * stride];
  s_p[ty][n] = acc;
  __syncthreads();
  if (ty == 0) {
    const float t = ((s_p[0][n] + s_p[1][n]) + (s_p[2][n] + s_p[3][n])) + ((s_p[4][n] + s_p[5][n]) + (s_p[6][n] + s_p[7][n]));
    if (bias_row) db[n] += t;
    else dW[(int64_t)n * ldw + j] += t;
  }
}

// stage 2 for SEVERAL weight gradients in one launch (blockIdx.y = gradient): a training step's weight gradients are only
// needed by the optimizer, so their stage-1 partials can wait and be summed together (31 launches of ~7 us -> one).
struct WgradDesc { const float* part; float* dW; float* db; int64_t ldw; int ncta, Kx; };
constexpr int kMaxWgradBatch = 32;
struct WgradBatch { WgradDesc d[kMaxWgradBatch]; };
__global__ void __launch_bounds__(1024) k_wgrad_reduce_batch(const WgradBatch b) {
  __shared__ float s_p[8][128];
  pdl_trigger();
  pdl_wait();
  const WgradDesc& g = b.d[blockIdx.y];
  const int j = blockIdx.x, n = threadIdx.x & 127, ty = threadIdx.x >> 7;
  if (j > g.Kx || (j == g.Kx && !g.db)) return;
  const bool bias_row = j >= g.Kx;
  const float* src = bias_row ? g.part + (size_t)g.ncta * g.Kx * 128 + n : g.part + (size_t)j * 128 + n;
  const size_t stride = bias_row ? 128 : (size_t)g.Kx * 128;
  float acc = 0.f;
  for (int c = ty; c < g.ncta; c += 8) acc += src[(size_t)c * stride];
  s_p[ty][n] = acc;
  __syncthreads();
  if (ty == 0) {
    const float t = ((s_p[0][n] + s_p[1][n]) + (s_p[2][n] + s_p[3][n])) + ((s_p[4][n] + s_p[5][n]) + (s_p[6][n] + s_p[7][n]));
    if (bias_row) g.db[n] += t;
    else g.dW[(int64_t)n * g.ldw + j] += t;
  }
}

constexpr size_t kMaxSmem = 227 * 1024;

int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

inline bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

}  // namespace

// ---- eligibility + launchers (called from linear.cu) -------------------------------------------
// rows kernel: contraction Kc % 32 == 0, output columns Nb % 16 == 0 and <= 128 per launch, weights resident.
static size_t rows_smem(int Kc, int Nb, int stages, int lo_stages) {
  const size_t halfB = (size_t)(Kc / kChunkK) * Nb * 128;
  return 2 * halfB + (size_t)(stages + lo_stages) * kStageBytes + 512 + 1024;
}

bool lcao_tc_rows_ok(int64_t M, int Kc, int Nb, int64_t lda, int64_t ldy, const void* A, const void* Y) {
  return M >= 512 && Kc % 32 == 0 && Kc >= 32 && Nb % 16 == 0 && Nb >= 16 && Nb <= 128 && lda % 4 == 0 && ldy % 4 == 0 &&
         al16(A) && al16(Y) && rows_smem(Kc, Nb, 2, 2) <= kMaxSmem;
}

int lcao_tc_rows(const float* A, int64_t lda, const float* W, int64_t ldw, int b_trans, const float* bias, const float* G,
                 int64_t ldg, float* Y, int64_t ldy, float* pre, int64_t ldp, int64_t M, int Kc, int Nb, int act,
                 int accumulate, int x3, cudaStream_t st) {
  RowsArgs g{};
  g.A = A; g.lda = lda; g.W = W; g.ldw = ldw; g.bias = bias; g.G = G; g.ldg = ldg; g.Y = Y; g.ldy = ldy;
  g.pre = pre; g.ldp = ldp; g.M = M; g.Kc = Kc; g.Nb = Nb; g.b_trans = b_trans; g.act = act; g.accumulate = accumulate;
  g.x3 = x3;
  g.wide_store = ((reinterpret_cast<uintptr_t>(Y) | (uintptr_t)(ldy * 4)) & 31u) == 0 &&
                 (!pre || ((reinterpret_cast<uintptr_t>(pre) | (uintptr_t)(ldp * 4)) & 31u) == 0);
  // the 3xTF32 weight (hi + lo) takes 128 KB at K = N = 128: 6 operand stages of 16 KB remain -> 3 hi + 3 lo
  int lo_stages = x3 ? 3 : 0;
  int stages = 8;
  while (stages > 2 && rows_smem(Kc, Nb, stages, lo_stages) > kMaxSmem) --stages;
  if (x3 && stages < 3 && lo_stages > 2) {  // keep the two rings balanced
    lo_stages = 2;
    stages = 8;
    while (stages > 2 && rows_smem(Kc, Nb, stages, lo_stages) > kMaxSmem) --stages;
  }
  g.stages = stages;
  g.lo_stages = x3 ? lo_stages : 1;  // (modulo operand only; no buffer is touched in 1x mode)
  const size_t smem = rows_smem(Kc, Nb, stages, lo_stages);
  static bool attr_set = false;
  if (!attr_set) {
    LCAO_CUDA(cudaFuncSetAttribute(k_tc_rows<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
    LCAO_CUDA(cudaFuncSetAttribute(k_tc_rows<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
    attr_set = true;
  }
  const int64_t nblocks = (M + kBlockM - 1) / kBlockM;
  const unsigned grid = (unsigned)(nblocks < num_sms() ? nblocks : num_sms());
  // eight epilogue warps pay when a CTA has a single tile (node- and table-sized layers: the drain is on the critical
  // path, 20.5 -> 18.4 us); with many tiles per CTA the drain overlaps the next tile's MMAs and they do not (85 -> 88 us)
  const bool epi8 = nblocks <= num_sms();
  // many tiles per CTA in 3xTF32 mode: the A-operand-in-tensor-memory kernel (twice the bytes in flight)
  if (x3 && nblocks >= 2 * num_sms() && Nb <= 128 && Kc % kChunkK == 0 &&
      2 * (size_t)(Kc / kChunkK) * Nb * 128 + 3 * kStageBytes + 512 + 1024 <= kMaxSmem) {
    static bool ta_attr = false;
    if (!ta_attr) {
      LCAO_CUDA(cudaFuncSetAttribute(k_tc_rows_ta, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
      ta_attr = true;
    }
    const size_t halfB = (size_t)(Kc / kChunkK) * Nb * 128;
    int R = 8;
    while (R > 2 && 2 * halfB + (size_t)R * kStageBytes + 512 + 1024 > kMaxSmem) --R;
    g.stages = R;
    const size_t smem_ta = 2 * halfB + (size_t)R * kStageBytes + 512 + 1024;
    LCAO_CUDA(launch_pdl(k_tc_rows_ta, grid, kTaThreads, smem_ta, st, g));
    LCAO_LAUNCH_CHECK();
    return LCAO_OK;
  }
  if (epi8) LCAO_CUDA(launch_pdl(k_tc_rows<true>, grid, kRowsThreads + 128, smem, st, g));
  else LCAO_CUDA(launch_pdl(k_tc_rows<false>, grid, kRowsThreads, smem, st, g));
  LCAO_LAUNCH_CHECK();
  return LCAO_OK;
}

static size_t wgrad_smem(int Kx, int x3, int raw_stages, int op_stages) {
  const size_t raw = (size_t)kChunkK * (512 + Kx * 4), op = (size_t)(x3 ? 2 : 1) * (128 * 128 + Kx * 128);
  return (size_t)raw_stages * raw + (size_t)op_stages * op + 512 + 1024;
}

bool lcao_tc_wgrad_ok(int64_t M, int Kx, int64_t ldy, int64_t ldx, const void* dY, const void* X) {
  return M >= 512 && Kx % 32 == 0 && Kx >= 32 && Kx <= 128 && ldy % 4 == 0 && ldx % 4 == 0 && al16(dY) && al16(X) &&
         wgrad_smem(Kx, 1, 2, 2) <= kMaxSmem;
}

// CTAs of the weight-gradient kernel: at least 128 rows (4 pipeline chunks) each; the per-CTA cost is one 64 KB
// partial tile, the per-chunk cost ~1.5 us of transform latency, so small M wants many CTAs
static unsigned wgrad_grid(int64_t M) {
  const int64_t want = (M + 127) / 128;
  return (unsigned)(want < 1 ? 1 : want < num_sms() ? want : num_sms());
}
// floats of scratch lcao_tc_wgrad needs
int64_t lcao_tc_wgrad_scratch(int64_t M, int Kx) { return (int64_t)wgrad_grid(M) * ((int64_t)Kx * 128 + 128); }

// dW (128 rows of the weight gradient, row stride ldw) += dY[:, 0:128]^T X[:, 0:Kx]
int lcao_tc_wgrad(const float* dY, int64_t ldy, const float* X, int64_t ldx, float* dW, int64_t ldw, float* db, int64_t M,
                  int Kx, int x3, float* part, cudaStream_t st, int64_t* defer_desc) {
  WgradArgs g{};
  g.dY = dY; g.ldy = ldy; g.X = X; g.ldx = ldx; g.dW = dW; g.ldw = ldw; g.db = db; g.part = part;
  g.M = M; g.Kx = Kx; g.x3 = x3;
  g.op_stages = 2;
  int raw_stages = 6;
  while (raw_stages > 2 && wgrad_smem(Kx, x3, raw_stages, g.op_stages) > kMaxSmem) --raw_stages;
  g.raw_stages = raw_stages;
  static bool attr_set = false;
  if (!attr_set) {
    LCAO_CUDA(cudaFuncSetAttribute(k_tc_wgrad, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
    attr_set = true;
  }
  const unsigned grid = wgrad_grid(M);
  LCAO_CUDA(launch_pdl(k_tc_wgrad, grid, kRowsThreads, wgrad_smem(Kx, x3, raw_stages, g.op_stages), st, g));
  LCAO_LAUNCH_CHECK();
  if (defer_desc) {  // stage 2 is left to lcao_wgrad_reduce_batch: {part, dW, db, ldw, ncta, Kx}
    defer_desc[0] = (int64_t)(uintptr_t)part; defer_desc[1] = (int64_t)(uintptr_t)dW; defer_desc[2] = (int64_t)(uintptr_t)db;
    defer_desc[3] = ldw; defer_desc[4] = (int64_t)grid; defer_desc[5] = Kx;
    return LCAO_OK;
  }
  LCAO_CUDA(launch_pdl(k_wgrad_reduce, Kx + (db ? 1 : 0), 1024, 0, st, (const float*)part, (int)grid, Kx, dW, ldw, db));
  LCAO_LAUNCH_CHECK();
  return LCAO_OK;
}

// sums the partial tiles of n deferred weight gradients (descriptors of 6 int64 written by lcao_tc_wgrad) into their dW / db
int lcao_tc_wgrad_reduce_batch(const int64_t* desc, int n, cudaStream_t st) {
  for (int i0 = 0; i0 < n; i0 += kMaxWgradBatch) {
    WgradBatch b{};
    const int m = n - i0 < kMaxWgradBatch ? n - i0 : kMaxWgradBatch;
    int kmax = 0;
    for (int i = 0; i < m; ++i) {
      const int64_t* d = desc + 6 * (int64_t)(i0 + i);
      b.d[i].part = reinterpret_cast<const float*>((uintptr_t)d[0]);
      b.d[i].dW = reinterpret_cast<float*>((uintptr_t)d[1]);
      b.d[i].db = reinterpret_cast<float*>((uintptr_t)d[2]);
      b.d[i].ldw = d[3]; b.d[i].ncta = (int)d[4]; b.d[i].Kx = (int)d[5];
      kmax = b.d[i].Kx > kmax ? b.d[i].Kx : kmax;
    }
    LCAO_CUDA(launch_pdl(k_wgrad_reduce_batch, dim3((unsigned)(kmax + 1), (unsigned)m), 1024, 0, st, b));
    LCAO_LAUNCH_CHECK();
  }
  return LCAO_OK;
}
