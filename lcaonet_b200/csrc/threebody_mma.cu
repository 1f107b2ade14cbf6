// Three-body message passing (lcaonet.py:173-189 + shbf.py:75-87 + lcaonet.py:431-435) with the per-node dense
// products on the warp-level tensor-core path (mma.sync m16n8k8 TF32, FP32 accumulate), forward and backward.
//
// Per centre node s with in-edges i (k->s) and out-edges j (s->t), and per pair coefficients
//   a[j,i,l] = Y_l(cos(j,i)) / max(|v_ji|, eps),  |v_ji|^2 = Y^T G_i Y  (Gram form, see threebody.cu / DESIGN.md R3)
// the whole layer is three small dense products per node (GB = gate[k_i] * B[i]):
//   forward   tbw[j,:]      = sum_{i,l} a[j,i,l] GB[i,l,:]                   (dO x dI*NL) . (dI*NL x C)
//   backward  D[(i,l),j]    = sum_c GB[i,l,c] Gt[j,c]                        (dI*NL x C) . (C x dO)      Gt = d tbw
//             dGB[(i,l),:]  = sum_j a[j,i,l] Gt[j,:]                         (dI*NL x dO) . (dO x C)
// plus O(pairs) scalar work (the coefficient chain, the norm path H_i = -sum_j dot_ij a a^T, cos gradients).
// On the FP32 pipe these products were 35 of the 91 warp instructions per triplet and the kernels were issue/latency
// bound at a third of the HBM roofline (profiles/r01_notes.md).  Here they are m16n8k8 TF32 MMAs with the 3xTF32
// operand split (x = hi + lo, hi = RN to TF32; lo.hi + hi.lo + hi.hi, FP32 accumulate: FP32-equivalent, as in the dense
// layers): ~3 MMAs per pair, and the coefficient of a pair is computed by exactly the thread whose A-fragment
// needs it, so there is no shared-memory broadcast and no block barrier on the energy path.
//
// Fragment <-> data mapping (g = lane >> 2, t = lane & 3; PTX ISA m16n8k8 .tf32 layouts):
//   forward   M = 16 out-edges, K-step = (l, 8 in-edges), N-tile = 8 channels.  Thread (g,t) owns the pairs
//             (j in {g, g+8}) x (i in {t, t+4}) of a block and, for every l, builds A = a[.,.,l] from them.
//             Channel of column n in tile nt:  (nt>>2)*32 + n*4 + (nt&3)  -> every B-fragment load and every
//             output store is a float4, and a warp-wide load instruction covers 4 rows x 128 contiguous bytes.
//   backward  M = 16 rows (l, i) of a tile of IPT in-edges (IPT = 4 for NL in {3,4}, 8 for NL in {1,2}; rows g and
//             g + 8 belong to the SAME in-edge), phase 1: K = channels, N = 8 out-edges -> D; thread (g,t) then holds
//             D for the pairs (i = g % IPT) x (j in {2t, 2t+1}) whose coefficients it computes, which is exactly
//             the A-fragment of phase 2 (K = out-edges permuted k=t <-> j=2t, k=t+4 <-> j=2t+1, N = channels).
// Sums over triplets stay in accumulator registers and are written once: no atomics (forces: see kJS), deterministic.
//
// C <= 128 (one 128-channel accumulator block per warp); wider layers take the FP32-pipe kernels in threebody.cu.
#include "common.cuh"
#include "tb_common.cuh"
#include "tb_async.cuh"
#include "tb_mma.cuh"

namespace {

__device__ __forceinline__ float f4c(const float4& v, int i) { return i == 0 ? v.x : i == 1 ? v.y : i == 2 ? v.z : v.w; }

constexpr int kIB = 8;      // in-edges per forward stage = one K-block of the MMAs
constexpr int kStages = 2;  // forward ring depth: one item in flight behind the one being multiplied (41 KB per CTA: five CTAs per SM; three stages / three CTAs: 0.248 ms, two / five: 0.190 ms, one: 0.203 ms)

// Shared-memory plan of one forward CTA: two stages of
//   [B rows | gate rows | unit + edge id of the in-edges | their Gram rows | unit + edge id of the 16 out-edge rows | item]
// plus two buffers of A fragments (coefficients, hi and lo).  Rows are padded by 8 floats so that the four in-edges a
// quarter-warp reads in one LDS.128 fall into different banks.
struct FwdPlan {
  int pB, pG;                 // row pitches in floats: B (NL*C + 8), gate (C + 8)
  int oG, oU, oGm, oR, oD;    // offsets inside a stage (floats); B rows start the stage
  int stage, oA, total;       // floats
};
__host__ __device__ inline FwdPlan fwd_plan(int C, int NL) {
  FwdPlan p;
  p.pB = NL * C + 8;
  p.pG = C + 8;
  p.oG = kIB * p.pB;
  p.oU = p.oG + kIB * p.pG;
  p.oGm = p.oU + kIB * 4;                 // (8-byte aligned: every term above is a multiple of 4 floats)
  p.oR = p.oGm + kIB * NL * (NL + 1);     // NP doubles per in-edge
  p.oD = p.oR + 16 * 4;
  p.stage = p.oD + 4;
  p.oA = 16 + kStages * p.stage;          // [0, 64 B): full[kStages] and empty[kStages] mbarriers
  p.total = p.oA + 2 * NL * 2 * 128;
  return p;
}
enum { kItemFirst = 1, kItemLast = 2, kItemEnd = 4 };

// ---------------------------------------------------------------------------------------------
// forward: CTA = 4 consumer warps (the four 32-channel quarters of C <= 128) + 1 producer warp.
// Work items = (node, M-tile of <= 16 out-edges, block of <= 8 in-edges), walked in order by the producer, which
// keeps the copy engine ahead through a ring of kStages stages (full / empty mbarriers): while item n is multiplied,
// the bulk copies of item n+1 are in flight, and the unit vectors / Gram rows / edge ids of the items after it sit in
// the producer's registers.  The ring is kept SHALLOW (two stages, 41 KB per CTA) so that five CTAs are resident per SM:
// the bytes in flight (a B200 SM needs ~100 KB of row gathers in flight to reach the HBM rate,
// scripts/micro/bulk_copy.cu) come from the number of CTAs, and so do the warps that hide each other's latencies.  The 128 coefficients of an item are computed one per consumer thread and exchanged
// through shared memory in fragment order (one named barrier among the consumers per item).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void consumer_sync() { asm volatile("bar.sync 1, 128;" ::: "memory"); }

template <int NL>
__global__ void __launch_bounds__(160) k_tb_fwd_mma(
    const float* __restrict__ B, int NG, const double* __restrict__ gram, const float* __restrict__ unit,
    const float* __restrict__ gate, int64_t ldg, const int32_t* __restrict__ in_ptr, const int32_t* __restrict__ in_edge,
    const int32_t* __restrict__ in_src, const int32_t* __restrict__ out_ptr, const int32_t* __restrict__ out_edge, int N,
    int C, float* __restrict__ tbw) {
  pdl_trigger();  // (programmatic dependent launch: the next kernel may start its set-up; common.cuh)
  constexpr int NP = NL * (NL + 1) / 2;
  extern __shared__ __align__(16) float smem[];
  const FwdPlan pl = fwd_plan(C, NL);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, tig = lane & 3;
  const uint32_t bar_full = smem_u32(smem), bar_empty = bar_full + 8 * kStages;
  if (threadIdx.x == 0) {
    for (int i = 0; i < kStages; ++i) { mbar_init(bar_full + 8 * i, 1); mbar_init(bar_empty + 8 * i, 4); }
  }
  __syncthreads();
  pdl_wait();  // (launched through launch_pdl: the set-up above may overlap the previous kernel's tail)
  // every CTA walks a CONTIGUOUS range of nodes: CSR pointers and in-edge id lists are read front to back
  const int per_cta = (N + (int)gridDim.x - 1) / (int)gridDim.x;
  const int s_end = min(N, ((int)blockIdx.x + 1) * per_cta);

  if (warp == 4) {
    // ------------------------------------------------------------------ producer
    struct Cur { int s, ib, dI, ob, dO, jb, i0; bool valid; };
    struct Ids { int ep, k, ej; };                                  // lane < 8: in-edge i0 + lane ; lane < 16: out-edge row
    struct Dat { float vx, vy, vz, ux, uy, uz; double gm[NP]; };    // unit + Gram of the in-edge, unit of the out-edge row
    auto load_node = [&](Cur& c) {  // first node at or after c.s that has out-edges
      c.valid = false;
      while (c.s < s_end) {
        c.ib = in_ptr[c.s]; c.dI = in_ptr[c.s + 1] - c.ib; c.ob = out_ptr[c.s]; c.dO = out_ptr[c.s + 1] - c.ob;
        if (c.dO > 0) { c.valid = true; return; }
        c.s += 1;
      }
    };
    auto advance = [&](Cur& c) {
      if (!c.valid) return;
      c.i0 += kIB;
      if (c.i0 < c.dI) return;
      c.i0 = 0;
      c.jb += 16;
      if (c.jb < c.dO) return;
      c.jb = 0;
      c.s += 1;
      load_node(c);
    };
    auto load_ids = [&](const Cur& c, Ids& r) {
      r.ep = 0; r.k = 0; r.ej = 0;
      if (!c.valid) return;
      if (lane < kIB && c.i0 + lane < c.dI) { r.ep = in_edge[c.ib + c.i0 + lane]; r.k = in_src[c.ib + c.i0 + lane]; }
      if (lane < 16) r.ej = out_edge[c.ob + c.jb + min(lane, min(16, c.dO - c.jb) - 1)];
    };
    auto load_dat = [&](const Cur& c, const Ids& r, Dat& d) {
      if (!c.valid) return;
      if (lane < kIB && c.i0 + lane < c.dI) {
        d.vx = unit[3 * (int64_t)r.ep]; d.vy = unit[3 * (int64_t)r.ep + 1]; d.vz = unit[3 * (int64_t)r.ep + 2];
#pragma unroll
        for (int x = 0; x < NP; ++x) d.gm[x] = gram[(int64_t)r.ep * NP + x];
      }
      if (lane < 16) { d.ux = unit[3 * (int64_t)r.ej]; d.uy = unit[3 * (int64_t)r.ej + 1]; d.uz = unit[3 * (int64_t)r.ej + 2]; }
    };
    auto issue = [&](int st, const Cur& c, const Ids& r, const Dat& d) {  // fill stage st with item c (or the END marker)
      float* sS = smem + 16 + st * pl.stage;
      const uint32_t bar = bar_full + 8 * st;
      const int n = c.valid ? max(0, min(kIB, c.dI - c.i0)) : 0;
      if (c.valid) {
        if (lane < n) {
          *reinterpret_cast<float4*>(sS + pl.oU + lane * 4) = make_float4(d.vx, d.vy, d.vz, __int_as_float(r.ep));
          double* sGm = reinterpret_cast<double*>(sS + pl.oGm);
#pragma unroll
          for (int x = 0; x < NP; ++x) sGm[lane * NP + x] = d.gm[x];
        }
        if (lane < 16) *reinterpret_cast<float4*>(sS + pl.oR + lane * 4) = make_float4(d.ux, d.uy, d.uz, __int_as_float(r.ej));
      }
      if (lane == 0) {
        const int flags = !c.valid ? kItemEnd : ((c.i0 == 0 ? kItemFirst : 0) | (c.i0 + kIB >= c.dI ? kItemLast : 0));
        *reinterpret_cast<int4*>(sS + pl.oD) = make_int4(n, c.valid ? min(16, c.dO - c.jb) : 0, flags, 0);
      }
      __syncwarp();
      if (lane == 0) mbar_expect_tx(bar, (uint32_t)n * (uint32_t)(NL * C + C) * 4u);  // (release: the stores above are visible to the waiters)
      __syncwarp();
      if (lane < n) {
        bulk_g2s(smem_u32(sS + lane * pl.pB), B + (int64_t)r.ep * NG * C, (uint32_t)(NL * C) * 4u, bar);
        bulk_g2s(smem_u32(sS + pl.oG + lane * pl.pG), gate + (int64_t)r.k * ldg, (uint32_t)C * 4u, bar);
      }
    };
    Cur c0, c1, c2;
    Ids i0r, i1, i2;
    Dat d0, d1;
    c0.s = (int)blockIdx.x * per_cta; c0.jb = 0; c0.i0 = 0;
    load_node(c0);
    load_ids(c0, i0r);
    load_dat(c0, i0r, d0);
    c1 = c0; advance(c1); load_ids(c1, i1);
    c2 = c1;
    for (int it = 0;; ++it) {
      const int st = it % kStages;
      if (it >= kStages) mbar_wait(bar_empty + 8 * st, ((it / kStages) - 1) & 1u);  // the consumers are done with this stage
      issue(st, c0, i0r, d0);
      if (!c0.valid) break;
      // shift: item n+1 becomes current (its ids arrived an iteration ago -> its data loads go out now); ids of n+2
      c0 = c1; i0r = i1;
      load_dat(c0, i0r, d1);
      d0 = d1;
      advance(c2);
      load_ids(c2, i2);
      c1 = c2; i1 = i2;
    }
    return;
  }

  // ------------------------------------------------------------------ consumers (warp w = channels [32w, 32w+32))
  float acc[4][4];
  const int q0 = warp * 32;
  // coefficient duty of this thread: the pair whose A-fragment slot is (lane, warp): row j, in-edge i
  const int cj = (lane >> 2) + 8 * (warp & 1), ci = (lane & 3) + 4 * (warp >> 1);
  for (int it = 0;; ++it) {
    const int st = it % kStages;
    const float* sS = smem + 16 + st * pl.stage;
    mbar_wait(bar_full + 8 * st, (it / kStages) & 1u);
    const int4 item = *reinterpret_cast<const int4*>(sS + pl.oD);
    const int n = item.x, nr = item.y, flags = item.z;
    if (flags & kItemEnd) break;
    float* sA = smem + pl.oA + (it & 1) * (NL * 2 * 128);
    // ---- coefficient of this thread's pair -> its slot of the A fragments (hi | lo) of the NL K-steps
    {
      const float4 rv = lds4f(sS + pl.oR + min(cj, max(nr, 1) - 1) * 4);
      const float4 uv = lds4f(sS + pl.oU + min(ci, max(n, 1) - 1) * 4);
      float w = 0.f;
      float Y[4] = {0.f, 0.f, 0.f, 0.f};
      if (cj < nr && ci < n && __float_as_int(uv.w) != __float_as_int(rv.w)) {
        const double* sGm = reinterpret_cast<const double*>(sS + pl.oGm) + ci * NP;
        double gm[NP];
#pragma unroll
        for (int x = 0; x < NP; ++x) gm[x] = sGm[x];
        const float c = fmaf(rv.x, uv.x, fmaf(rv.y, uv.y, rv.z * uv.z));
        sph_harm<NL>(c, Y);
        w = 1.0f / fmaxf(sqrtf(fmaxf((float)quad_form<NL>(gm, Y), 0.f)), kEps);
      }
#pragma unroll
      for (int l = 0; l < NL; ++l) {
        uint32_t hi, lo;
        split_tf32(w * Y[l], hi, lo);
        sA[(l * 2) * 128 + lane * 4 + warp] = __uint_as_float(hi);
        sA[(l * 2 + 1) * 128 + lane * 4 + warp] = __uint_as_float(lo);
      }
    }
    consumer_sync();  // A fragments complete (and every consumer is done with the A buffer of item it - 1)
    if (flags & kItemFirst) {
#pragma unroll
      for (int t = 0; t < 4; ++t)
#pragma unroll
        for (int x = 0; x < 4; ++x) acc[t][x] = 0.f;
    }
    if (n > 0 && q0 < C) {
      const int il0 = min(tig, n - 1), il1 = min(tig + 4, n - 1);
      const bool ok = q0 + g * 4 < C;
      const float* b0p = sS + il0 * pl.pB + q0 + g * 4;
      const float* b1p = sS + il1 * pl.pB + q0 + g * 4;
      const float4 gt0 = ok ? lds4f(sS + pl.oG + il0 * pl.pG + q0 + g * 4) : zero4();
      const float4 gt1 = ok ? lds4f(sS + pl.oG + il1 * pl.pG + q0 + g * 4) : zero4();
#pragma unroll
      for (int l = 0; l < NL; ++l) {
        const float4 a_hi = lds4f(sA + (l * 2) * 128 + lane * 4), a_lo = lds4f(sA + (l * 2 + 1) * 128 + lane * 4);
        const uint32_t ah[4] = {__float_as_uint(a_hi.x), __float_as_uint(a_hi.y), __float_as_uint(a_hi.z), __float_as_uint(a_hi.w)};
        const uint32_t al[4] = {__float_as_uint(a_lo.x), __float_as_uint(a_lo.y), __float_as_uint(a_lo.z), __float_as_uint(a_lo.w)};
        const float4 x0 = ok ? mul4(gt0, lds4f(b0p + l * C)) : zero4();
        const float4 x1 = ok ? mul4(gt1, lds4f(b1p + l * C)) : zero4();
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          uint32_t bh0, bl0, bh1, bl1;
          split_tf32(f4c(x0, r), bh0, bl0);
          split_tf32(f4c(x1, r), bh1, bl1);
          mma_3x(acc[r], ah, al, bh0, bh1, bl0, bl1);
        }
      }
    }
    int e0 = 0, e1 = 0;
    if (flags & kItemLast) {
      e0 = __float_as_int(sS[pl.oR + min(g, nr - 1) * 4 + 3]);
      e1 = __float_as_int(sS[pl.oR + min(g + 8, nr - 1) * 4 + 3]);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(bar_empty + 8 * st);  // this warp is done with the stage
    if ((flags & kItemLast) && q0 < C) {
      // ---- tile finished: accumulator (row g / g+8, columns 2t, 2t+1 of N-tile r) -> channels q0 + 8t + r and + 4 + r
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        const int ch = q0 + 8 * tig + 4 * hh;
        if (ch < C) {
          if (g < nr) st4(tbw + (int64_t)e0 * C + ch, make_float4(acc[0][hh], acc[1][hh], acc[2][hh], acc[3][hh]));
          if (g + 8 < nr) st4(tbw + (int64_t)e1 * C + ch, make_float4(acc[0][2 + hh], acc[1][2 + hh], acc[2][2 + hh], acc[3][2 + hh]));
        }
      }
    }
  }
}

// (A backward kernel in the same formulation — tile of 4 in-edges x all out-edges per warp, D = GB.Gt^T and dGB = a^T.Gt as
//  m16n8k8 MMAs, per-thread LDGs — was built and verified in round 2: 232 M warp instructions against 302 M for the
//  FP32-pipe kernel, but 168 registers + spills, 10 resident warps per SM and a 240 KB instruction footprint made it
//  2x SLOWER (0.97 ms against 0.46 ms at config 2).  It is not shipped; profiles/r02_notes.md has the numbers.)

constexpr int kFwdCtasPerSm = 40;  // grid cap per SM; each CTA takes a contiguous range of nodes

}  // namespace

// (argument checks are done by the C entry points in threebody.cu, which dispatch here for C <= 128)
int lcao_tb_mma_fwd(const float* B, int32_t NG, const double* gram, const float* unit, const float* gate, int64_t ldg,
                    const int32_t* in_ptr, const int32_t* in_edge, const int32_t* in_src, const int32_t* out_ptr,
                    const int32_t* out_edge, int64_t N, int32_t C, int32_t NL, float* tbw, cudaStream_t st) {
  const int64_t want = (N + 1) / 2;  // at least two nodes per CTA
  const unsigned grid = (unsigned)(want < 148ll * kFwdCtasPerSm ? (want > 0 ? want : 1) : 148ll * kFwdCtasPerSm);
  const size_t smem = sizeof(float) * (size_t)fwd_plan(C, NL).total;
#define CALL(nl)                                                                                                     \
  {                                                                                                                  \
    static bool attr_done = false;                                                                                   \
    if (!attr_done) {                                                                                                \
      LCAO_CUDA(cudaFuncSetAttribute(k_tb_fwd_mma<nl>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));      \
      attr_done = true;                                                                                              \
    }                                                                                                                \
    LCAO_CUDA(launch_pdl(k_tb_fwd_mma<nl>, grid, 160, smem, st, B, NG, gram, unit, gate, ldg, in_ptr, in_edge, in_src, out_ptr, out_edge, \
                                              (int)N, C, tbw));                                                       \
  }
  switch (NL) {
    case 1: CALL(1) break;
    case 2: CALL(2) break;
    case 3: CALL(3) break;
    default: CALL(4) break;
  }
#undef CALL
  LCAO_LAUNCH_CHECK();
  return LCAO_OK;
}

