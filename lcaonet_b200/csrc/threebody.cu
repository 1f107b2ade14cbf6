// Fused three-body message passing (lcaonet.py:173-189 + shbf.py:75-87 + lcaonet.py:431-435),
// forward and backward, one CTA per centre node s.
//
// All out-edges e=(s->t) of a node share the same set of in-edges e'=(k->s).  With
//   B[e',l,:]  = sum_{o in l} rb[e',o] cst'[e',o,:]        (orbital contraction grouped by l, pair_table.cu)
//   GB[e',l,:] = sigmoid(xk[k,:]) * B[e',l,:]              (gate folded in once per in-edge)
//   G[e']      = Gram matrix B[e',l,:].B[e',l',:]          (NL x NL, FP64, once per in-edge)
// the reference's per-triplet chain  v = sum_l Y_l(c) B_l ; y = v / max(|v|, eps) ; tbw[e] += y * gate
// becomes, exactly,
//   |v|^2 = Y^T G Y   (a 3x3 quadratic form per triplet instead of a C-wide reduction)
//   tbw[e,:] = sum_{e'} sum_l  a[e,e',l] * GB[e',l,:],      a = Y_l(c) / max(|v|, eps)
// i.e. per node one small dense product (deg_out x deg_in*NL) x (deg_in*NL x C) on the FP32 pipes:
// NL FMAs per triplet-channel, no cross-lane reduction in the forward at all.  No triplet-sized tensor
// (the reference's (T,O,C) gather, cos(theta), Y_l(T,O)) exists; cos(theta) = unit[e].unit[e'] and Y_l
// are recomputed per (e,e') pair by one thread and broadcast through shared memory.
//
// These FP32-pipe kernels serve 128 < C <= 256; C <= 128 goes to threebody_mma.cu (forward) and threebody_staged.cu
// (backward).  Both entry points require 16-byte-aligned B, gate and d_tbw (read in float4 rows or by bulk copies)
// and tbw, dB, q and dP (written or read in float4 rows).
//
// Thread mapping: lane <-> float4 channel columns (lane and lane + 32), warp <-> 8 out-edges of a node
// (forward: 8 register accumulators) or one in-edge (backward).  Warps are independent: B / gate / d_tbw
// rows are read straight from global memory (L1/L2 serve the re-reads by the sibling warps of the same
// node), the per-pair coefficients are computed by the lanes of the warp itself (one pair per lane)
// and broadcast through a 512-byte per-warp scratch.  There is no block-level staging and no
// __syncthreads on the energy path, so many nodes are in flight per SM and the latency of one node's
// index -> row chain is hidden by the others.  Sums over triplets accumulate in registers and are
// written once: no atomics, deterministic.
//
// `gate` is sigmoid(xk) per NODE (N x C, computed once per layer by lcao_sigmoid_rows).
#include "common.cuh"
#include "tb_common.cuh"

namespace {

constexpr int kFwdWarps = 2;   // forward CTA: 2 warps x 8 out-edges per pass
constexpr int kBwdWarps = 4;   // backward CTA: 4 warps, one in-edge per warp at a time (2 measured slower: 168 vs 128 registers)
constexpr int kR = 8;          // forward: out-edge accumulators per warp
constexpr int kIB = 4;         // forward: in-edges per coefficient batch (kR * kIB = 32 pairs = one per lane)
constexpr int kV4 = 2;         // float4 channel columns per lane: these kernels serve 128 < C <= 256
constexpr int kFwdCtasPerSm = 48, kBwdCtasPerSm = 24;  // grid caps (grid-stride over the centre nodes)

// (Packed FP32 pairs — fma.rn.f32x2 / FFMA2 — were tried for the FMA blocks: same FP32 pipe rate (measured 36.8 vs
// 36.2 TFMA/s, scripts/micro/ffma2.cu) and the forward kernel ran 2x SLOWER with them; see profiles/r01_notes.md.)

// ---------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------
// Out-of-range slots (out-edge r >= nr, in-edge beyond the node's list) are handled by CLAMPING the
// index to a valid row and zeroing the pair's coefficient, so the row loads and the FMA block are
// branch- and predicate-free.  (Fitting the slot grid to the node — R = 8 / 6 / 4 accumulator rows, skipping the
// FMA block of in-edges beyond the tail, per-row guards — removed up to 30 % of the issued FMAs and did not make the
// kernel faster: it is bound by the latency of each warp's dependent chain, not by issue slots; profiles/r01_notes.md.)

// One block of nr <= kR out-edges (positions ob + jb ..) of a node against all its dI in-edges.
template <int NL>
__device__ __forceinline__ void tb_fwd_block(const float* __restrict__ B, int NG, const double* __restrict__ gram,
                                             const float* __restrict__ unit, const float* __restrict__ gate, int64_t ldg,
                                             const int32_t* __restrict__ in_edge, const int32_t* __restrict__ in_src,
                                             const int32_t* __restrict__ out_edge, int C, float* __restrict__ tbw,
                                             float* sa, int lane, const bool (&okc)[kV4], int ib, int dI, int ob, int jb,
                                             int nr) {
  constexpr int NP = NL * (NL + 1) / 2;
  const int r_mine = lane % kR, t_mine = lane / kR;  // coefficient duty: pair (in-edge t, out-edge r)
  // lane (r, t) keeps out-edge r of this block: id and direction
  const int e_mine = out_edge[ob + jb + min(r_mine, nr - 1)];
  const float ux = unit[3 * (int64_t)e_mine], uy = unit[3 * (int64_t)e_mine + 1], uz = unit[3 * (int64_t)e_mine + 2];
  float4 acc[kR][kV4];
#pragma unroll
  for (int r = 0; r < kR; ++r)
#pragma unroll
    for (int v = 0; v < kV4; ++v) acc[r][v] = zero4();

  for (int ic = 0; ic < dI; ic += 32) {  // the node's in-edge ids, 32 at a time, one per lane
    const int nI = min(32, dI - ic);
    const int my_ep = in_edge[ib + ic + min(lane, nI - 1)];
    const int my_k = in_src[ib + ic + min(lane, nI - 1)];
    for (int i0 = 0; i0 < nI; i0 += kIB) {
      // ---- coefficients of the kR x kIB pairs of this batch, one per lane
      const int ep_c = __shfl_sync(0xffffffffu, my_ep, min(i0 + t_mine, nI - 1));
      float4 a = zero4();
      {
        const float c = fmaf(ux, unit[3 * (int64_t)ep_c], fmaf(uy, unit[3 * (int64_t)ep_c + 1], uz * unit[3 * (int64_t)ep_c + 2]));
        float Y[4];
        sph_harm<NL>(c, Y);
        double g[NP];
#pragma unroll
        for (int p = 0; p < NP; ++p) g[p] = gram[(int64_t)ep_c * NP + p];
        float w = 1.0f / fmaxf(sqrtf(fmaxf((float)quad_form<NL>(g, Y), 0.f)), kEps);
        if (r_mine >= nr || i0 + t_mine >= nI || ep_c == e_mine) w = 0.f;
        a = make_float4(w * Y[0], w * Y[1], w * Y[2], w * Y[3]);
      }
      __syncwarp();  // previous batch's readers are done
      st4(sa + (t_mine * 8 + r_mine) * 4, a);
      __syncwarp();
      // ---- rows of the batch: issue every load first, then the FMAs
      float4 gb[kIB][NL][kV4];
#pragma unroll
      for (int t = 0; t < kIB; ++t) {
        const int src = min(i0 + t, nI - 1);
        const int ep = __shfl_sync(0xffffffffu, my_ep, src);
        const int k = __shfl_sync(0xffffffffu, my_k, src);
#pragma unroll
        for (int v = 0; v < kV4; ++v) {
          const int c = (lane + 32 * v) * 4;
          const float4 gt = okc[v] ? ldg4(gate + (int64_t)k * ldg + c) : zero4();
#pragma unroll
          for (int l = 0; l < NL; ++l) gb[t][l][v] = okc[v] ? mul4(gt, ldg4(B + ((int64_t)ep * NG + l) * C + c)) : zero4();
        }
      }
#pragma unroll
      for (int t = 0; t < kIB; ++t) {
#pragma unroll
        for (int r = 0; r < kR; ++r) {
          const float4 ar = lds4(sa + (t * 8 + r) * 4);
#pragma unroll
          for (int v = 0; v < kV4; ++v) {
            acc[r][v] = fma4(ar.x, gb[t][0][v], acc[r][v]);
            if (NL > 1) acc[r][v] = fma4(ar.y, gb[t][1][v], acc[r][v]);
            if (NL > 2) acc[r][v] = fma4(ar.z, gb[t][2][v], acc[r][v]);
            if (NL > 3) acc[r][v] = fma4(ar.w, gb[t][3][v], acc[r][v]);
          }
        }
      }
    }
  }
#pragma unroll
  for (int r = 0; r < kR; ++r) {
    const int e = __shfl_sync(0xffffffffu, e_mine, r);
    if (r < nr) {
#pragma unroll
      for (int v = 0; v < kV4; ++v) {
        const int c = (lane + 32 * v) * 4;
        if (okc[v]) st4(tbw + (int64_t)e * C + c, acc[r][v]);
      }
    }
  }
}

template <int NL>
__global__ void __launch_bounds__(kFwdWarps * 32, 8) k_threebody_fwd(
    const float* __restrict__ B, int NG, const double* __restrict__ gram, const float* __restrict__ unit,
    const float* __restrict__ gate, int64_t ldg, const int32_t* __restrict__ in_ptr,
    const int32_t* __restrict__ in_edge, const int32_t* __restrict__ in_src, const int32_t* __restrict__ out_ptr,
    const int32_t* __restrict__ out_edge, int N, int C, float* __restrict__ tbw) {
  pdl_trigger();  // (programmatic dependent launch: the next kernel may start its set-up; common.cuh)
  __shared__ __align__(16) float s_a[kFwdWarps][32 * 4];  // per-warp coefficient scratch: pair (t, r) at slot t*8 + r
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* sa = s_a[warp];
  bool okc[kV4];
#pragma unroll
  for (int v = 0; v < kV4; ++v) okc[v] = (lane + 32 * v) * 4 < C;

  // Grid-stride over the centre nodes as a software pipeline that takes the dependent latency of the CSR row
  // pointers off every node's critical path: while node s is processed, the row pointers of node s + 2G are fetched.
  const int G = gridDim.x;
  int s = blockIdx.x;
  if (s >= N) return;
  int c_ib = in_ptr[s], c_ie = in_ptr[s + 1], c_ob = out_ptr[s], c_oe = out_ptr[s + 1];
  int n_ib = 0, n_ie = 0, n_ob = 0, n_oe = 0;
  if (s + G < N) { n_ib = in_ptr[s + G]; n_ie = in_ptr[s + G + 1]; n_ob = out_ptr[s + G]; n_oe = out_ptr[s + G + 1]; }
  for (; s < N; s += G) {
    const int ib = c_ib, dI = c_ie - c_ib, ob = c_ob, dO = c_oe - c_ob;
    int f_ib = 0, f_ie = 0, f_ob = 0, f_oe = 0;
    if ((int64_t)s + 2 * G < N) {
      const int sn = s + 2 * G;
      f_ib = in_ptr[sn]; f_ie = in_ptr[sn + 1]; f_ob = out_ptr[sn]; f_oe = out_ptr[sn + 1];
    }
    // the node's out-edges are split into ceil(dO / 8) blocks of (almost) equal size <= 8, one block per warp and pass
    const int nblk = (dO + kR - 1) / kR, per = nblk ? (dO + nblk - 1) / nblk : 0;
    for (int blk = warp; blk < nblk; blk += kFwdWarps) {
      const int jb = blk * per, nr = min(per, dO - jb);
      tb_fwd_block<NL>(B, NG, gram, unit, gate, ldg, in_edge, in_src, out_edge, C, tbw, sa, lane, okc, ib, dI, ob, jb, nr);
    }
    c_ib = n_ib; c_ie = n_ie; c_ob = n_ob; c_oe = n_oe;
    n_ib = f_ib; n_ie = f_ie; n_ob = f_ob; n_oe = f_oe;
  }
}

// ---------------------------------------------------------------------------------------------
// backward.  Given Gt[e,:] = d tbw[e,:], per pair (e = out j, e' = in i) with a_l = w Y_l, w = 1/max(|v|,eps):
//   dGB[i,l,:] += a_l Gt[j,:]                                   (gate and B gradients follow per in-edge)
//   dot = Gt[j,:] . sum_l a_l GB[i,l,:]  (= w * dL/dw)           one C-wide dot per pair, butterfly-reduced
//   H_i[l,l'] -= dot a_l a_l'            (norm path; skipped when |v| <= eps)  ->  dB[i,l] += sum_l' H[l,l'] B[i,l']
//   dB[i,l,:] += gate * dGB[i,l,:] ;  q[i,:] = gate (1-gate) sum_l B[i,l,:] dGB[i,l,:]   (d xk[k] = sum_{e' in out(k)} q[e'])
//   FORCES: dc = Gt[j,:] . sum_l (w Y'_l) GB[i,l,:] - w^2 dot sum_l Y'_l (G Y)_l ;  d unit[e_j] += dc unit[e_i] and v.v.
// Same clamping convention as the forward: dead slots read a valid row and carry zero coefficients.
// ---------------------------------------------------------------------------------------------
template <int NL, bool FORCES, bool FULL>
__global__ void __launch_bounds__(kBwdWarps * 32) k_threebody_bwd(
    const float* __restrict__ B, int NG, const double* __restrict__ gram, const float* __restrict__ unit,
    const float* __restrict__ gate, int64_t ldg, const int32_t* __restrict__ in_ptr,
    const int32_t* __restrict__ in_edge, const int32_t* __restrict__ in_src, const int32_t* __restrict__ out_ptr,
    const int32_t* __restrict__ out_edge, int N, int C, const float* __restrict__ d_tbw, const float* __restrict__ dP,
    float* __restrict__ dB, float* __restrict__ q, float* __restrict__ du_ks, float* __restrict__ du_st) {
  pdl_trigger();  // (programmatic dependent launch: the next kernel may start its set-up; common.cuh)
  constexpr int NP = NL * (NL + 1) / 2;
  const int NGP = NG - NL + 1;  // rows of the compact two-body gradient dP: [all l < NL | valence slot]
  // per-warp scratch, one slot per out-edge of the current chunk of 32: a_l = w Y_l | norm-path flag | (forces) w Y'_l
  __shared__ __align__(16) float s_a[kBwdWarps][33 * 4];  // (+1: the coefficient prefetch reads one slot ahead)
  __shared__ float s_f[kBwdWarps][32];
  __shared__ __align__(16) float s_a2[FORCES ? kBwdWarps : 1][FORCES ? 33 * 4 : 4];
  __shared__ float s_st[FORCES ? kBwdWarps : 1][FORCES ? kJS * 3 : 1];  // per-warp partials of d unit[e_j] (s->t role)

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // grid-stride over the centre nodes with the next node's CSR row in flight (see the forward kernel)
  int s = blockIdx.x;
  if (s >= N) return;
  int n_ib = in_ptr[s], n_ie = in_ptr[s + 1], n_ob = out_ptr[s], n_oe = out_ptr[s + 1];
  for (; s < N; s += gridDim.x) {
  const int ib = n_ib, dI = n_ie - n_ib, ob = n_ob, dO = n_oe - n_ob;
  if (s + (int)gridDim.x < N) {
    const int sn = s + gridDim.x;
    n_ib = in_ptr[sn]; n_ie = in_ptr[sn + 1]; n_ob = out_ptr[sn]; n_oe = out_ptr[sn + 1];
  }
  if (FORCES) __syncthreads();  // the previous node's d_unit partials have been consumed
  if (dI == 0) {  // no in-edges: only the s->t role gradients of the out-edges exist, and they are zero
    if (FORCES)
      for (int t = threadIdx.x; t < dO * 3; t += kBwdWarps * 32) du_st[3 * (int64_t)out_edge[ob + t / 3] + t % 3] = 0.f;
    continue;
  }
  if (dO == 0) {  // in-edges that feed no triplet: zero gradients
    for (int i = warp; i < dI; i += kBwdWarps) {
      const int ep = in_edge[ib + i];
      for (int c = lane * 4; c < C; c += 128) {
        for (int l = 0; l < NG; ++l)
          st4(dB + ((int64_t)ep * NG + l) * C + c, dP ? ldg4(dP + ((int64_t)ep * NGP + (l < NL ? 0 : 1)) * C + c) : zero4());
        st4(q + (int64_t)ep * C + c, zero4());
      }
      if (FORCES && lane < 3) du_ks[3 * (int64_t)ep + lane] = 0.f;
    }
    continue;
  }
  if constexpr (FORCES) {
    for (int t = lane; t < kJS * 3; t += 32) s_st[warp][t] = 0.f;
    for (int t = threadIdx.x; t < dO * 3; t += kBwdWarps * 32)
      if (t >= kJS * 3) du_st[3 * (int64_t)out_edge[ob + t / 3] + t % 3] = 0.f;  // rare overflow rows: global atomics below
    __syncthreads();
  }
  float* sa = s_a[warp];
  float* sf = s_f[warp];
  const int jsub = bfly8_index(lane);
  bool okc[kV4];
#pragma unroll
  for (int v = 0; v < kV4; ++v) okc[v] = FULL || (lane + 32 * v) * 4 < C;

  for (int i = warp; i < dI; i += kBwdWarps) {  // one in-edge per warp at a time
    const int ep = in_edge[ib + i], k = in_src[ib + i];
    float4 gb[NL][kV4], dacc[NL][kV4], gt[kV4];
    float h[NP];
#pragma unroll
    for (int v = 0; v < kV4; ++v) {
      const int c = (lane + 32 * v) * 4;
      gt[v] = okc[v] ? ldg4(gate + (int64_t)k * ldg + c) : zero4();
#pragma unroll
      for (int l = 0; l < NL; ++l) {
        gb[l][v] = okc[v] ? mul4(gt[v], ldg4(B + ((int64_t)ep * NG + l) * C + c)) : zero4();
        dacc[l][v] = zero4();
      }
    }
#pragma unroll
    for (int p = 0; p < NP; ++p) h[p] = 0.f;
    const float vx = unit[3 * (int64_t)ep], vy = unit[3 * (int64_t)ep + 1], vz = unit[3 * (int64_t)ep + 2];
    double g[NP];
#pragma unroll
    for (int p = 0; p < NP; ++p) g[p] = gram[(int64_t)ep * NP + p];
    float ks_x = 0.f, ks_y = 0.f, ks_z = 0.f;  // FORCES: d unit[e_i] partial of this lane (k->s role)

    for (int oc = 0; oc < dO; oc += 32) {  // the node's out-edges, 32 at a time: lane <-> out-edge oc + lane
      const int nO = min(32, dO - oc);
      const int my_ej = out_edge[ob + oc + min(lane, nO - 1)];
      // ---- coefficients of the pairs (out-edge oc + lane, this in-edge): one pair per lane, once per chunk
      const float ox = unit[3 * (int64_t)my_ej], oy = unit[3 * (int64_t)my_ej + 1], oz = unit[3 * (int64_t)my_ej + 2];
      const float cc = fmaf(ox, vx, fmaf(oy, vy, oz * vz));
      float Y[4];
      sph_harm<NL>(cc, Y);
      const float nrm = sqrtf(fmaxf((float)quad_form<NL>(g, Y), 0.f));
      const bool live = lane < nO && my_ej != ep;
      const float ww = live ? 1.0f / fmaxf(nrm, kEps) : 0.f;
      const float fl = (live && nrm > kEps) ? 1.f : 0.f;
      __syncwarp();  // the previous chunk's readers are done
      st4(sa + lane * 4, make_float4(ww * Y[0], ww * Y[1], ww * Y[2], ww * Y[3]));
      sf[lane] = fl;
      if constexpr (FORCES) {
        float dY[4];
        sph_harm_grad<NL>(cc, dY);
        st4(s_a2[warp] + lane * 4, make_float4(ww * dY[0], ww * dY[1], ww * dY[2], ww * dY[3]));
      }
      __syncwarp();
      for (int j0 = 0; j0 < nO; j0 += 8) {
        const int nj = min(8, nO - j0);
        // ---- d_tbw rows of the batch (all loads first); dead slots (jj >= nj) read a clamped row and carry zero
        //      coefficients (branch-free)
        float4 gr[8][kV4];
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) {
          const int e = __shfl_sync(0xffffffffu, my_ej, min(j0 + jj, nO - 1));
#pragma unroll
          for (int v = 0; v < kV4; ++v) gr[jj][v] = okc[v] ? ldg4(d_tbw + (int64_t)e * C + (lane + 32 * v) * 4) : zero4();
        }
        // FORCES needs two contractions of Gt with the in-edge's rows per pair (weights w Y_l and w Y'_l): instead of
        // forming both combined rows, the NL dots D_l = Gt . GB_l are taken once (NL FMAs per channel) and both scalars
        // follow from them after the butterfly: 24 instead of 44 arithmetic instructions per pair and lane.
        float part[FORCES ? 1 : 8], partD[FORCES ? NL : 1][8];
        float4 ar = lds4(sa + j0 * 4);
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) {
          const float4 ar_next = lds4(sa + (j0 + jj + 1) * 4);  // (one slot ahead: no block starts by waiting on shared memory)
          float d = 0.f, dl[NL];
#pragma unroll
          for (int l = 0; l < NL; ++l) dl[l] = 0.f;
#pragma unroll
          for (int v = 0; v < kV4; ++v) {
            if constexpr (FORCES) {
#pragma unroll
              for (int l = 0; l < NL; ++l) dl[l] += dot4(gb[l][v], gr[jj][v]);
            } else {
              float4 t = scale4(ar.x, gb[0][v]);
              if (NL > 1) t = fma4(ar.y, gb[1][v], t);
              if (NL > 2) t = fma4(ar.z, gb[2][v], t);
              if (NL > 3) t = fma4(ar.w, gb[3][v], t);
              d += dot4(t, gr[jj][v]);
            }
            dacc[0][v] = fma4(ar.x, gr[jj][v], dacc[0][v]);
            if (NL > 1) dacc[1][v] = fma4(ar.y, gr[jj][v], dacc[1][v]);
            if (NL > 2) dacc[2][v] = fma4(ar.z, gr[jj][v], dacc[2][v]);
            if (NL > 3) dacc[3][v] = fma4(ar.w, gr[jj][v], dacc[3][v]);
          }
          if constexpr (FORCES) {
#pragma unroll
            for (int l = 0; l < NL; ++l) partD[l][jj] = dl[l];
          } else {
            part[jj] = d;
          }
          ar = ar_next;
        }
        // ---- per pair scalars: the quad `jsub` of the warp finishes pair (out j0 + jsub, this in-edge)
        float dotv, dot2v = 0.f;
        {
          const int slot = j0 + jsub;  // dead slots carry a = 0, flag = 0 and a zero dot
          const float4 as = lds4(sa + slot * 4);
          if constexpr (FORCES) {
            const float4 as2 = lds4(s_a2[warp] + slot * 4);
            dotv = 0.f;
#pragma unroll
            for (int l = 0; l < NL; ++l) {
              const float D = bfly8(partD[l], lane);
              dotv = fmaf(comp4(as, l), D, dotv);
              dot2v = fmaf(comp4(as2, l), D, dot2v);
            }
          } else {
            dotv = bfly8(part, lane);
          }
          const float sc = -sf[slot] * dotv;
          int p = 0;
#pragma unroll
          for (int x = 0; x < NL; ++x)
#pragma unroll
            for (int y = x; y < NL; ++y) h[p++] += sc * comp4(as, x) * comp4(as, y);
        }
        if constexpr (FORCES) {
          // dL/dcos of pair (j0 + jl) is finished on its coefficient lane j0 + jl, which still holds the pair's cos /
          // w / flag and both directions; the two dots come from the quad that owns butterfly element jl (lane bits
          // 4,3,2 = bits 2,1,0 of jl).
          const int jl = (lane - j0) & 7;
          const int srcl = (((jl >> 2) & 1) << 4) | (((jl >> 1) & 1) << 3) | ((jl & 1) << 2);
          const float dt = __shfl_sync(0xffffffffu, dotv, srcl);
          const float dt2 = __shfl_sync(0xffffffffu, dot2v, srcl);
          if (lane >= j0 && lane < j0 + nj && live) {
            float dY[4];
            sph_harm_grad<NL>(cc, dY);
            const float corr = (float)bilin_form<NL>(g, dY, Y);
            const float dc = dt2 - fl * ww * ww * dt * corr;
            ks_x = fmaf(dc, ox, ks_x); ks_y = fmaf(dc, oy, ks_y); ks_z = fmaf(dc, oz, ks_z);
            const int j = oc + lane;
            if (j < kJS) {  // slot j of this warp's partials is only ever touched by this lane
              s_st[warp][3 * j] = fmaf(dc, vx, s_st[warp][3 * j]);
              s_st[warp][3 * j + 1] = fmaf(dc, vy, s_st[warp][3 * j + 1]);
              s_st[warp][3 * j + 2] = fmaf(dc, vz, s_st[warp][3 * j + 2]);
            } else {
              atomicAdd(du_st + 3 * (int64_t)my_ej, dc * vx);
              atomicAdd(du_st + 3 * (int64_t)my_ej + 1, dc * vy);
              atomicAdd(du_st + 3 * (int64_t)my_ej + 2, dc * vz);
            }
          }
        }
      }
    }
    // ---- finish this in-edge
    if constexpr (FORCES) {
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        ks_x += __shfl_xor_sync(0xffffffffu, ks_x, o);
        ks_y += __shfl_xor_sync(0xffffffffu, ks_y, o);
        ks_z += __shfl_xor_sync(0xffffffffu, ks_z, o);
      }
      if (lane == 0) {
        du_ks[3 * (int64_t)ep] = ks_x; du_ks[3 * (int64_t)ep + 1] = ks_y; du_ks[3 * (int64_t)ep + 2] = ks_z;
      }
    }
#pragma unroll
    for (int p = 0; p < NP; ++p) {  // h was accumulated by one lane quad per out-edge slot: add the 8 slots
      float x = h[p];
      x += __shfl_xor_sync(0xffffffffu, x, 4);
      x += __shfl_xor_sync(0xffffffffu, x, 8);
      x += __shfl_xor_sync(0xffffffffu, x, 16);
      h[p] = x;
    }
    float H[NL][NL];
    {
      int p = 0;
#pragma unroll
      for (int x = 0; x < NL; ++x)
#pragma unroll
        for (int y = x; y < NL; ++y) { H[x][y] = h[p]; H[y][x] = h[p]; ++p; }
    }
#pragma unroll
    for (int v = 0; v < kV4; ++v) {
      const int c = (lane + 32 * v) * 4;
      if (okc[v]) {
        float4 b[NL];
#pragma unroll
        for (int l = 0; l < NL; ++l) b[l] = ldg4(B + ((int64_t)ep * NG + l) * C + c);
        float4 qq = zero4();
        const float4 two_body = dP ? ldg4(dP + (int64_t)ep * NGP * C + c) : zero4();  // same for every l < NL
#pragma unroll
        for (int l = 0; l < NL; ++l) {
          float4 o4 = fma4(1.0f, mul4(gt[v], dacc[l][v]), two_body);
#pragma unroll
          for (int l2 = 0; l2 < NL; ++l2) o4 = fma4(H[l][l2], b[l2], o4);
          st4(dB + ((int64_t)ep * NG + l) * C + c, o4);
          qq = add4(qq, mul4(b[l], dacc[l][v]));
        }
        const float4 sg = gt[v];
        qq = mul4(qq, make_float4(sg.x * (1.f - sg.x), sg.y * (1.f - sg.y), sg.z * (1.f - sg.z), sg.w * (1.f - sg.w)));
        st4(q + (int64_t)ep * C + c, qq);
        for (int l = NL; l < NG; ++l)
          st4(dB + ((int64_t)ep * NG + l) * C + c, dP ? ldg4(dP + ((int64_t)ep * NGP + 1) * C + c) : zero4());
      }
    }
  }
  if constexpr (FORCES) {
    __syncthreads();
    for (int t = threadIdx.x; t < min(dO, kJS) * 3; t += kBwdWarps * 32) {
      float x = 0.f;
#pragma unroll
      for (int w = 0; w < kBwdWarps; ++w) x += s_st[w][t];
      du_st[3 * (int64_t)out_edge[ob + t / 3] + t % 3] = x;
    }
  }
  }
}

}  // namespace

// warp-level tensor-core formulation with bulk-copy staging (threebody_mma.cu): the forward for C <= 128
int lcao_tb_mma_fwd(const float* B, int32_t NG, const double* gram, const float* unit, const float* gate, int64_t ldg,
                    const int32_t* in_ptr, const int32_t* in_edge, const int32_t* in_src, const int32_t* out_ptr,
                    const int32_t* out_edge, int64_t N, int32_t C, int32_t NL, float* tbw, cudaStream_t st);
// staged backward (threebody_staged.cu): bulk-copy staging + producer warp, the backward for C <= 128
int lcao_tb_staged_bwd(const float* B, int32_t NG, const double* gram, const float* unit, const float* gate, int64_t ldg,
                       const int32_t* in_ptr, const int32_t* in_edge, const int32_t* in_src, const int32_t* out_ptr,
                       const int32_t* out_edge, int64_t N, int32_t C, int32_t NL, const float* d_tbw, const float* dP,
                       float* dB, float* q, float* du_ks, float* du_st, cudaStream_t st);

// every kernel reads or writes these rows with 16-byte accesses or bulk copies
static bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

#define TB_DISPATCH(NL, CALL)     \
  switch (NL) {                   \
    case 1: { CALL(1); } break;   \
    case 2: { CALL(2); } break;   \
    case 3: { CALL(3); } break;   \
    default: { CALL(4); } break;  \
  }

extern "C" int lcao_threebody_fwd(const float* B, int32_t NG, const double* gram, const float* unit, const float* gate,
                                  int64_t ldg, const int32_t* in_ptr, const int32_t* in_edge, const int32_t* in_src,
                                  const int32_t* out_ptr, const int32_t* out_edge, int64_t N, int64_t E, int32_t C,
                                  int32_t NL, float* tbw, void* stream) {
  if (N == 0 || E == 0) return LCAO_OK;
  LCAO_REQUIRE(B && gram && unit && gate && in_ptr && in_edge && in_src && out_ptr && out_edge && tbw,
               "lcao_threebody_fwd: null buffer");
  LCAO_REQUIRE(C % 4 == 0 && C > 0 && C <= 256 && NL >= 1 && NL <= 4 && NG >= NL && ldg % 4 == 0,
               "lcao_threebody_fwd: need C %% 4 == 0, C <= 256, 1 <= NL <= 4, NG >= NL (C=%d NL=%d NG=%d)", C, NL, NG);
  LCAO_REQUIRE(al16(B) && al16(gate) && al16(tbw), "lcao_threebody_fwd: B, gate and tbw must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  if (C <= 128) return lcao_tb_mma_fwd(B, NG, gram, unit, gate, ldg, in_ptr, in_edge, in_src, out_ptr, out_edge, N, C, NL, tbw, st);
  const unsigned grid = (unsigned)(N < 148ll * kFwdCtasPerSm ? N : 148ll * kFwdCtasPerSm);
  // (unlike the backward, the forward has no predicate-free C == 256 specialisation: it measured SLOWER, 0.291 vs 0.260 ms)
#define CALL(nl)                                                                                                   \
  k_threebody_fwd<nl><<<grid, kFwdWarps * 32, 0, st>>>(B, NG, gram, unit, gate, ldg, in_ptr, in_edge, in_src, out_ptr, \
                                                        out_edge, (int)N, C, tbw)
  TB_DISPATCH(NL, CALL)
#undef CALL
  LCAO_LAUNCH_CHECK();
  return LCAO_OK;
}

extern "C" int lcao_threebody_bwd(const float* B, int32_t NG, const double* gram, const float* unit, const float* gate,
                                  int64_t ldg, const int32_t* in_ptr, const int32_t* in_edge, const int32_t* in_src,
                                  const int32_t* out_ptr, const int32_t* out_edge, int64_t N, int64_t E, int32_t C,
                                  int32_t NL, const float* d_tbw, const float* dP, float* dB, float* q, float* d_unit_ks,
                                  float* d_unit_st, void* stream) {
  if (N == 0 || E == 0) return LCAO_OK;
  LCAO_REQUIRE(B && gram && unit && gate && in_ptr && in_edge && in_src && out_ptr && out_edge && d_tbw && dB && q,
               "lcao_threebody_bwd: null buffer");
  LCAO_REQUIRE(C % 4 == 0 && C > 0 && C <= 256 && NL >= 1 && NL <= 4 && NG >= NL && ldg % 4 == 0,
               "lcao_threebody_bwd: need C %% 4 == 0, C <= 256, 1 <= NL <= 4, NG >= NL");
  LCAO_REQUIRE((d_unit_ks == nullptr) == (d_unit_st == nullptr), "lcao_threebody_bwd: pass both d_unit buffers or neither");
  LCAO_REQUIRE(NG <= NL + 1, "lcao_threebody_bwd: at most one valence group (NG <= NL + 1)");
  LCAO_REQUIRE(al16(B) && al16(gate) && al16(d_tbw) && al16(dB) && al16(q) && al16(dP),
               "lcao_threebody_bwd: B, gate, d_tbw, dP, dB and q must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const bool forces = d_unit_ks != nullptr;
  if (C <= 128)
    return lcao_tb_staged_bwd(B, NG, gram, unit, gate, ldg, in_ptr, in_edge, in_src, out_ptr, out_edge, N, C, NL, d_tbw, dP, dB,
                              q, d_unit_ks, d_unit_st, st);
  const bool full = C == 128 * kV4;
  const unsigned grid = (unsigned)(N < 148ll * kBwdCtasPerSm ? N : 148ll * kBwdCtasPerSm);
#define TB_BWD_ARGS B, NG, gram, unit, gate, ldg, in_ptr, in_edge, in_src, out_ptr, out_edge, (int)N, C, d_tbw, dP, dB, q
#define CALL(nl)                                                                                            \
  if (forces)                                                                                               \
    k_threebody_bwd<nl, true, false><<<grid, kBwdWarps * 32, 0, st>>>(TB_BWD_ARGS, d_unit_ks, d_unit_st);  \
  else if (full)                                                                                            \
    k_threebody_bwd<nl, false, true><<<grid, kBwdWarps * 32, 0, st>>>(TB_BWD_ARGS, nullptr, nullptr);      \
  else                                                                                                      \
    k_threebody_bwd<nl, false, false><<<grid, kBwdWarps * 32, 0, st>>>(TB_BWD_ARGS, nullptr, nullptr)
  TB_DISPATCH(NL, CALL)
#undef CALL
#undef TB_BWD_ARGS
  LCAO_LAUNCH_CHECK();
  return LCAO_OK;
}
