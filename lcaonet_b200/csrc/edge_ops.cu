// Edge-sized streaming kernels of the LCAO hot path (all HBM-bound, float4-vectorised, one warp
// per edge row): orbital contraction against the radial basis, two-body weight normalisation,
// node->edge gathers, sorted-segment sums (no atomics), row gathers and keyed reductions.
// Reference sites: lcaonet.py:180-183,192-214 (einsum / normalize / scatter), embed.py:122-133,245-249.
#include "common.cuh"

namespace {

constexpr int kWarpsPerCta = 8;

__device__ __forceinline__ float4 f4_fma(float a, float4 x, float4 acc) {
  acc.x = fmaf(a, x.x, acc.x); acc.y = fmaf(a, x.y, acc.y); acc.z = fmaf(a, x.z, acc.z); acc.w = fmaf(a, x.w, acc.w);
  return acc;
}
__device__ __forceinline__ float4 f4_zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ float4 f4_add(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }
__device__ __forceinline__ float4 f4_sub(float4 a, float4 b) { return make_float4(a.x - b.x, a.y - b.y, a.z - b.z, a.w - b.w); }
__device__ __forceinline__ float4 f4_mul(float4 a, float4 b) { return make_float4(a.x * b.x, a.y * b.y, a.z * b.z, a.w * b.w); }
__device__ __forceinline__ float4 f4_scale(float a, float4 b) { return make_float4(a * b.x, a * b.y, a * b.z, a * b.w); }
__device__ __forceinline__ float f4_dot(float4 a, float4 b) { return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w; }

// ---------------------------------------------------------------------------------------------
// B[e,l,:] = sum_{o in l} rb[e,o] (A[e,o,:] + m[e,o] V[e,o,:]) ; B[e,NL,:] = sum_o rb m V
// one warp per edge, lane owns float4 column c4 = lane (+32 per extra pass).
// ---------------------------------------------------------------------------------------------
template <int NL, bool VAL>
__global__ void __launch_bounds__(kWarpsPerCta * 32) k_coeff_contract_fwd(
    const float* __restrict__ cst1, const float* __restrict__ rb, const float* __restrict__ vmask,
    const int32_t* __restrict__ lgrp, int64_t E, int O, int C, float* __restrict__ B) {
  __shared__ int s_l[LCAO_MAX_ORB];
  if (threadIdx.x < O) s_l[threadIdx.x] = lgrp[threadIdx.x];
  __syncthreads();
  const int64_t e = blockIdx.x * (int64_t)kWarpsPerCta + (threadIdx.x >> 5);
  if (e >= E) return;
  const int lane = threadIdx.x & 31;
  const int Cp = VAL ? 2 * C : C, NG = NL + (VAL ? 1 : 0);
  const float* row = cst1 + e * (int64_t)O * Cp;
  for (int c = lane * 4; c < C; c += 128) {
    float4 acc[NL + 1];
#pragma unroll
    for (int l = 0; l <= NL; ++l) acc[l] = f4_zero();
#pragma unroll 4
    for (int o = 0; o < O; ++o) {
      const float r = __ldg(rb + e * O + o);
      float4 t = f4_scale(r, ldg4(row + (int64_t)o * Cp + c));
      if (VAL) {
        const float rm = r * __ldg(vmask + e * O + o);
        const float4 v = f4_scale(rm, ldg4(row + (int64_t)o * Cp + C + c));
        acc[NL] = f4_add(acc[NL], v);
        t = f4_add(t, v);
      }
      const int l = s_l[o];
#pragma unroll
      for (int k = 0; k < NL; ++k)
        if (l == k) acc[k] = f4_add(acc[k], t);
    }
#pragma unroll
    for (int l = 0; l < NG; ++l) st4(B + (e * NG + l) * (int64_t)C + c, acc[l]);
  }
}

template <int NL, bool VAL>
__global__ void __launch_bounds__(kWarpsPerCta * 32) k_coeff_contract_bwd(
    const float* __restrict__ cst1, const float* __restrict__ rb, const float* __restrict__ vmask,
    const int32_t* __restrict__ lgrp, const float* __restrict__ dB, int64_t E, int O, int C,
    float* __restrict__ d_cst1, float* __restrict__ d_rb) {
  __shared__ int s_l[LCAO_MAX_ORB];
  if (threadIdx.x < O) s_l[threadIdx.x] = lgrp[threadIdx.x];
  __syncthreads();
  const int64_t e = blockIdx.x * (int64_t)kWarpsPerCta + (threadIdx.x >> 5);
  if (e >= E) return;
  const int lane = threadIdx.x & 31;
  const int Cp = VAL ? 2 * C : C, NG = NL + (VAL ? 1 : 0);
  const int64_t rowo = e * (int64_t)O * Cp;
  for (int o = 0; o < O; ++o) {
    const float r = __ldg(rb + e * O + o);
    const float m = VAL ? __ldg(vmask + e * O + o) : 0.f;
    const int l = s_l[o];
    float dot = 0.f;
    for (int c = lane * 4; c < C; c += 128) {
      const float4 g = ldg4(dB + (e * NG + l) * (int64_t)C + c);
      st4(d_cst1 + rowo + (int64_t)o * Cp + c, f4_scale(r, g));
      if (d_rb) dot += f4_dot(ldg4(cst1 + rowo + (int64_t)o * Cp + c), g);
      if (VAL) {
        const float4 gv = f4_add(g, ldg4(dB + (e * NG + NL) * (int64_t)C + c));
        st4(d_cst1 + rowo + (int64_t)o * Cp + C + c, f4_scale(r * m, gv));
        if (d_rb) dot += m * f4_dot(ldg4(cst1 + rowo + (int64_t)o * Cp + C + c), gv);
      }
    }
    if (d_rb) {
      dot = warp_sum(dot);
      if (lane == 0) d_rb[e * O + o] = dot;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// two-body weight: p = (1+gA) PA + (1+gV) PV ; lw = p / max(|p|, eps).  C <= 256 (2 float4 / lane)
// ---------------------------------------------------------------------------------------------
template <bool VAL>
__device__ __forceinline__ void twobody_load(const float* __restrict__ B, const float* __restrict__ g, int64_t e,
                                             int NG, int NL, int C, int c, float4& PA, float4& PV, float4& gA,
                                             float4& gV) {
  float4 s = f4_zero();
  for (int l = 0; l < NL; ++l) s = f4_add(s, ldg4(B + (e * NG + l) * (int64_t)C + c));
  if (VAL) {
    PV = ldg4(B + (e * NG + NL) * (int64_t)C + c);
    PA = f4_sub(s, PV);
    gA = ldg4(g + e * 2 * (int64_t)C + c);
    gV = ldg4(g + e * 2 * (int64_t)C + C + c);
  } else {
    PA = s; PV = f4_zero(); gV = f4_zero();
    gA = ldg4(g + e * (int64_t)C + c);
  }
}

// NV = float4 column slices per lane (1 for C <= 128, 2 up to 256): the register arrays are sized by it, which keeps
// the common C = 128 case at 5+ resident CTAs per SM (73 registers with two slices limited it to 3)
template <bool VAL, int NV>
__global__ void __launch_bounds__(kWarpsPerCta * 32) k_twobody_fwd(const float* __restrict__ B, int NG,
                                                                   const float* __restrict__ g, int64_t E, int C,
                                                                   int NL, float* __restrict__ lw) {
  pdl_trigger();  // (programmatic dependent launch: the next kernel may start its set-up; common.cuh)
  pdl_wait();     // launched through launch_pdl: nothing of the stream's earlier work is touched before this
  const int64_t e = blockIdx.x * (int64_t)kWarpsPerCta + (threadIdx.x >> 5);
  if (e >= E) return;
  const int lane = threadIdx.x & 31;
  float4 p[NV];
  float n2 = 0.f;
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const int c = lane * 4 + v * 128;
    p[v] = f4_zero();
    if (c < C) {
      float4 PA, PV, gA, gV;
      twobody_load<VAL>(B, g, e, NG, NL, C, c, PA, PV, gA, gV);
      p[v] = make_float4(fmaf(gA.x, PA.x, PA.x), fmaf(gA.y, PA.y, PA.y), fmaf(gA.z, PA.z, PA.z), fmaf(gA.w, PA.w, PA.w));
      if (VAL) p[v] = f4_add(p[v], make_float4(fmaf(gV.x, PV.x, PV.x), fmaf(gV.y, PV.y, PV.y), fmaf(gV.z, PV.z, PV.z), fmaf(gV.w, PV.w, PV.w)));
      n2 += f4_dot(p[v], p[v]);
    }
  }
  n2 = warp_sum(n2);
  const float inv = 1.0f / fmaxf(sqrtf(n2), 1e-12f);
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const int c = lane * 4 + v * 128;
    if (c < C) st4(lw + e * (int64_t)C + c, f4_scale(inv, p[v]));
  }
}

// backward: dp = (dlw - lw (lw.dlw)) / |p|  (or dlw/eps when clamped);
// dgA = dp*PA, dgV = dp*PV ; dPA = (1+gA) dp, dPV = (1+gV) dp ;
// stored groups: dB[l] = dPA for every l < NL ; dB[NL] = dPV - dPA   (PA = sum_l B_l - B_NL)
template <bool VAL, int NV>
__global__ void __launch_bounds__(kWarpsPerCta * 32) k_twobody_bwd(const float* __restrict__ B, int NG,
                                                                   const float* __restrict__ g,
                                                                   const float* __restrict__ d_lw, int64_t E, int C,
                                                                   int NL, int compact, float* __restrict__ dB,
                                                                   float* __restrict__ d_g) {
  pdl_trigger();  // (programmatic dependent launch: the next kernel may start its set-up; common.cuh)
  pdl_wait();     // launched through launch_pdl: nothing of the stream's earlier work is touched before this
  const int64_t e = blockIdx.x * (int64_t)kWarpsPerCta + (threadIdx.x >> 5);
  if (e >= E) return;
  const int lane = threadIdx.x & 31;
  float4 p[NV], PA[NV], PV[NV], gA[NV], gV[NV], dl[NV];
  float n2 = 0.f, pd = 0.f;
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const int c = lane * 4 + v * 128;
    p[v] = f4_zero(); dl[v] = f4_zero();
    if (c < C) {
      twobody_load<VAL>(B, g, e, NG, NL, C, c, PA[v], PV[v], gA[v], gV[v]);
      p[v] = make_float4(fmaf(gA[v].x, PA[v].x, PA[v].x), fmaf(gA[v].y, PA[v].y, PA[v].y), fmaf(gA[v].z, PA[v].z, PA[v].z), fmaf(gA[v].w, PA[v].w, PA[v].w));
      if (VAL) p[v] = f4_add(p[v], make_float4(fmaf(gV[v].x, PV[v].x, PV[v].x), fmaf(gV[v].y, PV[v].y, PV[v].y), fmaf(gV[v].z, PV[v].z, PV[v].z), fmaf(gV[v].w, PV[v].w, PV[v].w)));
      dl[v] = ldg4(d_lw + e * (int64_t)C + c);
      n2 += f4_dot(p[v], p[v]);
      pd += f4_dot(p[v], dl[v]);
    }
  }
  n2 = warp_sum(n2);
  pd = warp_sum(pd);
  const float nrm = sqrtf(n2);
  const bool clamped = !(nrm > 1e-12f);
  const float inv = 1.0f / fmaxf(nrm, 1e-12f);
  // lw = p*inv ; lw.dlw = pd*inv ; dp = (dl - p*inv*pd*inv) * inv
  const float coef = clamped ? 0.f : pd * inv * inv;
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const int c = lane * 4 + v * 128;
    if (c < C) {
      float4 dp = f4_scale(inv, f4_sub(dl[v], f4_scale(coef, p[v])));
      const float4 dPA = make_float4(fmaf(gA[v].x, dp.x, dp.x), fmaf(gA[v].y, dp.y, dp.y), fmaf(gA[v].z, dp.z, dp.z), fmaf(gA[v].w, dp.w, dp.w));
      const int NGo = compact ? (VAL ? 2 : 1) : NG, NLo = compact ? 1 : NL;  // compact: one row for all l < NL
      for (int l = 0; l < NLo; ++l) st4(dB + (e * NGo + l) * (int64_t)C + c, dPA);
      if (VAL) {
        const float4 dPV = make_float4(fmaf(gV[v].x, dp.x, dp.x), fmaf(gV[v].y, dp.y, dp.y), fmaf(gV[v].z, dp.z, dp.z), fmaf(gV[v].w, dp.w, dp.w));
        st4(dB + (e * NGo + NLo) * (int64_t)C + c, f4_sub(dPV, dPA));
        st4(d_g + e * 2 * (int64_t)C + c, f4_mul(dp, PA[v]));
        st4(d_g + e * 2 * (int64_t)C + C + c, f4_mul(dp, PV[v]));
      } else {
        st4(d_g + e * (int64_t)C + c, f4_mul(dp, PA[v]));
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// out[e,:] = act(a[src[e],:] + b[dst[e],:] + bias)
// ---------------------------------------------------------------------------------------------
template <bool GEN>
__global__ void __launch_bounds__(kWarpsPerCta * 32) k_edge_pair_fwd(
    const float* __restrict__ a, int64_t lda, const float* __restrict__ b, int64_t ldb, const float* __restrict__ bias,
    const int32_t* __restrict__ src32, const int32_t* __restrict__ dst32, int64_t E, int C, int act,
    float* __restrict__ out, float* __restrict__ pre) {
  pdl_trigger();  // (programmatic dependent launch: the next kernel may start its set-up; common.cuh)
  pdl_wait();     // launched through launch_pdl: nothing of the stream's earlier work is touched before this
  const int64_t e = blockIdx.x * (int64_t)kWarpsPerCta + (threadIdx.x >> 5);
  if (e >= E) return;
  const int lane = threadIdx.x & 31;
  const float* pa = a + src32[e] * lda;
  const float* pb = b + dst32[e] * ldb;
  for (int c = lane * 4; c < C; c += 128) {
    float4 v = f4_add(ldg4(pa + c), ldg4(pb + c));
    if (bias) v = f4_add(v, ldg4(bias + c));
    if (pre) st4(pre + e * (int64_t)C + c, v);
    if (act != LCAO_ACT_NONE) v = act_fwd4<GEN>(act, v);
    st4(out + e * (int64_t)C + c, v);
  }
}

// ---------------------------------------------------------------------------------------------
// sorted-segment sum: out[r,:] = scale_r * sum_{j in seg r} x[perm[j],:] (* y[perm[j],:])
// warp per output row; vector path when C % 4 == 0 and all strides % 4 == 0, scalar path otherwise
// ---------------------------------------------------------------------------------------------
template <bool VEC, bool GEN>
__global__ void __launch_bounds__(kWarpsPerCta * 32) k_segment_sum(
    const float* __restrict__ x, int64_t ldx, const float* __restrict__ y, int64_t ldy, const int32_t* __restrict__ ptr,
    const int32_t* __restrict__ perm, int64_t R, int C, int mean, float* __restrict__ out, int64_t ldo) {
  pdl_trigger();  // (programmatic dependent launch: the next kernel may start its set-up; common.cuh)
  pdl_wait();     // launched through launch_pdl: nothing of the stream's earlier work is touched before this
  const int64_t r = blockIdx.x * (int64_t)kWarpsPerCta + (threadIdx.x >> 5);
  if (r >= R) return;
  const int lane = threadIdx.x & 31;
  const int32_t lo = ptr[r], hi = ptr[r + 1];
  const float scale = (mean & 1) ? 1.0f / (float)max(hi - lo, 1) : 1.0f;
  const bool ysilu = (mean & 2) != 0;   // y holds a pre-activation: the factor is act(y)
  const bool ygrad = (mean & 4) != 0;   // ... or act'(y) (backward through an activation, folded into the reduction)
  const int act = ((mean >> 4) & 15) ? ((mean >> 4) & 15) : LCAO_ACT_SILU;
  if (VEC) {
    for (int c = lane * 4; c < C; c += 128) {
      float4 acc = f4_zero();
      for (int32_t j = lo; j < hi; ++j) {
        const int64_t i = perm ? perm[j] : j;
        float4 v = ldg4(x + i * ldx + c);
        if (y) {
          float4 w = ldg4(y + i * ldy + c);
          if (ysilu) w = act_fwd4<GEN>(act, w);
          if (ygrad) w = act_grad4<GEN>(act, w);
          v = f4_mul(v, w);
        }
        acc = f4_add(acc, v);
      }
      st4(out + r * ldo + c, f4_scale(scale, acc));
    }
  } else {
    for (int c = lane; c < C; c += 32) {
      float acc = 0.f;
      for (int32_t j = lo; j < hi; ++j) {
        const int64_t i = perm ? perm[j] : j;
        float v = x[i * ldx + c];
        if (y) v *= ysilu ? act_fwd_t<GEN>(act, y[i * ldy + c]) : ygrad ? act_grad_t<GEN>(act, y[i * ldy + c]) : y[i * ldy + c];
        acc += v;
      }
      out[r * ldo + c] = scale * acc;
    }
  }
}

template <typename IdxT, bool VEC>
__global__ void k_gather_rows(const float* __restrict__ table, int64_t ldt, const IdxT* __restrict__ idx,
                              const float* __restrict__ mul, int64_t ldm, int64_t n, int W, float* __restrict__ out,
                              int64_t ldo) {
  pdl_trigger();  // (programmatic dependent launch: the next kernel may start its set-up; common.cuh)
  const int WV = VEC ? W / 4 : W;
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= n * WV) return;
  const int64_t i = t / WV;
  const int c = (int)(t - i * WV) * (VEC ? 4 : 1);
  if (VEC) {
    float4 v = ldg4(table + (int64_t)idx[i] * ldt + c);
    if (mul) v = f4_mul(v, ldg4(mul + i * ldm + c));
    st4(out + i * ldo + c, v);
  } else {
    float v = __ldg(table + (int64_t)idx[i] * ldt + c);
    if (mul) v *= __ldg(mul + i * ldm + c);
    out[i * ldo + c] = v;
  }
}

// acc[key,:] += x[i,:] over the key-sorted permutation; CTA = 32 consecutive sorted entries,
// thread = one float4 column, register accumulation between key changes, one atomic flush per run.
__global__ void __launch_bounds__(256) k_reduce_by_key(const float* __restrict__ x, int64_t ldx,
                                                       const int32_t* __restrict__ kptr,
                                                       const int32_t* __restrict__ kperm, int nkeys, int64_t n,
                                                       int W, float* __restrict__ acc) {
  const int64_t j0 = blockIdx.x * 32ll, j1 = (j0 + 32 < n) ? j0 + 32 : n;
  // bucket of j0: last key with kptr[key] <= j0
  int lo = 0, hi = nkeys;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (kptr[mid] <= j0) lo = mid; else hi = mid;
  }
  for (int c = threadIdx.x * 4; c < W; c += 256 * 4) {
    int key = lo;
    float4 a = f4_zero();
    for (int64_t j = j0; j < j1; ++j) {
      while (j >= kptr[key + 1]) {
        if (a.x != 0.f || a.y != 0.f || a.z != 0.f || a.w != 0.f) {
          float* d = acc + (int64_t)key * W + c;
          atomicAdd(d, a.x); atomicAdd(d + 1, a.y); atomicAdd(d + 2, a.z); atomicAdd(d + 3, a.w);
        }
        a = f4_zero();
        ++key;
      }
      a = f4_add(a, ldg4(x + (int64_t)kperm[j] * ldx + c));
    }
    float* d = acc + (int64_t)key * W + c;
    atomicAdd(d, a.x); atomicAdd(d + 1, a.y); atomicAdd(d + 2, a.z); atomicAdd(d + 3, a.w);
  }
}

// Y = act(X) elementwise (the activations the tcgen05 epilogue does not fuse); X may alias Y
__global__ void k_act_fwd(const float* X, int64_t ldx, float* Y, int64_t ldy, int64_t M, int C4, int act) {
  pdl_trigger();  // (programmatic dependent launch: the next kernel may start its set-up; common.cuh)
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= M * C4) return;
  const int64_t i = t / C4;
  const int c = (int)(t - i * C4) * 4;
  st4(Y + i * ldy + c, act_fwd4<true>(act, *reinterpret_cast<const float4*>(X + i * ldx + c)));
}

template <bool GEN>
__global__ void k_act_bwd(const float* __restrict__ dY, int64_t ldy, const float* __restrict__ H, int64_t ldh,
                          float* __restrict__ dH, int64_t ldd, int64_t M, int C4, int act) {
  pdl_trigger();  // (programmatic dependent launch: the next kernel may start its set-up; common.cuh)
  pdl_wait();     // launched through launch_pdl: nothing of the stream's earlier work is touched before this
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= M * C4) return;
  const int64_t i = t / C4;
  const int c = (int)(t - i * C4) * 4;
  float4 g = *reinterpret_cast<const float4*>(dY + i * ldy + c);
  if (act != LCAO_ACT_NONE) g = f4_mul(g, act_grad4<GEN>(act, ldg4(H + i * ldh + c)));
  st4(dH + i * ldd + c, g);
}

// the same, one element per thread, for rows that are not 16-byte aligned or widths / strides that are not multiples of 4
// (the CUDA-core fallback of lcao_linear_dgrad_act applies the factor in place with the caller's G and dX)
__global__ void k_act_bwd_any(const float* dY, int64_t ldy, const float* __restrict__ H, int64_t ldh, float* dH,
                              int64_t ldd, int64_t M, int C, int act) {
  pdl_trigger();
  pdl_wait();
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= M * C) return;
  const int64_t i = t / C;
  const int c = (int)(t - i * C);
  float g = dY[i * ldy + c];
  if (act != LCAO_ACT_NONE) g *= act_gradf(act, __ldg(H + i * ldh + c));
  dH[i * ldd + c] = g;
}

// backward of  agg[s] = sum_{e in out(s)} bw[e] * h[e]  with  h = SiLU(pre_h):
//   d_bw[e] = d_agg[src[e]] * h[e] ;  d_pre_h[e] = d_agg[src[e]] * bw[e] * SiLU'(pre_h[e])
template <bool GEN>
__global__ void __launch_bounds__(kWarpsPerCta * 32) k_msg_bwd(
    const float* __restrict__ d_agg, int64_t lda, const int32_t* __restrict__ src32, const float* __restrict__ h,
    const float* __restrict__ bw, const float* __restrict__ pre_h, int64_t E, int C, int act, float* __restrict__ d_bw,
    float* __restrict__ d_pre_h) {
  pdl_trigger();  // (programmatic dependent launch: the next kernel may start its set-up; common.cuh)
  pdl_wait();     // launched through launch_pdl: nothing of the stream's earlier work is touched before this
  const int64_t e = blockIdx.x * (int64_t)kWarpsPerCta + (threadIdx.x >> 5);
  if (e >= E) return;
  const int lane = threadIdx.x & 31;
  const float* pa = d_agg + src32[e] * lda;
  for (int c = lane * 4; c < C; c += 128) {
    const float4 g = ldg4(pa + c), b = ldg4(bw + e * (int64_t)C + c);
    const float4 p = ldg4(pre_h + e * (int64_t)C + c);
    const float4 hv = h ? ldg4(h + e * (int64_t)C + c) : act_fwd4<GEN>(act, p);
    st4(d_bw + e * (int64_t)C + c, f4_mul(g, hv));
    st4(d_pre_h + e * (int64_t)C + c, f4_mul(f4_mul(g, b), act_grad4<GEN>(act, p)));
  }
}

__global__ void k_sigmoid_rows(const float* __restrict__ x, int64_t ldx, float* __restrict__ out, int64_t ldo, int64_t M,
                               int C4) {
  pdl_trigger();  // (programmatic dependent launch: the next kernel may start its set-up; common.cuh)
  pdl_wait();     // launched through launch_pdl: nothing of the stream's earlier work is touched before this
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= M * C4) return;
  const int64_t i = t / C4;
  const int c = (int)(t - i * C4) * 4;
  const float4 v = ldg4(x + i * ldx + c);
  st4(out + i * ldo + c, make_float4(sigmoidf_acc(v.x), sigmoidf_acc(v.y), sigmoidf_acc(v.z), sigmoidf_acc(v.w)));
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

}  // namespace

#define DISPATCH_NL_VAL(NL, VAL, FN, ...)                                          \
  do {                                                                             \
    if (VAL) {                                                                     \
      switch (NL) {                                                                \
        case 1: FN<1, true> __VA_ARGS__; break;                                    \
        case 2: FN<2, true> __VA_ARGS__; break;                                    \
        case 3: FN<3, true> __VA_ARGS__; break;                                    \
        default: FN<4, true> __VA_ARGS__; break;                                   \
      }                                                                            \
    } else {                                                                       \
      switch (NL) {                                                                \
        case 1: FN<1, false> __VA_ARGS__; break;                                   \
        case 2: FN<2, false> __VA_ARGS__; break;                                   \
        case 3: FN<3, false> __VA_ARGS__; break;                                   \
        default: FN<4, false> __VA_ARGS__; break;                                  \
      }                                                                            \
    }                                                                              \
  } while (0)

extern "C" int lcao_coeff_contract_fwd(const float* cst1, const float* rb, const float* vmask, const int32_t* lgrp,
                                       int64_t E, int32_t O, int32_t C, int32_t NL, int32_t valence, float* B,
                                       void* stream) {
  if (E == 0) return LCAO_OK;
  LCAO_REQUIRE(cst1 && rb && lgrp && B && (!valence || vmask), "lcao_coeff_contract_fwd: null buffer");
  LCAO_REQUIRE(C % 4 == 0 && C > 0 && O > 0 && O <= LCAO_MAX_ORB && NL >= 1 && NL <= 4,
               "lcao_coeff_contract_fwd: need C %% 4 == 0, O <= %d, 1 <= NL <= 4 (got C=%d O=%d NL=%d)", LCAO_MAX_ORB, C, O, NL);
  LCAO_REQUIRE(aligned16(cst1) && aligned16(B), "lcao_coeff_contract_fwd: cst1 and B must be 16-byte aligned");
  const unsigned grid = (unsigned)ceil_div64(E, kWarpsPerCta);
  cudaStream_t st = (cudaStream_t)stream;
  DISPATCH_NL_VAL(NL, valence != 0, k_coeff_contract_fwd, <<<grid, kWarpsPerCta * 32, 0, st>>>(cst1, rb, vmask, lgrp, E, O, C, B));
  LCAO_LAUNCH_CHECK();
  return LCAO_OK;
}

extern "C" int lcao_coeff_contract_bwd(const float* cst1, const float* rb, const float* vmask, const int32_t* lgrp,
                                       const float* dB, int64_t E, int32_t O, int32_t C, int32_t NL, int32_t valence,
                                       float* d_cst1, float* d_rb, void* stream) {
  if (E == 0) return LCAO_OK;
  LCAO_REQUIRE(rb && lgrp && dB && d_cst1 && (!valence || vmask) && (!d_rb || cst1), "lcao_coeff_contract_bwd: null buffer");
  LCAO_REQUIRE(C % 4 == 0 && C > 0 && O > 0 && O <= LCAO_MAX_ORB && NL >= 1 && NL <= 4,
               "lcao_coeff_contract_bwd: need C %% 4 == 0, O <= %d, 1 <= NL <= 4", LCAO_MAX_ORB);
  LCAO_REQUIRE(aligned16(dB) && aligned16(d_cst1) && (!d_rb || aligned16(cst1)),
               "lcao_coeff_contract_bwd: dB, d_cst1 and (with d_rb) cst1 must be 16-byte aligned");
  const unsigned grid = (unsigned)ceil_div64(E, kWarpsPerCta);
  cudaStream_t st = (cudaStream_t)stream;
  DISPATCH_NL_VAL(NL, valence != 0, k_coeff_contract_bwd, <<<grid, kWarpsPerCta * 32, 0, st>>>(cst1, rb, vmask, lgrp, dB, E, O, C, d_cst1, d_rb));
  LCAO_LAUNCH_CHECK();
  return LCAO_OK;
}

extern "C" int lcao_twobody_fwd(const float* B, int32_t NG, const float* g, int64_t E, int32_t C, int32_t NL,
                                int32_t valence, float* lw, void* stream) {
  if (E == 0) return LCAO_OK;
  LCAO_REQUIRE(B && g && lw, "lcao_twobody_fwd: null buffer");
  LCAO_REQUIRE(C % 4 == 0 && C > 0 && C <= 256 && NG == NL + (valence ? 1 : 0),
               "lcao_twobody_fwd: need C %% 4 == 0, C <= 256, NG == NL + valence (C=%d NG=%d NL=%d)", C, NG, NL);
  const unsigned grid = (unsigned)ceil_div64(E, kWarpsPerCta);
  cudaStream_t st = (cudaStream_t)stream;
  if (C <= 128) {
    if (valence) LCAO_CUDA(launch_pdl(k_twobody_fwd<true, 1>, grid, kWarpsPerCta * 32, 0, st, B, NG, g, E, C, NL, lw));
    else LCAO_CUDA(launch_pdl(k_twobody_fwd<false, 1>, grid, kWarpsPerCta * 32, 0, st, B, NG, g, E, C, NL, lw));
  } else {
    if (valence) LCAO_CUDA(launch_pdl(k_twobody_fwd<true, 2>, grid, kWarpsPerCta * 32, 0, st, B, NG, g, E, C, NL, lw));
    else LCAO_CUDA(launch_pdl(k_twobody_fwd<false, 2>, grid, kWarpsPerCta * 32, 0, st, B, NG, g, E, C, NL, lw));
  }
  LCAO_LAUNCH_CHECK();
  return LCAO_OK;
}

extern "C" int lcao_twobody_bwd(const float* B, int32_t NG, const float* g, const float* d_lw, int64_t E, int32_t C,
                                int32_t NL, int32_t valence, int32_t compact, float* dB, float* d_g, void* stream) {
  if (E == 0) return LCAO_OK;
  LCAO_REQUIRE(B && g && d_lw && dB && d_g, "lcao_twobody_bwd: null buffer");
  LCAO_REQUIRE(C % 4 == 0 && C > 0 && C <= 256 && NG == NL + (valence ? 1 : 0),
               "lcao_twobody_bwd: need C %% 4 == 0, C <= 256, NG == NL + valence");
  const unsigned grid = (unsigned)ceil_div64(E, kWarpsPerCta);
  cudaStream_t st = (cudaStream_t)stream;
  if (C <= 128) {
    if (valence) LCAO_CUDA(launch_pdl(k_twobody_bwd<true, 1>, grid, kWarpsPerCta * 32, 0, st, B, NG, g, d_lw, E, C, NL, compact, dB, d_g));
    else LCAO_CUDA(launch_pdl(k_twobody_bwd<false, 1>, grid, kWarpsPerCta * 32, 0, st, B, NG, g, d_lw, E, C, NL, compact, dB, d_g));
  } else {
    if (valence) LCAO_CUDA(launch_pdl(k_twobody_bwd<true, 2>, grid, kWarpsPerCta * 32, 0, st, B, NG, g, d_lw, E, C, NL, compact, dB, d_g));
    else LCAO_CUDA(launch_pdl(k_twobody_bwd<false, 2>, grid, kWarpsPerCta * 32, 0, st, B, NG, g, d_lw, E, C, NL, compact, dB, d_g));
  }
  LCAO_LAUNCH_CHECK();
  return LCAO_OK;
}

extern "C" int lcao_edge_pair_fwd(const float* a, int64_t lda, const float* b, int64_t ldb, const float* bias,
                                  const int32_t* src32, const int32_t* dst32, int64_t E, int32_t C, int32_t act,
                                  float* out, float* pre, void* stream) {
  if (E == 0) return LCAO_OK;
  LCAO_REQUIRE(a && b && src32 && dst32 && out, "lcao_edge_pair_fwd: null buffer");
  LCAO_REQUIRE(C % 4 == 0 && lda % 4 == 0 && ldb % 4 == 0 && aligned16(a) && aligned16(b) && aligned16(out),
               "lcao_edge_pair_fwd: need C, lda, ldb multiples of 4 and 16-byte aligned buffers");
  if (act == LCAO_ACT_NONE || act == LCAO_ACT_SILU)
    LCAO_CUDA(launch_pdl(k_edge_pair_fwd<false>, (unsigned)ceil_div64(E, kWarpsPerCta), kWarpsPerCta * 32, 0, (cudaStream_t)stream, 
        a, lda, b, ldb, bias, src32, dst32, E, C, act, out, pre));
  else
    LCAO_CUDA(launch_pdl(k_edge_pair_fwd<true>, (unsigned)ceil_div64(E, kWarpsPerCta), kWarpsPerCta * 32, 0, (cudaStream_t)stream, 
        a, lda, b, ldb, bias, src32, dst32, E, C, act, out, pre));
  LCAO_LAUNCH_CHECK();
  return LCAO_OK;
}

extern "C" int lcao_segment_sum(const float* x, int64_t ldx, const float* y, int64_t ldy, const int32_t* ptr,
                                const int32_t* perm, int64_t R, int32_t C, int32_t mean, float* out, int64_t ldo,
                                void* stream) {
  if (R == 0 || C == 0) return LCAO_OK;
  // x may be NULL when there are no items at all (an edge-less batch): every segment is empty and out is zero-filled
  LCAO_REQUIRE(ptr && out, "lcao_segment_sum: null buffer");
  const bool vec = C % 4 == 0 && ldx % 4 == 0 && ldo % 4 == 0 && (!y || ldy % 4 == 0) && aligned16(x) &&
                   aligned16(out) && (!y || aligned16(y));
  const unsigned grid = (unsigned)ceil_div64(R, kWarpsPerCta);
  cudaStream_t st = (cudaStream_t)stream;
  const int kind = (mean >> 4) & 15;
  LCAO_REQUIRE(kind <= LCAO_ACT_LAST, "lcao_segment_sum: unsupported activation %d", kind);
  const bool gen = (mean & 6) != 0 && kind > LCAO_ACT_SILU;  // only the non-default activations take the generic kernel
  if (vec && !gen) LCAO_CUDA(launch_pdl(k_segment_sum<true, false>, grid, kWarpsPerCta * 32, 0, st, x, ldx, y, ldy, ptr, perm, R, C, mean, out, ldo));
  else if (vec) LCAO_CUDA(launch_pdl(k_segment_sum<true, true>, grid, kWarpsPerCta * 32, 0, st, x, ldx, y, ldy, ptr, perm, R, C, mean, out, ldo));
  else LCAO_CUDA(launch_pdl(k_segment_sum<false, true>, grid, kWarpsPerCta * 32, 0, st, x, ldx, y, ldy, ptr, perm, R, C, mean, out, ldo));
  LCAO_LAUNCH_CHECK();
  return LCAO_OK;
}

extern "C" int lcao_gather_rows(const float* table, int64_t ldt, const void* idx, int32_t idx_is64, const float* mul,
                                int64_t ldm, int64_t n, int32_t W, float* out, int64_t ldo, void* stream) {
  if (n == 0 || W == 0) return LCAO_OK;
  LCAO_REQUIRE(table && idx && out, "lcao_gather_rows: null buffer");
  const bool vec = W % 4 == 0 && ldt % 4 == 0 && ldo % 4 == 0 && aligned16(table) && aligned16(out) &&
                   (!mul || (ldm % 4 == 0 && aligned16(mul)));
  const int WV = vec ? W / 4 : W;
  const unsigned grid = (unsigned)ceil_div64(n * WV, 256);
  cudaStream_t st = (cudaStream_t)stream;
  if (idx_is64) {
    if (vec) k_gather_rows<int64_t, true><<<grid, 256, 0, st>>>(table, ldt, (const int64_t*)idx, mul, ldm, n, W, out, ldo);
    else k_gather_rows<int64_t, false><<<grid, 256, 0, st>>>(table, ldt, (const int64_t*)idx, mul, ldm, n, W, out, ldo);
  } else {
    if (vec) k_gather_rows<int32_t, true><<<grid, 256, 0, st>>>(table, ldt, (const int32_t*)idx, mul, ldm, n, W, out, ldo);
    else k_gather_rows<int32_t, false><<<grid, 256, 0, st>>>(table, ldt, (const int32_t*)idx, mul, ldm, n, W, out, ldo);
  }
  LCAO_LAUNCH_CHECK();
  return LCAO_OK;
}

extern "C" int lcao_reduce_by_key(const float* x, int64_t ldx, const int32_t* kptr, const int32_t* kperm,
                                  int64_t nkeys, int64_t n, int32_t W, float* acc, void* stream) {
  if (n == 0) return LCAO_OK;
  LCAO_REQUIRE(x && kptr && kperm && acc && nkeys > 0, "lcao_reduce_by_key: null buffer");
  LCAO_REQUIRE(W % 4 == 0 && ldx % 4 == 0 && aligned16(x) && aligned16(acc), "lcao_reduce_by_key: need W, ldx multiples of 4");
  k_reduce_by_key<<<(unsigned)ceil_div64(n, 32), 256, 0, (cudaStream_t)stream>>>(x, ldx, kptr, kperm, (int)nkeys, n, W, acc);
  LCAO_LAUNCH_CHECK();
  return LCAO_OK;
}

extern "C" int lcao_act_bwd(const float* dY, int64_t ldy, const float* H, int64_t ldh, float* dH, int64_t ldd,
                            int64_t M, int32_t C, int32_t act, void* stream) {
  if (M == 0 || C == 0) return LCAO_OK;
  LCAO_REQUIRE(dY && dH && (act == LCAO_ACT_NONE || H), "lcao_act_bwd: null buffer");
  const bool vec = C % 4 == 0 && ldy % 4 == 0 && ldd % 4 == 0 && aligned16(dY) && aligned16(dH) &&
                   (act == LCAO_ACT_NONE || (ldh % 4 == 0 && aligned16(H)));
  if (!vec) {
    LCAO_CUDA(launch_pdl(k_act_bwd_any, (unsigned)ceil_div64(M * C, 256), 256, 0, (cudaStream_t)stream, dY, ldy, H, ldh, dH,
                         ldd, M, C, act));
    LCAO_LAUNCH_CHECK();
    return LCAO_OK;
  }
  const unsigned grid = (unsigned)ceil_div64(M * (C / 4), 256);
  if (act <= LCAO_ACT_SILU) LCAO_CUDA(launch_pdl(k_act_bwd<false>, grid, 256, 0, (cudaStream_t)stream, dY, ldy, H, ldh, dH, ldd, M, C / 4, act));
  else LCAO_CUDA(launch_pdl(k_act_bwd<true>, grid, 256, 0, (cudaStream_t)stream, dY, ldy, H, ldh, dH, ldd, M, C / 4, act));
  LCAO_LAUNCH_CHECK();
  return LCAO_OK;
}

extern "C" int lcao_act_fwd(const float* X, int64_t ldx, float* Y, int64_t ldy, int64_t M, int32_t C, int32_t act,
                            void* stream) {
  if (M == 0 || C == 0) return LCAO_OK;
  LCAO_REQUIRE(X && Y && act >= LCAO_ACT_NONE && act <= LCAO_ACT_LAST, "lcao_act_fwd: bad arguments");
  LCAO_REQUIRE(C % 4 == 0 && ldx % 4 == 0 && ldy % 4 == 0 && aligned16(X) && aligned16(Y),
               "lcao_act_fwd: need C and strides multiples of 4, 16-byte aligned buffers");
  k_act_fwd<<<(unsigned)ceil_div64(M * (C / 4), 256), 256, 0, (cudaStream_t)stream>>>(X, ldx, Y, ldy, M, C / 4, act);
  LCAO_LAUNCH_CHECK();
  return LCAO_OK;
}

extern "C" int lcao_sigmoid_rows(const float* x, int64_t ldx, float* out, int64_t ldo, int64_t M, int32_t C, void* stream) {
  if (M == 0 || C == 0) return LCAO_OK;
  LCAO_REQUIRE(x && out, "lcao_sigmoid_rows: null buffer");
  LCAO_REQUIRE(C % 4 == 0 && ldx % 4 == 0 && ldo % 4 == 0 && aligned16(x) && aligned16(out),
               "lcao_sigmoid_rows: need C and strides multiples of 4, 16-byte aligned buffers");
  LCAO_CUDA(launch_pdl(k_sigmoid_rows, (unsigned)ceil_div64(M * (C / 4), 256), 256, 0, (cudaStream_t)stream, x, ldx, out, ldo, M, C / 4));
  LCAO_LAUNCH_CHECK();
  return LCAO_OK;
}

extern "C" int lcao_msg_bwd(const float* d_agg, int64_t lda, const int32_t* src32, const float* h, const float* bw,
                            const float* pre_h, int64_t E, int32_t C, int32_t act, float* d_bw, float* d_pre_h,
                            void* stream) {
  if (E == 0) return LCAO_OK;
  LCAO_REQUIRE(d_agg && src32 && bw && pre_h && d_bw && d_pre_h, "lcao_msg_bwd: null buffer");
  LCAO_REQUIRE(C % 4 == 0 && lda % 4 == 0 && aligned16(d_agg) && (!h || aligned16(h)) && aligned16(bw) && aligned16(pre_h) &&
                   aligned16(d_bw) && aligned16(d_pre_h),
               "lcao_msg_bwd: need C, lda multiples of 4 and 16-byte aligned buffers");
  LCAO_REQUIRE(act > LCAO_ACT_NONE && act <= LCAO_ACT_LAST, "lcao_msg_bwd: unsupported activation %d", act);
  const unsigned grid = (unsigned)ceil_div64(E, kWarpsPerCta);
  if (act == LCAO_ACT_SILU)
    LCAO_CUDA(launch_pdl(k_msg_bwd<false>, grid, kWarpsPerCta * 32, 0, (cudaStream_t)stream, d_agg, lda, src32, h, bw, pre_h, E, C, act, d_bw, d_pre_h));
  else
    LCAO_CUDA(launch_pdl(k_msg_bwd<true>, grid, kWarpsPerCta * 32, 0, (cudaStream_t)stream, d_agg, lda, src32, h, bw, pre_h, E, C, act, d_bw, d_pre_h));
  LCAO_LAUNCH_CHECK();
  return LCAO_OK;
}
