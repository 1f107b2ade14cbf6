// Orbital contraction against the SPECIES-PAIR coefficient table (lcaonet.py:170,180-183,200-203).
//
// The reference evaluates f_coeffs on all E*O coefficient rows.  Those rows are a function of the
// element pair (z_s, z_t) only (embed.py:234-249: cst[e] = BN(fe[z_t] * (1 + fz[z_s, z_t])), and
// f_coeffs has no bias and acts row-wise), so the same numbers are obtained by running f_coeffs on the
// P = (max_z+1)^2 table rows (a few thousand GEMM rows instead of E*O ~ 2 M) and contracting
//     B[e,l,:] = sum_{o in l} rb[e,o] * tab[pair_e, o, :]
// per edge.  The table (P*O*C' floats, 5.6 MB at the default sizes) is L2 resident, so this kernel's
// HBM traffic is the B it writes.  Backward: d_tab[p,o,:] = sum_{e: pair_e = p} rb[e,o] dB[e,l(o),:]
// is a keyed reduction done in two deterministic stages (per-chunk partials in sorted order, then a
// per-key sum in chunk order): no atomics.
//
// The kernel also emits the per-edge Gram matrix G[e,l,l'] = B[e,l,:].B[e,l',:] (FP64, upper
// triangle) that the three-body kernels use for the triplet norms (threebody.cu).
#include "common.cuh"

namespace {

constexpr int kWarps = 8;
constexpr int kChunk = 256;  // sorted entries per stage-1 CTA of the keyed reduction

__device__ __forceinline__ float4 f4z() { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ float4 f4fma(float a, float4 x, float4 acc) {
  acc.x = fmaf(a, x.x, acc.x); acc.y = fmaf(a, x.y, acc.y); acc.z = fmaf(a, x.z, acc.z); acc.w = fmaf(a, x.w, acc.w);
  return acc;
}
__device__ __forceinline__ float4 f4add(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }
__device__ __forceinline__ double dot4d(float4 a, float4 b) {
  return (double)a.x * b.x + (double)a.y * b.y + (double)a.z * b.z + (double)a.w * b.w;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Sum up to 8 per-lane FP64 partials over the 32 lanes with 9 shuffles (see bfly8 in threebody.cu);
// lane L ends up with the total of element 4*bit4(L) + 2*bit3(L) + bit2(L).
__device__ __forceinline__ double bfly8d(const double (&p)[8], int lane) {
  double q4[4], q2[2];
  bool up = (lane & 16) != 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const double recv = __shfl_xor_sync(0xffffffffu, up ? p[k] : p[k + 4], 16);
    q4[k] = (up ? p[k + 4] : p[k]) + recv;
  }
  up = (lane & 8) != 0;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const double recv = __shfl_xor_sync(0xffffffffu, up ? q4[k] : q4[k + 2], 8);
    q2[k] = (up ? q4[k + 2] : q4[k]) + recv;
  }
  up = (lane & 4) != 0;
  const double recv = __shfl_xor_sync(0xffffffffu, up ? q2[0] : q2[1], 4);
  double r = (up ? q2[1] : q2[0]) + recv;
  r += __shfl_xor_sync(0xffffffffu, r, 2);
  r += __shfl_xor_sync(0xffffffffu, r, 1);
  return r;
}
__device__ __forceinline__ int bfly8_index(int lane) { return ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1); }

// Writes the NP <= 10 Gram entries of one edge from per-lane FP64 partials.
template <int NP>
__device__ __forceinline__ void store_gram(const double (&g)[NP], int lane, double* __restrict__ out) {
  double p[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) p[i] = i < NP ? g[i] : 0.0;
  const double r = bfly8d(p, lane);
  const int idx = bfly8_index(lane);
  if ((lane & 3) == 0 && idx < NP) out[idx] = r;
  if (NP > 8) {  // NL = 4: entries 8, 9
    double p2[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) p2[i] = (8 + i) < NP ? g[(8 + i) < NP ? 8 + i : 0] : 0.0;
    const double r2 = bfly8d(p2, lane);
    if ((lane & 3) == 0 && 8 + idx < NP) out[8 + idx] = r2;
  }
}

// one warp per edge; lane owns float4 column lane (+32 for C > 128).  The group selection is folded into
// the scale factor (rb[e,o] for the orbital's own l, 0 otherwise): NL FMAs per orbital, no branches.
template <int NL, bool VAL>
__global__ void __launch_bounds__(kWarps * 32) k_pair_contract_fwd(
    const float* __restrict__ tab, const int64_t* __restrict__ pair, const float* __restrict__ rb,
    const float* __restrict__ vmask, const int32_t* __restrict__ lgrp, int64_t E, int O, int C, float* __restrict__ B,
    double* __restrict__ gram, float* __restrict__ psum) {
  pdl_trigger();  // (programmatic dependent launch: the next kernel may start its set-up; common.cuh)
  pdl_wait();     // launched through launch_pdl: nothing of the stream's earlier work is touched before this
  __shared__ int s_l[LCAO_MAX_ORB];
  if (threadIdx.x < O) s_l[threadIdx.x] = lgrp[threadIdx.x];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  constexpr int NG = NL + (VAL ? 1 : 0), NP = NL * (NL + 1) / 2;
  const int Cp = VAL ? 2 * C : C;
  // grid-stride over edges: the per-CTA set-up above is paid once, and a warp's next pair id is already in flight
  for (int64_t e = blockIdx.x * (int64_t)kWarps + (threadIdx.x >> 5); e < E; e += (int64_t)gridDim.x * kWarps) {
  const float* row = tab + pair[e] * (int64_t)O * Cp;
  double g[NP];
#pragma unroll
  for (int i = 0; i < NP; ++i) g[i] = 0.0;
  for (int c = lane * 4; c < C; c += 128) {
    float4 acc[NL + 1];
#pragma unroll
    for (int l = 0; l <= NL; ++l) acc[l] = f4z();
#pragma unroll 8
    for (int o = 0; o < O; ++o) {
      const float r = __ldg(rb + e * O + o);
      const int l = s_l[o];
      const float4 t = ldg4(row + (int64_t)o * Cp + c);
      if (VAL) {
        const float rm = r * __ldg(vmask + e * O + o);
        const float4 v = ldg4(row + (int64_t)o * Cp + C + c);
        acc[NL] = f4fma(rm, v, acc[NL]);
#pragma unroll
        for (int k = 0; k < NL; ++k) {
          acc[k] = f4fma(l == k ? r : 0.f, t, acc[k]);
          acc[k] = f4fma(l == k ? rm : 0.f, v, acc[k]);
        }
      } else {
#pragma unroll
        for (int k = 0; k < NL; ++k) acc[k] = f4fma(l == k ? r : 0.f, t, acc[k]);
      }
    }
#pragma unroll
    for (int l = 0; l < NG; ++l) st4(B + (e * NG + l) * (int64_t)C + c, acc[l]);
    if (psum) {  // [sum_{l<NL} B_l | B_NL]: all the two-body weight needs (lcao_twobody_* with NG = 1 + valence, NL = 1)
      float4 t = acc[0];
#pragma unroll
      for (int l = 1; l < NL; ++l) t = f4add(t, acc[l]);
      st4(psum + e * (int64_t)(VAL ? 2 : 1) * C + c, t);
      if (VAL) st4(psum + (e * 2 + 1) * (int64_t)C + c, acc[NL]);
    }
    if (gram) {
      int i = 0;
#pragma unroll
      for (int a = 0; a < NL; ++a)
#pragma unroll
        for (int b = a; b < NL; ++b) g[i++] += dot4d(acc[a], acc[b]);
    }
  }
  if (gram) store_gram<NP>(g, lane, gram + e * NP);
  }
}

// Gram matrix of an existing B (E,NG,C): upper triangle over the first NL groups, FP64
template <int NL>
__global__ void __launch_bounds__(kWarps * 32) k_gram(const float* __restrict__ B, int NG, int64_t E, int C,
                                                      double* __restrict__ gram) {
  const int64_t e = blockIdx.x * (int64_t)kWarps + (threadIdx.x >> 5);
  if (e >= E) return;
  const int lane = threadIdx.x & 31;
  constexpr int NP = NL * (NL + 1) / 2;
  double g[NP];
#pragma unroll
  for (int i = 0; i < NP; ++i) g[i] = 0.0;
  for (int c = lane * 4; c < C; c += 128) {
    float4 b[NL];
#pragma unroll
    for (int l = 0; l < NL; ++l) b[l] = ldg4(B + (e * NG + l) * (int64_t)C + c);
    int i = 0;
#pragma unroll
    for (int a = 0; a < NL; ++a)
#pragma unroll
      for (int bb = a; bb < NL; ++bb) g[i++] += dot4d(b[a], b[bb]);
  }
  store_gram<NP>(g, lane, gram + e * NP);
}

// d_rb[e,o] = tab[p,o,:C].dB[e,l(o),:] + m[e,o] tab[p,o,C:].(dB[e,l(o),:] + dB[e,NL,:])   (autograd forces)
template <bool VAL>
__global__ void __launch_bounds__(kWarps * 32) k_pair_contract_drb(
    const float* __restrict__ tab, const int64_t* __restrict__ pair, const float* __restrict__ vmask,
    const int32_t* __restrict__ lgrp, const float* __restrict__ dB, int64_t E, int O, int C, int NL,
    float* __restrict__ d_rb) {
  const int64_t e = blockIdx.x * (int64_t)kWarps + (threadIdx.x >> 5);
  if (e >= E) return;
  const int lane = threadIdx.x & 31;
  const int Cp = VAL ? 2 * C : C, NG = NL + (VAL ? 1 : 0);
  const float* row = tab + pair[e] * (int64_t)O * Cp;
  // eight orbitals at a time: the edge's gradient rows are read once per 128-column slice, the eight table rows are
  // independent loads, and the eight dots are reduced together by one 9-shuffle butterfly (the per-orbital form paid
  // a dependent load + 5 shuffles per orbital)
  for (int ob = 0; ob < O; ob += 8) {
    float part[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) part[u] = 0.f;
    for (int c = lane * 4; c < C; c += 128) {
      float4 g[4], gv = f4z();
#pragma unroll
      for (int l = 0; l < 4; ++l) g[l] = l < NL ? ldg4(dB + (e * NG + l) * (int64_t)C + c) : f4z();
      if (VAL) gv = ldg4(dB + (e * NG + NL) * (int64_t)C + c);
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int o = ob + u;
        if (o < O) {  // warp-uniform
          const int l = lgrp[o];
          const float4 gl = l == 0 ? g[0] : l == 1 ? g[1] : l == 2 ? g[2] : g[3];
          const float4 a = ldg4(row + (int64_t)o * Cp + c);
          part[u] += a.x * gl.x + a.y * gl.y + a.z * gl.z + a.w * gl.w;
          if (VAL) {
            const float4 s = f4add(gl, gv);
            const float4 v = ldg4(row + (int64_t)o * Cp + C + c);
            part[u] += __ldg(vmask + e * O + o) * (v.x * s.x + v.y * s.y + v.z * s.z + v.w * s.w);
          }
        }
      }
    }
    const float tot = bfly8(part, lane);
    const int o = ob + bfly8_index(lane);
    if ((lane & 3) == 0 && o < O) d_rb[e * O + o] = tot;
  }
}

// The same for C <= 128, walking the edges in PAIR-SORTED order (kperm): a warp takes 16 consecutive sorted positions
// and keeps the eight table rows of the current pair in registers, so the 4 KB of table rows are fetched once per run
// of equal pairs instead of once per edge (crystals with 36 species: 824 MB of L2 reads per call, 280 us -> see notes).
template <bool VAL>
__global__ void __launch_bounds__(kWarps * 32) k_pair_contract_drb_sorted(
    const float* __restrict__ tab, const int64_t* __restrict__ pair, const int32_t* __restrict__ kperm,
    const float* __restrict__ vmask, const int32_t* __restrict__ lgrp, const float* __restrict__ dB, int64_t E, int O,
    int C, int NL, float* __restrict__ d_rb) {
  constexpr int kRun = 16;
  const int64_t j0 = (blockIdx.x * (int64_t)kWarps + (threadIdx.x >> 5)) * kRun;
  if (j0 >= E) return;
  const int lane = threadIdx.x & 31;
  const int n = (int)min((int64_t)kRun, E - j0);
  const int Cp = VAL ? 2 * C : C, NG = NL + (VAL ? 1 : 0);
  const bool ok = lane * 4 < C;
  const int c = lane * 4;
  const int my_e = kperm[j0 + min(lane, n - 1)];
  const int64_t my_p = pair[my_e];
  for (int ob = 0; ob < O; ob += 8) {
    int lg[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) lg[u] = lgrp[min(ob + u, O - 1)];
    int64_t cur = -1;
    float4 trow[8], vrow[VAL ? 8 : 1];
    for (int t = 0; t < n; ++t) {
      const int64_t e = __shfl_sync(0xffffffffu, my_e, t);
      const int64_t pk = __shfl_sync(0xffffffffu, my_p, t);
      if (pk != cur) {  // warp-uniform
        cur = pk;
        const float* row = tab + pk * (int64_t)O * Cp;
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const bool live = ok && ob + u < O;
          trow[u] = live ? ldg4(row + (int64_t)(ob + u) * Cp + c) : f4z();
          if (VAL) vrow[u] = live ? ldg4(row + (int64_t)(ob + u) * Cp + C + c) : f4z();
        }
      }
      float4 g[4], gv = f4z();
#pragma unroll
      for (int l = 0; l < 4; ++l) g[l] = (l < NL && ok) ? ldg4(dB + (e * NG + l) * (int64_t)C + c) : f4z();
      if (VAL && ok) gv = ldg4(dB + (e * NG + NL) * (int64_t)C + c);
      float part[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const float4 gl = lg[u] == 0 ? g[0] : lg[u] == 1 ? g[1] : lg[u] == 2 ? g[2] : g[3];
        part[u] = trow[u].x * gl.x + trow[u].y * gl.y + trow[u].z * gl.z + trow[u].w * gl.w;
        if (VAL) {
          const float4 s = f4add(gl, gv);
          const float m = __ldg(vmask + e * O + min(ob + u, O - 1));
          part[u] += m * (vrow[u].x * s.x + vrow[u].y * s.y + vrow[u].z * s.z + vrow[u].w * s.w);
        }
      }
      const float tot = bfly8(part, lane);
      const int o = ob + bfly8_index(lane);
      if ((lane & 3) == 0 && o < O) d_rb[e * O + o] = tot;
    }
  }
}

// ---- keyed reduction, stage 0: cptr[k] = exclusive scan of ceil(count_k / kChunk)   (single CTA)
__global__ void __launch_bounds__(1024) k_chunk_ptr(const int32_t* __restrict__ kptr, int P, int32_t* __restrict__ cptr) {
  __shared__ int32_t part[1024];
  const int per = (P + 1023) / 1024;
  const int lo = min(P, (int)threadIdx.x * per), hi = min(P, lo + per);
  int32_t s = 0;
  for (int k = lo; k < hi; ++k) s += (kptr[k + 1] - kptr[k] + kChunk - 1) / kChunk;
  part[threadIdx.x] = s;
  __syncthreads();
  for (int o = 1; o < 1024; o <<= 1) {  // Hillis-Steele inclusive scan
    const int32_t v = (threadIdx.x >= (unsigned)o) ? part[threadIdx.x - o] : 0;
    __syncthreads();
    part[threadIdx.x] += v;
    __syncthreads();
  }
  int32_t run = part[threadIdx.x] - s;
  for (int k = lo; k < hi; ++k) {
    cptr[k] = run;
    run += (kptr[k + 1] - kptr[k] + kChunk - 1) / kChunk;
  }
  if (threadIdx.x == 1023) cptr[P] = part[1023];
}

// ---- stage 1: CTA = one chunk of one key; thread = one (o, float4 column); partial[chunk][o][Cp].
// The chunk's edge ids and radial values are staged in shared memory first, so the main loop's dB loads
// are independent of each other and 8 of them are in flight per thread.
template <bool VAL>
__global__ void __launch_bounds__(256) k_pair_reduce_partial(
    const int32_t* __restrict__ kptr, const int32_t* __restrict__ kperm, const int32_t* __restrict__ cptr, int P,
    const float* __restrict__ rb, const float* __restrict__ vmask, const int32_t* __restrict__ lgrp,
    const float* __restrict__ dB, int O, int C, int NL, float* __restrict__ partial) {
  pdl_trigger();  // (programmatic dependent launch: the next kernel may start its set-up; common.cuh)
  pdl_wait();     // launched through launch_pdl: nothing of the stream's earlier work is touched before this
  extern __shared__ __align__(16) unsigned char smem_raw[];
  int32_t* s_e = reinterpret_cast<int32_t*>(smem_raw);            // kChunk
  float* s_r = reinterpret_cast<float*>(s_e + kChunk);            // O x kChunk   rb[e,o]
  float* s_m = s_r + (size_t)O * kChunk;                          // VAL: O x kChunk   rb[e,o] * vmask[e,o]
  const int chunk = blockIdx.x;
  if (chunk >= cptr[P]) return;
  int lo = 0, hi = P;  // last key with cptr[key] <= chunk (keys without entries have empty chunk ranges)
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (cptr[mid] <= chunk) lo = mid; else hi = mid;
  }
  const int key = lo;
  const int32_t j0 = kptr[key] + (chunk - cptr[key]) * kChunk;
  const int n = min(kChunk, kptr[key + 1] - j0);
  for (int t = threadIdx.x; t < n; t += 256) {
    const int64_t e = kperm[j0 + t];
    s_e[t] = (int32_t)e;
    for (int o = 0; o < O; ++o) {
      const float r = __ldg(rb + e * O + o);
      s_r[o * kChunk + t] = r;
      if (VAL) s_m[o * kChunk + t] = r * __ldg(vmask + e * O + o);
    }
  }
  __syncthreads();
  const int C4 = C >> 2;
  const int NG = NL + (VAL ? 1 : 0), Cp = VAL ? 2 * C : C;
  for (int w = threadIdx.x; w < O * C4; w += 256) {
    const int o = w / C4, c = (w - o * C4) * 4;
    const int l = lgrp[o];
    const float* sr = s_r + o * kChunk;
    const float* sm = s_m + o * kChunk;
    float4 accA = f4z(), accV = f4z();
    int t = 0;
    for (; t + 8 <= n; t += 8) {
      float4 g[8], gv[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        g[u] = ldg4(dB + ((int64_t)s_e[t + u] * NG + l) * C + c);
        if (VAL) gv[u] = ldg4(dB + ((int64_t)s_e[t + u] * NG + NL) * C + c);
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        accA = f4fma(sr[t + u], g[u], accA);
        if (VAL) accV = f4fma(sm[t + u], f4add(g[u], gv[u]), accV);
      }
    }
    for (; t < n; ++t) {
      const float4 g = ldg4(dB + ((int64_t)s_e[t] * NG + l) * C + c);
      accA = f4fma(sr[t], g, accA);
      if (VAL) accV = f4fma(sm[t], f4add(g, ldg4(dB + ((int64_t)s_e[t] * NG + NL) * C + c)), accV);
    }
    float* out = partial + ((int64_t)chunk * O + o) * Cp + c;
    st4(out, accA);
    if (VAL) st4(out + C, accV);
  }
}

// ---- stage 2: d_tab[key][o][:] = sum of the key's partials (zeros for absent keys).  CTA = (key, 32 float4 columns);
// its 8 sub-rows each add every 8th chunk of the key in chunk order and the 8 sub-sums are combined in a fixed order:
// deterministic, and a key that owns hundreds of chunks (one or two species in the batch: crystals) is summed by 8
// independent chains of loads instead of one (355 us -> see profiles/r01_notes.md).
__global__ void __launch_bounds__(256) k_pair_reduce_final(const int32_t* __restrict__ cptr, int P, int W4,
                                                           const float* __restrict__ partial,
                                                           float* __restrict__ d_tab) {
  pdl_trigger();  // (programmatic dependent launch: the next kernel may start its set-up; common.cuh)
  pdl_wait();     // launched through launch_pdl: nothing of the stream's earlier work is touched before this
  __shared__ float4 s_part[8][32];
  const int key = blockIdx.x, col = blockIdx.y * 32 + (threadIdx.x & 31), sub = threadIdx.x >> 5;
  const int32_t q0 = cptr[key], q1 = cptr[key + 1];
  float4 acc = f4z();
  if (col < W4)
    for (int32_t q = q0 + sub; q < q1; q += 8) acc = f4add(acc, ldg4(partial + ((int64_t)q * W4 + col) * 4));
  s_part[sub][threadIdx.x & 31] = acc;
  __syncthreads();
  if (sub == 0 && col < W4) {
#pragma unroll
    for (int u = 1; u < 8; ++u) acc = f4add(acc, s_part[u][threadIdx.x]);
    st4(d_tab + ((int64_t)key * W4 + col) * 4, acc);
  }
}

inline bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

}  // namespace

extern "C" int lcao_pair_contract_fwd(const float* tab, const int64_t* pair, const float* rb, const float* vmask,
                                      const int32_t* lgrp, int64_t E, int32_t O, int32_t C, int32_t NL,
                                      int32_t valence, float* B, double* gram, float* psum, void* stream) {
  if (E == 0) return LCAO_OK;
  LCAO_REQUIRE(tab && pair && rb && lgrp && B && (!valence || vmask), "lcao_pair_contract_fwd: null buffer");
  LCAO_REQUIRE(C % 4 == 0 && C > 0 && O > 0 && O <= LCAO_MAX_ORB && NL >= 1 && NL <= 4,
               "lcao_pair_contract_fwd: need C %% 4 == 0, O <= %d, 1 <= NL <= 4 (got C=%d O=%d NL=%d)", LCAO_MAX_ORB, C, O, NL);
  LCAO_REQUIRE(al16(tab) && al16(B) && al16(psum), "lcao_pair_contract_fwd: tab, B and psum must be 16-byte aligned");
  const int64_t want = ceil_div64(E, kWarps);
  const unsigned grid = (unsigned)(want < 148 * 16 ? want : 148 * 16);
  cudaStream_t st = (cudaStream_t)stream;
#define PC_CALL(nl, val) LCAO_CUDA(launch_pdl(k_pair_contract_fwd<nl, val>, grid, kWarps * 32, 0, st, tab, pair, rb, vmask, lgrp, E, O, C, B, gram, psum))
  if (valence) {
    switch (NL) { case 1: PC_CALL(1, true); break; case 2: PC_CALL(2, true); break; case 3: PC_CALL(3, true); break; default: PC_CALL(4, true); }
  } else {
    switch (NL) { case 1: PC_CALL(1, false); break; case 2: PC_CALL(2, false); break; case 3: PC_CALL(3, false); break; default: PC_CALL(4, false); }
  }
#undef PC_CALL
  LCAO_LAUNCH_CHECK();
  return LCAO_OK;
}

extern "C" int lcao_coeff_gram(const float* B, int32_t NG, int64_t E, int32_t C, int32_t NL, double* gram, void* stream) {
  if (E == 0) return LCAO_OK;
  LCAO_REQUIRE(B && gram, "lcao_coeff_gram: null buffer");
  LCAO_REQUIRE(C % 4 == 0 && C > 0 && NL >= 1 && NL <= 4 && NG >= NL && al16(B), "lcao_coeff_gram: need C %% 4 == 0, 1 <= NL <= 4, NG >= NL");
  const unsigned grid = (unsigned)ceil_div64(E, kWarps);
  cudaStream_t st = (cudaStream_t)stream;
  switch (NL) {
    case 1: k_gram<1><<<grid, kWarps * 32, 0, st>>>(B, NG, E, C, gram); break;
    case 2: k_gram<2><<<grid, kWarps * 32, 0, st>>>(B, NG, E, C, gram); break;
    case 3: k_gram<3><<<grid, kWarps * 32, 0, st>>>(B, NG, E, C, gram); break;
    default: k_gram<4><<<grid, kWarps * 32, 0, st>>>(B, NG, E, C, gram); break;
  }
  LCAO_LAUNCH_CHECK();
  return LCAO_OK;
}

extern "C" int64_t lcao_pair_contract_bwd_scratch(int64_t E, int64_t P, int32_t O, int32_t C, int32_t valence) {
  const int64_t chunks = ceil_div64(E, kChunk) + P;
  const int64_t Cp = valence ? 2 * (int64_t)C : C;
  return ((P + 1 + 3) / 4) * 16 + chunks * O * Cp * (int64_t)sizeof(float);  // bytes: cptr (padded to 16) + partials
}

extern "C" int lcao_pair_contract_bwd(const float* tab, const int64_t* pair, const int32_t* kptr, const int32_t* kperm,
                                      const float* rb, const float* vmask, const int32_t* lgrp, const float* dB,
                                      int64_t E, int64_t P, int32_t O, int32_t C, int32_t NL, int32_t valence,
                                      float* d_tab, float* d_rb, void* scratch, void* stream) {
  LCAO_REQUIRE(P > 0 && P < (1 << 30) && (d_tab || d_rb) && (!d_tab || scratch) && kptr, "lcao_pair_contract_bwd: null buffer");
  LCAO_REQUIRE(E == 0 || (kperm && rb && lgrp && dB && (!valence || vmask)), "lcao_pair_contract_bwd: null buffer");
  LCAO_REQUIRE(C % 4 == 0 && C > 0 && O > 0 && O <= LCAO_MAX_ORB && NL >= 1 && NL <= 4,
               "lcao_pair_contract_bwd: need C %% 4 == 0, O <= %d, 1 <= NL <= 4", LCAO_MAX_ORB);
  LCAO_REQUIRE(!d_rb || E == 0 || (tab && pair), "lcao_pair_contract_bwd: d_rb needs tab and pair");
  LCAO_REQUIRE(al16(dB) && al16(d_tab) && al16(scratch) && (!d_rb || al16(tab)),
               "lcao_pair_contract_bwd: dB, d_tab, scratch and (with d_rb) tab must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  int32_t* cptr = static_cast<int32_t*>(scratch);
  float* partial = reinterpret_cast<float*>(static_cast<char*>(scratch) + ((P + 1 + 3) / 4) * 16);
  const int Cp = valence ? 2 * C : C;
  const int64_t chunks = ceil_div64(E, kChunk) + P;
  if (d_tab) {  // (d_tab == NULL: only d_rb is wanted — the positions-only pass of autograd forces)
  k_chunk_ptr<<<1, 1024, 0, st>>>(kptr, (int)P, cptr);
  LCAO_LAUNCH_CHECK();
  if (E > 0) {
    const size_t smem = sizeof(int32_t) * kChunk + sizeof(float) * (size_t)O * kChunk * (valence ? 2 : 1);
    if (smem > 48 * 1024) {
      LCAO_CUDA(cudaFuncSetAttribute(valence ? k_pair_reduce_partial<true> : k_pair_reduce_partial<false>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    if (valence) LCAO_CUDA(launch_pdl(k_pair_reduce_partial<true>, (unsigned)chunks, 256, smem, st, kptr, kperm, cptr, (int)P, rb, vmask, lgrp, dB, O, C, NL, partial));
    else LCAO_CUDA(launch_pdl(k_pair_reduce_partial<false>, (unsigned)chunks, 256, smem, st, kptr, kperm, cptr, (int)P, rb, vmask, lgrp, dB, O, C, NL, partial));
    LCAO_LAUNCH_CHECK();
  }
  const int W4 = O * Cp / 4;
  LCAO_CUDA(launch_pdl(k_pair_reduce_final, dim3((unsigned)P, (unsigned)((W4 + 31) / 32)), 256, 0, st, cptr, (int)P, W4, partial, d_tab));
  LCAO_LAUNCH_CHECK();
  }
  if (d_rb && E > 0) {
    if (C <= 128) {  // pair-sorted walk: table rows stay in registers across a run of equal pairs
      const unsigned grid = (unsigned)ceil_div64(ceil_div64(E, 16), kWarps);
      if (valence) k_pair_contract_drb_sorted<true><<<grid, kWarps * 32, 0, st>>>(tab, pair, kperm, vmask, lgrp, dB, E, O, C, NL, d_rb);
      else k_pair_contract_drb_sorted<false><<<grid, kWarps * 32, 0, st>>>(tab, pair, kperm, vmask, lgrp, dB, E, O, C, NL, d_rb);
    } else {
      const unsigned grid = (unsigned)ceil_div64(E, kWarps);
      if (valence) k_pair_contract_drb<true><<<grid, kWarps * 32, 0, st>>>(tab, pair, vmask, lgrp, dB, E, O, C, NL, d_rb);
      else k_pair_contract_drb<false><<<grid, kWarps * 32, 0, st>>>(tab, pair, vmask, lgrp, dB, E, O, C, NL, d_rb);
    }
    LCAO_LAUNCH_CHECK();
  }
  return LCAO_OK;
}
