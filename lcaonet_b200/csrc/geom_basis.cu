// Edge geometry + hydrogen-like radial basis with smooth cutoff, forward and position-backward.
// Reference: base.py:27-43 (vectors under PBC), cutoff.py:32-67, rbf.py:92-103,129-142,164-182.
// One thread per edge; arithmetic in fp64 (E-sized, negligible cost) so that the fp32 outputs are
// correctly rounded images of the fp64 oracle: the cutoff is evaluated in its factored form
// fc = (1-q)^3 (1+3q+6q^2) which has no cancellation at the cutoff shell (SURVEY.md Appendix B).
#include "common.cuh"

namespace {

struct CutVal { double f, df; };

__device__ __forceinline__ CutVal cutoff_eval(int kind, double r, double rc) {
  CutVal c{0.0, 0.0};
  if (!(r <= rc)) return c;
  const double q = r / rc, u = 1.0 - q;
  if (kind == LCAO_CUT_POLYNOMIAL) {
    c.f = u * u * u * (1.0 + q * (3.0 + 6.0 * q));
    c.df = -30.0 * q * q * u * u / rc;
  } else if (kind == LCAO_CUT_ENVELOPE) {  // p = 5
    c.f = u * u * u * (1.0 + q * (3.0 + q * (6.0 + q * (10.0 + 15.0 * q))));
    c.df = -105.0 * q * q * q * q * u * u / rc;
  } else {  // cosine
    const double a = 3.14159265358979323846 / rc;
    c.f = 0.5 * (cos(a * r) + 1.0);
    c.df = -0.5 * a * sin(a * r);
  }
  return c;
}

__global__ void __launch_bounds__(128) k_geom_basis_fwd(
    const float* __restrict__ pos, const float* __restrict__ shift, const float* __restrict__ lattice,
    const int64_t* __restrict__ batch, const int32_t* __restrict__ src32, const int32_t* __restrict__ dst32,
    int64_t E, const __grid_constant__ lcao_basis_spec sp, float* __restrict__ dist, float* __restrict__ unit,
    float* __restrict__ rb, float* __restrict__ drb) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= E) return;
  const int32_t s = src32[e], t = dst32[e];
  const float* L = lattice + 9 * (batch ? batch[s] : 0);
  const double s0 = shift[3 * e], s1 = shift[3 * e + 1], s2 = shift[3 * e + 2];
  double v[3];
#pragma unroll
  for (int j = 0; j < 3; ++j)
    v[j] = ((double)pos[3 * t + j] - (double)pos[3 * s + j]) + (s0 * L[j] + s1 * L[3 + j] + s2 * L[6 + j]);
  const double r = sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
  dist[e] = (float)r;
#pragma unroll
  for (int j = 0; j < 3; ++j) unit[3 * e + j] = (float)(v[j] / r);
  const CutVal fc = cutoff_eval(sp.cutoff_kind, r, sp.rc);
  const int O = sp.n_unique * sp.n_rep;
  for (int u = 0; u < sp.n_unique; ++u) {
    double R, dR;
    if (sp.rbf_kind == LCAO_RBF_HYDROGEN) {
      const double zs = 2.0 / (sp.n[u] * sp.a0), zeta = zs * r;
      double p = 0.0, dp = 0.0;
      for (int i = sp.deg[u]; i >= 0; --i) {  // Horner for value and derivative
        dp = dp * zeta + p;
        p = p * zeta + sp.poly[u][i];
      }
      const int l = sp.l[u];
      double zl = 1.0, zlm1 = 0.0;  // zeta^l and l*zeta^(l-1)
      for (int i = 0; i < l; ++i) { zlm1 = zl * (i + 1); zl *= zeta; }
      if (l == 0) zlm1 = 0.0;
      const double ex = exp(-0.5 * zeta);
      R = sp.norm[u] * p * zl * ex;
      dR = sp.norm[u] * ex * (dp * zl + p * zlm1 - 0.5 * p * zl) * zs;
    } else {  // spherical Bessel j0-like: sin(pi n r / rc) / r
      const double w = 3.14159265358979323846 * sp.n[u] / sp.rc;
      R = sin(w * r) / r;
      dR = w * cos(w * r) / r - sin(w * r) / (r * r);
    }
    const float val = (float)(fc.f * R), dval = (float)(fc.df * R + fc.f * dR);
    for (int k = 0; k < sp.n_rep; ++k) {
      rb[e * O + u * sp.n_rep + k] = val;
      if (drb) drb[e * O + u * sp.n_rep + k] = dval;
    }
  }
}

// dvec[e] = (d_unit - unit (unit . d_unit)) / r + (d_dist + sum_o d_rb * drb) unit
__global__ void k_geom_edge_bwd(const float* __restrict__ dist, const float* __restrict__ unit,
                                const float* __restrict__ drb, const float* __restrict__ d_dist,
                                const float* __restrict__ d_unit, const float* __restrict__ d_rb, int64_t E, int O,
                                float* __restrict__ dvec) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= E) return;
  const float ux = unit[3 * e], uy = unit[3 * e + 1], uz = unit[3 * e + 2];
  float gr = d_dist ? d_dist[e] : 0.f;
  if (d_rb)
    for (int o = 0; o < O; ++o) gr += d_rb[e * O + o] * drb[e * O + o];
  float gx = gr * ux, gy = gr * uy, gz = gr * uz;
  if (d_unit) {
    const float ax = d_unit[3 * e], ay = d_unit[3 * e + 1], az = d_unit[3 * e + 2];
    const float dot = ax * ux + ay * uy + az * uz, inv = 1.0f / dist[e];
    gx += (ax - ux * dot) * inv;
    gy += (ay - uy * dot) * inv;
    gz += (az - uz * dot) * inv;
  }
  dvec[3 * e] = gx; dvec[3 * e + 1] = gy; dvec[3 * e + 2] = gz;
}

// d_pos[n] = sum_{e in in(n)} dvec[e] - sum_{e in out(n)} dvec[e]   (vec = pos[t] - pos[s] + ...)
__global__ void k_geom_node_bwd(const float* __restrict__ dvec, const int32_t* __restrict__ in_ptr,
                                const int32_t* __restrict__ in_edge, const int32_t* __restrict__ out_ptr,
                                const int32_t* __restrict__ out_edge, int64_t N, float* __restrict__ d_pos) {
  const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (idx >= N * 3) return;
  const int64_t n = idx / 3;
  const int j = (int)(idx - n * 3);
  float acc = 0.f;
  for (int32_t p = in_ptr[n]; p < in_ptr[n + 1]; ++p) acc += dvec[3 * (int64_t)in_edge[p] + j];
  for (int32_t p = out_ptr[n]; p < out_ptr[n + 1]; ++p) acc -= dvec[3 * (int64_t)out_edge[p] + j];
  d_pos[idx] = acc;
}

// ---- cell derivatives: d E / d lattice and the virial, per graph (lcao_geom_cell_bwd), and the per-atom virials
// (lcao_geom_atom_virial_bwd).
// A graph's nodes (seg_perm[seg_ptr[g] .. seg_ptr[g+1]), or that range itself when seg_perm is NULL) are cut into chunks of
// LCAO_CELL_CHUNK; chunk j of graph g owns partial slot  seg_ptr[g] / LCAO_CELL_CHUNK + g + j.  These ranges are disjoint
// (the slots of g end at or before the first slot of g + 1), their union lies in [0, N / LCAO_CELL_CHUNK + B), and a slot
// finds its graph by a binary search over seg_ptr: no scan kernel, no atomics.
constexpr int kCellWarps = 8;
constexpr int kCellVals = 18;  // 9 of d E / d L, then 9 of the virial

__device__ __forceinline__ int64_t cell_slot_base(const int32_t* seg_ptr, int g) {
  return seg_ptr[g] / LCAO_CELL_CHUNK + g;
}

// vec = pos[t] - pos[s] + shift . L in FP64, formed exactly as k_geom_basis_fwd forms it (not dist * unit: that would carry
// the FP32 rounding of unit into the virial); ps = pos[s], L = the lattice of the graph of s.  Both virial reductions below
// form vec here, so the per-atom virials of a graph add up to its virial up to the rounding of the sums.
__device__ __forceinline__ void edge_vec(const float* __restrict__ pos, int32_t t, const double ps[3], const double sh[3],
                                         const float* __restrict__ L, double v[3]) {
#pragma unroll
  for (int c = 0; c < 3; ++c)
    v[c] = ((double)pos[3 * t + c] - ps[c]) + (sh[0] * L[c] + sh[1] * L[3 + c] + sh[2] * L[6 + c]);
}

// Per-atom virial of node n (one warp): W_n = 1/2 sum_{e: s_e = n} vec_e (x) dvec_e + 1/2 sum_{e: t_e = n} vec_e (x) dvec_e.
// Lane l takes the node's out-edges l, l + 32, ... in out-CSR order, then its in-edges the same way in in-CSR order, so a
// node of any degree is one warp's loop.  FP64 accumulation, a fixed xor butterfly and one rounding after the 1/2: the row
// is a fixed function of the inputs (bitwise reproducible), and no atomics.
__device__ __forceinline__ void atom_virial_row(
    const float* __restrict__ pos, const float* __restrict__ shift, const float* __restrict__ lattice,
    const int64_t* __restrict__ batch, const int32_t* __restrict__ dst32, const float* __restrict__ dvec,
    const int32_t* __restrict__ out_ptr, const int32_t* __restrict__ out_edge, const int32_t* __restrict__ in_ptr,
    const int32_t* __restrict__ in_edge, const int32_t* __restrict__ in_src, int64_t n, int lane,
    float* __restrict__ atom_virial) {
  double acc[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) acc[k] = 0.0;
  const int32_t o0 = out_ptr[n], o1 = out_ptr[n + 1], i0 = in_ptr[n], i1 = in_ptr[n + 1];
  if (o0 < o1 || i0 < i1) {  // (an atom without edges reads nothing: edge buffers may be NULL when E == 0)
    const double pn[3] = {pos[3 * n], pos[3 * n + 1], pos[3 * n + 2]};
    const float* Ln = lattice + 9 * (batch ? batch[n] : 0);
    for (int32_t p = o0 + lane; p < o1; p += 32) {  // s = n: vec = pos[t] - pos[n] + shift . L[batch[n]]
      const int64_t e = out_edge[p];
      const double sh[3] = {shift[3 * e], shift[3 * e + 1], shift[3 * e + 2]};
      const double dv[3] = {dvec[3 * e], dvec[3 * e + 1], dvec[3 * e + 2]};
      double v[3];
      edge_vec(pos, dst32[e], pn, sh, Ln, v);
#pragma unroll
      for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int c = 0; c < 3; ++c) acc[3 * a + c] = fma(v[a], dv[c], acc[3 * a + c]);
    }
    for (int32_t p = i0 + lane; p < i1; p += 32) {  // t = n: vec = pos[n] - pos[s] + shift . L[batch[s]]
      const int64_t e = in_edge[p];
      const int32_t s = in_src[p];
      const double ps[3] = {pos[3 * s], pos[3 * s + 1], pos[3 * s + 2]};
      const double sh[3] = {shift[3 * e], shift[3 * e + 1], shift[3 * e + 2]};
      const double dv[3] = {dvec[3 * e], dvec[3 * e + 1], dvec[3 * e + 2]};
      double v[3];
      edge_vec(pos, (int32_t)n, ps, sh, lattice + 9 * (batch ? batch[s] : 0), v);
#pragma unroll
      for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int c = 0; c < 3; ++c) acc[3 * a + c] = fma(v[a], dv[c], acc[3 * a + c]);
    }
  }
  float out = 0.f;
#pragma unroll
  for (int k = 0; k < 9; ++k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
    if (lane == k) out = (float)(0.5 * acc[k]);
  }
  if (lane < 9) atom_virial[9 * n + lane] = out;
}

// Two reductions of the same dvec, with the same vec (edge_vec), in one kernel:
//  - atom_virial != NULL (lcao_geom_atom_virial_bwd): warp w of CTA b is node 8 b + w (atom_virial_row); the cell arguments
//    (seg_ptr, seg_perm, B, partial) are unused.
//  - otherwise, stage 1 of lcao_geom_cell_bwd: CTA = one chunk; warp w takes the chunk's nodes w, w + 8, ...; lane l the
//    out-edges l, l + 32, ... of each node in out-CSR order.  Every lane accumulates shift (x) dvec and vec (x) dvec in
//    FP64; the lanes are combined by a fixed xor butterfly and the warps in warp order: the partial is a fixed function of
//    the inputs (bitwise reproducible).
__global__ void __launch_bounds__(kCellWarps * 32) k_geom_cell_partial(
    const float* __restrict__ pos, const float* __restrict__ shift, const float* __restrict__ lattice,
    const int64_t* __restrict__ batch, const int32_t* __restrict__ dst32, const float* __restrict__ dvec,
    const int32_t* __restrict__ out_ptr, const int32_t* __restrict__ out_edge, const int32_t* __restrict__ seg_ptr,
    const int32_t* __restrict__ seg_perm, int B, double* __restrict__ partial, const int32_t* __restrict__ in_ptr,
    const int32_t* __restrict__ in_edge, const int32_t* __restrict__ in_src, int64_t N, float* __restrict__ atom_virial) {
  pdl_trigger();  // (programmatic dependent launch: the next kernel may start its set-up; common.cuh)
  pdl_wait();     // launched through launch_pdl: nothing of the stream's earlier work is touched before this
  if (atom_virial) {
    const int64_t n = blockIdx.x * (int64_t)kCellWarps + (threadIdx.x >> 5);
    if (n < N)
      atom_virial_row(pos, shift, lattice, batch, dst32, dvec, out_ptr, out_edge, in_ptr, in_edge, in_src, n,
                      threadIdx.x & 31, atom_virial);
    return;
  }
  __shared__ double s_red[kCellWarps][kCellVals];
  const int64_t slot = blockIdx.x;
  int lo = 0, hi = B;  // the graph: last g with cell_slot_base(g) <= slot (strictly increasing in g)
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (cell_slot_base(seg_ptr, mid) <= slot) lo = mid; else hi = mid;
  }
  const int g = lo;
  const int64_t j0 = seg_ptr[g] + (slot - cell_slot_base(seg_ptr, g)) * LCAO_CELL_CHUNK;
  const int64_t j1 = min(j0 + LCAO_CELL_CHUNK, (int64_t)seg_ptr[g + 1]);
  if (j0 >= j1) return;  // a slot no chunk owns: never read
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double acc[kCellVals];
#pragma unroll
  for (int k = 0; k < kCellVals; ++k) acc[k] = 0.0;
  for (int64_t j = j0 + warp; j < j1; j += kCellWarps) {
    const int32_t n = seg_perm ? seg_perm[j] : (int32_t)j;
    const int32_t p0 = out_ptr[n], p1 = out_ptr[n + 1];
    if (p0 >= p1) continue;
    const float* L = lattice + 9 * (batch ? batch[n] : 0);
    const double ps0 = pos[3 * n], ps1 = pos[3 * n + 1], ps2 = pos[3 * n + 2];
    for (int32_t p = p0 + lane; p < p1; p += 32) {
      const int64_t e = out_edge[p];
      const int32_t t = dst32[e];
      const double sh[3] = {shift[3 * e], shift[3 * e + 1], shift[3 * e + 2]};
      const double ps[3] = {ps0, ps1, ps2};
      const double dv[3] = {dvec[3 * e], dvec[3 * e + 1], dvec[3 * e + 2]};
      double v[3];
      edge_vec(pos, t, ps, sh, L, v);
#pragma unroll
      for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          acc[3 * a + c] = fma(sh[a], dv[c], acc[3 * a + c]);
          acc[9 + 3 * a + c] = fma(v[a], dv[c], acc[9 + 3 * a + c]);
        }
    }
  }
#pragma unroll
  for (int k = 0; k < kCellVals; ++k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
  }
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < kCellVals; ++k) s_red[warp][k] = acc[k];
  }
  __syncthreads();
  if (threadIdx.x < kCellVals) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < kCellWarps; ++w) s += s_red[w][threadIdx.x];
    partial[slot * kCellVals + threadIdx.x] = s;
  }
}

// Stage 2: warp = graph; lane k < 18 adds component k of the graph's chunk partials in chunk order and rounds once.
// Graphs without nodes or without edges get zeros.
__global__ void __launch_bounds__(kCellWarps * 32) k_geom_cell_final(const int32_t* __restrict__ seg_ptr, int B,
                                                                     const double* __restrict__ partial,
                                                                     float* __restrict__ d_lattice,
                                                                     float* __restrict__ virial) {
  pdl_trigger();
  pdl_wait();  // the partials come from the kernel before this one
  const int g = blockIdx.x * kCellWarps + (threadIdx.x >> 5), k = threadIdx.x & 31;
  if (g >= B || k >= kCellVals) return;
  const int64_t base = cell_slot_base(seg_ptr, g);
  const int64_t chunks = ((int64_t)seg_ptr[g + 1] - seg_ptr[g] + LCAO_CELL_CHUNK - 1) / LCAO_CELL_CHUNK;
  double s = 0.0;
  for (int64_t c = 0; c < chunks; ++c) s += partial[(base + c) * kCellVals + k];
  if (k < 9) {
    if (d_lattice) d_lattice[9 * (int64_t)g + k] = (float)s;
  } else if (virial) {
    virial[9 * (int64_t)g + k - 9] = (float)s;
  }
}

}  // namespace

extern "C" int lcao_geom_basis_fwd(const float* pos, const float* shift, const float* lattice, const int64_t* batch,
                                   const int32_t* src32, const int32_t* dst32, int64_t E,
                                   const lcao_basis_spec* sp, float* dist, float* unit, float* rb, float* drb,
                                   void* stream) {
  if (E == 0) return LCAO_OK;
  LCAO_REQUIRE(pos && shift && lattice && src32 && dst32 && sp && dist && unit && rb, "lcao_geom_basis_fwd: null buffer");
  LCAO_REQUIRE(sp->n_unique >= 1 && sp->n_unique <= LCAO_MAX_UNIQUE_ORB && sp->n_rep >= 1,
               "lcao_geom_basis_fwd: bad orbital count");
  LCAO_REQUIRE(sp->cutoff_kind >= LCAO_CUT_POLYNOMIAL && sp->cutoff_kind <= LCAO_CUT_COSINE &&
                   (sp->rbf_kind == LCAO_RBF_HYDROGEN || sp->rbf_kind == LCAO_RBF_SPHERICAL_BESSEL),
               "lcao_geom_basis_fwd: unknown cutoff_kind %d or rbf_kind %d", sp->cutoff_kind, sp->rbf_kind);
  for (int u = 0; u < sp->n_unique; ++u)
    LCAO_REQUIRE(sp->deg[u] >= 0 && sp->deg[u] < LCAO_MAX_POLY && sp->l[u] >= 0 && sp->l[u] <= 3,
                 "lcao_geom_basis_fwd: bad orbital entry %d", u);
  k_geom_basis_fwd<<<(unsigned)ceil_div64(E, 128), 128, 0, (cudaStream_t)stream>>>(pos, shift, lattice, batch, src32,
                                                                                  dst32, E, *sp, dist, unit, rb, drb);
  LCAO_LAUNCH_CHECK();
  return LCAO_OK;
}

extern "C" int lcao_geom_basis_bwd(const float* dist, const float* unit, const float* drb, const float* d_dist,
                                   const float* d_unit, const float* d_rb, int64_t E, int64_t N, int32_t O,
                                   const int32_t* in_ptr, const int32_t* in_edge, const int32_t* out_ptr,
                                   const int32_t* out_edge, float* dvec, float* d_pos, void* stream) {
  LCAO_REQUIRE(d_pos && in_ptr && out_ptr, "lcao_geom_basis_bwd: null buffer");
  LCAO_REQUIRE(!d_rb || drb, "lcao_geom_basis_bwd: d_rb needs the saved drb");
  cudaStream_t st = (cudaStream_t)stream;
  if (E > 0) {
    LCAO_REQUIRE(dist && unit && dvec && in_edge && out_edge, "lcao_geom_basis_bwd: null edge buffer");
    k_geom_edge_bwd<<<(unsigned)ceil_div64(E, 256), 256, 0, st>>>(dist, unit, drb, d_dist, d_unit, d_rb, E, O, dvec);
    LCAO_LAUNCH_CHECK();
  }
  if (N > 0) {
    k_geom_node_bwd<<<(unsigned)ceil_div64(N * 3, 256), 256, 0, st>>>(dvec, in_ptr, in_edge, out_ptr, out_edge, N, d_pos);
    LCAO_LAUNCH_CHECK();
  }
  return LCAO_OK;
}

extern "C" int lcao_geom_cell_bwd(const float* pos, const float* shift, const float* lattice, const int64_t* batch,
                                  const int32_t* dst32, const float* dvec, int64_t E, int64_t N, const int32_t* out_ptr,
                                  const int32_t* out_edge, const int32_t* seg_ptr, const int32_t* seg_perm, int64_t B,
                                  double* scratch, float* d_lattice, float* virial, void* stream) {
  if (B == 0 || (!d_lattice && !virial)) return LCAO_OK;
  LCAO_REQUIRE(B > 0 && B < (1 << 30) && N >= 0 && N < ((int64_t)1 << 31), "lcao_geom_cell_bwd: bad sizes (N=%lld, B=%lld)",
               (long long)N, (long long)B);
  LCAO_REQUIRE(lattice && out_ptr && seg_ptr && scratch, "lcao_geom_cell_bwd: null buffer");
  LCAO_REQUIRE(E == 0 || (pos && shift && dst32 && dvec && out_edge), "lcao_geom_cell_bwd: null edge buffer");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t slots = N / LCAO_CELL_CHUNK + B;
  LCAO_CUDA(launch_pdl(k_geom_cell_partial, (unsigned)slots, kCellWarps * 32, 0, st, pos, shift, lattice, batch, dst32, dvec,
                       out_ptr, out_edge, seg_ptr, seg_perm, (int)B, scratch, (const int32_t*)nullptr,
                       (const int32_t*)nullptr, (const int32_t*)nullptr, (int64_t)0, (float*)nullptr));
  LCAO_LAUNCH_CHECK();
  LCAO_CUDA(launch_pdl(k_geom_cell_final, (unsigned)ceil_div64(B, kCellWarps), kCellWarps * 32, 0, st, seg_ptr, (int)B,
                       (const double*)scratch, d_lattice, virial));
  LCAO_LAUNCH_CHECK();
  return LCAO_OK;
}

extern "C" int lcao_geom_atom_virial_bwd(const float* pos, const float* shift, const float* lattice, const int64_t* batch,
                                         const int32_t* dst32, const int32_t* in_ptr, const int32_t* in_edge,
                                         const int32_t* in_src, const int32_t* out_ptr, const int32_t* out_edge,
                                         const float* dvec, int64_t E, int64_t N, float* atom_virial, void* stream) {
  LCAO_REQUIRE(N >= 0 && N < ((int64_t)1 << 31) && E >= 0 && E < ((int64_t)1 << 31),
               "lcao_geom_atom_virial_bwd: bad sizes (N=%lld, E=%lld)", (long long)N, (long long)E);
  if (N == 0) return LCAO_OK;
  LCAO_REQUIRE(in_ptr && out_ptr && atom_virial, "lcao_geom_atom_virial_bwd: null buffer");
  LCAO_REQUIRE(E == 0 || (pos && shift && lattice && dst32 && in_edge && in_src && out_edge && dvec),
               "lcao_geom_atom_virial_bwd: null edge buffer");
  LCAO_CUDA(launch_pdl(k_geom_cell_partial, (unsigned)ceil_div64(N, kCellWarps), kCellWarps * 32, 0, (cudaStream_t)stream,
                       pos, shift, lattice, batch, dst32, dvec, out_ptr, out_edge, (const int32_t*)nullptr,
                       (const int32_t*)nullptr, 0, (double*)nullptr, in_ptr, in_edge, in_src, N, atom_virial));
  LCAO_LAUNCH_CHECK();
  return LCAO_OK;
}
