// Three-body backward (autograd of lcaonet.py:173-189 + shbf.py:75-87, see threebody.cu for the algebra) with EVERY
// operand staged in shared memory by bulk asynchronous copies (TMA unit) and a producer warp, so that the consumers'
// inner loop is nothing but shared-memory loads at immediate offsets and FMAs.
//
// Why: the register/LDG formulation in threebody.cu issues 91 warp instructions per triplet of which 28 are the
// arithmetic minimum (profiles/r01_notes.md) — 64-bit address arithmetic, id shuffles, clamps and the dependent
// id -> row load chains are the rest — and sits at a third of the HBM roofline, issue/latency bound.  Here
//   * a producer warp walks the CTA's contiguous node range and emits ITEMS = (node, block of <= 4 in-edges, chunk of
//     <= 32 out-edges): per item the in-edges' B rows (NL*C floats, contiguous) and gate rows arrive by two bulk
//     copies per in-edge into a ring of stages (full / empty mbarriers), the chunk's d_tbw rows by one bulk copy per
//     out-edge into one of two chunk buffers that stay resident while the node's in-edge blocks stream past;
//     unit vectors / Gram rows / edge ids travel through the producer's registers one item ahead;
//   * consumer warp w owns in-edge slot w of the item: its gate*B rows live in registers, the coefficients of the
//     <= 32 (in-edge, out-edge) pairs are computed one per lane, and the pair loop is  LDS.128 (d_tbw row) +
//     LDS.128 (coefficient broadcast) + 28 FMAs,  eight pairs per butterfly;
//   * dead slots (chunk tail) carry zero coefficients and read whatever finite rows the buffer holds (the buffers are
//     zero-filled once), so the loop is branch-free.
// Results are identical in structure to threebody.cu (same per-pair formulas, sums in registers, no atomics except the
// out-degree > kJS overflow of d_unit); C <= 128 only — wider layers keep the register kernels.
#include <type_traits>

#include "common.cuh"
#include "tb_common.cuh"
#include "tb_async.cuh"

namespace {

constexpr int kSlots = 4;   // in-edges per item = consumer warps
constexpr int kJC = 32;     // out-edges per chunk (lane <-> out-edge in the coefficient phase)
constexpr int kGtBufs = 2;  // resident d_tbw chunks
constexpr int kCtasPerSm = 16;  // grid cap per SM; each CTA takes a contiguous range of nodes
enum { kFirst = 1, kLast = 2, kEnd = 4, kNodeFirst = 8, kNodeLast = 16 };

// Shared-memory plan (floats).  [0, 128 B): mbarriers full_in[4] | empty_in[4] | full_gt[2].
struct BwdPlan {
  int slot, oMeta, oGram, oItem, stage, nst;
  int oGt, gtbuf, oSa, oSf, oSa2, oSst, total;
};
__host__ __device__ inline BwdPlan bwd_plan(int C, int NL, bool forces, int nst) {
  BwdPlan p;
  const int NP = NL * (NL + 1) / 2;
  p.nst = nst;
  p.slot = NL * C + C;                 // B rows of the in-edge | gate row of its source node
  p.oMeta = kSlots * p.slot;           // kSlots x float4 (unit vector, edge id)
  p.oGram = p.oMeta + kSlots * 4;      // kSlots x NP doubles (8-byte aligned: every term is a multiple of 4 floats)
  p.oItem = p.oGram + kSlots * NP * 2; // two int4: {n_in, nO, flags, gt buffer | parity << 1}, {ob, dO, jc, 0}
  p.stage = p.oItem + 8;
  p.oGt = 32 + nst * p.stage;
  p.gtbuf = kJC * C + kJC * 4;         // d_tbw rows | float4 (unit vector, edge id) per out-edge
  p.oSa = p.oGt + kGtBufs * p.gtbuf;   // per-warp coefficient scratch: a_l = w Y_l (33 slots: one-ahead reads)
  p.oSf = p.oSa + kSlots * 33 * 4;     // norm-path flags
  p.oSa2 = p.oSf + kSlots * 32;        // (forces) w Y'_l
  p.oSst = p.oSa2 + (forces ? kSlots * 33 * 4 : 0);  // (forces) per-warp partials of d unit[e_j]
  p.total = p.oSst + (forces ? kSlots * kJS * 3 : 0);
  return p;
}

// Sum 4 per-lane partials over the 32 lanes; every lane ends up with the total of element 2*bit4(lane) + bit3(lane).
__device__ __forceinline__ float bfly4(const float (&p)[4], int lane) {
  float q2[2];
  bool up = (lane & 16) != 0;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const float recv = __shfl_xor_sync(0xffffffffu, up ? p[k] : p[k + 2], 16);
    q2[k] = (up ? p[k + 2] : p[k]) + recv;
  }
  up = (lane & 8) != 0;
  const float recv = __shfl_xor_sync(0xffffffffu, up ? q2[0] : q2[1], 8);
  float r = (up ? q2[1] : q2[0]) + recv;
  r += __shfl_xor_sync(0xffffffffu, r, 4);
  r += __shfl_xor_sync(0xffffffffu, r, 2);
  r += __shfl_xor_sync(0xffffffffu, r, 1);
  return r;
}
__device__ __forceinline__ int bfly4_index(int lane) { return ((lane >> 4) & 1) * 2 + ((lane >> 3) & 1); }

__device__ __forceinline__ void consumer_bar() { asm volatile("bar.sync 1, 128;" ::: "memory"); }

template <int NL, bool FORCES, int CT>
__global__ void __launch_bounds__(160, FORCES ? 3 : 4) k_tb_bwd_staged(
    const float* __restrict__ B, int NG, const double* __restrict__ gram, const float* __restrict__ unit,
    const float* __restrict__ gate, int64_t ldg, const int32_t* __restrict__ in_ptr, const int32_t* __restrict__ in_edge,
    const int32_t* __restrict__ in_src, const int32_t* __restrict__ out_ptr, const int32_t* __restrict__ out_edge, int N,
    int C_rt, int nst, const float* __restrict__ d_tbw, const float* __restrict__ dP, float* __restrict__ dB,
    float* __restrict__ q, float* __restrict__ du_ks, float* __restrict__ du_st) {
  pdl_trigger();  // (programmatic dependent launch: the next kernel may start its set-up; common.cuh)
  constexpr int NP = NL * (NL + 1) / 2;
  const int C = CT ? CT : C_rt;
  const int NGP = NG - NL + 1;
  extern __shared__ __align__(128) float smem[];
  const BwdPlan pl = bwd_plan(C, NL, FORCES, nst);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t bar_full = smem_u32(smem), bar_empty = bar_full + 32, bar_gt = bar_full + 64;
  // zero fill: dead chunk rows / columns are multiplied by zero coefficients and must be finite
  for (int i = 32 + threadIdx.x; i < pl.total; i += blockDim.x) smem[i] = 0.f;
  if (threadIdx.x == 0) {
    for (int i = 0; i < 4; ++i) { mbar_init(bar_full + 8 * i, 1); mbar_init(bar_empty + 8 * i, kSlots); }
    for (int i = 0; i < kGtBufs; ++i) mbar_init(bar_gt + 8 * i, 1);
  }
  fence_proxy_async();  // the zero fill (generic proxy) is ordered before the bulk copies (async proxy) into the same bytes
  __syncthreads();
  pdl_wait();  // (launched through launch_pdl: the set-up above may overlap the previous kernel's tail)
  const int per_cta = (N + (int)gridDim.x - 1) / (int)gridDim.x;
  const int s_end = min(N, ((int)blockIdx.x + 1) * per_cta);

  if (warp == kSlots) {
    // ------------------------------------------------------------------ producer
    // Metadata (edge ids, unit vectors, Gram rows) is fetched per PANEL = (node, <= 32 of its in-edges; lane <-> in-edge)
    // together with the node's first out-edge chunk (lane <-> out-edge), one panel ahead of the copies, so that the
    // dependent chain  CSR row -> edge ids -> unit / Gram rows  is paid once per panel and off the critical path.
    struct Node { int s, ib, dI, ob, dO; bool valid; };
    struct Ids { int ep, k, ej; };
    struct Dat { float vx, vy, vz, ux, uy, uz; double gm[NP]; };
    auto next_node = [&](Node& n) {  // first node at or after n.s that has in-edges
      n.valid = false;
      while (n.s < s_end) {
        n.ib = in_ptr[n.s]; n.dI = in_ptr[n.s + 1] - n.ib; n.ob = out_ptr[n.s]; n.dO = out_ptr[n.s + 1] - n.ob;
        if (n.dI > 0) { n.valid = true; return; }
        if (FORCES)  // no in-edges: the s->t role gradients of the out-edges are zero
          for (int t = lane; t < n.dO * 3; t += 32) du_st[3 * (int64_t)out_edge[n.ob + t / 3] + t % 3] = 0.f;
        n.s += 1;
      }
    };
    auto next_panel = [&](Node& n, int& ic) {
      if (!n.valid) return;
      ic += 32;
      if (ic < n.dI) return;
      ic = 0;
      n.s += 1;
      next_node(n);
    };
    auto load_ids = [&](const Node& n, int ic, Ids& r) {
      r.ep = 0; r.k = 0; r.ej = 0;
      if (!n.valid) return;
      if (ic + lane < n.dI) { r.ep = in_edge[n.ib + ic + lane]; r.k = in_src[n.ib + ic + lane]; }
      if (lane < n.dO) r.ej = out_edge[n.ob + lane];
    };
    auto load_dat = [&](const Node& n, int ic, const Ids& r, Dat& d) {
      if (!n.valid) return;
      if (ic + lane < n.dI) {
        d.vx = unit[3 * (int64_t)r.ep]; d.vy = unit[3 * (int64_t)r.ep + 1]; d.vz = unit[3 * (int64_t)r.ep + 2];
#pragma unroll
        for (int x = 0; x < NP; ++x) d.gm[x] = gram[(int64_t)r.ep * NP + x];
      }
      if (lane < n.dO) { d.ux = unit[3 * (int64_t)r.ej]; d.uy = unit[3 * (int64_t)r.ej + 1]; d.uz = unit[3 * (int64_t)r.ej + 2]; }
    };
    // ring position of the next item, and the resident d_tbw chunks: which (node, chunk) each buffer holds, how often
    // it was filled, and the last item that read it (index | stage | phase)
    int it = 0, st = 0, ph = 0;
    int tagS0 = -1, tagJ0 = 0, cnt0 = 0, use0 = -1, ust0 = 0, uph0 = 0, tagS1 = -1, tagJ1 = 0, cnt1 = 0, use1 = -1, ust1 = 0, uph1 = 0;
    auto stage_wait = [&]() {  // the consumers have released the stage's previous item
      if (it >= nst) mbar_wait_backoff(bar_empty + 8 * st, (uint32_t)(ph ^ 1));
    };
    auto stage_next = [&]() {
      it += 1;
      if (++st == nst) { st = 0; ph ^= 1; }
    };
    // item (block b of the panel's in-edges, out-edge chunk jc)
    auto issue = [&](const Node& n, int ic, const Ids& r, const Dat& d, int b, int jc) {
      stage_wait();
      float* sS = smem + 32 + st * pl.stage;
      const uint32_t bar = bar_full + 8 * st;
      const int nI = min(32, n.dI - ic), cnt = min(kSlots, nI - kSlots * b), nO = max(0, min(kJC, n.dO - jc));
      int bsel = 0, par = 0;
      if (nO > 0) {
        if (tagS0 == n.s && tagJ0 == jc) bsel = 0;
        else if (tagS1 == n.s && tagJ1 == jc) bsel = 1;
        else {
          bsel = (use0 <= use1) ? 0 : 1;  // least recently used
          const int x = bsel ? use1 : use0;
          if (x >= 0 && x > it - nst) mbar_wait_backoff(bar_empty + 8 * (bsel ? ust1 : ust0), (uint32_t)(bsel ? uph1 : uph0));  // its last readers are done
          float* gbuf = smem + pl.oGt + bsel * pl.gtbuf;
          int ej = r.ej;
          float ux = d.ux, uy = d.uy, uz = d.uz;
          if (jc > 0 && lane < nO) {  // later chunks of a wide node: fetched on demand
            ej = out_edge[n.ob + jc + lane];
            ux = unit[3 * (int64_t)ej]; uy = unit[3 * (int64_t)ej + 1]; uz = unit[3 * (int64_t)ej + 2];
          }
          if (lane < nO) st4(gbuf + kJC * C + lane * 4, make_float4(ux, uy, uz, __int_as_float(ej)));
          __syncwarp();
          if (lane == 0) mbar_expect_tx(bar_gt + 8 * bsel, (uint32_t)nO * (uint32_t)C * 4u);
          __syncwarp();
          if (lane < nO) bulk_g2s(smem_u32(gbuf + lane * C), d_tbw + (int64_t)ej * C, (uint32_t)C * 4u, bar_gt + 8 * bsel);
          if (bsel) { tagS1 = n.s; tagJ1 = jc; cnt1 += 1; } else { tagS0 = n.s; tagJ0 = jc; cnt0 += 1; }
        }
        par = ((bsel ? cnt1 : cnt0) - 1) & 1;
        if (bsel) { use1 = it; ust1 = st; uph1 = ph; } else { use0 = it; ust0 = st; uph0 = ph; }
      }
      const bool first = jc == 0, last = jc + kJC >= n.dO;
      const bool rows = first || last;  // gate*B -> registers at the first chunk, raw B for the epilogue at the last
      const bool mine = (lane >> 2) == b && lane < nI;  // lane <-> in-edge ic + lane -> slot lane & 3 of block lane >> 2
      const int slot = lane & 3;
      if (mine) {
        st4(sS + pl.oMeta + slot * 4, make_float4(d.vx, d.vy, d.vz, __int_as_float(r.ep)));
        double* sG = reinterpret_cast<double*>(sS + pl.oGram);
#pragma unroll
        for (int x = 0; x < NP; ++x) sG[slot * NP + x] = d.gm[x];
      }
      if (lane == 0) {
        const bool nfirst = first && ic == 0 && b == 0;
        const bool nlast = last && ic + 32 >= n.dI && kSlots * (b + 1) >= nI;
        const int flags = (first ? kFirst : 0) | (last ? kLast : 0) | (nfirst ? kNodeFirst : 0) | (nlast ? kNodeLast : 0);
        *reinterpret_cast<int4*>(sS + pl.oItem) = make_int4(cnt, nO, flags, bsel | (par << 1));
        *reinterpret_cast<int4*>(sS + pl.oItem + 4) = make_int4(n.ob, n.dO, jc, 0);
      }
      __syncwarp();
      if (lane == 0) mbar_expect_tx(bar, rows ? (uint32_t)cnt * (uint32_t)pl.slot * 4u : 0u);
      __syncwarp();
      if (rows && mine) {
        bulk_g2s(smem_u32(sS + slot * pl.slot), B + (int64_t)r.ep * NG * C, (uint32_t)(NL * C) * 4u, bar);
        bulk_g2s(smem_u32(sS + slot * pl.slot + NL * C), gate + (int64_t)r.k * ldg, (uint32_t)C * 4u, bar);
      }
      stage_next();
    };
    Node cur, nxt;
    int cic = 0, nic = 0;
    Ids ci, ni;
    Dat cd, nd;
    cur.s = (int)blockIdx.x * per_cta;
    next_node(cur);
    load_ids(cur, cic, ci);
    load_dat(cur, cic, ci, cd);
    while (cur.valid) {
      nxt = cur; nic = cic;
      next_panel(nxt, nic);
      load_ids(nxt, nic, ni);  // (in flight while this panel's first item is issued)
      const int nI = min(32, cur.dI - cic);
      bool pending = true;
      for (int b = 0; b * kSlots < nI; ++b) {
        int jc = 0;
        do {
          issue(cur, cic, ci, cd, b, jc);
          if (pending) { load_dat(nxt, nic, ni, nd); pending = false; }  // next panel's rows: in flight during the rest of this one
          jc += kJC;
        } while (jc < cur.dO);
      }
      cur = nxt; cic = nic; ci = ni; cd = nd;
    }
    // END marker
    stage_wait();
    if (lane == 0) {
      *reinterpret_cast<int4*>(smem + 32 + st * pl.stage + pl.oItem) = make_int4(0, 0, kEnd, 0);
      mbar_expect_tx(bar_full + 8 * st, 0u);
    }
    return;
  }

  // ------------------------------------------------------------------ consumers: warp w <-> in-edge slot w
  const bool okc = lane * 4 < C;
  const int loff = okc ? lane * 4 : 0;  // lanes beyond C read column 0 (finite) and are masked
  float* sa = smem + pl.oSa + warp * 33 * 4;
  float* sf = smem + pl.oSf + warp * 32;
  float* sa2 = smem + pl.oSa2 + warp * 33 * 4;
  float* sst = smem + pl.oSst + warp * kJS * 3;
  float4 gb[NL], dacc[NL], gtv = zero4(), two_body = zero4();
  float h[NP];
  float ks_x = 0.f, ks_y = 0.f, ks_z = 0.f;
#pragma unroll
  for (int l = 0; l < NL; ++l) { gb[l] = zero4(); dacc[l] = zero4(); }
#pragma unroll
  for (int p = 0; p < NP; ++p) h[p] = 0.f;

  for (int st = 0, ph = 0;; ph ^= (st + 1 == nst), st = (st + 1 == nst) ? 0 : st + 1) {
    const float* sS = smem + 32 + st * pl.stage;
    mbar_wait(bar_full + 8 * st, (uint32_t)ph);
    const int4 item = *reinterpret_cast<const int4*>(sS + pl.oItem);
    const int n_in = item.x, nO = item.y, flags = item.z;
    if (flags & kEnd) break;
    const int4 item2 = *reinterpret_cast<const int4*>(sS + pl.oItem + 4);
    const int ob = item2.x, dO = item2.y, jc = item2.z;
    if (FORCES && (flags & kNodeFirst)) {
      for (int t = lane; t < kJS * 3; t += 32) sst[t] = 0.f;
      if (dO > kJS) {  // rare overflow rows: global atomics below
        for (int t = kJS * 3 + (int)threadIdx.x; t < dO * 3; t += 128) du_st[3 * (int64_t)out_edge[ob + t / 3] + t % 3] = 0.f;
        consumer_bar();
      }
    }
    if (warp < n_in) {
      const float* slot = sS + warp * pl.slot;
      const float4 vm = lds4f(sS + pl.oMeta + warp * 4);
      const int ep = __float_as_int(vm.w);
      if (flags & kFirst) {
        gtv = okc ? lds4f(slot + NL * C + loff) : zero4();
#pragma unroll
        for (int l = 0; l < NL; ++l) { gb[l] = okc ? mul4(gtv, lds4f(slot + l * C + loff)) : zero4(); dacc[l] = zero4(); }
#pragma unroll
        for (int p = 0; p < NP; ++p) h[p] = 0.f;
        ks_x = 0.f; ks_y = 0.f; ks_z = 0.f;
        two_body = (dP && okc) ? ldg4(dP + (int64_t)ep * NGP * C + loff) : zero4();  // same for every l < NL
      }
      if (nO > 0) {
        const int gi = item.w;
        mbar_wait(bar_gt + 8 * (gi & 1), (uint32_t)(gi >> 1));
        const float* gtb = smem + pl.oGt + (gi & 1) * pl.gtbuf;
        // ---- coefficients of the pairs (out-edge jc + lane, this in-edge), one per lane
        const float4 om = lds4f(gtb + kJC * C + lane * 4);
        const float ox = om.x, oy = om.y, oz = om.z;
        const int my_ej = __float_as_int(om.w);
        double g[NP];
        {
          const double* sG = reinterpret_cast<const double*>(sS + pl.oGram) + warp * NP;
#pragma unroll
          for (int p = 0; p < NP; ++p) g[p] = sG[p];
        }
        const float cc = fmaf(ox, vm.x, fmaf(oy, vm.y, oz * vm.z));
        float Y[4];
        sph_harm<NL>(cc, Y);
        const float nrm = sqrtf(fmaxf((float)quad_form<NL>(g, Y), 0.f));
        const bool live = lane < nO && my_ej != ep;
        const float ww = live ? 1.0f / fmaxf(nrm, kEps) : 0.f;
        const float fl = (live && nrm > kEps) ? 1.f : 0.f;
        __syncwarp();  // the previous chunk's readers are done
        st4(sa + lane * 4, live ? make_float4(ww * Y[0], ww * Y[1], ww * Y[2], ww * Y[3]) : zero4());
        sf[lane] = fl;
        if constexpr (FORCES) {
          float dY[4];
          sph_harm_grad<NL>(cc, dY);
          st4(sa2 + lane * 4, live ? make_float4(ww * dY[0], ww * dY[1], ww * dY[2], ww * dY[3]) : zero4());
        }
        __syncwarp();
        const float* grow = gtb + loff;
        // G pairs (out-edges j0 .. j0 + G) against this in-edge: G = 8, or 4 for a short tail
        auto group = [&](auto Gc, const int j0) {
          constexpr int G = decltype(Gc)::value;
          float4 gr[G];
#pragma unroll
          for (int jj = 0; jj < G; ++jj) gr[jj] = lds4f(grow + (j0 + jj) * C);
          float part[FORCES ? 1 : G], partD[FORCES ? NL : 1][G];
#pragma unroll
          for (int jj = 0; jj < G; ++jj) {
            const float4 ar = lds4f(sa + (j0 + jj) * 4);
            if constexpr (FORCES) {
#pragma unroll
              for (int l = 0; l < NL; ++l) partD[l][jj] = dot4(gb[l], gr[jj]);
            } else {
              float4 t = scale4(ar.x, gb[0]);
              if (NL > 1) t = fma4(ar.y, gb[1], t);
              if (NL > 2) t = fma4(ar.z, gb[2], t);
              if (NL > 3) t = fma4(ar.w, gb[3], t);
              part[jj] = dot4(t, gr[jj]);
            }
            dacc[0] = fma4(ar.x, gr[jj], dacc[0]);
            if (NL > 1) dacc[1] = fma4(ar.y, gr[jj], dacc[1]);
            if (NL > 2) dacc[2] = fma4(ar.z, gr[jj], dacc[2]);
            if (NL > 3) dacc[3] = fma4(ar.w, gr[jj], dacc[3]);
          }
          // ---- per pair scalars: the lanes that end up with the sums of pair j0 + jsub finish it (G = 8: one lane
          //      quad per pair; G = 4: two quads per pair, the upper one is masked out of the norm path)
          const int jsub = G == 8 ? bfly8_index(lane) : bfly4_index(lane);
          const int slt = j0 + jsub;  // dead slots carry a = 0, flag = 0
          const float4 as = lds4f(sa + slt * 4);
          float dotv, dot2v = 0.f;
          if constexpr (FORCES) {
            const float4 as2 = lds4f(sa2 + slt * 4);
            dotv = 0.f;
#pragma unroll
            for (int l = 0; l < NL; ++l) {
              float D;
              if constexpr (G == 8) D = bfly8(partD[l], lane); else D = bfly4(partD[l], lane);
              dotv = fmaf(comp4(as, l), D, dotv);
              dot2v = fmaf(comp4(as2, l), D, dot2v);
            }
          } else {
            if constexpr (G == 8) dotv = bfly8(part, lane); else dotv = bfly4(part, lane);
          }
          {
            float sc = -sf[slt] * dotv;
            if (G == 4 && (lane & 4)) sc = 0.f;
            int p = 0;
#pragma unroll
            for (int x = 0; x < NL; ++x)
#pragma unroll
              for (int y = x; y < NL; ++y) h[p++] += sc * comp4(as, x) * comp4(as, y);
          }
          if constexpr (FORCES) {
            // dL/dcos of pair (j0 + jl) is finished on its coefficient lane j0 + jl (threebody.cu), fed by the lane
            // whose butterfly element is jl
            const int jl = (lane - j0) & (G - 1);
            const int srcl = G == 8 ? ((((jl >> 2) & 1) << 4) | (((jl >> 1) & 1) << 3) | ((jl & 1) << 2))
                                    : ((((jl >> 1) & 1) << 4) | ((jl & 1) << 3));
            const float dt = __shfl_sync(0xffffffffu, dotv, srcl);
            const float dt2 = __shfl_sync(0xffffffffu, dot2v, srcl);
            if (lane >= j0 && lane < j0 + G && live) {
              float dY[4];
              sph_harm_grad<NL>(cc, dY);
              const float corr = (float)bilin_form<NL>(g, dY, Y);
              const float dc = dt2 - fl * ww * ww * dt * corr;
              ks_x = fmaf(dc, ox, ks_x); ks_y = fmaf(dc, oy, ks_y); ks_z = fmaf(dc, oz, ks_z);
              const int j = jc + lane;
              if (j < kJS) {  // slot j of this warp's partials is only ever touched by this lane
                sst[3 * j] = fmaf(dc, vm.x, sst[3 * j]);
                sst[3 * j + 1] = fmaf(dc, vm.y, sst[3 * j + 1]);
                sst[3 * j + 2] = fmaf(dc, vm.z, sst[3 * j + 2]);
              } else {
                atomicAdd(du_st + 3 * (int64_t)my_ej, dc * vm.x);
                atomicAdd(du_st + 3 * (int64_t)my_ej + 1, dc * vm.y);
                atomicAdd(du_st + 3 * (int64_t)my_ej + 2, dc * vm.z);
              }
            }
          }
        };
        int j0 = 0;
        for (; j0 + 4 < nO; j0 += 8) group(std::integral_constant<int, 8>{}, j0);
        if (j0 < nO) group(std::integral_constant<int, 4>{}, j0);
      }
      if (flags & kLast) {
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
        if (okc) {
          const int c = lane * 4;
          float4 b[NL];
#pragma unroll
          for (int l = 0; l < NL; ++l) b[l] = lds4f(slot + l * C + c);
          float4 qq = zero4();
#pragma unroll
          for (int l = 0; l < NL; ++l) {
            float4 o4 = fma4(1.0f, mul4(gtv, dacc[l]), two_body);
#pragma unroll
            for (int l2 = 0; l2 < NL; ++l2) o4 = fma4(H[l][l2], b[l2], o4);
            st4(dB + ((int64_t)ep * NG + l) * C + c, o4);
            qq = add4(qq, mul4(b[l], dacc[l]));
          }
          const float4 sg = gtv;
          qq = mul4(qq, make_float4(sg.x * (1.f - sg.x), sg.y * (1.f - sg.y), sg.z * (1.f - sg.z), sg.w * (1.f - sg.w)));
          st4(q + (int64_t)ep * C + c, qq);
          for (int l = NL; l < NG; ++l)
            st4(dB + ((int64_t)ep * NG + l) * C + c, dP ? ldg4(dP + ((int64_t)ep * NGP + 1) * C + c) : zero4());
        }
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(bar_empty + 8 * st);  // this warp is done with the stage (and with the chunk buffer)
    if (FORCES && (flags & kNodeLast)) {
      consumer_bar();
      for (int t = threadIdx.x; t < min(dO, kJS) * 3; t += 128) {
        float x = 0.f;
#pragma unroll
        for (int w = 0; w < kSlots; ++w) x += smem[pl.oSst + w * kJS * 3 + t];
        du_st[3 * (int64_t)out_edge[ob + t / 3] + t % 3] = x;
      }
      consumer_bar();
    }
  }
}

template <int NL, bool FORCES, int CT>
int launch_bwd(const float* B, int NG, const double* gram, const float* unit, const float* gate, int64_t ldg,
               const int32_t* in_ptr, const int32_t* in_edge, const int32_t* in_src, const int32_t* out_ptr,
               const int32_t* out_edge, int64_t N, int C, const float* d_tbw, const float* dP, float* dB, float* q,
               float* du_ks, float* du_st, cudaStream_t st) {
  // ring depth: as many stages (<= 4) as keep four CTAs (energy path: 96 registers) or three (forces: 128) resident per
  // SM (227 KB of shared memory, 1 KB reserved per CTA).  Four CTAs with a two-stage ring measured 0.402 ms against
  // 0.428 ms for three with four stages; the forces variant spills at 96 registers and stays at three.
  int nst = 4;
  while (nst > 2 && sizeof(float) * (size_t)bwd_plan(C, NL, FORCES, nst).total > (FORCES ? 74 : 55) * 1024) --nst;
  const size_t smem = sizeof(float) * (size_t)bwd_plan(C, NL, FORCES, nst).total;
  static bool attr_done = false;
  if (!attr_done) {
    LCAO_CUDA(cudaFuncSetAttribute(k_tb_bwd_staged<NL, FORCES, CT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 120 * 1024));
    attr_done = true;
  }
  const int64_t want = (N + 1) / 2;  // at least two nodes per CTA
  const unsigned grid = (unsigned)(want < 148ll * kCtasPerSm ? (want > 0 ? want : 1) : 148ll * kCtasPerSm);
  LCAO_CUDA(launch_pdl(k_tb_bwd_staged<NL, FORCES, CT>, grid, 160, smem, st, B, NG, gram, unit, gate, ldg, in_ptr, in_edge, in_src, out_ptr,
                                                          out_edge, (int)N, C, nst, d_tbw, dP, dB, q, du_ks, du_st));
  LCAO_LAUNCH_CHECK();
  return LCAO_OK;
}

}  // namespace

// (argument checks are done by lcao_threebody_bwd in threebody.cu, which dispatches here for C <= 128)
int lcao_tb_staged_bwd(const float* B, int32_t NG, const double* gram, const float* unit, const float* gate, int64_t ldg,
                       const int32_t* in_ptr, const int32_t* in_edge, const int32_t* in_src, const int32_t* out_ptr,
                       const int32_t* out_edge, int64_t N, int32_t C, int32_t NL, const float* d_tbw, const float* dP,
                       float* dB, float* q, float* du_ks, float* du_st, cudaStream_t st) {
  const bool forces = du_ks != nullptr;
#define ARGS B, NG, gram, unit, gate, ldg, in_ptr, in_edge, in_src, out_ptr, out_edge, N, C, d_tbw, dP, dB, q, du_ks, du_st, st
#define CALL(nl)                                                               \
  {                                                                            \
    if (forces) return C == 128 ? launch_bwd<nl, true, 128>(ARGS) : launch_bwd<nl, true, 0>(ARGS);   \
    return C == 128 ? launch_bwd<nl, false, 128>(ARGS) : launch_bwd<nl, false, 0>(ARGS);             \
  }
  switch (NL) {
    case 1: CALL(1)
    case 2: CALL(2)
    case 3: CALL(3)
    default: CALL(4)
  }
#undef CALL
#undef ARGS
}
