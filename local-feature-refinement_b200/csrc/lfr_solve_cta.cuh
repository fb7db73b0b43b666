// lfr_solve_cta.cuh — one CTA solves one LARGE component (more than 96
// unknowns: Madrid-scale scenes cap a component at #images = 1000 nodes,
// solve.cc:586), or every component when lfr_options.linear_solver = 2.
//
// Same trust-region loop as the warp kernels (SURVEY Appendix A.6), but the
// damped normal equations (S H S + D^2) y = S g are never formed: they are
// solved matrix-free by conjugate gradients preconditioned with the inverse of
// the 2x2 diagonal blocks (block-Jacobi), iterated to a relative residual of
// 1e-14 and then refined on the true residual to 2e-15, so that the step is, to working precision, the exact solve Ceres'
// SPARSE_NORMAL_CHOLESKY (solve.cc:147) returns:
//
//   q_e = a_e (x_d~ - M_e x_s~)             one thread per directed edge
//   w_v = S_v ( sum_out -M_e^T q_e + sum_in q_e ) + D_v^2 p_v   one thread per free node
//
// with x~ = S p, a_e = sim rho', M_e = I + grad(flow) staged by the evaluation.
// The kept-edge lists, in-edge lists and free-variable numbering of the large
// components live in HBM and are built on the device by cta_prepare_kernel
// (below; the host only lays out per-component offsets from row_ptr).
#pragma once
#include "lfr_solve_warp.cuh"

namespace lfr {

struct CtaComp {
  uint32_t slot, Nc, Ec, nf;
  uint64_t e_off, n_off, f_off;  // offsets of this component in the per-edge / per-node / per-free-node arrays
  uint32_t comp_index, regular;  // ordinal among the large components; 1 = every kept edge has exactly one twin
  uint64_t ell_off, s_off;       // offsets into the sliced-ELL slot arrays / the ell_base array
};

struct CtaArrays {
  // per kept edge
  const float4* rec;       // the edge's 80-byte record (5 x float4), copied once from the caller's array (HBM or pinned host)
  const uint32_t* meta;    // src_local | dst_local << 14 | kind << 28
  const uint32_t* inlist;  // kept-edge indices sorted by destination
  const uint32_t* twin;    // index of the reverse edge (regular components)
  const int32_t* fdst;     // free index of the edge's destination node, or -1
  // sliced ELL (see cta_matvec_bcsr), per padded slot
  double2* bE01;           // scaled off-diagonal block S_s H_sd S_d, first row (regular components)
  double2* bE23;           // ... second row
  const int32_t* fdstE;    // free index of the block's column node, or -1
  const uint32_t* ell_base;  // [slices + 1 per component] first slot of each 32-row slice, relative to the component
  double* scr;             // 7 doubles per edge (a, r0, r1, m00, m01, m10, m11), SoA per component
  double* q;               // 2 doubles per edge (matvec scratch)
  // per node
  const uint32_t* node;    // global node index
  const uint32_t* outptr;  // [Nc + 1] per component
  const uint32_t* inptr;   // [Nc + 1] per component
  const int32_t* freeof;   // free index or -1
  double* x;               // 2 per node
  double* xc;              // 2 per node
  // per free node
  const uint32_t* lof;     // local node of free index
  double* vec;             // 13 vectors of 2 doubles per free node + 2 of 3 doubles, see offsets below
  uint64_t total_free;     // sum of nf over all large components (stride between vectors)
};

constexpr int kCtaThreads = 256;     // preparation kernel; smallest solve variant
constexpr int kCtaMaxThreads = 512;  // largest solve variant (CtaCtx::nt)
enum { V_G = 0, V_S, V_DL, V_D2, V_R, V_Z, V_P, V_W, V_Y, V_COUNT };  // 2-doubles-per-node vectors
// then three 3-doubles-per-node arrays: diagonal blocks (d00, d01, d11), their damped scaled form, its inverse

constexpr int kCtaRowsCached = 4;  // covers components up to 1024 nodes (solve.cc:586 caps them at #images)

struct CtaCtx {
  int tid, nt, Nc, Ec, nf, n;  // nt = threads of this CTA (256 or 512: compile-time in every instantiation)
  const uint32_t *meta, *inlist, *node, *outptr, *inptr, *lof;
  const int32_t* freeof;
  double *scr, *q, *x, *xc, *g, *S, *dl, *D2, *r, *z, *p, *w, *y, *diag, *pinv, *pblk;
  double2 *bE01, *bE23;
  const int32_t* fdstE;
  const uint32_t* ell_base;
  int row_f[kCtaRowsCached];        // block rows tid, tid + 256, ...: free index (-1: none), degree, first ELL slot
  uint32_t row_deg[kCtaRowsCached], row_slot[kCtaRowsCached];
  const uint32_t* twin;
  const int32_t* fdst;
  bool regular;
  const float4* rec;
  double* red;   // shared: 3 * 8 doubles
  double* red2;  // shared: 2 parities x 2 values x 8 warps (block_sum_db)
};

__device__ __forceinline__ double2* P2(double* p) { return reinterpret_cast<double2*>(p); }  // per-node pairs are 16-byte aligned

__device__ __forceinline__ void block_sum3(const CtaCtx& C, double& a, double& b, double& c) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_xor_sync(kFull, a, o);
    b += __shfl_xor_sync(kFull, b, o);
    c += __shfl_xor_sync(kFull, c, o);
  }
  const int w = C.tid >> 5, nw = C.nt >> 5;
  __syncthreads();  // previous users of `red` are done
  if ((C.tid & 31) == 0) {
    C.red[w] = a;
    C.red[nw + w] = b;
    C.red[2 * nw + w] = c;
  }
  __syncthreads();
  a = b = c = 0.0;
#pragma unroll
  for (int i = 0; i < nw; ++i) {  // fixed order: identical in every thread, reproducible
    a += C.red[i];
    b += C.red[nw + i];
    c += C.red[2 * nw + i];
  }
}
// N sums with ONE barrier: partials go to the `parity` half of a double-buffered line, so the next
// call (other parity) may write while stragglers still read this one; calls with the same parity
// must be separated by another barrier (the CG loop alternates 0, 1 and ends each iteration with one).
template <int N>
__device__ __forceinline__ void block_sum_db(const CtaCtx& C, double (&v)[N], int parity) {
  static_assert(N <= 2, "red2 holds two values per warp and parity");
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
    for (int k = 0; k < N; ++k) v[k] += __shfl_xor_sync(kFull, v[k], o);
  }
  const int nw = C.nt >> 5;
  double* line = C.red2 + parity * 2 * nw;
  if ((C.tid & 31) == 0) {
#pragma unroll
    for (int k = 0; k < N; ++k) line[k * nw + (C.tid >> 5)] = v[k];
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < N; ++k) {
    double a = 0.0;
#pragma unroll
    for (int i = 0; i < nw; ++i) a += line[k * nw + i];  // fixed order: identical in every thread, reproducible
    v[k] = a;
  }
}

__device__ __forceinline__ double block_max(const CtaCtx& C, double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(kFull, v, o));
  const int w = C.tid >> 5, nw = C.nt >> 5;
  __syncthreads();
  if ((C.tid & 31) == 0) C.red[w] = v;
  __syncthreads();
  v = C.red[0];
#pragma unroll
  for (int i = 1; i < nw; ++i) v = fmax(v, C.red[i]);
  return v;
}

__device__ __forceinline__ double cta_eval(const CtaCtx& C, const double* xe, const DevConsts& K) {
  double cost = 0.0, z1 = 0.0, z2 = 0.0;
  const int E = C.Ec;
  for (int j = C.tid; j < E; j += C.nt) {
    const uint32_t mt = C.meta[j];
    const int s = mt & 0x3fff, d = (mt >> 14) & 0x3fff, kind = mt >> 28;
    const float4* qp = C.rec + 5 * (size_t)j;
    float4 q[5];
#pragma unroll
    for (int t = 0; t < 5; ++t) q[t] = __ldg(qp + t);
    const EdgeEval ev = eval_edge(q, kind, xe[2 * s], xe[2 * s + 1], xe[2 * d], xe[2 * d + 1], K);
    double* sc = C.scr + j;
    sc[0] = ev.a;
    sc[E] = ev.r0;
    sc[2 * (size_t)E] = ev.r1;
    sc[3 * (size_t)E] = ev.m00;
    sc[4 * (size_t)E] = ev.m01;
    sc[5 * (size_t)E] = ev.m10;
    sc[6 * (size_t)E] = ev.m11;
    cost += ev.half_rho;
  }
  block_sum3(C, cost, z1, z2);
  return cost;
}

// Diagonal blocks + gradient from the staged evaluation (GRAD_ONLY: returns grad . dl).
template <bool GRAD_ONLY>
__device__ __forceinline__ double cta_assemble(const CtaCtx& C, bool first, const DevConsts& K) {
  const size_t E = C.Ec;
  double acc = 0.0, gmax = 0.0;
  for (int f = C.tid; f < C.nf; f += C.nt) {
    const int l = C.lof[f];
    double d00 = 0., d01 = 0., d11 = 0., g0 = 0., g1 = 0.;
    for (uint32_t j = C.outptr[l]; j < C.outptr[l + 1]; ++j) {
      const double a = C.scr[j], r0 = C.scr[E + j], r1 = C.scr[2 * E + j];
      const double m00 = C.scr[3 * E + j], m01 = C.scr[4 * E + j], m10 = C.scr[5 * E + j], m11 = C.scr[6 * E + j];
      g0 -= a * (m00 * r0 + m10 * r1);
      g1 -= a * (m01 * r0 + m11 * r1);
      if (!GRAD_ONLY) {
        d00 += a * (m00 * m00 + m10 * m10);
        d01 += a * (m00 * m01 + m10 * m11);
        d11 += a * (m01 * m01 + m11 * m11);
      }
    }
    for (uint32_t t = C.inptr[l]; t < C.inptr[l + 1]; ++t) {
      const uint32_t j = C.inlist[t];
      const double a = C.scr[j];
      g0 += a * C.scr[E + j];
      g1 += a * C.scr[2 * E + j];
      if (!GRAD_ONLY) {
        d00 += a;
        d11 += a;
      }
    }
    if (GRAD_ONLY) {
      acc += g0 * C.dl[2 * f] + g1 * C.dl[2 * f + 1];
    } else {
      C.diag[3 * f] = d00;
      C.diag[3 * f + 1] = d01;
      C.diag[3 * f + 2] = d11;
      C.g[2 * f] = g0;
      C.g[2 * f + 1] = g1;
      if (first) {
        C.S[2 * f] = 1.0 / (1.0 + sqrt(d00));
        C.S[2 * f + 1] = 1.0 / (1.0 + sqrt(d11));
      }
      const double x0 = C.x[2 * l], x1 = C.x[2 * l + 1];
      const double p0 = fmin(fmax(x0 - g0, -K.bound), K.bound), p1 = fmin(fmax(x1 - g1, -K.bound), K.bound);
      gmax = fmax(gmax, fmax(fabs(x0 - p0), fabs(x1 - p1)));
    }
  }
  if (GRAD_ONLY) {
    double z1 = 0.0, z2 = 0.0;
    block_sum3(C, acc, z1, z2);
    return acc;
  }
  gmax = block_max(C, gmax);  // (also makes S visible to every thread)
  if (C.regular) {
    // block-CSR form of S H S: one scaled 2x2 block per out-edge, edge + twin combined
    for (int j = C.tid; j < C.Ec; j += C.nt) {
      const uint32_t mt = C.meta[j];
      const int fs = C.freeof[mt & 0x3fff], fd = C.fdst[j];
      if (fs < 0 || fd < 0) continue;
      const uint32_t t = C.twin[j];
      const double a = C.scr[j], at = C.scr[t];
      const double m00 = C.scr[3 * E + j], m01 = C.scr[4 * E + j], m10 = C.scr[5 * E + j], m11 = C.scr[6 * E + j];
      const double t00 = C.scr[3 * E + t], t01 = C.scr[4 * E + t], t10 = C.scr[5 * E + t], t11 = C.scr[6 * E + t];
      const double s0 = C.S[2 * fs], s1 = C.S[2 * fs + 1], d0 = C.S[2 * fd], d1 = C.S[2 * fd + 1];
      const uint32_t sl = mt & 0x3fff;
      const size_t slot = (size_t)C.ell_base[sl >> 5] + (sl & 31u) + 32u * (size_t)((uint32_t)j - C.outptr[sl]);
      // block (s, d) = -a M^T - a_t M_t
      C.bE01[slot] = make_double2(s0 * (-a * m00 - at * t00) * d0, s0 * (-a * m10 - at * t01) * d1);
      C.bE23[slot] = make_double2(s1 * (-a * m01 - at * t10) * d0, s1 * (-a * m11 - at * t11) * d1);
    }
    __syncthreads();
  }
  return gmax;
}

// w = (S H S + D^2) v, matrix-free.
__device__ __forceinline__ void cta_matvec(const CtaCtx& C, const double* v, double* w) {
  const size_t E = C.Ec;
#pragma unroll 4
  for (int j = C.tid; j < C.Ec; j += C.nt) {
    const uint32_t mt = C.meta[j];
    const int fs = C.freeof[mt & 0x3fff], fd = C.freeof[(mt >> 14) & 0x3fff];
    double s0 = 0., s1 = 0., t0 = 0., t1 = 0.;
    if (fs >= 0) {
      s0 = C.S[2 * fs] * v[2 * fs];
      s1 = C.S[2 * fs + 1] * v[2 * fs + 1];
    }
    if (fd >= 0) {
      t0 = C.S[2 * fd] * v[2 * fd];
      t1 = C.S[2 * fd + 1] * v[2 * fd + 1];
    }
    const double a = C.scr[j];
    const double m00 = C.scr[3 * E + j], m01 = C.scr[4 * E + j], m10 = C.scr[5 * E + j], m11 = C.scr[6 * E + j];
    C.q[2 * (size_t)j] = a * (t0 - (m00 * s0 + m01 * s1));      // a (J x~)_0,  J = [-M | I]
    C.q[2 * (size_t)j + 1] = a * (t1 - (m10 * s0 + m11 * s1));
  }
  __syncthreads();
  for (int f = C.tid; f < C.nf; f += C.nt) {
    const int l = C.lof[f];
    double a0 = 0., a1 = 0.;
#pragma unroll 4
    for (uint32_t j = C.outptr[l]; j < C.outptr[l + 1]; ++j) {
      const double q0 = C.q[2 * (size_t)j], q1 = C.q[2 * (size_t)j + 1];
      a0 -= C.scr[3 * E + j] * q0 + C.scr[5 * E + j] * q1;   // -M^T q
      a1 -= C.scr[4 * E + j] * q0 + C.scr[6 * E + j] * q1;
    }
#pragma unroll 4
    for (uint32_t t = C.inptr[l]; t < C.inptr[l + 1]; ++t) {
      const uint32_t j = C.inlist[t];
      a0 += C.q[2 * (size_t)j];
      a1 += C.q[2 * (size_t)j + 1];
    }
    w[2 * f] = C.S[2 * f] * a0 + C.D2[2 * f] * v[2 * f];
    w[2 * f + 1] = C.S[2 * f + 1] * a1 + C.D2[2 * f + 1] * v[2 * f + 1];
  }
  __syncthreads();
}

// Regular components: w = (S H S + D^2) v in ONE node-parallel pass over the block rows (damped
// diagonal block `pblk` + one 2x2 block per out-edge); returns this thread's share of v . w.
// The blocks live in a sliced-ELL layout: the k-th block of local node l sits at
// ell_base[l / 32] + 32 k + l % 32, i.e. the 32 rows a warp walks together are interleaved, so the
// warp's k-th loads (destination index, two 16-byte halves of the block) are each ONE contiguous
// 128 / 512-byte access.  ncu (round 2, cfg5): with the blocks in CSR order every lane strode through
// its own row — L1/TEX at 85 % of peak on uncoalesced 8-byte loads bounded the whole tier.
// One block row: w_f = P_f v_f + sum_k B_k v_col(k), blocks k = 0 .. deg-1 at slot0 + 32 k.
// The row is walked in groups of four slots with NO branch on the column index: a slot past the row's
// end, or whose column is a root, holds a zero block and column -1 (the preparation kernel fills
// every slot of the slice, whose width is a multiple of 4), so the twelve loads of a group — four
// column indices, eight block halves — are all in flight before the first one is needed, and a
// group costs one L2 round trip (+ the shared-memory gathers) instead of one per block.
__device__ __forceinline__ double cta_block_row(const CtaCtx& C, const double2* v2, double2* w2, const double* pblk,
                                                int f, uint32_t deg, size_t s) {
  const double2 vv = v2[f];
  double a0 = pblk[3 * f] * vv.x + pblk[3 * f + 1] * vv.y, a1 = pblk[3 * f + 1] * vv.x + pblk[3 * f + 2] * vv.y;
  for (uint32_t k = 0; k < deg; k += 4, s += 128) {
    int fd[4];
    double2 b01[4], b23[4], u[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      fd[t] = C.fdstE[s + 32 * t];
      b01[t] = C.bE01[s + 32 * t];
      b23[t] = C.bE23[s + 32 * t];
    }
#pragma unroll
    for (int t = 0; t < 4; ++t) u[t] = v2[max(fd[t], 0)];
#pragma unroll
    for (int t = 0; t < 4; ++t) {  // same order as a slot-by-slot walk; a zero block adds +0.0
      a0 += b01[t].x * u[t].x + b01[t].y * u[t].y;
      a1 += b23[t].x * u[t].x + b23[t].y * u[t].y;
    }
  }
  w2[f] = make_double2(a0, a1);
  return vv.x * a0 + vv.y * a1;
}

template <bool SYNC = true>
__device__ __forceinline__ double cta_matvec_bcsr(const CtaCtx& C, const double* v, double* w, const double* pblk) {
  const double2* v2 = reinterpret_cast<const double2*>(v);
  double2* w2 = reinterpret_cast<double2*>(w);
  double dot = 0.0;
  // the first kCtaRowsCached rows of this thread: free index, degree and first slot sit in registers
  // (they never change), which takes two dependent L2 round trips out of every CG iteration
#pragma unroll
  for (int i = 0; i < kCtaRowsCached; ++i)
    if (C.row_f[i] >= 0) dot += cta_block_row(C, v2, w2, pblk, C.row_f[i], C.row_deg[i], C.row_slot[i]);
  for (int l = C.tid + kCtaRowsCached * C.nt; l < C.Nc; l += C.nt) {
    const int f = C.freeof[l];
    if (f < 0) continue;
    dot += cta_block_row(C, v2, w2, pblk, f, C.outptr[l + 1] - C.outptr[l],
                         (size_t)C.ell_base[l >> 5] + (uint32_t)(l & 31));
  }
  if (SYNC) __syncthreads();  // (else the caller's reduction barrier publishes w)
  return dot;
}

// Block-Jacobi PCG for (S H S + D^2) y = S g; dl = -S y.  Returns validity and
// {model_cost_change, g . dl, |dl|_inf}.  tph (LFR_DBG_PROFILE only, else nullptr) accumulates the
// cycles of the four phases of a CG iteration.
__device__ __forceinline__ bool cta_lm_step(const CtaCtx& C, double radius, const DevConsts& K, double* model_change,
                                            double* gd, double* dmax, unsigned* cg_iters, long long* tph) {
  // damping, preconditioner, initial residual
  double bb = 0.0, rz = 0.0, bad = 0.0;
  for (int f = C.tid; f < C.nf; f += C.nt) {
    const double s0 = C.S[2 * f], s1 = C.S[2 * f + 1];
    const double h00 = C.diag[3 * f] * s0 * s0, h01 = C.diag[3 * f + 1] * s0 * s1, h11 = C.diag[3 * f + 2] * s1 * s1;
    const double e0 = fmin(fmax(h00, K.min_diag), K.max_diag) / radius;
    const double e1 = fmin(fmax(h11, K.min_diag), K.max_diag) / radius;
    C.D2[2 * f] = e0;
    C.D2[2 * f + 1] = e1;
    const double p00 = h00 + e0, p11 = h11 + e1;
    const double det = p00 * p11 - h01 * h01;
    if (!(det > 0.0) || !(p00 > 0.0)) bad = 1.0;
    const double id = 1.0 / det;
    C.pblk[3 * f] = p00;
    C.pblk[3 * f + 1] = h01;
    C.pblk[3 * f + 2] = p11;
    C.pinv[3 * f] = p11 * id;
    C.pinv[3 * f + 1] = -h01 * id;
    C.pinv[3 * f + 2] = p00 * id;
    const double b0 = s0 * C.g[2 * f], b1 = s1 * C.g[2 * f + 1];
    C.y[2 * f] = 0.0;
    C.y[2 * f + 1] = 0.0;
    C.r[2 * f] = b0;
    C.r[2 * f + 1] = b1;
    const double z0 = C.pinv[3 * f] * b0 + C.pinv[3 * f + 1] * b1, z1 = C.pinv[3 * f + 1] * b0 + C.pinv[3 * f + 2] * b1;
    C.z[2 * f] = z0;
    C.z[2 * f + 1] = z1;
    C.p[2 * f] = z0;
    C.p[2 * f + 1] = z1;
    bb += b0 * b0 + b1 * b1;
    rz += b0 * z0 + b1 * z1;
  }
  block_sum3(C, bb, rz, bad);
  bool ok = (bad == 0.0) && isfinite(bb);
  const double tol2 = 1e-28 * bb;  // recurrence residual |r| <= 1e-14 |b| ...
  const int max_it = 8 * C.n + 100;
  int it = 0, restarts = 0;
  // ... then iterative refinement: the recurrence residual drifts away from b - A y by ~cond * eps,
  // so CG is restarted from the TRUE residual until that is <= 2e-15 |b| (at most twice): the step is
  // the exact solve of Ceres' SPARSE_NORMAL_CHOLESKY to working precision, which keeps the line
  // search's discontinuous decisions on the oracle's side
  while (ok && bb > 0.0) {
    for (; it < max_it; ++it) {
      // three barriers per iteration: (1) inside the p.w reduction (also publishes w), (2) inside the
      // {r.r, r.z} reduction, (3) after the update of p, which the next product gathers
      long long c0 = 0, c1 = 0, c2 = 0, c3 = 0, c4 = 0;
      if (tph) c0 = clock64();
      double s1[1] = {0.0};
      if (C.regular) {
        s1[0] = cta_matvec_bcsr<false>(C, C.p, C.w, C.pblk);
      } else {
        cta_matvec(C, C.p, C.w);
        for (int i = C.tid; i < C.n; i += C.nt) s1[0] += C.p[i] * C.w[i];
      }
      if (tph) c1 = clock64();
      block_sum_db(C, s1, 0);
      if (tph) c2 = clock64();
      const double pw = s1[0];
      if (!(pw > 0.0) || !isfinite(pw)) {  // not positive definite in working precision
        ok = false;
        break;
      }
      const double alpha = rz / pw;
      double s2[2] = {0.0, 0.0};  // r.r, r.z
      for (int f = C.tid; f < C.nf; f += C.nt) {  // one 16-byte access per vector and node
        const double2 pf = P2(C.p)[f], wf = P2(C.w)[f], yf = P2(C.y)[f], rf = P2(C.r)[f];
        const double y0 = yf.x + alpha * pf.x, y1 = yf.y + alpha * pf.y;
        const double r0 = rf.x - alpha * wf.x, r1 = rf.y - alpha * wf.y;
        P2(C.y)[f] = make_double2(y0, y1);
        P2(C.r)[f] = make_double2(r0, r1);
        const double z0 = C.pinv[3 * f] * r0 + C.pinv[3 * f + 1] * r1, zz1 = C.pinv[3 * f + 1] * r0 + C.pinv[3 * f + 2] * r1;
        P2(C.z)[f] = make_double2(z0, zz1);
        s2[0] += r0 * r0 + r1 * r1;
        s2[1] += r0 * z0 + r1 * zz1;
      }
      if (tph) c3 = clock64();
      block_sum_db(C, s2, 1);
      if (tph) c4 = clock64();
      if (tph) {
        tph[0] += c1 - c0;  // product
        tph[1] += c2 - c1;  // reduction 1
        tph[2] += c3 - c2;  // vector update
        tph[3] += c4 - c3;  // reduction 2
      }
      const double rr = s2[0], rz_new = s2[1];
      if (rr <= tol2) {
        ++it;
        break;
      }
      const double beta = rz_new / rz;
      rz = rz_new;
      for (int f = C.tid; f < C.nf; f += C.nt) {  // same thread <-> node mapping as above: z[f] is this thread's own
        const double2 zf = P2(C.z)[f], pf = P2(C.p)[f];
        P2(C.p)[f] = make_double2(zf.x + beta * pf.x, zf.y + beta * pf.y);
      }
      __syncthreads();
    }
    if (!ok || it >= max_it || restarts >= 2) break;
    // true residual r = S g - A y, z = M^-1 r, p = z
    if (C.regular) cta_matvec_bcsr(C, C.y, C.w, C.pblk); else cta_matvec(C, C.y, C.w);
    double rt = 0.0, rzt = 0.0, z3 = 0.0;
    for (int f = C.tid; f < C.nf; f += C.nt) {
      const double r0 = C.S[2 * f] * C.g[2 * f] - C.w[2 * f], r1 = C.S[2 * f + 1] * C.g[2 * f + 1] - C.w[2 * f + 1];
      const double z0 = C.pinv[3 * f] * r0 + C.pinv[3 * f + 1] * r1, z1 = C.pinv[3 * f + 1] * r0 + C.pinv[3 * f + 2] * r1;
      C.r[2 * f] = r0;
      C.r[2 * f + 1] = r1;
      C.z[2 * f] = z0;
      C.z[2 * f + 1] = z1;
      C.p[2 * f] = z0;
      C.p[2 * f + 1] = z1;
      rt += r0 * r0 + r1 * r1;
      rzt += r0 * z0 + r1 * z1;
    }
    block_sum3(C, rt, rzt, z3);
    if (rt <= 4e-30 * bb || !(rzt > 0.0)) break;  // |b - A y| <= 2e-15 |b|
    rz = rzt;
    ++restarts;
  }
  *cg_iters += (unsigned)it;
  double mc = 0.0, dot = 0.0, nonfinite = 0.0, mx = 0.0;
  for (int i = C.tid; i < C.n; i += C.nt) {
    const double y = C.y[i], si = C.S[i], gi = C.g[i];
    const double d = -si * y;
    C.dl[i] = d;
    mc += y * (si * gi + C.D2[i] * y);
    dot += gi * d;
    mx = fmax(mx, fabs(d));
    if (!isfinite(y)) nonfinite = 1.0;
  }
  block_sum3(C, mc, dot, nonfinite);
  mx = block_max(C, mx);
  *model_change = 0.5 * mc;
  *gd = dot;
  *dmax = mx;
  return ok && nonfinite == 0.0;
}

__device__ __forceinline__ void cta_candidate(const CtaCtx& C, double alpha, const DevConsts& K) {
  for (int i = C.tid; i < 2 * C.Nc; i += C.nt) {
    const int f = C.freeof[i >> 1];
    double v = C.x[i];
    if (f >= 0) v = fmin(fmax(v + alpha * C.dl[2 * f + (i & 1)], -K.bound), K.bound);
    C.xc[i] = v;
  }
  __syncthreads();
}

// MINB = CTAs per SM the register allocation is capped for (65536 / (256 x MINB) registers per thread;
// ptxas: 128 registers at MINB = 2 spill no more than 255 do, profiles/): the CG loop is a chain of
// block reductions, so an SM needs several resident CTAs to stay busy.  The host picks MINB and the
// dynamic shared memory per size class of components.
template <int NT, int MINB>
__global__ void __launch_bounds__(NT, MINB)
solve_cta_kernel(const DevProblem P, const DevConsts K, const CtaArrays A, const CtaComp* comps, unsigned smem_doubles) {
  static_assert(NT == kCtaThreads || NT == kCtaMaxThreads, "reduction lines are sized for 8 or 16 warps");
  __shared__ double red[3 * (NT / 32)];
  __shared__ double red2[4 * (NT / 32)];
  const CtaComp cc = comps[blockIdx.x];
  CtaCtx C;
  C.tid = threadIdx.x;
  C.nt = NT;
  C.Nc = (int)cc.Nc;
  C.Ec = (int)cc.Ec;
  C.nf = (int)cc.nf;
  C.n = 2 * C.nf;
  C.rec = A.rec + 5 * cc.e_off;
  C.meta = A.meta + cc.e_off;
  C.inlist = A.inlist + cc.e_off;
  C.scr = A.scr + 7 * cc.e_off;
  C.q = A.q + 2 * cc.e_off;
  C.node = A.node + cc.n_off;
  C.outptr = A.outptr + cc.n_off + cc.comp_index;
  C.inptr = A.inptr + cc.n_off + cc.comp_index;
  C.freeof = A.freeof + cc.n_off;
  C.x = A.x + 2 * cc.n_off;
  C.xc = A.xc + 2 * cc.n_off;
  C.lof = A.lof + cc.f_off;
  const uint64_t stride = 2 * A.total_free;
  double* v0 = A.vec + 2 * cc.f_off;
  C.g = v0 + V_G * stride;
  C.S = v0 + V_S * stride;
  C.dl = v0 + V_DL * stride;
  C.D2 = v0 + V_D2 * stride;
  C.r = v0 + V_R * stride;
  C.z = v0 + V_Z * stride;
  C.p = v0 + V_P * stride;  // (replaced by shared memory below when it fits)
  C.w = v0 + V_W * stride;
  C.y = v0 + V_Y * stride;
  C.diag = A.vec + V_COUNT * stride + 3 * cc.f_off;
  C.pblk = A.vec + V_COUNT * stride + 3 * A.total_free + 3 * cc.f_off;
  C.pinv = A.vec + V_COUNT * stride + 6 * A.total_free + 3 * cc.f_off;
  C.bE01 = A.bE01 + cc.ell_off;
  C.bE23 = A.bE23 + cc.ell_off;
  C.fdstE = A.fdstE + cc.ell_off;
  C.ell_base = A.ell_base + cc.s_off;
  C.twin = A.twin + cc.e_off;
  C.fdst = A.fdst + cc.e_off;
  C.regular = cc.regular != 0;
#pragma unroll
  for (int i = 0; i < kCtaRowsCached; ++i) {
    const int l = (int)threadIdx.x + i * NT;
    C.row_f[i] = l < C.Nc ? C.freeof[l] : -1;
    C.row_deg[i] = l < C.Nc ? C.outptr[l + 1] - C.outptr[l] : 0u;
    C.row_slot[i] = l < C.Nc ? C.ell_base[l >> 5] + (uint32_t)(l & 31) : 0u;
  }
  // CG vectors on chip while they fit in the launch's dynamic shared memory, in order of how often an
  // iteration touches them: p (randomly gathered by the matvec), w, r, z, y, then the preconditioner
  extern __shared__ __align__(16) double cg_smem[];
  {
    size_t used = 0;
    const size_t cap = smem_doubles;
    auto take = [&](double*& ptr, size_t n_doubles) {
      if (used + n_doubles <= cap) {
        ptr = cg_smem + used;
        used += n_doubles;
      }
    };
    take(C.p, (size_t)C.n);
    take(C.w, (size_t)C.n);
    take(C.r, (size_t)C.n);
    take(C.z, (size_t)C.n);
    take(C.y, (size_t)C.n);
    take(C.pinv, 3 * (size_t)C.nf);
  }
  C.red = red;
  C.red2 = red2;
  const uint32_t c = cc.slot;
  const int tid = C.tid, lane = tid & 31;
  if (P.st_times && tid == 0) {
    unsigned long long ns;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
    P.st_times[2 * (size_t)c] = ns;
  }

  // start point: IterationZero projects the free blocks onto the box
  for (int l = tid; l < C.Nc; l += C.nt) {
    const uint32_t v = C.node[l];
    double p0 = P.positions[2 * (size_t)v], p1 = P.positions[2 * (size_t)v + 1];
    if (C.freeof[l] >= 0) {
      p0 = fmin(fmax(p0, -K.bound), K.bound);
      p1 = fmin(fmax(p1, -K.bound), K.bound);
    }
    C.x[2 * l] = p0;
    C.x[2 * l + 1] = p1;
  }
  __syncthreads();
  if (tid == 0) P.st_kept[c] = cc.Ec;
  if (C.nf == 0) {
    if (tid == 0) {
      P.st_iter[c] = 0;
      P.st_term[c] = LFR_TERM_EMPTY;
      P.st_cost0[c] = 0.0;
      P.st_cost1[c] = 0.0;
      P.st_ls[c] = 0;
    }
    return;
  }
  const bool prof = P.st_cycles != nullptr;
  long long t_begin = 0, t_lm = 0, t_eval = 0, t_mark = 0;
  long long tph[4] = {0, 0, 0, 0};
  if (prof) t_begin = clock64();
  double cost = cta_eval(C, C.x, K);
  double gmax = cta_assemble<false>(C, true, K);
  const double cost0 = cost;
  double radius = K.radius0, nu = 2.0;
  int iter = 0, n_invalid = 0, term = LFR_TERM_NO_CONVERGENCE;
  unsigned ls_steps = 0, cg_iters = 0;
  bool success = true;
  auto norms = [&](double* xn2, double* dn2) {
    double a = 0.0, b = 0.0, z = 0.0;
    for (int i = tid; i < C.n; i += C.nt) {
      const int l = C.lof[i >> 1];
      const double xv = C.x[2 * l + (i & 1)], dv = xv - C.xc[2 * l + (i & 1)];
      a += xv * xv;
      b += dv * dv;
    }
    block_sum3(C, a, b, z);
    *xn2 = a;
    *dn2 = b;
  };
  double x_norm;
  {
    double a = 0.0, b = 0.0, z = 0.0;
    for (int i = tid; i < C.n; i += C.nt) {
      const int l = C.lof[i >> 1];
      const double xv = C.x[2 * l + (i & 1)];
      a += xv * xv;
    }
    block_sum3(C, a, b, z);
    x_norm = sqrt(a);
  }
  for (;;) {
    if (iter >= K.max_iter) { term = LFR_TERM_NO_CONVERGENCE; break; }
    if (success && gmax <= K.g_tol) { term = LFR_TERM_GRADIENT_TOL; break; }
    if (radius <= K.radius_min) { term = LFR_TERM_MIN_RADIUS; break; }
    ++iter;
    success = false;
    double model_change = 0.0, gd = 0.0, dmax = 0.0;
    if (prof) t_mark = clock64();
    bool valid = cta_lm_step(C, radius, K, &model_change, &gd, &dmax, &cg_iters, prof ? tph : nullptr);
    if (prof) t_lm += clock64() - t_mark;
    valid = valid && (model_change > 0.0);
    if (!valid) {
      if (++n_invalid >= K.max_invalid) { term = LFR_TERM_FAILURE; break; }
      radius /= nu;
      nu *= 2.0;
      continue;
    }
    n_invalid = 0;
    cta_candidate(C, 1.0, K);
    if (prof) t_mark = clock64();
    double cost_c = cta_eval(C, C.xc, K);
    if (prof) t_eval += clock64() - t_mark;
    bool c_valid = isfinite(cost_c);
    if (!c_valid || cost_c > cost + K.ls_suff * gd * 1.0) {
      LsSample initial{0.0, cost, gd, true, true};
      LsSample previous{0.0, 0.0, 0.0, false, false};
      LsSample current{1.0, cost_c, 0.0, c_valid, false};
      if (c_valid) {
        current.gradient = cta_assemble<true>(C, false, K);
        current.gradient_valid = isfinite(current.gradient);
      }
      int ls_iter = 0;
      bool ls_ok = false;
      for (;;) {
        ++ls_iter;
        ++ls_steps;
        if (ls_iter >= K.max_ls_iter) break;
        const double step = ls_next_step(initial, previous, current, K, lane);
        if (step * dmax < K.ls_min_step) break;
        previous = current;
        cta_candidate(C, step, K);
        cost_c = cta_eval(C, C.xc, K);
        c_valid = isfinite(cost_c);
        current = LsSample{step, cost_c, 0.0, c_valid, false};
        if (c_valid) {
          current.gradient = cta_assemble<true>(C, false, K);
          current.gradient_valid = isfinite(current.gradient);
        }
        if (c_valid && !(cost_c > cost + K.ls_suff * gd * step)) { ls_ok = true; break; }
      }
      if (ls_ok) {
        for (int i = tid; i < C.n; i += C.nt) C.dl[i] *= current.x;
        __syncthreads();
      } else {
        cta_candidate(C, 1.0, K);
        cost_c = cta_eval(C, C.xc, K);
        c_valid = isfinite(cost_c);
      }
    }
    if (!c_valid) cost_c = 1.7976931348623157e308;
    double xn2, dn2;
    norms(&xn2, &dn2);
    const double step_norm = sqrt(dn2);
    if (step_norm <= K.p_tol * (x_norm + K.p_tol)) { term = LFR_TERM_PARAMETER_TOL; break; }
    if (fabs(cost - cost_c) <= K.f_tol * cost) { term = LFR_TERM_FUNCTION_TOL; break; }
    const double rho = (cost - cost_c) / model_change;
    if (rho > K.min_rel_decrease) {
      double a2 = 0.0, z1 = 0.0, z2 = 0.0;
      for (int i = tid; i < 2 * C.Nc; i += C.nt) {
        const double v = C.xc[i];
        C.x[i] = v;
        if (C.freeof[i >> 1] >= 0) a2 += v * v;
      }
      block_sum3(C, a2, z1, z2);
      x_norm = sqrt(a2);
      cost = cost_c;
      gmax = cta_assemble<false>(C, false, K);
      success = true;
      const double t = 2.0 * rho - 1.0;
      radius = fmin(K.radius_max, radius / fmax(1.0 / 3.0, 1.0 - t * t * t));
      nu = 2.0;
    } else {
      radius /= nu;
      nu *= 2.0;
    }
  }
  // (not after FAILURE: Ceres only commits a usable solution, solver.cc Minimize / IsSolutionUsable)
  if (term != LFR_TERM_FAILURE) {
    for (int i = tid; i < C.n; i += C.nt) {
      const int l = C.lof[i >> 1];
      P.positions_out[2 * (size_t)C.node[l] + (i & 1)] = C.x[2 * l + (i & 1)];
    }
  }
  if (tid == 0) {
    P.st_iter[c] = iter;
    P.st_term[c] = term;
    P.st_cost0[c] = cost0;
    P.st_cost1[c] = cost;
    P.st_ls[c] = ls_steps;
    if (P.st_cycles) {
      unsigned long long* o = P.st_cycles + 8 * (size_t)c;
      o[0] = (unsigned long long)(clock64() - t_begin);  // total, of which o[2] in the PCG solves
      o[2] = (unsigned long long)t_lm;
      o[3] = ((unsigned long long)(tph[0] >> 8) << 32) | (unsigned long long)min((long long)0xffffffffll, tph[1] >> 8);  // product | reduction 1, 256-cycle units
      o[5] = ((unsigned long long)(tph[2] >> 8) << 32) | (unsigned long long)min((long long)0xffffffffll, tph[3] >> 8);  // update | reduction 2
      o[4] = cg_iters;
      o[1] = 1;  // marks a CTA-tier component
      o[6] = ((unsigned long long)ls_steps << 32) | (unsigned long long)min((long long)0xffffffffll, t_eval >> 10);  // + first-candidate evaluations, kcycles
      unsigned smid;
      asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
      o[7] = smid;
    }
    if (P.st_times) {
      unsigned long long ns;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
      P.st_times[2 * (size_t)c + 1] = ns;
    }
  }
}

// ---- device-side preparation of the CTA-tier components (solve.cc:98-143 for each) --------------
// One CTA per large component builds, in HBM: the kept-edge list in CSR order (a compact copy of the
// 80-byte records + src_local | dst_local << 14 | kind << 28), out- and in-edge row pointers, the in-edge list (stable:
// ascending kept-edge index per destination, so every later summation order is fixed), the
// free-variable numbering, every kept edge's twin and its destination's free index.  The host hands
// in only offsets (upper bounds from row_ptr / is_root: cc.e_off counts CANDIDATE edges).
// Exclusive prefix over per-thread segment sums; returns the grand total.  `sh` holds kCtaThreads + 1 words.
__device__ __forceinline__ uint32_t cta_scan_partials(uint32_t mine, uint32_t* sh, uint32_t* total) {
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  uint32_t v = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_up_sync(kFull, v, o);
    if (lane >= o) v += t;
  }
  __syncthreads();  // `sh` may still be read from a previous call
  if (lane == 31) sh[w] = v;
  __syncthreads();
  if (tid == 0) {
    uint32_t run = 0;
    for (int k = 0; k < kCtaThreads / 32; ++k) {
      const uint32_t t = sh[k];
      sh[k] = run;
      run += t;
    }
    sh[kCtaThreads / 32] = run;
  }
  __syncthreads();
  *total = sh[kCtaThreads / 32];
  return sh[w] + v - mine;
}

struct CtaEdgeClass {
  bool keep;
  uint32_t kind, dl;
};

__device__ __forceinline__ CtaEdgeClass cta_classify(const DevProblem& P, const uint32_t* node, uint32_t Nc, uint32_t v,
                                                     uint32_t e) {
  CtaEdgeClass r{false, 0u, 0u};
  const uint32_t dst = reinterpret_cast<const uint32_t*>(P.edges)[20 * (size_t)e + 19];
  if (dst >= P.n_nodes || dst == v) {
    *P.err_flag = 1;  // malformed input: reported by the host as LFR_EINVAL
    return r;
  }
  if (P.track[v] == P.track[dst]) r.kind = LFR_EDGE_CAUCHY;        // solve.cc:105
  else if (P.comp[v] == P.comp[dst]) r.kind = LFR_EDGE_TUKEY;      // solve.cc:114
  else return r;                                                   // solve.cc:123
  if (P.is_root[v] && P.is_root[dst]) return r;                    // all-constant block (A.1)
  r.dl = P.local_of[dst];
  if (r.dl >= Nc || node[r.dl] != dst) {
    *P.err_flag = 1;  // component_idx and nodes_in_component disagree
    return r;
  }
  r.keep = true;
  return r;
}

__global__ void __launch_bounds__(kCtaThreads)
cta_prepare_kernel(const DevProblem P, const CtaArrays A, CtaComp* comps) {
  __shared__ uint32_t sh[kCtaThreads + 1];
  CtaComp& cc = comps[blockIdx.x];
  const uint32_t Nc = cc.Nc, nbeg = P.comp_ptr[cc.slot];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  constexpr int kWarps = kCtaThreads / 32;
  float4* rec = const_cast<float4*>(A.rec) + 5 * cc.e_off;
  uint32_t* meta = const_cast<uint32_t*>(A.meta) + cc.e_off;
  uint32_t* inlist = const_cast<uint32_t*>(A.inlist) + cc.e_off;
  uint32_t* twin = const_cast<uint32_t*>(A.twin) + cc.e_off;
  int32_t* fdst = const_cast<int32_t*>(A.fdst) + cc.e_off;
  uint32_t* node = const_cast<uint32_t*>(A.node) + cc.n_off;
  uint32_t* outptr = const_cast<uint32_t*>(A.outptr) + cc.n_off + cc.comp_index;
  uint32_t* inptr = const_cast<uint32_t*>(A.inptr) + cc.n_off + cc.comp_index;
  int32_t* freeof = const_cast<int32_t*>(A.freeof) + cc.n_off;
  uint32_t* lof = const_cast<uint32_t*>(A.lof) + cc.f_off;

  for (uint32_t l = tid; l <= Nc; l += kCtaThreads) {
    if (l < Nc) node[l] = P.comp_nodes[nbeg + l];
    inptr[l] = 0;
    outptr[l] = 0;
  }
  __syncthreads();
  // kept out-degree of every node: one warp per node, lanes over its out-edges
  for (uint32_t l = wid; l < Nc; l += kWarps) {
    const uint32_t v = node[l], rs = P.row_ptr[v], re = P.row_ptr[v + 1];
    uint32_t cnt = 0;
    for (uint32_t e0 = rs; e0 < re; e0 += 32) {
      const uint32_t e = e0 + lane;
      const bool keep = e < re && cta_classify(P, node, Nc, v, e).keep;
      cnt += __popc(__ballot_sync(kFull, keep));
    }
    if (lane == 0) outptr[l + 1] = cnt;
  }
  __syncthreads();
  // row pointers: thread t owns the contiguous node range [t*seg, (t+1)*seg)
  const uint32_t seg = (Nc + kCtaThreads - 1) / kCtaThreads;
  const uint32_t lb = min(Nc, (uint32_t)tid * seg), le = min(Nc, lb + seg);
  uint32_t Ec = 0;
  {
    uint32_t mine = 0;
    for (uint32_t l = lb; l < le; ++l) mine += outptr[l + 1];
    uint32_t run = cta_scan_partials(mine, sh, &Ec);
    for (uint32_t l = lb; l < le; ++l) {
      run += outptr[l + 1];
      outptr[l + 1] = run;  // inclusive at l + 1 == exclusive start of node l + 1
    }
  }
  __syncthreads();
  // sliced-ELL geometry: slice s = local nodes [32 s, 32 s + 32), width = its largest kept out-degree
  uint32_t* ell_base = const_cast<uint32_t*>(A.ell_base) + cc.s_off;
  int32_t* fdstE = const_cast<int32_t*>(A.fdstE) + cc.ell_off;
  {
    const uint32_t S = (Nc + 31) / 32, sseg = (S + kCtaThreads - 1) / kCtaThreads;
    const uint32_t sb = min(S, (uint32_t)tid * sseg), se = min(S, sb + sseg);
    uint32_t mine = 0, tot;
    for (uint32_t sidx = sb; sidx < se; ++sidx) {
      uint32_t wmax = 0;
      for (uint32_t l = 32 * sidx; l < min(Nc, 32 * sidx + 32); ++l) wmax = max(wmax, outptr[l + 1] - outptr[l]);
      wmax = (wmax + 3u) & ~3u;  // rows are walked in groups of four slots
      ell_base[sidx + 1] = 32 * wmax;
      mine += 32 * wmax;
    }
    uint32_t run = cta_scan_partials(mine, sh, &tot);
    if (tid == 0) ell_base[0] = 0;
    for (uint32_t sidx = sb; sidx < se; ++sidx) {
      run += ell_base[sidx + 1];
      ell_base[sidx + 1] = run;
    }
  }
  __syncthreads();
  {  // every slot starts as "zero block, no column": real blocks are written by the assembly each iteration
    double2* bE01 = const_cast<double2*>(A.bE01) + cc.ell_off;
    double2* bE23 = const_cast<double2*>(A.bE23) + cc.ell_off;
    const uint32_t n_slots = ell_base[(Nc + 31) / 32];
    for (uint32_t i = tid; i < n_slots; i += kCtaThreads) {
      fdstE[i] = -1;
      bE01[i] = make_double2(0.0, 0.0);
      bE23[i] = make_double2(0.0, 0.0);
    }
  }
  // kept-edge records in CSR order + in-degree counts
  for (uint32_t l = wid; l < Nc; l += kWarps) {
    const uint32_t v = node[l], rs = P.row_ptr[v], re = P.row_ptr[v + 1];
    uint32_t at = outptr[l];
    for (uint32_t e0 = rs; e0 < re; e0 += 32) {
      const uint32_t e = e0 + lane;
      CtaEdgeClass k{false, 0u, 0u};
      if (e < re) k = cta_classify(P, node, Nc, v, e);
      const unsigned m = __ballot_sync(kFull, k.keep);
      if (k.keep) {
        const uint32_t j = at + __popc(m & ((1u << lane) - 1u));
        meta[j] = l | (k.dl << 14) | (k.kind << 28);
        atomicAdd(&inptr[k.dl + 1], 1u);  // integer count: order-independent
      }
      // the kept records of this chunk, copied by the whole warp word by word: the 32 candidates are
      // contiguous (a node's out-edges, 80 bytes each), so every load instruction reads one <= 512-byte
      // span — from HBM, or from the caller's pinned array, where it is what keeps the PCIe pull at
      // link rate (a lane fetching its own record in five 16-byte pieces ran at ~12 GB/s)
      {
        const float4* src = P.edges + 5 * (size_t)e0;
        const uint32_t n_words = 5u * min(32u, re - e0);
        float4 q[5];
        uint32_t dst[5];
#pragma unroll
        for (int t = 0; t < 5; ++t) {
          const uint32_t w = (uint32_t)lane + 32u * t, i = w / 5u;
          const bool take = w < n_words && ((m >> i) & 1u);
          dst[t] = take ? 5u * (at + __popc(m & ((1u << i) - 1u))) + (w - 5u * i) : 0xffffffffu;
          if (take) q[t] = __ldg(src + w);
        }
#pragma unroll
        for (int t = 0; t < 5; ++t)
          if (dst[t] != 0xffffffffu) rec[dst[t]] = q[t];
      }
      at += __popc(m);
    }
  }
  __syncthreads();
  {
    uint32_t mine = 0, tot;
    for (uint32_t l = lb; l < le; ++l) mine += inptr[l + 1];
    uint32_t run = cta_scan_partials(mine, sh, &tot);
    for (uint32_t l = lb; l < le; ++l) {
      run += inptr[l + 1];
      inptr[l + 1] = run;
    }
  }
  __syncthreads();
  // in-edge lists, stable.  `freeof` serves as the per-destination fill cursor; warp w owns the
  // destinations with dl % kWarps == w and walks ALL kept edges in ascending order, so each list
  // comes out in ascending kept-edge index whatever the warp timing.
  for (uint32_t l = tid; l < Nc; l += kCtaThreads) freeof[l] = (int32_t)inptr[l];
  __syncthreads();
  for (uint32_t j0 = 0; j0 < Ec; j0 += 32) {
    const uint32_t j = j0 + lane;
    uint32_t dl = 0;
    bool mine = false;
    if (j < Ec) {
      dl = (meta[j] >> 14) & 0x3fffu;
      mine = (dl % kWarps) == (uint32_t)wid;
    }
    const unsigned m = __match_any_sync(kFull, mine ? dl : (0x10000u + (uint32_t)lane));
    int base = 0;
    if (mine) base = freeof[dl];
    __syncwarp();
    if (mine) {
      const int rank = __popc(m & ((1u << lane) - 1u)), n_same = __popc(m);
      inlist[base + rank] = j;
      if (rank == n_same - 1) freeof[dl] = base + n_same;
    }
    __syncwarp();
  }
  __syncthreads();
  // free-variable numbering: a node is free when it has a kept edge and is not a root
  uint32_t nf = 0;
  {
    uint32_t mine = 0;
    for (uint32_t l = lb; l < le; ++l) {
      const bool is_free = (outptr[l + 1] - outptr[l]) + (inptr[l + 1] - inptr[l]) > 0 && !P.is_root[node[l]];
      mine += is_free ? 1u : 0u;
    }
    uint32_t run = cta_scan_partials(mine, sh, &nf);
    for (uint32_t l = lb; l < le; ++l) {
      const bool is_free = (outptr[l + 1] - outptr[l]) + (inptr[l + 1] - inptr[l]) > 0 && !P.is_root[node[l]];
      freeof[l] = is_free ? (int32_t)run : -1;
      if (is_free) lof[run++] = l;
    }
  }
  __syncthreads();
  // twin (reverse edge) of every kept edge and the destination's free index
  int regular = 1;
  for (uint32_t j = tid; j < Ec; j += kCtaThreads) {
    const uint32_t sl = meta[j] & 0x3fffu, dl = (meta[j] >> 14) & 0x3fffu;
    uint32_t found = 0, tw = j;
    for (uint32_t t = outptr[dl]; t < outptr[dl + 1]; ++t)
      if (((meta[t] >> 14) & 0x3fffu) == sl) {
        tw = t;
        ++found;
      }
    if (found != 1) regular = 0;
    twin[j] = tw;
    fdst[j] = freeof[dl];
    fdstE[(size_t)ell_base[sl >> 5] + (sl & 31u) + 32u * (size_t)(j - outptr[sl])] = freeof[dl];
  }
  regular = __syncthreads_and(regular);
  if (tid == 0) {
    cc.Ec = Ec;
    cc.nf = nf;
    cc.regular = regular ? 1u : 0u;
  }
}

}  // namespace lfr
