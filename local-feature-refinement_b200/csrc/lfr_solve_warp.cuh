// lfr_solve_warp.cuh — one warp solves one component (one ceres::Problem of
// solve.cc:79-160) start to finish: residual/Jacobian evaluation, J^T J block
// assembly, exact linear solve, LM damping / projected Armijo line search /
// termination (SURVEY Appendix A.6), with no host round trip inside the loop.
//
// Mapping (SURVEY 7 "device-mapping notes"):
//   * lanes <-> directed edges for the evaluation: each lane reads its 80-byte
//     edge record as five 128-bit loads, evaluates cost.cc's interpolator and
//     the robust loss in fp64 registers and stages {a, r, M} (7 doubles) in
//     shared memory;
//   * lanes <-> free nodes for the assembly: each lane gathers its node's
//     out-edges (contiguous, CSR by source) and in-edges (index list built once)
//     from shared memory into the node's 2x2 diagonal block, its gradient pair
//     and its block row of the packed lower-triangular normal matrix — row
//     ownership makes the sums atomics-free and bit-reproducible;
//   * the warp factorises the (<= 96 x 96) damped normal matrix in shared
//     memory (Cholesky with the right-hand side carried as an extra row), and
//     all trust-region scalars live in registers, identical in every lane.
#pragma once
#include "lfr_math.cuh"

namespace lfr {

struct DevProblem {
  uint32_t n_nodes;
  int* err_flag;  // set when a malformed edge (dst out of range, self edge) is met
  const uint32_t* row_ptr;
  const float4* edges;  // 5 x float4 per edge
  const uint32_t* track;
  const uint32_t* comp;
  const uint8_t* is_root;
  const uint32_t* comp_ptr;
  const uint32_t* comp_nodes;
  const uint32_t* local_of;  // node -> index inside its component's node list
  double* positions;         // [2N] start point (device memory)
  double* positions_out;     // [2N] results: `positions` itself, or the caller's pinned host buffer
                             // (zero-copy write-back: only free nodes are written, solve.cc:131-141)
  unsigned long long* pull_ctr;  // [2] bytes of staging pulls {ticketed, arrived} (zero-copy pacing, see stage_edges)
  unsigned pull_window;      // 0 = unpaced; else at most this many bytes of staging pulls are outstanding per device
  // per dispatch slot
  int32_t* st_iter;
  int32_t* st_term;
  double* st_cost0;
  double* st_cost1;
  uint32_t* st_ls;
  uint32_t* st_kept;  // kept directed edges E_c
  unsigned long long* st_cycles;  // optional [8 per slot]: total, setup, eval, assemble, lm_step, line search (LFR_DBG_PROFILE)
  unsigned long long* st_times;   // optional [2 per slot]: %globaltimer (ns) when the component's warp started / finished
};

struct WarpBucket {
  const uint32_t* list;  // dispatch slots handled by this launch
  uint32_t n;
  int emax;    // max candidate out-edges of a component in this bucket
  int ncmax;   // max nodes
  int n2max;   // max unknowns (2 x free nodes)
  int smem_per_warp;
};

__host__ __device__ inline int tri(int n) { return n * (n + 1) / 2; }
__host__ __device__ inline int align_up(int v, int a) { return (v + a - 1) / a * a; }

// Per-warp shared-memory carve-up; host and device must agree.
struct WarpLayout {
  int x, xc, g, S, dl, dinv, H, A, scr;             // doubles (byte offsets)
  int eidx, meta, node, rowstart, candptr;          // u32
  int inlist, outptr, inptr, freeof, lof;           // u16 / i16
  int total;
  __host__ __device__ WarpLayout(int emax, int ncmax, int n2max) {
    int o = 0;
    x = o; o += 16 * ncmax;
    xc = o; o += 16 * ncmax;
    g = o; o += 8 * n2max;
    S = o; o += 8 * n2max;
    dl = o; o += 8 * n2max;
    dinv = o; o += 8 * n2max;
    H = o; o += 8 * tri(n2max);
    A = o; o += 8 * tri(n2max + 1);
    scr = o; o += 8 * 7 * emax;
    eidx = o; o += 4 * emax;
    meta = o; o += 4 * emax;
    node = o; o += 4 * ncmax;
    rowstart = o; o += 4 * ncmax;
    candptr = o; o += 4 * (ncmax + 1);
    inlist = o; o += 2 * emax;
    outptr = o; o += 2 * (ncmax + 1);
    inptr = o; o += 2 * (ncmax + 1);
    freeof = o; o += 2 * ncmax;
    lof = o; o += 2 * (n2max / 2 + 1);
    total = align_up(o, 16);
  }
};

constexpr unsigned kFull = 0xffffffffu;
constexpr int kMaxWarpN2 = 96;      // unknowns a warp handles
constexpr int kMaxWarpNodes = 4095; // 12-bit local indices in `meta`

struct WarpCtx {
  int lane, Nc, Ec, nf, n, emax;
  double *x, *xc, *g, *S, *dl, *dinv, *H, *A, *scr;
  uint32_t *eidx, *meta, *node;
  uint16_t *inlist, *outptr, *inptr, *lof;
  int16_t* freeof;
  const float4* edges;
};

// Evaluate every kept edge at positions `xe` ([2*Nc], component-local); stage
// {a, r0, r1, m00, m01, m10, m11} in shared memory; return the cost (A.1).
__device__ __forceinline__ double eval_pass(const WarpCtx& C, const double* xe, const DevConsts& K) {
  double cost = 0.0;
  for (int j = C.lane; j < C.Ec; j += 32) {
    const uint32_t mt = C.meta[j];
    const int s = mt & 0xfff, d = (mt >> 12) & 0xfff, kind = mt >> 24;
    const float4* qp = C.edges + 5 * (size_t)C.eidx[j];
    float4 q[5];
#pragma unroll
    for (int t = 0; t < 5; ++t) q[t] = __ldg(qp + t);
    const EdgeEval ev = eval_edge(q, kind, xe[2 * s], xe[2 * s + 1], xe[2 * d], xe[2 * d + 1], K);
    double* sc = C.scr + j;
    sc[0] = ev.a;
    sc[C.emax] = ev.r0;
    sc[2 * C.emax] = ev.r1;
    sc[3 * C.emax] = ev.m00;
    sc[4 * C.emax] = ev.m01;
    sc[5 * C.emax] = ev.m10;
    sc[6 * C.emax] = ev.m11;
    cost += ev.half_rho;
  }
  cost = warp_sum(cost);
  __syncwarp();
  return cost;
}

// Gradient of the cost at the staged evaluation, dotted with dl (phi'(alpha)
// of the line search).
__device__ __forceinline__ double staged_grad_dot(const WarpCtx& C) {
  double acc = 0.0;
  const int E = C.emax;
  for (int f = C.lane; f < C.nf; f += 32) {
    const int l = C.lof[f];
    double g0 = 0., g1 = 0.;
    for (int j = C.outptr[l]; j < C.outptr[l + 1]; ++j) {
      const double a = C.scr[j], r0 = C.scr[E + j], r1 = C.scr[2 * E + j];
      g0 -= a * (C.scr[3 * E + j] * r0 + C.scr[5 * E + j] * r1);
      g1 -= a * (C.scr[4 * E + j] * r0 + C.scr[6 * E + j] * r1);
    }
    for (int t = C.inptr[l]; t < C.inptr[l + 1]; ++t) {
      const int j = C.inlist[t];
      const double a = C.scr[j];
      g0 += a * C.scr[E + j];
      g1 += a * C.scr[2 * E + j];
    }
    acc += g0 * C.dl[2 * f] + g1 * C.dl[2 * f + 1];
  }
  return warp_sum(acc);
}

// J^T J and J^T r from the staged evaluation.  On the first call also fixes the
// Jacobi column scaling S = 1/(1 + sqrt(diag)) (A.6 iter 0).  Leaves H = S H S
// (packed lower triangle), g = raw gradient.  Returns the projected-gradient
// max norm  |x - P(x - g)|_inf.
__device__ __forceinline__ double assemble(const WarpCtx& C, bool first, const DevConsts& K) {
  const int E = C.emax;
  for (int i = C.lane; i < tri(C.n); i += 32) C.H[i] = 0.0;
  __syncwarp();
  for (int f = C.lane; f < C.nf; f += 32) {
    const int l = C.lof[f];
    double d00 = 0., d01 = 0., d11 = 0., g0 = 0., g1 = 0.;
    double* H0 = C.H + tri(2 * f);
    double* H1 = C.H + tri(2 * f + 1);
    for (int j = C.outptr[l]; j < C.outptr[l + 1]; ++j) {
      const double a = C.scr[j], r0 = C.scr[E + j], r1 = C.scr[2 * E + j];
      const double m00 = C.scr[3 * E + j], m01 = C.scr[4 * E + j], m10 = C.scr[5 * E + j],
                   m11 = C.scr[6 * E + j];
      d00 += a * (m00 * m00 + m10 * m10);
      d01 += a * (m00 * m01 + m10 * m11);
      d11 += a * (m01 * m01 + m11 * m11);
      g0 -= a * (m00 * r0 + m10 * r1);
      g1 -= a * (m01 * r0 + m11 * r1);
      const int fd = C.freeof[(C.meta[j] >> 12) & 0xfff];
      if (fd >= 0 && fd < f) {  // block (f, fd) = a J_s^T J_d = -a M^T
        H0[2 * fd] -= a * m00;
        H0[2 * fd + 1] -= a * m10;
        H1[2 * fd] -= a * m01;
        H1[2 * fd + 1] -= a * m11;
      }
    }
    for (int t = C.inptr[l]; t < C.inptr[l + 1]; ++t) {
      const int j = C.inlist[t];
      const double a = C.scr[j];
      d00 += a;
      d11 += a;
      g0 += a * C.scr[E + j];
      g1 += a * C.scr[2 * E + j];
      const int fs = C.freeof[C.meta[j] & 0xfff];
      if (fs >= 0 && fs < f) {  // block (f, fs) = a J_d^T J_s = -a M
        H0[2 * fs] -= a * C.scr[3 * E + j];
        H0[2 * fs + 1] -= a * C.scr[4 * E + j];
        H1[2 * fs] -= a * C.scr[5 * E + j];
        H1[2 * fs + 1] -= a * C.scr[6 * E + j];
      }
    }
    H0[2 * f] = d00;
    H1[2 * f] = d01;
    H1[2 * f + 1] = d11;
    C.g[2 * f] = g0;
    C.g[2 * f + 1] = g1;
    if (first) {
      C.S[2 * f] = 1.0 / (1.0 + sqrt(d00));
      C.S[2 * f + 1] = 1.0 / (1.0 + sqrt(d11));
    }
  }
  __syncwarp();
  double gmax = 0.0;
  for (int i = C.lane; i < C.n; i += 32) {  // scale row i, projected gradient
    double* Hi = C.H + tri(i);
    const double si = C.S[i];
    for (int j = 0; j <= i; ++j) Hi[j] *= si * C.S[j];
    const int l = C.lof[i >> 1];
    const double xi = C.x[2 * l + (i & 1)];
    const double p = fmin(fmax(xi - C.g[i], -K.bound), K.bound);
    gmax = fmax(gmax, fabs(xi - p));
  }
  gmax = warp_max(gmax);
  __syncwarp();
  return gmax;
}

// Solve (S H S + D^2) y = S g exactly (dense Cholesky, rhs as extra row),
// write dl = -S y.  Returns false on a non-positive pivot / non-finite step.
// model_cost_change = y'Sg - y'(SHS)y/2 = (y'Sg + y'D^2 y)/2.
__device__ __forceinline__ bool lm_step(const WarpCtx& C, double radius, const DevConsts& K,
                                        double* model_change) {
  const int n = C.n;
  for (int i = C.lane; i < tri(n); i += 32) C.A[i] = C.H[i];
  __syncwarp();
  double* An = C.A + tri(n);
  for (int i = C.lane; i < n; i += 32) {
    const double hii = C.H[tri(i) + i];
    const double d2 = fmin(fmax(hii, K.min_diag), K.max_diag) / radius;
    C.A[tri(i) + i] = hii + d2;
    An[i] = C.S[i] * C.g[i];
  }
  __syncwarp();
  bool ok = true;
  for (int j = 0; j < n; ++j) {
    const double* Aj = C.A + tri(j);
    // rows j + lane + 32 p of this column, all passes in ONE k-loop: four
    // independent accumulators share the broadcast load of A[j][k]
    double s[4];
    const double* Ar[4];
    const int npass = (n - j) / 32 + 1;  // passes that have at least one live row (warp-uniform)
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      const int i = j + C.lane + 32 * p;
      const bool live = i <= n;
      Ar[p] = C.A + tri(live ? i : j);  // dead lanes shadow row j (harmless, never stored)
      s[p] = Ar[p][j];
    }
    if (npass == 1) {
      for (int k = 0; k < j; ++k) s[0] -= Ar[0][k] * Aj[k];
    } else if (npass == 2) {
      for (int k = 0; k < j; ++k) {
        const double ajk = Aj[k];
        s[0] -= Ar[0][k] * ajk;
        s[1] -= Ar[1][k] * ajk;
      }
    } else {
      for (int k = 0; k < j; ++k) {
        const double ajk = Aj[k];
#pragma unroll
        for (int p = 0; p < 4; ++p) s[p] -= Ar[p][k] * ajk;
      }
    }
    const double sjj = __shfl_sync(kFull, s[0], 0);
    if (!(sjj > 0.0) || !isfinite(sjj)) {
      ok = false;
      break;
    }
    const double rs = rsqrt(sjj);
    __syncwarp();  // every lane's reads of column j / row j are done before the column is overwritten
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      const int i = j + C.lane + 32 * p;
      if (i <= n) C.A[tri(i) + j] = s[p] * rs;
    }
    if (C.lane == 0) C.dinv[j] = rs;
    __syncwarp();
  }
  if (!ok) return false;
  // back substitution L^T y = z, z = row n of A; lane holds y[lane + 32 p]
  double z[3];
#pragma unroll
  for (int p = 0; p < 3; ++p) z[p] = (C.lane + 32 * p < n) ? An[C.lane + 32 * p] : 0.0;
  for (int i = n - 1; i >= 0; --i) {
    const double* Li = C.A + tri(i);
    const int slot = i >> 5;
    double yi = (slot == 0 ? z[0] : (slot == 1 ? z[1] : z[2])) * C.dinv[i];
    yi = __shfl_sync(kFull, yi, i & 31);
#pragma unroll
    for (int p = 0; p < 3; ++p)
      if (C.lane + 32 * p < i) z[p] -= Li[C.lane + 32 * p] * yi;
    if (C.lane == (i & 31)) {
      if (slot == 0) z[0] = yi; else if (slot == 1) z[1] = yi; else z[2] = yi;
    }
  }
  double mc = 0.0;
  bool finite = true;
#pragma unroll
  for (int p = 0; p < 3; ++p) {
    const int i = C.lane + 32 * p;
    if (i < n) {
      const double y = z[p];
      const double hii = C.H[tri(i) + i];
      const double d2 = fmin(fmax(hii, K.min_diag), K.max_diag) / radius;
      const double si = C.S[i];
      mc += y * (si * C.g[i] + d2 * y);
      C.dl[i] = -si * y;
      finite = finite && isfinite(y);
    }
  }
  *model_change = 0.5 * warp_sum(mc);
  finite = __all_sync(kFull, finite);
  __syncwarp();
  return finite;
}

// xc = P(x + alpha dl) for free nodes, x for constants.
__device__ __forceinline__ void make_candidate(const WarpCtx& C, double alpha, const DevConsts& K) {
  for (int i = C.lane; i < 2 * C.Nc; i += 32) {
    const int f = C.freeof[i >> 1];
    double v = C.x[i];
    if (f >= 0) v = fmin(fmax(v + alpha * C.dl[2 * f + (i & 1)], -K.bound), K.bound);
    C.xc[i] = v;
  }
  __syncwarp();
}

template <int WARPS>
__global__ void __launch_bounds__(WARPS * 32, 16 / WARPS)
solve_warp_kernel(const DevProblem P, const DevConsts K, const WarpBucket B) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const uint32_t item = blockIdx.x * WARPS + wib;
  if (item >= B.n) return;  // warps are independent: no block-level barrier anywhere
  const uint32_t c = B.list[item];
  unsigned char* base = smem_raw + (size_t)wib * B.smem_per_warp;
  const WarpLayout L(B.emax, B.ncmax, B.n2max);
  WarpCtx C;
  C.lane = lane;
  C.emax = B.emax;
  C.x = (double*)(base + L.x);
  C.xc = (double*)(base + L.xc);
  C.g = (double*)(base + L.g);
  C.S = (double*)(base + L.S);
  C.dl = (double*)(base + L.dl);
  C.dinv = (double*)(base + L.dinv);
  C.H = (double*)(base + L.H);
  C.A = (double*)(base + L.A);
  C.scr = (double*)(base + L.scr);
  C.eidx = (uint32_t*)(base + L.eidx);
  C.meta = (uint32_t*)(base + L.meta);
  C.node = (uint32_t*)(base + L.node);
  uint32_t* rowstart = (uint32_t*)(base + L.rowstart);
  uint32_t* candptr = (uint32_t*)(base + L.candptr);
  C.inlist = (uint16_t*)(base + L.inlist);
  C.outptr = (uint16_t*)(base + L.outptr);
  C.inptr = (uint16_t*)(base + L.inptr);
  C.freeof = (int16_t*)(base + L.freeof);
  C.lof = (uint16_t*)(base + L.lof);
  C.edges = P.edges;

  const bool prof = (P.st_cycles != nullptr);
  long long t_begin = prof ? clock64() : 0, t_mark = t_begin;
  long long cyc_eval = 0, cyc_asm = 0, cyc_lm = 0, cyc_ls = 0, cyc_setup = 0;
#define LFR_TICK(acc) do { if (prof) { const long long now__ = clock64(); acc += now__ - t_mark; t_mark = now__; } } while (0)
  // ---- component setup (solve.cc:98-143) --------------------------------------
  const uint32_t nbeg = P.comp_ptr[c];
  const int Nc = (int)(P.comp_ptr[c + 1] - nbeg);
  C.Nc = Nc;
  int run = 0;
  for (int l0 = 0; l0 < Nc; l0 += 32) {
    const int l = l0 + lane;
    int d = 0;
    if (l < Nc) {
      const uint32_t v = P.comp_nodes[nbeg + l];
      const uint32_t rs = P.row_ptr[v];
      d = (int)(P.row_ptr[v + 1] - rs);
      C.node[l] = v;
      rowstart[l] = rs;
      double p0 = P.positions[2 * (size_t)v], p1 = P.positions[2 * (size_t)v + 1];
      if (!P.is_root[v]) {  // IterationZero: x <- Plus(x, 0) projects the start point
        p0 = fmin(fmax(p0, -K.bound), K.bound);
        p1 = fmin(fmax(p1, -K.bound), K.bound);
      }
      C.x[2 * l] = p0;
      C.x[2 * l + 1] = p1;
    }
    const int inc = warp_incl_scan(d, lane);
    if (l < Nc) candptr[l] = run + inc - d;
    run += __shfl_sync(kFull, inc, 31);
  }
  if (lane == 0) candptr[Nc] = run;
  __syncwarp();
  const int Eup = run;
  // keep same-track (Cauchy) and same-component (Tukey) out-edges; drop blocks
  // whose two ends are both constant (Ceres removes them, A.1)
  int kept = 0;
  for (int k0 = 0; k0 < Eup; k0 += 32) {
    const int k = k0 + lane;
    bool keep = false;
    uint32_t e = 0, mt = 0;
    if (k < Eup) {
      int lo = 0, hi = Nc - 1;
      while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if ((int)candptr[mid] <= k) lo = mid; else hi = mid - 1;
      }
      e = rowstart[lo] + (uint32_t)(k - (int)candptr[lo]);
      const uint32_t v = C.node[lo];
      const uint32_t dst = __float_as_uint(__ldg(&P.edges[5 * (size_t)e + 4].w));
      if (dst >= P.n_nodes || dst == v) {
        *P.err_flag = 1;  // malformed input: reported by the host as LFR_EINVAL
      } else {
        int kind = LFR_EDGE_SKIP;
        if (P.track[v] == P.track[dst]) kind = LFR_EDGE_CAUCHY;          // solve.cc:105
        else if (P.comp[v] == P.comp[dst]) kind = LFR_EDGE_TUKEY;        // solve.cc:114
        keep = (kind != LFR_EDGE_SKIP) && !(P.is_root[v] && P.is_root[dst]);
        mt = (uint32_t)lo | (P.local_of[dst] << 12) | ((uint32_t)kind << 24);
      }
    }
    const unsigned m = __ballot_sync(kFull, keep);
    if (keep) {
      const int pos = kept + __popc(m & ((1u << lane) - 1u));
      C.eidx[pos] = e;
      C.meta[pos] = mt;
    }
    kept += __popc(m);
  }
  __syncwarp();
  const int Ec = kept;
  C.Ec = Ec;
  // out/in edge ranges per node, free-variable numbering
  int orun = 0, irun = 0, frun = 0;
  for (int l0 = 0; l0 < Nc; l0 += 32) {
    const int l = l0 + lane;
    int co = 0, ci = 0;
    for (int j = 0; j < Ec; ++j) {
      const uint32_t mt = C.meta[j];
      co += ((int)(mt & 0xfff) == l);
      ci += ((int)((mt >> 12) & 0xfff) == l);
    }
    if (l >= Nc) co = ci = 0;
    const int so = warp_incl_scan(co, lane), si = warp_incl_scan(ci, lane);
    const bool is_free = (l < Nc) && (co + ci > 0) && !P.is_root[C.node[l < Nc ? l : 0]];
    const int sf = warp_incl_scan(is_free ? 1 : 0, lane);
    if (l < Nc) {
      C.outptr[l] = (uint16_t)(orun + so - co);
      C.inptr[l] = (uint16_t)(irun + si - ci);
      C.freeof[l] = is_free ? (int16_t)(frun + sf - 1) : (int16_t)-1;
      if (is_free) C.lof[frun + sf - 1] = (uint16_t)l;
    }
    orun += __shfl_sync(kFull, so, 31);
    irun += __shfl_sync(kFull, si, 31);
    frun += __shfl_sync(kFull, sf, 31);
  }
  if (lane == 0) {
    C.outptr[Nc] = (uint16_t)orun;
    C.inptr[Nc] = (uint16_t)irun;
  }
  __syncwarp();
  for (int l0 = 0; l0 < Nc; l0 += 32) {
    const int l = l0 + lane;
    int w = (l < Nc) ? C.inptr[l] : 0;
    for (int j = 0; j < Ec; ++j)
      if (l < Nc && (int)((C.meta[j] >> 12) & 0xfff) == l) C.inlist[w++] = (uint16_t)j;
  }
  const int nf = frun;
  C.nf = nf;
  C.n = 2 * nf;
  __syncwarp();
  if (lane == 0) P.st_kept[c] = (uint32_t)Ec;
  if (nf == 0) {  // "No non-constant parameter blocks found."
    if (lane == 0) {
      P.st_iter[c] = 0;
      P.st_term[c] = LFR_TERM_EMPTY;
      P.st_cost0[c] = 0.0;
      P.st_cost1[c] = 0.0;
      P.st_ls[c] = 0;
    }
    return;
  }

  LFR_TICK(cyc_setup);
  // ---- iteration 0 -----------------------------------------------------------------
  double cost = eval_pass(C, C.x, K);
  LFR_TICK(cyc_eval);
  double gmax = assemble(C, true, K);
  LFR_TICK(cyc_asm);
  const double cost0 = cost;
  double radius = K.radius0, nu = 2.0;
  int iter = 0, n_invalid = 0, term = LFR_TERM_NO_CONVERGENCE;
  unsigned ls_steps = 0;
  bool success = true;
  auto free_norm = [&](const double* a, const double* b) {  // |a - b|_2 over free coordinates (b may be null)
    double acc = 0.0;
    for (int i = lane; i < C.n; i += 32) {
      const int l = C.lof[i >> 1];
      const double v = a[2 * l + (i & 1)] - (b ? b[2 * l + (i & 1)] : 0.0);
      acc += v * v;
    }
    const double r = sqrt(warp_sum(acc));
    __syncwarp();  // reads above are ordered before later writes of x (shuffles are not a memory barrier)
    return r;
  };
  double x_norm = free_norm(C.x, nullptr);

  // ---- trust-region loop (A.6) ---------------------------------------------------------
  for (;;) {
    if (iter >= K.max_iter) { term = LFR_TERM_NO_CONVERGENCE; break; }
    if (success && gmax <= K.g_tol) { term = LFR_TERM_GRADIENT_TOL; break; }
    if (radius <= K.radius_min) { term = LFR_TERM_MIN_RADIUS; break; }
    ++iter;
    success = false;
    double model_change = 0.0;
    LFR_TICK(cyc_ls);
    bool valid = lm_step(C, radius, K, &model_change);
    LFR_TICK(cyc_lm);
    valid = valid && (model_change > 0.0);
    if (!valid) {
      if (++n_invalid >= K.max_invalid) { term = LFR_TERM_FAILURE; break; }
      radius /= nu;
      nu *= 2.0;
      continue;
    }
    n_invalid = 0;
    // projected Armijo line search along dl (bounds-constrained problem, A.7b)
    double gd = 0.0, dmax = 0.0;
    for (int i = lane; i < C.n; i += 32) {
      gd += C.g[i] * C.dl[i];
      dmax = fmax(dmax, fabs(C.dl[i]));
    }
    gd = warp_sum(gd);
    dmax = warp_max(dmax);
    LFR_TICK(cyc_ls);
    make_candidate(C, 1.0, K);
    double cost_c = eval_pass(C, C.xc, K);
    LFR_TICK(cyc_eval);
    bool c_valid = isfinite(cost_c);
    if (!c_valid || cost_c > cost + K.ls_suff * gd * 1.0) {
      LsSample initial{0.0, cost, gd, true, true};
      LsSample previous{0.0, 0.0, 0.0, false, false};
      LsSample current{1.0, cost_c, 0.0, c_valid, false};
      if (c_valid) {
        current.gradient = staged_grad_dot(C);
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
        make_candidate(C, step, K);
        cost_c = eval_pass(C, C.xc, K);
        c_valid = isfinite(cost_c);
        current = LsSample{step, cost_c, 0.0, c_valid, false};
        if (c_valid) {
          current.gradient = staged_grad_dot(C);
          current.gradient_valid = isfinite(current.gradient);
        }
        if (c_valid && !(cost_c > cost + K.ls_suff * gd * step)) { ls_ok = true; break; }
      }
      if (ls_ok) {
        for (int i = lane; i < C.n; i += 32) C.dl[i] *= current.x;
        __syncwarp();
      } else {  // line search failed: delta unchanged, candidate = P(x + delta)
        make_candidate(C, 1.0, K);
        cost_c = eval_pass(C, C.xc, K);
        c_valid = isfinite(cost_c);
      }
    }
    if (!c_valid) cost_c = 1.7976931348623157e308;
    const double step_norm = free_norm(C.x, C.xc);
    if (step_norm <= K.p_tol * (x_norm + K.p_tol)) { term = LFR_TERM_PARAMETER_TOL; break; }
    if (fabs(cost - cost_c) <= K.f_tol * cost) { term = LFR_TERM_FUNCTION_TOL; break; }
    const double rho = (cost - cost_c) / model_change;
    if (rho > K.min_rel_decrease) {
      for (int i = lane; i < 2 * Nc; i += 32) C.x[i] = C.xc[i];
      __syncwarp();
      x_norm = free_norm(C.x, nullptr);
      cost = cost_c;
      LFR_TICK(cyc_ls);
      gmax = assemble(C, false, K);
      LFR_TICK(cyc_asm);
      success = true;
      const double t = 2.0 * rho - 1.0;
      radius = fmin(K.radius_max, radius / fmax(1.0 / 3.0, 1.0 - t * t * t));
      nu = 2.0;
    } else {
      radius /= nu;
      nu *= 2.0;
    }
  }
  // ---- write back the last accepted x ---------------------------------------------------
  // (not after FAILURE: Ceres only commits a usable solution, solver.cc Minimize / IsSolutionUsable)
  if (term != LFR_TERM_FAILURE) {
    for (int i = lane; i < C.n; i += 32) {
      const int l = C.lof[i >> 1];
      P.positions_out[2 * (size_t)C.node[l] + (i & 1)] = C.x[2 * l + (i & 1)];
    }
  }
  if (lane == 0) {
    P.st_iter[c] = iter;
    P.st_term[c] = term;
    P.st_cost0[c] = cost0;
    P.st_cost1[c] = cost;
    P.st_ls[c] = ls_steps;
    if (prof) {
      LFR_TICK(cyc_ls);
      unsigned long long* o = P.st_cycles + 8 * (size_t)c;
      o[0] = (unsigned long long)(t_mark - t_begin);
      o[1] = cyc_setup; o[2] = cyc_eval; o[3] = cyc_asm; o[4] = cyc_lm; o[5] = cyc_ls;
      unsigned smid; asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
      o[6] = (unsigned long long)smid | ((unsigned long long)ls_steps << 32); o[7] = (unsigned long long)t_begin;
    }
  }
#undef LFR_TICK
}

// node -> index inside its component's node list
__global__ void local_index_kernel(const uint32_t* comp_ptr, const uint32_t* comp_nodes,
                                   uint32_t n_components, uint32_t total, uint32_t* local_of) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  uint32_t lo = 0, hi = n_components - 1;  // largest c with comp_ptr[c] <= i
  while (lo < hi) {
    const uint32_t mid = (lo + hi + 1) >> 1;
    if (comp_ptr[mid] <= i) lo = mid; else hi = mid - 1;
  }
  local_of[comp_nodes[i]] = i - comp_ptr[lo];
}

// Test hook: the line search's step-size selection (hermite_minimizer) on caller-supplied
// samples, one warp per case (lfr_debug_ls_minimizer).  in[c] = {f0, g0, x1, f1, g1, three,
// x2, f2, g2, lo, hi}.
__global__ void ls_minimizer_kernel(const double* __restrict__ in, int n, double* __restrict__ out) {
  const int wid = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (wid >= n) return;  // whole warps leave together
  const double* s = in + 11 * (size_t)wid;
  const double x = hermite_minimizer(s[0], s[1], s[2], s[3], s[4], s[5] != 0.0, s[6], s[7], s[8], s[9], s[10], lane);
  if (lane == 0) out[wid] = x;
}

// Test hook: the line search's quartic root finders on caller-supplied polynomials,
// one warp per polynomial (lfr_debug_quartic_roots).
__global__ void quartic_roots_kernel(const double* __restrict__ coef, const double* __restrict__ lohi, int n,
                                     int use_grid, double* __restrict__ roots, int* __restrict__ counts) {
  const int wid = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (wid >= n) return;  // whole warps leave together
  const double q[5] = {coef[5 * wid], coef[5 * wid + 1], coef[5 * wid + 2], coef[5 * wid + 3], coef[5 * wid + 4]};
  double out[4] = {0.0, 0.0, 0.0, 0.0};
  const int c = use_grid ? quartic_roots_grid(q, lohi[2 * wid], lohi[2 * wid + 1], out, lane)
                         : quartic_roots_in(q, lohi[2 * wid], lohi[2 * wid + 1], out, lane);
  if (lane == 0) {
    counts[wid] = c;
    for (int k = 0; k < 4; ++k) roots[4 * wid + k] = out[k];
  }
}

// K1 test hook: one thread per edge.
__global__ void edge_eval_kernel(const float4* edges, const uint8_t* kind, uint64_t n, const double* xs,
                                 const double* xd, const DevConsts K, double* r, double* jac, double* rho) {
  const uint64_t e = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (e >= n) return;
  float4 q[5];
#pragma unroll
  for (int t = 0; t < 5; ++t) q[t] = __ldg(edges + 5 * e + t);
  const EdgeEval ev = eval_edge(q, kind[e], xs[2 * e], xs[2 * e + 1], xd[2 * e], xd[2 * e + 1], K);
  r[2 * e] = ev.r0;
  r[2 * e + 1] = ev.r1;
  jac[4 * e] = -ev.m00;
  jac[4 * e + 1] = -ev.m01;
  jac[4 * e + 2] = -ev.m10;
  jac[4 * e + 3] = -ev.m11;
  rho[3 * e] = 2.0 * ev.half_rho;
  rho[3 * e + 1] = ev.a;
  rho[3 * e + 2] = 0.0;  // rho'' is not used by the solve (always <= 0, A.3)
}

}  // namespace lfr
