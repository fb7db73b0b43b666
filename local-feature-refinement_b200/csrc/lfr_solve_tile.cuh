// lfr_solve_tile.cuh — mid-size components (32 < n <= 80 unknowns: e.g. the
// 17..41-node components of an ETH3D-courtyard-scale scene): one CTA of T = 64
// or 128 threads solves one component.  Same scheme as the register warp kernel
// (lfr_solve_warp2.cuh) with the warp widened to a tile: thread i owns row i of
// the damped normal matrix in registers (Gauss-Jordan, pivot row broadcast
// through shared memory), evaluation is edge-parallel over T threads, assembly
// combines each directed edge with its twin.  Warp 0 performs the setup
// (ballot compaction), then the tile works in lock step with __syncthreads().
#pragma once
#include "lfr_solve_warp2.cuh"

namespace lfr {

struct TileLayout {
  int stage, bar;
  int x, xc, g, S, dl, H, scr, tup, prow, red, hdr;
  int eidx, meta, node, rowstart, candptr, cnt;
  int twin, outptr, freeof, lof;
  int ldh, total;
  __host__ __device__ TileLayout(int emax, int ncmax, int n2max) {
    ldh = n2max | 1;
    int o = 0;
    stage = o; o += 80 * emax;   // staged edge records (see Warp2Layout)
    bar = o; o += 16;
    x = o; o += 16 * ncmax;
    xc = o; o += 16 * ncmax;
    g = o; o += 8 * n2max;
    S = o; o += 8 * n2max;
    dl = o; o += 8 * n2max;
    H = o; o += 8 * n2max * ldh;
    // scr (7 doubles per candidate edge: the staged evaluation) and tup (5: the assembly tuples), 96 of
    // 186 bytes per edge.  Moving them to a per-CTA global area was measured on cfg4
    // (profiles/r02_tile_tier_occupancy.txt): 1.4x the resident components, each 1.3x slower -> same time.
    scr = o; o += 8 * 7 * emax;
    tup = o; o += 8 * 5 * emax;
    o = align_up(o, 16);
    prow = o; o += 8 * 4 * 84;   // double-buffered pair of pivot rows: 2 x 2 x (80 columns, rhs, spare)
    red = o; o += 8 * 3 * 4;     // block reductions (<= 4 warps)
    hdr = o; o += 16;            // Ec, nf, irregular broadcast by warp 0
    eidx = o; o += 4 * emax;
    meta = o; o += 4 * emax;
    node = o; o += 4 * ncmax;
    rowstart = o; o += 4 * ncmax;
    candptr = o; o += 4 * (ncmax + 1);
    cnt = o; o += 4 * 2 * ncmax;
    twin = o; o += 2 * emax;
    outptr = o; o += 2 * (ncmax + 1);
    freeof = o; o += 2 * ncmax;
    lof = o; o += 2 * (n2max / 2 + 1);
    total = align_up(o, 16);
  }
};

template <int T>
struct TileCtx {
  int tid, Nc, Ec, nf, n, emax, ldh;
  bool irregular;
  double *x, *xc, *g, *S, *dl, *H, *scr, *tup, *prow, *red;
  uint32_t *eidx, *meta, *node;
  uint16_t *twin, *outptr, *lof;
  int16_t* freeof;
  float4* stage;
  uint64_t* bar;
};

template <int T>
__device__ __forceinline__ void tile_sum3(const TileCtx<T>& C, double& a, double& b, double& c) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_xor_sync(kFull, a, o);
    b += __shfl_xor_sync(kFull, b, o);
    c += __shfl_xor_sync(kFull, c, o);
  }
  constexpr int NW = T / 32;
  const int w = C.tid >> 5;
  __syncthreads();
  if ((C.tid & 31) == 0) {
    C.red[w] = a;
    C.red[NW + w] = b;
    C.red[2 * NW + w] = c;
  }
  __syncthreads();
  a = b = c = 0.0;
#pragma unroll
  for (int i = 0; i < NW; ++i) {
    a += C.red[i];
    b += C.red[NW + i];
    c += C.red[2 * NW + i];
  }
}
template <int T>
__device__ __forceinline__ double tile_max(const TileCtx<T>& C, double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(kFull, v, o));
  constexpr int NW = T / 32;
  __syncthreads();
  if ((C.tid & 31) == 0) C.red[C.tid >> 5] = v;
  __syncthreads();
  v = C.red[0];
#pragma unroll
  for (int i = 1; i < NW; ++i) v = fmax(v, C.red[i]);
  return v;
}

// DIRDERIV: also grad f(xe) . dl, per edge from the same evaluation (see eval_pass2)
template <int T, bool DIRDERIV>
__device__ __forceinline__ double tile_eval(const TileCtx<T>& C, const double* xe, const DevConsts& K,
                                            double* dphi = nullptr) {
  double cost = 0.0, z1 = 0.0, z2 = 0.0;
  for (int j = C.tid; j < C.Ec; j += T) {
    const uint32_t mt = C.meta[j];
    const int s = mt & 0xfff, d = (mt >> 12) & 0xfff, kind = mt >> 24;
    const float4* qp = C.stage + 5 * C.eidx[j];
    float4 q[5];
#pragma unroll
    for (int t = 0; t < 5; ++t) q[t] = qp[t];
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
    if (DIRDERIV) {
      const int fs = C.freeof[s], fd = C.freeof[d];
      const double s0 = fs >= 0 ? C.dl[2 * fs] : 0.0, s1 = fs >= 0 ? C.dl[2 * fs + 1] : 0.0;
      const double d0 = fd >= 0 ? C.dl[2 * fd] : 0.0, d1 = fd >= 0 ? C.dl[2 * fd + 1] : 0.0;
      z1 += ev.a * (ev.r0 * (d0 - (ev.m00 * s0 + ev.m01 * s1)) + ev.r1 * (d1 - (ev.m10 * s0 + ev.m11 * s1)));
    }
  }
  tile_sum3(C, cost, z1, z2);  // (its barriers also publish the staged values)
  if (DIRDERIV) *dphi = z1;
  return cost;
}

template <int T, bool GRAD_ONLY>
__device__ __forceinline__ double tile_assemble(const TileCtx<T>& C, bool first, const DevConsts& K) {
  const int E = C.emax, ldh = C.ldh;
  if (!GRAD_ONLY) {
    for (int i = C.tid; i < C.n * ldh; i += T) C.H[i] = 0.0;
    __syncthreads();
  }
  if (!C.irregular) {
    for (int e = C.tid; e < C.Ec; e += T) {
      const uint32_t mt = C.meta[e];
      const int fs = C.freeof[mt & 0xfff], fd = C.freeof[(mt >> 12) & 0xfff];
      const int t = C.twin[e];
      const double a = C.scr[e], r0 = C.scr[E + e], r1 = C.scr[2 * E + e];
      const double m00 = C.scr[3 * E + e], m01 = C.scr[4 * E + e], m10 = C.scr[5 * E + e], m11 = C.scr[6 * E + e];
      const double at = C.scr[t], rt0 = C.scr[E + t], rt1 = C.scr[2 * E + t];
      C.tup[3 * E + e] = at * rt0 - a * (m00 * r0 + m10 * r1);
      C.tup[4 * E + e] = at * rt1 - a * (m01 * r0 + m11 * r1);
      if (!GRAD_ONLY) {
        C.tup[e] = a * (m00 * m00 + m10 * m10) + at;
        C.tup[E + e] = a * (m00 * m01 + m10 * m11);
        C.tup[2 * E + e] = a * (m01 * m01 + m11 * m11) + at;
        if (fs >= 0 && fd >= 0) {
          const double t00 = C.scr[3 * E + t], t01 = C.scr[4 * E + t], t10 = C.scr[5 * E + t], t11 = C.scr[6 * E + t];
          double* h0 = C.H + (2 * fs) * ldh + 2 * fd;
          h0[0] = -a * m00 - at * t00;
          h0[1] = -a * m10 - at * t01;
          h0[ldh] = -a * m01 - at * t10;
          h0[ldh + 1] = -a * m11 - at * t11;
        }
      }
    }
    __syncthreads();
  }
  double acc = 0.0, gmax = 0.0;
  if (!C.irregular) {
    for (int f = C.tid; f < C.nf; f += T) {
      const int l = C.lof[f];
      double d00 = 0., d01 = 0., d11 = 0., g0 = 0., g1 = 0.;
      for (int j = C.outptr[l]; j < C.outptr[l + 1]; ++j) {
        g0 += C.tup[3 * E + j];
        g1 += C.tup[4 * E + j];
        if (!GRAD_ONLY) {
          d00 += C.tup[j];
          d01 += C.tup[E + j];
          d11 += C.tup[2 * E + j];
        }
      }
      if (GRAD_ONLY) {
        acc += g0 * C.dl[2 * f] + g1 * C.dl[2 * f + 1];
      } else {
        double* hd = C.H + (2 * f) * ldh + 2 * f;
        hd[0] = d00;
        hd[1] = d01;
        hd[ldh] = d01;
        hd[ldh + 1] = d11;
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
  } else {
    if (C.tid == 0) {  // serial path for inputs without clean edge twins
      for (int i = 0; i < C.n; ++i) C.g[i] = 0.0;
      for (int e = 0; e < C.Ec; ++e) {
        const uint32_t mt = C.meta[e];
        const int fs = C.freeof[mt & 0xfff], fd = C.freeof[(mt >> 12) & 0xfff];
        const double a = C.scr[e], r0 = C.scr[E + e], r1 = C.scr[2 * E + e];
        const double m00 = C.scr[3 * E + e], m01 = C.scr[4 * E + e], m10 = C.scr[5 * E + e], m11 = C.scr[6 * E + e];
        if (fs >= 0) {
          C.g[2 * fs] -= a * (m00 * r0 + m10 * r1);
          C.g[2 * fs + 1] -= a * (m01 * r0 + m11 * r1);
          if (!GRAD_ONLY) {
            double* hd = C.H + (2 * fs) * ldh + 2 * fs;
            hd[0] += a * (m00 * m00 + m10 * m10);
            hd[1] += a * (m00 * m01 + m10 * m11);
            hd[ldh] += a * (m00 * m01 + m10 * m11);
            hd[ldh + 1] += a * (m01 * m01 + m11 * m11);
          }
        }
        if (fd >= 0) {
          C.g[2 * fd] += a * r0;
          C.g[2 * fd + 1] += a * r1;
          if (!GRAD_ONLY) {
            C.H[(2 * fd) * ldh + 2 * fd] += a;
            C.H[(2 * fd + 1) * ldh + 2 * fd + 1] += a;
          }
        }
        if (!GRAD_ONLY && fs >= 0 && fd >= 0) {
          double* h0 = C.H + (2 * fs) * ldh + 2 * fd;
          double* h1 = C.H + (2 * fd) * ldh + 2 * fs;
          h0[0] -= a * m00; h0[1] -= a * m10; h0[ldh] -= a * m01; h0[ldh + 1] -= a * m11;
          h1[0] -= a * m00; h1[1] -= a * m01; h1[ldh] -= a * m10; h1[ldh + 1] -= a * m11;
        }
      }
    }
    __syncthreads();
    for (int i = C.tid; i < C.n; i += T) {
      if (GRAD_ONLY) {
        acc += C.g[i] * C.dl[i];
      } else {
        if (first) C.S[i] = 1.0 / (1.0 + sqrt(C.H[i * ldh + i]));
        const int l = C.lof[i >> 1];
        const double xi = C.x[2 * l + (i & 1)];
        const double p = fmin(fmax(xi - C.g[i], -K.bound), K.bound);
        gmax = fmax(gmax, fabs(xi - p));
      }
    }
  }
  if (GRAD_ONLY) {
    double z1 = 0.0, z2 = 0.0;
    tile_sum3(C, acc, z1, z2);
    return acc;
  }
  return tile_max(C, gmax);
}

// Gauss-Jordan with thread i <-> row i (n <= NREG <= T).
template <int T, int NREG>
__device__ __forceinline__ bool tile_lm_step(const TileCtx<T>& C, double radius, const DevConsts& K,
                                             double* model_change, double* gd, double* dmax) {
  const int n = C.n, i = C.tid;
  const bool act = i < n;
  const double si = act ? C.S[i] : 0.0;
  const double gi = act ? C.g[i] : 0.0;
  const double* Hi = C.H + (act ? i : 0) * C.ldh;
  const double hii = act ? Hi[i] * si * si : 1.0;
  const double d2 = act ? fmin(fmax(hii, K.min_diag), K.max_diag) / radius : 0.0;
  double a[NREG];
#pragma unroll
  for (int k = 0; k < NREG; ++k) {
    double v = 0.0;
    if (k < n && act) v = Hi[k] * si * C.S[k];
    if (k == i) v = act ? v + d2 : 1.0;
    a[k] = v;
  }
  const double b0 = si * gi;
  double b = b0;
  bool ok = true;
  // 2x2 block pivots (see lm_step2 in lfr_solve_warp2.cuh): threads j, j+1 publish
  // their raw rows, every thread inverts the pivot block itself; half as many
  // block-wide barriers as scalar pivots.
  constexpr int R = 84;
  double inv0 = 0.0, inv1 = 0.0;
  for (int j = 0; j < n; j += 2) {
    double* buf = C.prow + ((j >> 1) & 1) * (2 * R);
    if (i == j || i == j + 1) {
      double* row = buf + (i - j) * R;
      double2* row2 = reinterpret_cast<double2*>(row);
#pragma unroll
      for (int k = 0; k < NREG; k += 2) row2[k / 2] = make_double2(a[k], a[k + 1]);
      row[NREG] = b;
    }
    __syncthreads();
    const double2* r0 = reinterpret_cast<const double2*>(buf);
    const double2* r1 = reinterpret_cast<const double2*>(buf + R);
    const double2 p0 = r0[0], p1 = r1[0];
    const double bj0 = buf[NREG], bj1 = buf[R + NREG];
    const double det = p0.x * p1.y - p0.y * p1.x;
    ok = ok && (p0.x > 0.0) && (det > 0.0) && isfinite(det);
    const double rdet = 1.0 / det;
    const bool piv_thread = (i == j) || (i == j + 1);
    if (i == j) { inv0 = p1.y * rdet; inv1 = -p0.y * rdet; }
    if (i == j + 1) { inv0 = -p1.x * rdet; inv1 = p0.x * rdet; }
    const double f0 = piv_thread ? 0.0 : (a[0] * p1.y - a[1] * p1.x) * rdet;
    const double f1 = piv_thread ? 0.0 : (a[1] * p0.x - a[0] * p0.y) * rdet;
#pragma unroll
    for (int k0 = 2; k0 < NREG; k0 += 4) {  // two 128-bit words of each row per group
      double2 u[2], v[2];
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        if (k0 + 2 * q < NREG) { u[q] = r0[k0 / 2 + q]; v[q] = r1[k0 / 2 + q]; }
      }
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        const int k = k0 + 2 * q;
        if (k < NREG) {
          a[k - 2] = a[k] - f0 * u[q].x - f1 * v[q].x;
          a[k - 1] = a[k + 1] - f0 * u[q].y - f1 * v[q].y;
        }
      }
    }
    a[NREG - 2] = 0.0;
    a[NREG - 1] = 0.0;
    b -= f0 * bj0 + f1 * bj1;
  }
  const double bp = __shfl_xor_sync(0xffffffffu, b, 1);
  const double y = (i & 1) ? inv0 * bp + inv1 * b : inv0 * b + inv1 * bp;
  double mc = 0.0, dot = 0.0, bad = 0.0, mx = 0.0;
  if (act) {
    const double d = -si * y;
    C.dl[i] = d;
    mc = y * (b0 + d2 * y);
    dot = gi * d;
    mx = fabs(d);
    if (!isfinite(y)) bad = 1.0;
  }
  tile_sum3(C, mc, dot, bad);
  mx = tile_max(C, mx);
  *model_change = 0.5 * mc;
  *gd = dot;
  *dmax = mx;
  return ok && bad == 0.0;
}

template <int T>
__device__ __forceinline__ void tile_candidate(const TileCtx<T>& C, double alpha, const DevConsts& K) {
  for (int i = C.tid; i < 2 * C.Nc; i += T) {
    const int f = C.freeof[i >> 1];
    double v = C.x[i];
    if (f >= 0) v = fmin(fmax(v + alpha * C.dl[2 * f + (i & 1)], -K.bound), K.bound);
    C.xc[i] = v;
  }
  __syncthreads();
}

template <int T, int NREG>
__global__ void __launch_bounds__(T)
solve_tile_kernel(const DevProblem P, const DevConsts K, const WarpBucket B) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int tid = threadIdx.x, lane = tid & 31;
  const uint32_t c = B.list[blockIdx.x];
  unsigned char* base = smem_raw;
  const TileLayout L(B.emax, B.ncmax, B.n2max);
  TileCtx<T> C;
  C.tid = tid;
  C.emax = B.emax;
  C.ldh = L.ldh;
  C.x = (double*)(base + L.x);
  C.xc = (double*)(base + L.xc);
  C.g = (double*)(base + L.g);
  C.S = (double*)(base + L.S);
  C.dl = (double*)(base + L.dl);
  C.H = (double*)(base + L.H);
  C.scr = (double*)(base + L.scr);
  C.tup = (double*)(base + L.tup);
  C.prow = (double*)(base + L.prow);
  C.red = (double*)(base + L.red);
  int* hdr = (int*)(base + L.hdr);
  C.eidx = (uint32_t*)(base + L.eidx);
  C.meta = (uint32_t*)(base + L.meta);
  C.node = (uint32_t*)(base + L.node);
  uint32_t* rowstart = (uint32_t*)(base + L.rowstart);
  uint32_t* candptr = (uint32_t*)(base + L.candptr);
  int* cnt = (int*)(base + L.cnt);
  C.twin = (uint16_t*)(base + L.twin);
  C.outptr = (uint16_t*)(base + L.outptr);
  C.freeof = (int16_t*)(base + L.freeof);
  C.lof = (uint16_t*)(base + L.lof);
  C.stage = (float4*)(base + L.stage);
  C.bar = (uint64_t*)(base + L.bar);

  const int Nc = (int)(P.comp_ptr[c + 1] - P.comp_ptr[c]);
  C.Nc = Nc;
  long long t_begin = 0, t_lm = 0, t_mark = 0;
  if (P.st_cycles) t_begin = clock64();
  if (P.st_times && tid == 0) {
    unsigned long long ns;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
    P.st_times[2 * (size_t)c] = ns;
  }
  // ---- setup by warp 0 (solve.cc:98-143), shared with the warp kernel -----------------------
  if (tid < 32) {
    int Ec = 0, nf = 0;
    bool irregular = false;
    warp_setup(C, rowstart, candptr, cnt, B.ncmax, P, K, c, lane, &Ec, &nf, &irregular);
    if (lane == 0) {
      hdr[0] = Ec;
      hdr[1] = nf;
      hdr[2] = irregular ? 1 : 0;
      P.st_kept[c] = (uint32_t)Ec;
    }
  }
  __syncthreads();
  C.Ec = hdr[0];
  C.nf = hdr[1];
  C.n = 2 * C.nf;
  C.irregular = hdr[2] != 0;
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

  double cost = tile_eval<T, false>(C, C.x, K);
  double gmax = tile_assemble<T, false>(C, true, K);
  const double cost0 = cost;
  double radius = K.radius0, nu = 2.0;
  int iter = 0, n_invalid = 0, term = LFR_TERM_NO_CONVERGENCE;
  unsigned ls_steps = 0;
  bool success = true;
  double x_norm;
  {
    double a = 0.0, z1 = 0.0, z2 = 0.0;
    for (int i = tid; i < C.n; i += T) {
      const int l = C.lof[i >> 1];
      const double xv = C.x[2 * l + (i & 1)];
      a += xv * xv;
    }
    tile_sum3(C, a, z1, z2);
    x_norm = sqrt(a);
  }
  for (;;) {
    if (iter >= K.max_iter) { term = LFR_TERM_NO_CONVERGENCE; break; }
    if (success && gmax <= K.g_tol) { term = LFR_TERM_GRADIENT_TOL; break; }
    if (radius <= K.radius_min) { term = LFR_TERM_MIN_RADIUS; break; }
    ++iter;
    success = false;
    double model_change = 0.0, gd = 0.0, dmax = 0.0;
    if (P.st_cycles) t_mark = clock64();
    bool valid = tile_lm_step<T, NREG>(C, radius, K, &model_change, &gd, &dmax);
    if (P.st_cycles) t_lm += clock64() - t_mark;
    valid = valid && (model_change > 0.0);
    if (!valid) {
      if (++n_invalid >= K.max_invalid) { term = LFR_TERM_FAILURE; break; }
      radius /= nu;
      nu *= 2.0;
      continue;
    }
    n_invalid = 0;
    tile_candidate(C, 1.0, K);
    double cost_c = tile_eval<T, false>(C, C.xc, K);
    bool c_valid = isfinite(cost_c);
    if (!c_valid || cost_c > cost + K.ls_suff * gd * 1.0) {
      LsSample initial{0.0, cost, gd, true, true};
      LsSample previous{0.0, 0.0, 0.0, false, false};
      LsSample current{1.0, cost_c, 0.0, c_valid, false};
      if (c_valid) {
        current.gradient = tile_assemble<T, true>(C, false, K);
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
        tile_candidate(C, step, K);
        double dphi;
        cost_c = tile_eval<T, true>(C, C.xc, K, &dphi);
        c_valid = isfinite(cost_c);
        current = LsSample{step, cost_c, 0.0, c_valid, false};
        if (c_valid) {
          current.gradient = dphi;
          current.gradient_valid = isfinite(dphi);
        }
        if (c_valid && !(cost_c > cost + K.ls_suff * gd * step)) { ls_ok = true; break; }
      }
      if (ls_ok) {
        for (int i = tid; i < C.n; i += T) C.dl[i] *= current.x;
        __syncthreads();
      } else {
        tile_candidate(C, 1.0, K);
        cost_c = tile_eval<T, false>(C, C.xc, K);
        c_valid = isfinite(cost_c);
      }
    }
    if (!c_valid) cost_c = 1.7976931348623157e308;
    double dn2 = 0.0, z1 = 0.0, z2 = 0.0;
    for (int i = tid; i < C.n; i += T) {
      const int l = C.lof[i >> 1];
      const double dv = C.x[2 * l + (i & 1)] - C.xc[2 * l + (i & 1)];
      dn2 += dv * dv;
    }
    tile_sum3(C, dn2, z1, z2);
    const double step_norm = sqrt(dn2);
    if (step_norm <= K.p_tol * (x_norm + K.p_tol)) { term = LFR_TERM_PARAMETER_TOL; break; }
    if (fabs(cost - cost_c) <= K.f_tol * cost) { term = LFR_TERM_FUNCTION_TOL; break; }
    const double rho = (cost - cost_c) / model_change;
    if (rho > K.min_rel_decrease) {
      double a2 = 0.0;
      z1 = z2 = 0.0;
      for (int i = tid; i < 2 * Nc; i += T) {
        const double v = C.xc[i];
        C.x[i] = v;
        if (C.freeof[i >> 1] >= 0) a2 += v * v;
      }
      tile_sum3(C, a2, z1, z2);
      x_norm = sqrt(a2);
      cost = cost_c;
      gmax = tile_assemble<T, false>(C, false, K);
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
    for (int i = tid; i < C.n; i += T) {
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
      o[2] = o[3] = o[5] = 0;
      o[0] = (unsigned long long)(clock64() - t_begin);
      o[4] = (unsigned long long)t_lm;  // of which in the linear solves
      o[1] = 2;  // marks a tile-tier component
      o[6] = (unsigned long long)ls_steps << 32;
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

}  // namespace lfr
