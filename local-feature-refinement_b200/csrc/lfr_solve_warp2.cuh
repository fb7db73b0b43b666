// lfr_solve_warp2.cuh — latency-optimised warp-per-component solve for
// components with <= 32 unknowns (all of the exhaustive-pair configs: a
// component has at most #images nodes, solve.cc:586).
//
// A solve of a Fountain-scale graph is a few thousand independent, strictly
// sequential LM trajectories; its duration is the latency of the slowest one,
// not bandwidth.  Compared with lfr_solve_warp.cuh (kept for 32 < n <= 64) this
// kernel shortens every dependent chain of one LM iteration:
//
//   * assembly is edge-parallel: each lane combines its directed edge with its
//     twin (the reverse edge, found once at setup) into the complete 2x2
//     off-diagonal block of the normal matrix and a 5-value contribution to its
//     source node's diagonal block / gradient; a node lane then adds its <= deg
//     contributions.  One owner per written word => no atomics, reproducible.
//   * the damped normal equations are solved in REGISTERS: lane i holds row i of
//     (S H S + D^2 | S g) and the warp runs a Gauss-Jordan elimination, the pivot
//     row broadcast through one shared-memory line (one reciprocal per pivot, no
//     square roots, no back substitution).  For an SPD matrix the pivots
//     are the LDL^T pivots, so "pivot <= 0" is exactly the Cholesky failure test.
//   * warp reductions are batched (several values per butterfly).
//
// Inputs whose edges do not come in (src->dst, dst->src) pairs, or that repeat a
// pair, are still solved (a serial assembly path), just slower.
#pragma once
#include "lfr_solve_warp.cuh"

namespace lfr {

struct Warp2Layout {
  int stage, bar;                                   // staged 80-byte edge records (float4 x 5 each), mbarrier
  int x, xc, g, S, dl, H, scr, tup, prow;           // doubles (byte offsets)
  int eidx, meta, node, rowstart, candptr, cnt;     // u32 / i32
  int twin, outptr, freeof, lof;                    // u16 / i16
  int ldh, total;
  __host__ __device__ Warp2Layout(int emax, int ncmax, int n2max) {
    ldh = n2max | 1;  // odd row stride (in doubles): lanes reading one column hit distinct banks
    int o = 0;
    stage = o; o += 80 * emax;  // 16-byte aligned: destination of the bulk copies
    bar = o; o += 16;
    x = o; o += 16 * ncmax;
    xc = o; o += 16 * ncmax;
    g = o; o += 8 * n2max;
    S = o; o += 8 * n2max;
    dl = o; o += 8 * n2max;
    H = o; o += 8 * n2max * ldh;
    scr = o; o += 8 * 7 * emax;
    tup = o; o += 8 * 5 * emax;
    o = align_up(o, 16);
    prow = o; o += 8 * 2 * 72;  // double-buffered pivot rows of the elimination: 2 rows x (32 columns, rhs, spare)
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

struct Warp2Ctx {
  int lane, Nc, Ec, nf, n, emax, ldh;
  bool irregular;
  double *x, *xc, *g, *S, *dl, *H, *scr, *tup, *prow;
  int prow_stride;
  uint32_t *eidx, *meta, *node;
  uint16_t *twin, *outptr, *lof;
  int16_t* freeof;
  float4* stage;   // this component's candidate out-edge records in shared memory, 5 x float4 each
  uint64_t* bar;   // mbarrier the bulk copies complete on
};

// ---- TMA 1-D bulk copy global -> shared, completion on an mbarrier (sm_90+; here sm_100a) -------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");  // make the init visible to the async proxy
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_copy_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  } while (!done);
}

template <int N>
__device__ __forceinline__ void warp_sum_n(double (&v)[N]) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    double t[N];
#pragma unroll
    for (int k = 0; k < N; ++k) t[k] = __shfl_xor_sync(kFull, v[k], o);
#pragma unroll
    for (int k = 0; k < N; ++k) v[k] += t[k];
  }
}

__device__ __forceinline__ void warp_sum2_max1(double& s0, double& s1, double& m0) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double a = __shfl_xor_sync(kFull, s0, o), b = __shfl_xor_sync(kFull, s1, o),
                 c = __shfl_xor_sync(kFull, m0, o);
    s0 += a;
    s1 += b;
    m0 = fmax(m0, c);
  }
}
__device__ __forceinline__ void warp_sum2(double& s0, double& s1) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double a = __shfl_xor_sync(kFull, s0, o), b = __shfl_xor_sync(kFull, s1, o);
    s0 += a;
    s1 += b;
  }
}

// Lane partials of |x - xc|^2 and |xc|^2 over the free coordinates, produced where the candidate
// is formed (make_candidate2) and summed in the evaluation pass's butterfly: the parameter-tolerance
// test and the accepted point's norm cost no reduction of their own.
struct CandNorms {
  double dn2, xn2;
};

// Evaluate every kept edge at positions `xe` ([2*Nc], component-local) from the records staged in
// shared memory (five conflict-free LDS.128 per edge: 80-byte stride = 20 banks, a quarter-warp of
// 16-byte accesses covers all 32 banks once); stage {a, r, M} (7 doubles, SoA) for the assembly.
// DIRDERIV = true additionally returns phi'(alpha) = grad f(xe) . dl of the line
// search, accumulated per edge from the same evaluation:
//   grad . dl = sum_e a_e r_e^T (dl_dst - M_e dl_src)      (J_src = -M, J_dst = I)
// so a line-search trial needs no separate gradient assembly pass.
template <bool DIRDERIV, bool NORMS>
__device__ __forceinline__ double eval_pass2(const Warp2Ctx& C, const double* xe, const DevConsts& K,
                                             double* dphi = nullptr, CandNorms* nrm = nullptr) {
  double cost = 0.0, dd = 0.0;
  for (int j = C.lane; j < C.Ec; j += 32) {
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
      dd += ev.a * (ev.r0 * (d0 - (ev.m00 * s0 + ev.m01 * s1)) + ev.r1 * (d1 - (ev.m10 * s0 + ev.m11 * s1)));
    }
  }
  if (DIRDERIV && NORMS) {
    double v[4] = {cost, dd, nrm->dn2, nrm->xn2};
    warp_sum_n<4>(v);
    cost = v[0];
    *dphi = v[1];
    nrm->dn2 = v[2];
    nrm->xn2 = v[3];
  } else if (NORMS) {
    double v[3] = {cost, nrm->dn2, nrm->xn2};
    warp_sum_n<3>(v);
    cost = v[0];
    nrm->dn2 = v[1];
    nrm->xn2 = v[2];
  } else if (DIRDERIV) {
    warp_sum2(cost, dd);
    *dphi = dd;
  } else {
    cost = warp_sum(cost);
  }
  __syncwarp();
  return cost;
}

// From the staged evaluation: GRAD_ONLY = false -> H (unscaled, full symmetric),
// g, on the first call the Jacobi scaling S; returns |x - P(x - g)|_inf.
// GRAD_ONLY = true -> returns grad . dl (phi'(alpha) of the line search).
template <bool GRAD_ONLY>
__device__ __forceinline__ double assemble2(const Warp2Ctx& C, bool first, const DevConsts& K) {
  const int E = C.emax, ldh = C.ldh;
  if (!GRAD_ONLY) {
    for (int i = C.lane; i < C.n * ldh; i += 32) C.H[i] = 0.0;
    __syncwarp();
  }
  if (!C.irregular) {
    for (int e = C.lane; e < C.Ec; e += 32) {
      const uint32_t mt = C.meta[e];
      const int fs = C.freeof[mt & 0xfff], fd = C.freeof[(mt >> 12) & 0xfff];
      const int t = C.twin[e];
      const double a = C.scr[e], r0 = C.scr[E + e], r1 = C.scr[2 * E + e];
      const double m00 = C.scr[3 * E + e], m01 = C.scr[4 * E + e], m10 = C.scr[5 * E + e],
                   m11 = C.scr[6 * E + e];
      const double at = C.scr[t], rt0 = C.scr[E + t], rt1 = C.scr[2 * E + t];
      // contribution of e (as out-edge of its source) and of its twin (as in-edge of the same node)
      C.tup[3 * E + e] = at * rt0 - a * (m00 * r0 + m10 * r1);
      C.tup[4 * E + e] = at * rt1 - a * (m01 * r0 + m11 * r1);
      if (!GRAD_ONLY) {
        C.tup[e] = a * (m00 * m00 + m10 * m10) + at;
        C.tup[E + e] = a * (m00 * m01 + m10 * m11);
        C.tup[2 * E + e] = a * (m01 * m01 + m11 * m11) + at;
        if (fs >= 0 && fd >= 0) {  // block (fs, fd) = -a M^T - a_t M_t
          const double t00 = C.scr[3 * E + t], t01 = C.scr[4 * E + t], t10 = C.scr[5 * E + t],
                       t11 = C.scr[6 * E + t];
          double* h0 = C.H + (2 * fs) * ldh + 2 * fd;
          h0[0] = -a * m00 - at * t00;
          h0[1] = -a * m10 - at * t01;
          h0[ldh] = -a * m01 - at * t10;
          h0[ldh + 1] = -a * m11 - at * t11;
        }
      }
    }
    __syncwarp();
  }
  double acc = 0.0, gmax = 0.0;
  if (!C.irregular) {
    for (int f = C.lane; f < C.nf; f += 32) {
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
    // serial path for inputs without clean edge twins: one lane accumulates every edge in order
    if (C.lane == 0) {
      for (int i = 0; i < C.n; ++i) C.g[i] = 0.0;
      for (int e = 0; e < C.Ec; ++e) {
        const uint32_t mt = C.meta[e];
        const int fs = C.freeof[mt & 0xfff], fd = C.freeof[(mt >> 12) & 0xfff];
        const double a = C.scr[e], r0 = C.scr[E + e], r1 = C.scr[2 * E + e];
        const double m00 = C.scr[3 * E + e], m01 = C.scr[4 * E + e], m10 = C.scr[5 * E + e],
                     m11 = C.scr[6 * E + e];
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
    __syncwarp();
    for (int i = C.lane; i < C.n; i += 32) {
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
  __syncwarp();
  if (GRAD_ONLY) return warp_sum(acc);
  return warp_max(gmax);
}

// (S H S + D^2) y = S g by Gauss-Jordan elimination with the rows in registers
// (lane i <-> row i, n <= NREG <= 32).  Writes dl = -S y; returns validity and
// {model_cost_change, g . dl, |dl|_inf}.
// NREG up to which lm_step2 eliminates with 2x2 block pivots (above: scalar pivots,
// kept for comparison; -DLFR_BLOCK_PIVOT_MAX_NREG=0 restores them everywhere)
#ifndef LFR_BLOCK_PIVOT_MAX_NREG
#define LFR_BLOCK_PIVOT_MAX_NREG 32
#endif
constexpr int kBlockPivotMaxNreg = LFR_BLOCK_PIVOT_MAX_NREG;

template <int NREG>
__device__ __forceinline__ bool lm_step2(const Warp2Ctx& C, double radius, const DevConsts& K,
                                         double* model_change, double* gd, double* dmax) {
  const int n = C.n, i = C.lane;
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
    if (k == i) v = act ? v + d2 : 1.0;  // idle lanes carry identity rows
    a[k] = v;
  }
  const double b0 = si * gi;
  double b = b0;
  bool ok = true;
  // Gauss-Jordan: the pivot lanes publish their raw rows through a double-buffered
  // shared-memory line (one broadcast LDS.128 per two elements instead of
  // shuffles); every other lane eliminates the pivot columns from its own row.
  // The register row is shifted left after every step, so the leading slots
  // always hold the current pivot columns and ONE compact loop body serves every
  // step (a fully unrolled elimination is ~100 KB of straight-line code and stalls
  // on instruction fetch).
  // No per-element guards: all NREG slots are processed every step (slots past
  // the live columns hold zeros), so the step is a straight run of 128-bit
  // shared-memory accesses and DFMAs that the scheduler can overlap freely.
  double y;
  if constexpr (NREG <= kBlockPivotMaxNreg) {
    // 2x2 block pivots (n = 2 x free nodes is even; the diagonal blocks of an SPD
    // matrix are SPD): half as many publish / synchronise / reciprocal rounds on
    // the dependent chain for the same number of DFMAs.  Lanes j, j+1 publish
    // their raw rows; every lane inverts the 2x2 pivot block B itself.
    constexpr int R = NREG + 2;  // second published row (16-byte aligned: NREG is even)
    double inv0 = 0.0, inv1 = 0.0;  // this lane's row of B^-1 (pivot lanes)
    for (int j = 0; j < n; j += 2) {
      double* buf = C.prow + ((j >> 1) & 1) * C.prow_stride;
      if (i == j || i == j + 1) {
        double* row = buf + (i - j) * R;
        double2* row2 = reinterpret_cast<double2*>(row);
#pragma unroll
        for (int k = 0; k < NREG; k += 2) row2[k / 2] = make_double2(a[k], a[k + 1]);
        row[NREG] = b;
      }
      __syncwarp();
      const double2* r0 = reinterpret_cast<const double2*>(buf);
      const double2* r1 = reinterpret_cast<const double2*>(buf + R);
      const double2 p0 = r0[0], p1 = r1[0];  // B = [p0.x p0.y; p1.x p1.y]
      const double bj0 = buf[NREG], bj1 = buf[R + NREG];
      const double det = p0.x * p1.y - p0.y * p1.x;
      ok = ok && (p0.x > 0.0) && (det > 0.0) && isfinite(det);
      const double rdet = 1.0 / det;
      const bool piv_lane = (i == j) || (i == j + 1);
      if (i == j) { inv0 = p1.y * rdet; inv1 = -p0.y * rdet; }
      if (i == j + 1) { inv0 = -p1.x * rdet; inv1 = p0.x * rdet; }
      // [f0 f1] B = [a0 a1]; the pivot rows themselves are kept (raw)
      const double f0 = piv_lane ? 0.0 : (a[0] * p1.y - a[1] * p1.x) * rdet;
      const double f1 = piv_lane ? 0.0 : (a[1] * p0.x - a[0] * p0.y) * rdet;
#pragma unroll
      for (int k = 2; k < NREG; k += 2) {
        const double2 u = r0[k / 2], v = r1[k / 2];
        a[k - 2] = a[k] - f0 * u.x - f1 * v.x;
        a[k - 1] = a[k + 1] - f0 * u.y - f1 * v.y;
      }
      a[NREG - 2] = 0.0;
      a[NREG - 1] = 0.0;
      b -= f0 * bj0 + f1 * bj1;
    }
    // rows j, j+1 now read  B [y_j y_j+1]^T = [b_j b_j+1]^T
    const double bp = __shfl_xor_sync(kFull, b, 1);
    y = (i & 1) ? inv0 * bp + inv1 * b : inv0 * b + inv1 * bp;
  } else {  // scalar pivots (kept for comparison: -DLFR_BLOCK_PIVOT_MAX_NREG=0)
  double myrp = 1.0;
  for (int j = 0; j < n; ++j) {
    double* buf = C.prow + (j & 1) * C.prow_stride;
    double2* buf2 = reinterpret_cast<double2*>(buf);
    if (i == j) {  // the pivot lane only publishes its registers (slot 0 = the pivot)
#pragma unroll
      for (int k = 0; k < NREG; k += 2) buf2[k / 2] = make_double2(a[k], a[k + 1]);
      buf[NREG] = b;
    }
    __syncwarp();
    double2 t[NREG / 2];
#pragma unroll
    for (int k = 0; k < NREG; k += 2) t[k / 2] = buf2[k / 2];
    const double bj = buf[NREG];
    const double piv = t[0].x;
    ok = ok && (piv > 0.0) && isfinite(piv);
    const double rp = 1.0 / piv;  // every lane: no serial work in the pivot lane
    if (i == j) myrp = rp;
    const double f = (i == j) ? 0.0 : a[0] * rp;  // the pivot row itself is kept (un-normalised)
#pragma unroll
    for (int k = 1; k < NREG; ++k) a[k - 1] = a[k] - f * ((k & 1) ? t[k / 2].y : t[k / 2].x);
    a[NREG - 1] = 0.0;
    b -= f * bj;
  }
  y = b * myrp;  // row i now reads  piv_i * y_i = b_i
  }
  double mc = 0.0, dot = 0.0, mx = 0.0;
  bool finite = true;
  if (act) {
    const double d = -si * y;
    C.dl[i] = d;
    mc = y * (b0 + d2 * y);
    dot = gi * d;
    mx = fabs(d);
    finite = isfinite(y);
  }
  warp_sum2_max1(mc, dot, mx);
  *model_change = 0.5 * mc;
  *gd = dot;
  *dmax = mx;
  finite = __all_sync(kFull, finite);
  __syncwarp();
  return ok && finite;
}

__device__ __forceinline__ CandNorms make_candidate2(const Warp2Ctx& C, double alpha, const DevConsts& K) {
  CandNorms nr{0.0, 0.0};
  for (int i = C.lane; i < 2 * C.Nc; i += 32) {
    const int f = C.freeof[i >> 1];
    const double xv = C.x[i];
    double v = xv;
    if (f >= 0) {
      v = fmin(fmax(xv + alpha * C.dl[2 * f + (i & 1)], -K.bound), K.bound);
      const double dv = xv - v;
      nr.dn2 += dv * dv;
      nr.xn2 += v * v;
    }
    C.xc[i] = v;
  }
  __syncwarp();
  return nr;
}

// Component setup by ONE warp (solve.cc:98-143): node list and start point,
// compaction of the kept out-edges (same track -> Cauchy, same component ->
// Tukey, other component or root-root -> dropped) with ballots, out-edge ranges,
// free-variable numbering, and the twin (reverse edge) of every kept edge.
// Shared by the warp kernel and the tile kernel (whose warp 0 runs it).
// Pull the candidate out-edge records of every node of the component into shared memory, once:
// a node's out-edges are contiguous in the CSR array, so each node is ONE 1-D bulk copy
// (cp.async.bulk, 80 * degree bytes, 16-byte aligned on both sides) completing on the warp's
// mbarrier; all copies are in flight together and no register is tied up.  `P.edges` may be device
// memory or the caller's pinned host buffer (zero-copy over PCIe: the records are read exactly
// once either way, every later evaluation runs from shared memory).
template <class Ctx>
__device__ __forceinline__ void stage_edges(Ctx& C, const uint32_t* rowstart, const uint32_t* candptr, int Nc,
                                            int Eup, const DevProblem& P, int lane) {
  if (Eup == 0) return;
  // Pacing of zero-copy pulls: every resident warp asking for its records at once makes the PCIe
  // link serve ~10 MB of requests round-robin, so the FIRST components (the largest, dispatched
  // first because they run longest) get their data last.  A ticket counter keeps at most
  // `pull_window` bytes outstanding: records arrive in dispatch order at the same link rate.
  const bool paced = P.pull_window != 0;
  if (paced) {
    if (lane == 0) {
      const unsigned long long ticket = atomicAdd(P.pull_ctr, 80ull * (unsigned)Eup);
      const volatile unsigned long long* arrived = P.pull_ctr + 1;
      while ((long long)(ticket - *arrived) >= (long long)P.pull_window) __nanosleep(64);
    }
    __syncwarp();
  }
  if (lane == 0) mbar_arrive_expect_tx(C.bar, 80u * (uint32_t)Eup);
  __syncwarp();
  for (int l = lane; l < Nc; l += 32) {
    const uint32_t d = candptr[l + 1] - candptr[l];
    if (d) bulk_copy_g2s(C.stage + 5 * candptr[l], P.edges + 5 * (size_t)rowstart[l], 80u * d, C.bar);
  }
  mbar_wait(C.bar, 0);
  if (paced && lane == 0) atomicAdd(P.pull_ctr + 1, 80ull * (unsigned)Eup);
  __syncwarp();
}

template <class Ctx>
__device__ __forceinline__ void warp_setup(Ctx& C, uint32_t* rowstart, uint32_t* candptr, int* cnt, int ncmax,
                                           const DevProblem& P, const DevConsts& K, uint32_t c, int lane,
                                           int* Ec_out, int* nf_out, bool* irregular_out) {
  const uint32_t nbeg = P.comp_ptr[c];
  const int Nc = (int)(P.comp_ptr[c + 1] - nbeg);
  C.Nc = Nc;
  if (lane == 0) mbar_init(C.bar, 1);
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
      cnt[l] = 0;
      cnt[ncmax + l] = 0;
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
  stage_edges(C, rowstart, candptr, Nc, Eup, P, lane);
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
      e = (uint32_t)k;  // index of the record in the staged array
      const uint32_t v = C.node[lo];
      const uint32_t dst = __float_as_uint(C.stage[5 * k + 4].w);
      if (dst >= P.n_nodes || dst == v) {
        *P.err_flag = 1;  // malformed input: reported by the host as LFR_EINVAL
      } else {
        int kind = LFR_EDGE_SKIP;
        if (P.track[v] == P.track[dst]) kind = LFR_EDGE_CAUCHY;          // solve.cc:105
        else if (P.comp[v] == P.comp[dst]) kind = LFR_EDGE_TUKEY;        // solve.cc:114
        keep = (kind != LFR_EDGE_SKIP) && !(P.is_root[v] && P.is_root[dst]);
        if (keep) {
          const uint32_t dl_ = P.local_of[dst];
          mt = (uint32_t)lo | (dl_ << 12) | ((uint32_t)kind << 24);
          atomicAdd(&cnt[lo], 1);              // kept out-degree (integer: order-independent)
          atomicAdd(&cnt[ncmax + dl_], 1);   // kept in-degree
        }
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
  int orun = 0, frun = 0;
  for (int l0 = 0; l0 < Nc; l0 += 32) {
    const int l = l0 + lane;
    const int co = (l < Nc) ? cnt[l] : 0, ci = (l < Nc) ? cnt[ncmax + l] : 0;
    const int so = warp_incl_scan(co, lane);
    const bool is_free = (l < Nc) && (co + ci > 0) && !P.is_root[C.node[l < Nc ? l : 0]];
    const int sf = warp_incl_scan(is_free ? 1 : 0, lane);
    if (l < Nc) {
      C.outptr[l] = (uint16_t)(orun + so - co);
      C.freeof[l] = is_free ? (int16_t)(frun + sf - 1) : (int16_t)-1;
      if (is_free) C.lof[frun + sf - 1] = (uint16_t)l;
    }
    orun += __shfl_sync(kFull, so, 31);
    frun += __shfl_sync(kFull, sf, 31);
  }
  if (lane == 0) C.outptr[Nc] = (uint16_t)orun;
  __syncwarp();
  // twin of every kept edge: the unique kept edge dst -> src
  bool irregular = false;
  for (int e = lane; e < Ec; e += 32) {
    const uint32_t mt = C.meta[e];
    const int s = mt & 0xfff, d = (mt >> 12) & 0xfff;
    int found = 0, tw = e;
    for (int j = C.outptr[d]; j < C.outptr[d + 1]; ++j)
      if ((int)((C.meta[j] >> 12) & 0xfff) == s) {
        tw = j;
        ++found;
      }
    irregular = irregular || (found != 1);
    C.twin[e] = (uint16_t)tw;
  }
  *irregular_out = __any_sync(kFull, irregular);
  *Ec_out = Ec;
  *nf_out = frun;
}

// (12 resident warps per SM = 168 registers for NREG <= 16; measured: 8 (255 registers, no spills)
// and 16 (128 registers) change neither the single-scene latency nor the throughput, profiles/README.md)
template <int WARPS, int NREG>
__global__ void __launch_bounds__(WARPS * 32, (NREG > 16 ? 8 : 12) / WARPS)
solve_warp2_kernel(const DevProblem P, const DevConsts K, const WarpBucket B) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const uint32_t item = blockIdx.x * WARPS + wib;
  if (item >= B.n) return;  // warps are independent: no block-level barrier anywhere
  const uint32_t c = B.list[item];
  unsigned char* base = smem_raw + (size_t)wib * B.smem_per_warp;
  const Warp2Layout L(B.emax, B.ncmax, B.n2max);
  Warp2Ctx C;
  C.lane = lane;
  C.emax = B.emax;
  C.ldh = L.ldh;
  C.stage = (float4*)(base + L.stage);
  C.bar = (uint64_t*)(base + L.bar);
  C.x = (double*)(base + L.x);
  C.xc = (double*)(base + L.xc);
  C.g = (double*)(base + L.g);
  C.S = (double*)(base + L.S);
  C.dl = (double*)(base + L.dl);
  C.H = (double*)(base + L.H);
  C.scr = (double*)(base + L.scr);
  C.tup = (double*)(base + L.tup);
  C.prow = (double*)(base + L.prow);
  C.prow_stride = 72;
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

  const bool prof = (P.st_cycles != nullptr);
  if (prof && lane == 0) {
    unsigned long long ns;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
    P.st_times[2 * (size_t)c] = ns;
  }
  long long t_begin = prof ? clock64() : 0, t_mark = t_begin;
  long long cyc_eval = 0, cyc_asm = 0, cyc_lm = 0, cyc_ls = 0, cyc_setup = 0, cyc_poly = 0;
#define LFR_TICK(acc) do { if (prof) { const long long now__ = clock64(); acc += now__ - t_mark; t_mark = now__; } } while (0)

  // ---- component setup (solve.cc:98-143) --------------------------------------
  int Ec = 0, nf_setup = 0;
  bool irregular_setup = false;
  warp_setup(C, rowstart, candptr, cnt, B.ncmax, P, K, c, lane, &Ec, &nf_setup, &irregular_setup);
  C.Ec = Ec;
  C.irregular = irregular_setup;
  const int Nc = C.Nc;
  const int frun = nf_setup;
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
  double cost = eval_pass2<false, false>(C, C.x, K);
  LFR_TICK(cyc_eval);
  double gmax = assemble2<false>(C, true, K);
  LFR_TICK(cyc_asm);
  const double cost0 = cost;
  double radius = K.radius0, nu = 2.0;
  int iter = 0, n_invalid = 0, term = LFR_TERM_NO_CONVERGENCE;
  unsigned ls_steps = 0;
  bool success = true;
  double x_norm;
  {
    double a = 0.0;
    for (int i = lane; i < C.n; i += 32) {
      const int l = C.lof[i >> 1];
      const double xv = C.x[2 * l + (i & 1)];
      a += xv * xv;
    }
    x_norm = sqrt(warp_sum(a));
  }

  // ---- trust-region loop (A.6) ---------------------------------------------------------
  for (;;) {
    if (iter >= K.max_iter) { term = LFR_TERM_NO_CONVERGENCE; break; }
    if (success && gmax <= K.g_tol) { term = LFR_TERM_GRADIENT_TOL; break; }
    if (radius <= K.radius_min) { term = LFR_TERM_MIN_RADIUS; break; }
    ++iter;
    success = false;
    double model_change = 0.0, gd = 0.0, dmax = 0.0;
    LFR_TICK(cyc_ls);
    bool valid = lm_step2<NREG>(C, radius, K, &model_change, &gd, &dmax);
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
    CandNorms nr = make_candidate2(C, 1.0, K);
    double cost_c = eval_pass2<false, true>(C, C.xc, K, nullptr, &nr);
    LFR_TICK(cyc_eval);
    bool c_valid = isfinite(cost_c);
    if (!c_valid || cost_c > cost + K.ls_suff * gd * 1.0) {
      LsSample initial{0.0, cost, gd, true, true};
      LsSample previous{0.0, 0.0, 0.0, false, false};
      LsSample current{1.0, cost_c, 0.0, c_valid, false};
      if (c_valid) {
        current.gradient = assemble2<true>(C, false, K);
        current.gradient_valid = isfinite(current.gradient);
      }
      int ls_iter = 0;
      bool ls_ok = false;
      for (;;) {
        ++ls_iter;
        ++ls_steps;
        if (ls_iter >= K.max_ls_iter) break;
        LFR_TICK(cyc_ls);
        const double step = ls_next_step(initial, previous, current, K, lane);
        LFR_TICK(cyc_poly);
        if (step * dmax < K.ls_min_step) break;
        previous = current;
        nr = make_candidate2(C, step, K);
        double dphi;
        cost_c = eval_pass2<true, true>(C, C.xc, K, &dphi, &nr);
        c_valid = isfinite(cost_c);
        current = LsSample{step, cost_c, 0.0, c_valid, false};
        if (c_valid) {
          current.gradient = dphi;
          current.gradient_valid = isfinite(dphi);
        }
        if (c_valid && !(cost_c > cost + K.ls_suff * gd * step)) { ls_ok = true; break; }
      }
      if (ls_ok) {
        for (int i = lane; i < C.n; i += 32) C.dl[i] *= current.x;
        __syncwarp();
      } else {  // line search failed: delta unchanged, candidate = P(x + delta)
        nr = make_candidate2(C, 1.0, K);
        cost_c = eval_pass2<false, true>(C, C.xc, K, nullptr, &nr);
        c_valid = isfinite(cost_c);
      }
    }
    if (!c_valid) cost_c = 1.7976931348623157e308;
    const double step_norm = sqrt(nr.dn2);
    if (step_norm <= K.p_tol * (x_norm + K.p_tol)) { term = LFR_TERM_PARAMETER_TOL; break; }
    if (fabs(cost - cost_c) <= K.f_tol * cost) { term = LFR_TERM_FUNCTION_TOL; break; }
    const double rho = (cost - cost_c) / model_change;
    if (rho > K.min_rel_decrease) {
      for (int i = lane; i < 2 * Nc; i += 32) C.x[i] = C.xc[i];
      __syncwarp();
      cost = cost_c;
      LFR_TICK(cyc_ls);
      gmax = assemble2<false>(C, false, K);
      x_norm = sqrt(nr.xn2);
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
      unsigned smid;
      asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
      o[6] = (unsigned long long)smid | ((unsigned long long)ls_steps << 32);
      o[7] = (unsigned long long)cyc_poly;
      unsigned long long ns;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
      P.st_times[2 * (size_t)c + 1] = ns;
    }
  }
#undef LFR_TICK
}

}  // namespace lfr
