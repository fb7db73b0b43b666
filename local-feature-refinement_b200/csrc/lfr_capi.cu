// lfr_capi.cu — the C ABI of include/lfr.h for the B200 backend: plan
// construction (problem -> HBM, size-bucketed launch schedule), the solve
// launches, and result download.  No CPU fallback: every entry point that
// computes fails with LFR_ENODEV / LFR_ECUDA when no device is usable.
#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "lfr_solve_cta.cuh"
#include "lfr_solve_tile.cuh"

namespace {

thread_local std::string g_last_error;

// host-side timeline of the calling thread's last lfr_solve(): microseconds since the call began at
// {small uploads queued, schedule built, plan filled, kernels queued, stats back, return}
thread_local double g_host_marks[8] = {};
thread_local std::chrono::steady_clock::time_point g_host_t0;
inline void host_mark(int i) {
  g_host_marks[i] = std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - g_host_t0).count();
}

int fail(int code, const std::string& msg) {
  g_last_error = msg;
  return code;
}

int cuda_code(cudaError_t e) {
  if (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver || e == cudaErrorInvalidDevice) return LFR_ENODEV;
  if (e == cudaErrorMemoryAllocation) return LFR_ENOMEM;
  return LFR_ECUDA;
}

#define LFR_CUDA(call)                                                              \
  do {                                                                              \
    cudaError_t err__ = (call);                                                     \
    if (err__ != cudaSuccess)                                                       \
      return fail(cuda_code(err__), std::string(#call) + ": " + cudaGetErrorString(err__)); \
  } while (0)

#define LFR_TRY(expr)        \
  do {                       \
    const int rc__ = (expr); \
    if (rc__) return rc__;   \
  } while (0)

constexpr int kMaxSmemPerBlock = 227 * 1024;
constexpr int kScheduleThreadsMax = 8;  // host threads that classify the dispatch list (build_buckets)
constexpr int kMaxStreams = 12;

lfr::DevConsts make_consts(const lfr_options& o) {
  lfr::DevConsts K;
  K.bound = o.bound;
  K.cauchy_b = o.cauchy_a * o.cauchy_a;
  K.cauchy_c = 1.0 / K.cauchy_b;
  K.tukey_a2 = o.tukey_a * o.tukey_a;
  K.tukey_inv_a2 = 1.0 / K.tukey_a2;
  if (o.tukey_variant == 2) {
    K.tukey_rho0 = K.tukey_a2 / 3.0;
    K.tukey_rho1 = 1.0;
  } else {
    K.tukey_rho0 = K.tukey_a2 / 6.0;
    K.tukey_rho1 = 0.5;
  }
  K.f_tol = o.function_tolerance;
  K.g_tol = o.gradient_tolerance;
  K.p_tol = o.parameter_tolerance;
  K.radius0 = o.initial_trust_region_radius;
  K.radius_max = o.max_trust_region_radius;
  K.radius_min = o.min_trust_region_radius;
  K.min_rel_decrease = o.min_relative_decrease;
  K.min_diag = o.min_lm_diagonal;
  K.max_diag = o.max_lm_diagonal;
  K.ls_suff = o.line_search_sufficient_function_decrease;
  K.ls_max_contraction = o.max_line_search_step_contraction;
  K.ls_min_contraction = o.min_line_search_step_contraction;
  K.ls_min_step = o.min_line_search_step_size;
  K.max_iter = o.max_num_iterations;
  K.max_invalid = o.max_num_consecutive_invalid_steps;
  K.max_ls_iter = o.max_num_line_search_step_size_iterations;
  K.linear_solver = o.linear_solver;
  return K;
}

// Grow-only device buffer: lfr_solve() re-uses its workspace across calls, so a
// steady stream of solves performs no cudaMalloc/cudaFree.
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  int reserve(size_t bytes) {
    if (bytes <= cap) return LFR_OK;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    const size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) return fail(cuda_code(e), std::string("cudaMalloc: ") + cudaGetErrorString(e));
    cap = want;
    return LFR_OK;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <typename T>
  T* as() const { return static_cast<T*>(p); }
};

// One launch of the CTA tier: a size class of large components (its dynamic shared memory and the
// register cap MINB decide how many of them an SM runs at once).
struct CtaGroup {
  uint32_t first = 0, n = 0, max_free = 0;
  int minb = 2;
};

struct Bucket {
  uint32_t offset = 0;  // into the bucket-list buffer
  uint32_t n = 0;
  int emax = 0, ncmax = 0, n2max = 0, smem_per_warp = 0, warps = 4;
  int variant = 0;  // 0: shared-memory Cholesky kernel (n <= 64); 16 / 32: register Gauss-Jordan kernel (n <= variant)
  bool stages_edges() const { return variant != 0; }  // warp2 / tile tiers pull their edge records into shared memory
};

int validate(const lfr_problem* p) {
  if (!p) return fail(LFR_EINVAL, "problem is NULL");
  if (p->n_nodes && (!p->row_ptr || !p->track || !p->comp || !p->is_root))
    return fail(LFR_EINVAL, "NULL per-node array");
  if (p->n_components && (!p->comp_ptr || !p->comp_nodes)) return fail(LFR_EINVAL, "NULL component list");
  if (p->n_nodes && p->row_ptr[p->n_nodes] != p->n_edges) return fail(LFR_EINVAL, "row_ptr[n_nodes] != n_edges");
  if (p->n_edges && !p->edges) return fail(LFR_EINVAL, "edges is NULL");
  if (p->n_edges >= (1ull << 32)) return fail(LFR_EUNSUPPORTED, "more than 2^32 directed edges");
  // per-edge checks (dst range, self edges) run on the device while the edges are
  // staged (solve_warp_kernel), so the host never walks the 80-byte records.
  return LFR_OK;
}

}  // namespace

struct lfr_plan {
  int device = 0;
  lfr_options opt;
  lfr::DevConsts K;
  uint32_t N = 0, C = 0;
  uint64_t E = 0;
  uint32_t total_slots = 0;
  DevBuf row_ptr, edges, track, comp, is_root, comp_ptr, comp_nodes, local_of, pos, pos_init, stats, cycles, times, lists;
  // `stats` is one block (one memset, one D2H copy): cost0[Cp] cost1[Cp] iter[Cp] term[Cp] ls[Cp] kept[Cp] err[2] pull[2 x u64]
  uint32_t Cp = 0;               // C rounded up to an even count
  bool pos_is_staged = false;    // lfr_solve(): the start point was uploaded straight into `pos`
  void* h_stage = nullptr;       // pinned host staging for the stats block
  size_t h_stage_cap = 0;
  double* d_cost0() const { return stats.as<double>(); }
  double* d_cost1() const { return stats.as<double>() + Cp; }
  int32_t* d_iter() const { return reinterpret_cast<int32_t*>(stats.as<double>() + 2 * (size_t)Cp); }
  int32_t* d_term() const { return d_iter() + Cp; }
  uint32_t* d_ls() const { return reinterpret_cast<uint32_t*>(d_term() + Cp); }
  uint32_t* d_kept() const { return d_ls() + Cp; }
  int* d_err() const { return reinterpret_cast<int*>(d_kept() + Cp); }
  unsigned long long* d_pull() const { return reinterpret_cast<unsigned long long*>(d_err() + 2); }  // {ticketed, arrived} bytes
  size_t stats_bytes() const { return 16 * (size_t)Cp + 16 * (size_t)Cp + 8 + 16; }
  std::vector<Bucket> buckets;
  std::vector<uint32_t> comp_size;  // nodes per dispatch slot
  std::vector<uint32_t> list_host;
  // CTA tier (block-Jacobi PCG): components with more than kMaxWarpN2 unknowns, or all with linear_solver = 2
  struct SchedDim { int e, nc, n2; };
  std::vector<uint16_t> sched_key;        // build_buckets scratch: (variant, shared-memory class) of every slot
  std::vector<SchedDim> sched_dim;
  std::vector<uint32_t> large_slots;
  std::vector<uint64_t> large_cand;       // candidate out-edges of each large component (row_ptr sums)
  std::vector<uint32_t> large_free;       // its non-root nodes (upper bound of the free nodes)
  std::vector<uint64_t> large_ell;        // its sliced-ELL slots (32 x the largest candidate out-degree of every 32-node slice)
  std::vector<lfr::CtaComp> L_comps_host;
  std::vector<CtaGroup> cta_groups;
  uint32_t n_large = 0;
  DevBuf L_comps, L_rec, L_meta, L_inlist, L_twin, L_fdst, L_bE01, L_bE23, L_fdstE, L_ell_base, L_scr, L_q, L_node, L_outptr, L_inptr, L_freeof, L_x, L_xc, L_lof, L_vec;
  uint64_t L_total_free = 0;
  uint32_t L_max_free = 0;
  uint32_t n_solved = 0;
  bool profile = false;
  // lfr_solve() zero-copy: staging tiers read the caller's pinned edge array / write the caller's
  // pinned positions directly (device-side addresses of those host buffers), nullptr = through HBM
  const float4* zc_edges = nullptr;
  double* zc_positions = nullptr;
  const uint8_t* slot_owner = nullptr;  // lfr_solve_multi(): owner[c] of every dispatch slot, this plan solves owner == owner_id
  uint8_t owner_id = 0;
  bool edges_in_hbm = false;       // the edge array was (or is being) copied to `edges`
  bool needs_hbm_edges = false;    // some bucket (smem-Cholesky warp tier) reads edge records from global memory by index
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_edges = nullptr;  // bulk edge copy done (only the non-staging tiers wait for it)
  cudaEvent_t ev_small = nullptr;  // fork / join of the second upload stream
  cudaEvent_t ev_prep = nullptr;   // small arrays + local_of ready (CTA-tier preparation on the copy stream)
  bool cta_from_hbm = false;       // zero-copy solve whose CTA tier reads the bulk HBM copy of the edge array
  cudaStream_t streams[kMaxStreams] = {};
  cudaEvent_t ev_fork = nullptr, ev_join[kMaxStreams] = {};
  int n_streams = 0;

  lfr::CtaArrays cta_arrays() const {
    lfr::CtaArrays A;
    A.rec = L_rec.as<float4>();
    A.meta = L_meta.as<uint32_t>();
    A.inlist = L_inlist.as<uint32_t>();
    A.twin = L_twin.as<uint32_t>();
    A.fdst = L_fdst.as<int32_t>();
    A.bE01 = L_bE01.as<double2>();
    A.bE23 = L_bE23.as<double2>();
    A.fdstE = L_fdstE.as<int32_t>();
    A.ell_base = L_ell_base.as<uint32_t>();
    A.scr = L_scr.as<double>();
    A.q = L_q.as<double>();
    A.node = L_node.as<uint32_t>();
    A.outptr = L_outptr.as<uint32_t>();
    A.inptr = L_inptr.as<uint32_t>();
    A.freeof = L_freeof.as<int32_t>();
    A.x = L_x.as<double>();
    A.xc = L_xc.as<double>();
    A.lof = L_lof.as<uint32_t>();
    A.vec = L_vec.as<double>();
    A.total_free = L_total_free;
    return A;
  }

  lfr::DevProblem dev() const {
    lfr::DevProblem P;
    P.n_nodes = N;
    P.row_ptr = row_ptr.as<uint32_t>();
    P.edges = edges.as<float4>();
    P.track = track.as<uint32_t>();
    P.comp = comp.as<uint32_t>();
    P.is_root = is_root.as<uint8_t>();
    P.comp_ptr = comp_ptr.as<uint32_t>();
    P.comp_nodes = comp_nodes.as<uint32_t>();
    P.local_of = local_of.as<uint32_t>();
    P.positions = pos.as<double>();
    P.positions_out = zc_positions ? zc_positions : pos.as<double>();
    P.pull_ctr = d_pull();
    P.pull_window = 0;  // set by launch_solve for zero-copy staging only
    P.st_iter = d_iter();
    P.st_term = d_term();
    P.st_cost0 = d_cost0();
    P.st_cost1 = d_cost1();
    P.st_ls = d_ls();
    P.st_kept = d_kept();
    P.st_cycles = profile ? cycles.as<unsigned long long>() : nullptr;
    P.st_times = profile ? times.as<unsigned long long>() : nullptr;
    P.err_flag = d_err();
    return P;
  }
};

namespace {

void free_plan(lfr_plan* pl) {
  if (!pl) return;
  DevBuf* bufs[] = {&pl->row_ptr, &pl->edges, &pl->track, &pl->comp, &pl->is_root, &pl->comp_ptr, &pl->comp_nodes,
                    &pl->local_of, &pl->pos, &pl->pos_init, &pl->stats, &pl->cycles, &pl->times, &pl->lists, &pl->L_comps, &pl->L_rec, &pl->L_meta,
                    &pl->L_inlist, &pl->L_twin, &pl->L_fdst, &pl->L_bE01, &pl->L_bE23, &pl->L_fdstE, &pl->L_ell_base, &pl->L_scr, &pl->L_q, &pl->L_node, &pl->L_outptr, &pl->L_inptr, &pl->L_freeof,
                    &pl->L_x, &pl->L_xc, &pl->L_lof, &pl->L_vec};
  for (DevBuf* b : bufs) b->release();
  if (pl->h_stage) cudaFreeHost(pl->h_stage);
  for (int i = 0; i < pl->n_streams; ++i) {
    if (pl->streams[i]) cudaStreamDestroy(pl->streams[i]);
    if (pl->ev_join[i]) cudaEventDestroy(pl->ev_join[i]);
  }
  if (pl->ev_fork) cudaEventDestroy(pl->ev_fork);
  if (pl->ev_edges) cudaEventDestroy(pl->ev_edges);
  if (pl->ev_small) cudaEventDestroy(pl->ev_small);
  if (pl->ev_prep) cudaEventDestroy(pl->ev_prep);
  if (pl->copy_stream) cudaStreamDestroy(pl->copy_stream);
  delete pl;
}

template <typename T>
int upload(DevBuf* d, const T* h, size_t count, cudaStream_t s) {
  LFR_TRY(d->reserve(std::max<size_t>(count, 1) * sizeof(T)));
  if (count) LFR_CUDA(cudaMemcpyAsync(d->p, h, count * sizeof(T), cudaMemcpyHostToDevice, s));
  return LFR_OK;
}

// Size-bucketed schedule: components are grouped by the shared memory one warp
// needs for them, so small tracks run at high occupancy and the few large
// components do not dictate the carve-up of everyone else.  Buckets are
// launched on concurrent streams, largest components first.
int build_buckets(lfr_plan* pl, const lfr_problem* p) {
  // shared-memory classes of a launch (finer classes — one per "one more CTA fits an SM" boundary — were
  // measured on cfg4: 26 launches instead of 15, same solve time; profiles/r02_tile_tier_occupancy.txt)
  static const int kClass[] = {2048, 3072, 4096, 6144, 8192, 12288, 16384, 24576, 32768, 57344, kMaxSmemPerBlock};
  constexpr int n_class = sizeof(kClass) / sizeof(kClass[0]);
  // register warp kernel (8..32), register tile kernel (48, 64: 64 threads; 80: 128 threads),
  // smem-Cholesky warp kernel (0)
  static const int kVariant[8] = {8, 16, 24, 32, 48, 64, 80, 0};
  constexpr int kNV = 8, kV1 = 7, kKeys = kNV * n_class;
  constexpr uint16_t kNoKey = 0xffff;
  auto is_tile = [](int vi) { return vi >= 4 && vi <= 6; };
  const int dbg = pl->opt.debug_flags;
  const bool no_tile = (dbg & LFR_DBG_NO_TILE) != 0;
  const bool force_v1 = (dbg & LFR_DBG_FORCE_SMEM_CHOLESKY) != 0;
  const bool force_pcg = pl->opt.linear_solver == 2;
  auto layout_bytes = [&](int vi, int e, int nc, int n2) {
    return (vi == kV1) ? lfr::WarpLayout(e, nc, n2).total
                       : (is_tile(vi) ? lfr::TileLayout(e, nc, n2).total : lfr::Warp2Layout(e, nc, n2).total);
  };
  // This runs on the calling thread while the GPU waits for its first launch: one pass over the
  // components into flat, reused arrays (no per-call allocation once the plan is warm), then a
  // counting sort of the slots by (variant, shared-memory class).
  const uint32_t C = p->n_components;
  pl->comp_size.resize(C);
  pl->sched_key.resize(C);
  pl->sched_dim.resize(C);
  pl->n_solved = 0;
  pl->buckets.clear();
  pl->large_slots.clear();
  pl->large_cand.clear();
  pl->large_free.clear();
  pl->large_ell.clear();
  const uint32_t* comp_ptr = p->comp_ptr;
  const uint32_t* comp_nodes = p->comp_nodes;
  const uint32_t* row_ptr = p->row_ptr;
  const uint8_t* is_root = p->is_root;
  const uint8_t* owner = pl->slot_owner;
  const uint32_t n_nodes = p->n_nodes;
  uint16_t* key_of = pl->sched_key.data();
  lfr_plan::SchedDim* dim = pl->sched_dim.data();
  // Pass 1 — classify the slots [c0, c1): a pure function of the problem arrays that writes only the
  // per-slot entries of its own range and its own accumulator, so ranges run on separate threads
  // (merged in range order: the schedule does not depend on the thread count).
  struct Acc {
    Bucket caps[kKeys];
    uint32_t count[kKeys] = {};
    uint32_t n_solved = 0;
    std::vector<uint32_t> large_slots, large_free;
    std::vector<uint64_t> large_cand, large_ell;
    int rc = LFR_OK;
    const char* msg = nullptr;
  };
  auto classify = [&](uint32_t c0, uint32_t c1, Acc& A) {
    auto bail = [&](int code, const char* m) {
      A.rc = code;
      A.msg = m;
    };
    for (uint32_t c = c0; c < c1; ++c) {
      const uint32_t beg = comp_ptr[c], end = comp_ptr[c + 1];
      if (end < beg || end > pl->total_slots) return bail(LFR_EINVAL, "comp_ptr not monotone");
      const uint32_t nc = end - beg;
      pl->comp_size[c] = nc;
      key_of[c] = kNoKey;
      if (nc <= 1) continue;  // solve.cc:619-622
      if (owner && owner[c] != pl->owner_id) continue;  // another device's component
      ++A.n_solved;
      uint64_t eup = 0;
      uint32_t nfree = 0;
      for (uint32_t i = beg; i < end; ++i) {
        const uint32_t v = comp_nodes[i];
        if (v >= n_nodes) return bail(LFR_EINVAL, "comp_nodes out of range");
        const uint32_t r0 = row_ptr[v], r1 = row_ptr[v + 1];
        if (r1 < r0) return bail(LFR_EINVAL, "row_ptr not monotone");
        eup += r1 - r0;
        nfree += is_root[v] ? 0 : 1;
      }
      const int n2 = std::max(2 * (int)nfree, 2);
      auto to_cta_tier = [&]() -> bool {
        if (nc > 16383) {
          bail(LFR_EUNSUPPORTED, "component with more than 16383 nodes");
          return false;
        }
        uint64_t slots = 0;
        for (uint32_t i0 = beg; i0 < end; i0 += 32) {
          uint32_t wmax = 0;
          for (uint32_t i = i0; i < std::min(end, i0 + 32); ++i) wmax = std::max(wmax, row_ptr[comp_nodes[i] + 1] - row_ptr[comp_nodes[i]]);
          slots += 32ull * ((wmax + 3u) & ~3u);  // slice width: a multiple of four slots (cta_block_row)
        }
        if (slots > 0xffffffffull) {
          bail(LFR_EUNSUPPORTED, "component too dense for the CTA tier's block layout");
          return false;
        }
        A.large_slots.push_back(c);
        A.large_cand.push_back(eup);
        A.large_free.push_back(nfree);
        A.large_ell.push_back(slots);
        return true;
      };
      if (force_pcg || n2 > lfr::kMaxWarpN2 || nc > (uint32_t)lfr::kMaxWarpNodes || eup > 65535) {
        if (!to_cta_tier()) return;
        continue;
      }
      const int e = std::max<int>(1, (int)eup);
      int vi = (n2 <= 8) ? 0 : (n2 <= 16 ? 1 : (n2 <= 24 ? 2 : (n2 <= 32 ? 3 : (n2 <= 48 ? 4 : (n2 <= 64 ? 5 : (n2 <= 80 ? 6 : kV1))))));
      if (is_tile(vi) && (no_tile || lfr::TileLayout(e, (int)nc, n2).total > kMaxSmemPerBlock)) vi = kV1;
      if (force_v1) vi = kV1;
      int need = layout_bytes(vi, e, (int)nc, n2);
      if (need > kMaxSmemPerBlock && vi != kV1) {  // the staged records do not fit: the Cholesky warp kernel reads them from global memory
        vi = kV1;
        need = layout_bytes(vi, e, (int)nc, n2);
      }
      if (need > kMaxSmemPerBlock) {
        // a dense, high-degree component (its per-edge scratch alone exceeds one SM's shared
        // memory): the CTA tier keeps its per-edge data in HBM
        if (!to_cta_tier()) return;
        continue;
      }
      int k = 0;
      while (need > kClass[k]) ++k;  // need <= kClass[n_class - 1] here
      const int key = vi * n_class + k;
      key_of[c] = (uint16_t)key;
      dim[c] = lfr_plan::SchedDim{e, (int)nc, n2};
      Bucket& cb = A.caps[key];
      ++A.count[key];
      cb.emax = std::max(cb.emax, e);
      cb.ncmax = std::max(cb.ncmax, (int)nc);
      cb.n2max = std::max(cb.n2max, n2);
    }
  };
  // ranges of about equal node counts; extra threads only where their start-up pays
  // (measured on the GPU box's host, profiles/r02_schedule_threads.txt: ~3 ns per listed node + ~16 ns
  // per slot on one thread, ~50 us to start a helper)
  const uint64_t work_ns = 3ull * pl->total_slots + 16ull * C;
  // (inside an application the helpers cost more than in the stand-alone timing — the CUDA runtime
  // hooks thread creation — so they start only from about half a millisecond of work)
  int n_thr = work_ns < 500000 ? 1 : (int)std::min<uint64_t>(kScheduleThreadsMax, work_ns / 150000);
  if (const char* e = std::getenv("LFR_SCHEDULE_THREADS")) n_thr = std::max(1, std::min(kScheduleThreadsMax, std::atoi(e)));
  std::vector<uint32_t> cut((size_t)n_thr + 1, C);
  cut[0] = 0;
  for (int t = 1; t < n_thr; ++t) {
    const uint32_t want = (uint32_t)((uint64_t)pl->total_slots * t / n_thr);
    cut[t] = (uint32_t)(std::upper_bound(comp_ptr, comp_ptr + C + 1, want) - comp_ptr);
    cut[t] = std::min(C, std::max(cut[t], cut[t - 1]));
  }
  std::vector<Acc> acc((size_t)n_thr);
  {
    std::vector<std::thread> workers;
    for (int t = 1; t < n_thr; ++t) workers.emplace_back([&, t] { classify(cut[t], cut[t + 1], acc[t]); });
    classify(cut[0], cut[1], acc[0]);
    for (std::thread& w : workers) w.join();
  }
  Bucket caps[kKeys];
  uint32_t count[kKeys] = {};
  for (const Acc& A : acc) {  // range order
    if (A.rc != LFR_OK) return fail(A.rc, A.msg);
    pl->n_solved += A.n_solved;
    for (int k = 0; k < kKeys; ++k) {
      count[k] += A.count[k];
      caps[k].emax = std::max(caps[k].emax, A.caps[k].emax);
      caps[k].ncmax = std::max(caps[k].ncmax, A.caps[k].ncmax);
      caps[k].n2max = std::max(caps[k].n2max, A.caps[k].n2max);
    }
    pl->large_slots.insert(pl->large_slots.end(), A.large_slots.begin(), A.large_slots.end());
    pl->large_cand.insert(pl->large_cand.end(), A.large_cand.begin(), A.large_cand.end());
    pl->large_free.insert(pl->large_free.end(), A.large_free.begin(), A.large_free.end());
    pl->large_ell.insert(pl->large_ell.end(), A.large_ell.begin(), A.large_ell.end());
  }
  // emission order: largest shared-memory class first, within a class the higher tiers first
  uint32_t start[kKeys], total = 0;
  for (int k = n_class - 1; k >= 0; --k)
    for (int vi = kNV - 1; vi >= 0; --vi) {
      start[vi * n_class + k] = total;
      total += count[vi * n_class + k];
    }
  pl->list_host.resize(total);
  {
    uint32_t fill[kKeys];
    std::memcpy(fill, start, sizeof(fill));
    uint32_t* list = pl->list_host.data();
    for (uint32_t c = 0; c < C; ++c)
      if (key_of[c] != kNoKey) list[fill[key_of[c]]++] = c;  // ascending slot index inside a bucket
  }
  pl->needs_hbm_edges = false;
  auto emit = [&](int vi, const Bucket& cap, uint32_t offset, uint32_t n_mem) {
    Bucket b = cap;
    b.variant = kVariant[vi];
    b.n = n_mem;
    b.offset = offset;
    b.smem_per_warp = layout_bytes(vi, b.emax, b.ncmax, b.n2max);
    b.warps = (4 * b.smem_per_warp <= kMaxSmemPerBlock) ? 4 : 1;
    if (b.variant >= 48) b.warps = 1;  // tile kernels: one component per CTA
    if (b.warps == 1 && b.variant != 0 && b.variant < 48) b.variant = 32;  // only <1,32> is instantiated for single-warp CTAs
    pl->buckets.push_back(b);
    if (!b.stages_edges()) pl->needs_hbm_edges = true;  // the Cholesky warp tier reads records from HBM by global index
  };
  for (int k = n_class - 1; k >= 0; --k) {
    for (int vi = kNV - 1; vi >= 0; --vi) {
      const int key = vi * n_class + k;
      if (!count[key]) continue;
      const Bucket& cap = caps[key];
      if (layout_bytes(vi, cap.emax, cap.ncmax, cap.n2max) <= kMaxSmemPerBlock) {
        emit(vi, cap, start[key], count[key]);
      } else {
        // every member fits on its own but the union of their maxima does not: one launch each
        for (uint32_t i = 0; i < count[key]; ++i) {
          const uint32_t c = pl->list_host[start[key] + i];
          Bucket one;
          one.emax = dim[c].e;
          one.ncmax = dim[c].nc;
          one.n2max = dim[c].n2;
          emit(vi, one, start[key] + i, 1);
        }
      }
    }
  }
  return LFR_OK;
}

// CTA-tier components: the host only lays out per-component offsets (upper bounds: candidate edges
// from row_ptr, non-root nodes) and sizes the HBM arrays; the kept-edge / in-edge lists, free-variable
// numbering and twins are built on the device by cta_prepare_kernel (launched by fill_plan once the
// edge records and local_of are in HBM).
int prepare_large(lfr_plan* pl, const lfr_problem* p, cudaStream_t s) {
  pl->n_large = (uint32_t)pl->large_slots.size();
  pl->L_total_free = 0;
  pl->L_max_free = 0;
  pl->cta_groups.clear();
  if (pl->n_large == 0) return LFR_OK;
  std::vector<lfr::CtaComp>& comps = pl->L_comps_host;  // plan member: the async upload reads it
  comps.assign(pl->n_large, lfr::CtaComp{});
  // size classes by free nodes (upper bound): 104 bytes of CG vectors per free node in shared memory
  // -> 1 / 2 / 4 / 8 components per SM by shared memory; registers cap it at MINB
  static const uint32_t kClassMaxFree[4] = {0xffffffffu, 1008, 504, 250};
  static const int kClassMinb[4] = {2, 2, 3, 4};
  auto class_of = [&](uint32_t nfree) { return nfree > kClassMaxFree[1] ? 0 : (nfree > kClassMaxFree[2] ? 1 : (nfree > kClassMaxFree[3] ? 2 : 3)); };
  pl->cta_groups.clear();
  uint64_t e_off = 0, n_off = 0, f_off = 0, ell_off = 0, s_off = 0;
  uint32_t k = 0;
  for (int cls = 0; cls < 4; ++cls) {
    CtaGroup g;
    g.first = k;
    g.minb = kClassMinb[cls];
    for (uint32_t i = 0; i < pl->n_large; ++i) {  // dispatch order (largest first) inside a class
      if (class_of(pl->large_free[i]) != cls) continue;
      const uint32_t c = pl->large_slots[i];
      const uint32_t nc = p->comp_ptr[c + 1] - p->comp_ptr[c];
      if (pl->large_cand[i] > 0xffffffffull) return fail(LFR_EUNSUPPORTED, "component with more than 2^32 out-edges");
      lfr::CtaComp& cc = comps[k];
      cc.slot = c;
      cc.Nc = nc;
      cc.Ec = 0;  // filled on the device, with nf and regular
      cc.nf = 0;
      cc.regular = 0;
      cc.e_off = e_off;
      cc.n_off = n_off;
      cc.f_off = f_off;
      cc.comp_index = k;
      cc.ell_off = ell_off;
      cc.s_off = s_off;
      ell_off += pl->large_ell[i];
      s_off += (nc + 31) / 32 + 1;
      g.max_free = std::max(g.max_free, pl->large_free[i]);
      pl->L_max_free = std::max(pl->L_max_free, pl->large_free[i]);
      e_off += pl->large_cand[i];
      n_off += nc;
      f_off += pl->large_free[i];
      ++k;
    }
    g.n = k - g.first;
    if (g.n) pl->cta_groups.push_back(g);
  }
  pl->L_total_free = f_off;
  const uint64_t E1 = std::max<uint64_t>(e_off, 1), N1 = std::max<uint64_t>(n_off, 1), F1 = std::max<uint64_t>(f_off, 1);
  const uint64_t L1 = std::max<uint64_t>(ell_off, 1), S1 = std::max<uint64_t>(s_off, 1);
  LFR_TRY(upload(&pl->L_comps, comps.data(), comps.size(), s));
  LFR_TRY(pl->L_rec.reserve(sizeof(float4) * 5 * E1));
  LFR_TRY(pl->L_meta.reserve(sizeof(uint32_t) * E1));
  LFR_TRY(pl->L_inlist.reserve(sizeof(uint32_t) * E1));
  LFR_TRY(pl->L_twin.reserve(sizeof(uint32_t) * E1));
  LFR_TRY(pl->L_fdst.reserve(sizeof(int32_t) * E1));
  LFR_TRY(pl->L_bE01.reserve(sizeof(double2) * L1));
  LFR_TRY(pl->L_bE23.reserve(sizeof(double2) * L1));
  LFR_TRY(pl->L_fdstE.reserve(sizeof(int32_t) * L1));
  LFR_TRY(pl->L_ell_base.reserve(sizeof(uint32_t) * S1));
  LFR_TRY(pl->L_node.reserve(sizeof(uint32_t) * N1));
  LFR_TRY(pl->L_outptr.reserve(sizeof(uint32_t) * (N1 + pl->n_large)));
  LFR_TRY(pl->L_inptr.reserve(sizeof(uint32_t) * (N1 + pl->n_large)));
  LFR_TRY(pl->L_freeof.reserve(sizeof(int32_t) * N1));
  LFR_TRY(pl->L_lof.reserve(sizeof(uint32_t) * F1));
  LFR_TRY(pl->L_scr.reserve(sizeof(double) * 7 * E1));
  LFR_TRY(pl->L_q.reserve(sizeof(double) * 2 * E1));
  LFR_TRY(pl->L_x.reserve(sizeof(double) * 2 * N1));
  LFR_TRY(pl->L_xc.reserve(sizeof(double) * 2 * N1));
  LFR_TRY(pl->L_vec.reserve(sizeof(double) * (2 * lfr::V_COUNT + 9) * F1));
  return LFR_OK;
}

// Device-side address of a page-locked (cudaHostAlloc / cudaHostRegister) host buffer, or nullptr
// when the memory is pageable (or not 16-byte aligned, which the 128-bit accesses need).
void* device_view_of_pinned(const void* host_ptr) {
  if (!host_ptr || (reinterpret_cast<uintptr_t>(host_ptr) & 15u)) return nullptr;
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, host_ptr) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  if (a.type != cudaMemoryTypeHost || !a.devicePointer) return nullptr;
  return a.devicePointer;
}

// (Re)fill a plan from host arrays: H2D copies + schedule.  Buffers only grow.
// zc_edges / zc_positions: device-side views of the caller's pinned buffers (lfr_solve() only):
// the staging tiers then read the edge records / write the results there, and the 80-byte records
// — 95 % of the input bytes — are copied to HBM only if some non-staging tier needs them.
int fill_plan(lfr_plan* pl, const lfr_problem* p, const lfr_options& o, const double* initial_positions,
              cudaStream_t s, bool stage_positions_directly = false, const float4* zc_edges = nullptr,
              double* zc_positions = nullptr) {
  pl->opt = o;
  pl->K = make_consts(o);
  pl->N = p->n_nodes;
  pl->C = p->n_components;
  pl->E = p->n_edges;
  pl->total_slots = p->n_components ? p->comp_ptr[p->n_components] : 0;
  pl->profile = (o.debug_flags & LFR_DBG_PROFILE) != 0;
  pl->zc_edges = zc_edges;
  pl->zc_positions = zc_positions;
  pl->edges_in_hbm = false;
  if (!zc_edges) {
    LFR_TRY(upload(&pl->edges, p->edges, (size_t)p->n_edges, s));  // the bulk first: the DMA runs while the host schedules
    pl->edges_in_hbm = true;
  }
  // the small per-node arrays gate the first launch: with zero-copy edges they ARE the upload, so they
  // go out on two streams (two copy engines) instead of queueing behind each other
  cudaStream_t s2 = s;
  if (zc_edges) {
    if (!pl->copy_stream) LFR_CUDA(cudaStreamCreateWithFlags(&pl->copy_stream, cudaStreamNonBlocking));
    if (!pl->ev_small) LFR_CUDA(cudaEventCreateWithFlags(&pl->ev_small, cudaEventDisableTiming));
    s2 = pl->copy_stream;
    LFR_CUDA(cudaEventRecord(pl->ev_small, s));          // orders s2's copies after whatever `s` ran before
    LFR_CUDA(cudaStreamWaitEvent(s2, pl->ev_small, 0));
  }
  LFR_TRY(upload(&pl->row_ptr, p->row_ptr, (size_t)p->n_nodes + 1, s));
  LFR_TRY(upload(&pl->track, p->track, (size_t)p->n_nodes, s2));
  LFR_TRY(upload(&pl->comp, p->comp, (size_t)p->n_nodes, s2));
  LFR_TRY(upload(&pl->is_root, p->is_root, (size_t)p->n_nodes, s2));
  LFR_TRY(upload(&pl->comp_ptr, p->comp_ptr, (size_t)p->n_components + 1, s));
  LFR_TRY(upload(&pl->comp_nodes, p->comp_nodes, (size_t)pl->total_slots, s));
  if (s2 != s) {
    LFR_CUDA(cudaEventRecord(pl->ev_small, s2));
    LFR_CUDA(cudaStreamWaitEvent(s, pl->ev_small, 0));
  }
  const size_t N = std::max<size_t>(pl->N, 1), C = std::max<size_t>(pl->C, 1);
  LFR_TRY(pl->local_of.reserve(sizeof(uint32_t) * N));
  LFR_TRY(pl->pos.reserve(sizeof(double) * 2 * N));
  pl->Cp = (uint32_t)((C + 1) & ~(size_t)1);
  LFR_TRY(pl->stats.reserve(pl->stats_bytes()));
  if (pl->profile) {
    LFR_TRY(pl->cycles.reserve(sizeof(unsigned long long) * 8 * C));
    LFR_TRY(pl->times.reserve(sizeof(unsigned long long) * 2 * C));
    LFR_CUDA(cudaMemsetAsync(pl->cycles.p, 0, sizeof(unsigned long long) * 8 * C, s));
    LFR_CUDA(cudaMemsetAsync(pl->times.p, 0, sizeof(unsigned long long) * 2 * C, s));
  }
  // per-slot stats default to "skipped" (size-1 components never run); also clears the error flag
  LFR_CUDA(cudaMemsetAsync(pl->stats.p, 0, pl->stats_bytes(), s));
  if (stage_positions_directly) {
    // lfr_solve(): the caller's start point goes straight into the working array
    if (pl->N)
      LFR_CUDA(cudaMemcpyAsync(pl->pos.p, initial_positions, sizeof(double) * 2 * (size_t)pl->N,
                               cudaMemcpyHostToDevice, s));
    pl->pos_is_staged = true;
  } else {
    LFR_TRY(pl->pos_init.reserve(sizeof(double) * 2 * N));
    if (initial_positions && pl->N)
      LFR_CUDA(cudaMemcpyAsync(pl->pos_init.p, initial_positions, sizeof(double) * 2 * (size_t)pl->N,
                               cudaMemcpyHostToDevice, s));
    else
      LFR_CUDA(cudaMemsetAsync(pl->pos_init.p, 0, sizeof(double) * 2 * N, s));
    pl->pos_is_staged = false;
  }
  host_mark(0);
  LFR_TRY(build_buckets(pl, p));  // host work overlaps the copies above
  host_mark(1);
  // Zero-copy and the CTA tier: its preparation kernel can pull the records it keeps straight from the
  // pinned array, but SM loads over PCIe run at ~15 GB/s against ~50 GB/s for the copy engine
  // (profiles/README.md), so that pays only while those components hold less than ~0.3 of the edges
  // (one device of a multi-device solve); otherwise the whole array goes to HBM on the copy stream.
  uint64_t cta_cand = 0;
  for (uint64_t e : pl->large_cand) cta_cand += e;
  pl->cta_from_hbm = zc_edges && 10 * cta_cand > 3 * (uint64_t)p->n_edges;
  if (zc_edges && (pl->needs_hbm_edges || pl->cta_from_hbm)) {
    // mixed schedule: the Cholesky-warp tier reads edge records from global memory by index, so the
    // array goes to HBM after all — on its own stream, and only that tier waits for it
    if (!pl->copy_stream) LFR_CUDA(cudaStreamCreateWithFlags(&pl->copy_stream, cudaStreamNonBlocking));
    if (!pl->ev_edges) LFR_CUDA(cudaEventCreateWithFlags(&pl->ev_edges, cudaEventDisableTiming));
    LFR_TRY(upload(&pl->edges, p->edges, (size_t)p->n_edges, pl->copy_stream));
    LFR_CUDA(cudaEventRecord(pl->ev_edges, pl->copy_stream));
    pl->edges_in_hbm = true;
  }
  LFR_TRY(prepare_large(pl, p, s));
  LFR_TRY(upload(&pl->lists, pl->list_host.data(), pl->list_host.size(), s));
  if (pl->total_slots) {
    lfr::local_index_kernel<<<(pl->total_slots + 255) / 256, 256, 0, s>>>(
        pl->comp_ptr.as<uint32_t>(), pl->comp_nodes.as<uint32_t>(), pl->C, pl->total_slots,
        pl->local_of.as<uint32_t>());
    LFR_CUDA(cudaGetLastError());
  }
  if (pl->n_large) {
    // kept-edge records / in-edge lists, free-variable numbering and twins of the CTA-tier components,
    // built on the device; with zero-copy edges the kernel either pulls exactly the records these
    // components keep from the caller's pinned array, or reads the bulk copy (see above)
    lfr::DevProblem P = pl->dev();
    cudaStream_t ps = s;
    if (zc_edges && !pl->cta_from_hbm) {
      P.edges = zc_edges;
    } else if (zc_edges) {
      // behind the bulk copy on the copy stream, once the small arrays and local_of (stream s) are
      // there; the CTA-tier launches wait for ev_edges, the staging tiers do not
      if (!pl->ev_prep) LFR_CUDA(cudaEventCreateWithFlags(&pl->ev_prep, cudaEventDisableTiming));
      LFR_CUDA(cudaEventRecord(pl->ev_prep, s));
      LFR_CUDA(cudaStreamWaitEvent(pl->copy_stream, pl->ev_prep, 0));
      ps = pl->copy_stream;
    }
    lfr::cta_prepare_kernel<<<pl->n_large, lfr::kCtaThreads, 0, ps>>>(P, pl->cta_arrays(), pl->L_comps.as<lfr::CtaComp>());
    LFR_CUDA(cudaGetLastError());
    if (ps != s) LFR_CUDA(cudaEventRecord(pl->ev_edges, pl->copy_stream));
  }
  // streams for concurrent bucket launches
  const int want = std::min<int>(kMaxStreams, std::max<int>(0, (int)pl->buckets.size() + (int)pl->cta_groups.size() - 1));
  if (!pl->ev_fork) LFR_CUDA(cudaEventCreateWithFlags(&pl->ev_fork, cudaEventDisableTiming));
  while (pl->n_streams < want) {
    LFR_CUDA(cudaStreamCreateWithFlags(&pl->streams[pl->n_streams], cudaStreamNonBlocking));
    LFR_CUDA(cudaEventCreateWithFlags(&pl->ev_join[pl->n_streams], cudaEventDisableTiming));
    ++pl->n_streams;
  }
  return LFR_OK;
}

// Bytes of zero-copy staging pulls kept outstanding per device (stage_edges): large enough to cover
// the PCIe bandwidth-delay product, small enough that records arrive in dispatch order.
constexpr unsigned kZeroCopyPullWindow = 512u * 1024u;

int set_kernel_attrs() {
  static bool done_for_device[16] = {};  // per device, guarded by that device's workspace mutex / idempotent otherwise
  int dev = 0;
  LFR_CUDA(cudaGetDevice(&dev));
  if (dev >= 0 && dev < 16 && done_for_device[dev]) return LFR_OK;
  LFR_CUDA(cudaFuncSetAttribute(lfr::solve_cta_kernel<256, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  LFR_CUDA(cudaFuncSetAttribute(lfr::solve_cta_kernel<256, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  LFR_CUDA(cudaFuncSetAttribute(lfr::solve_cta_kernel<256, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  LFR_CUDA(cudaFuncSetAttribute(lfr::solve_warp_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                kMaxSmemPerBlock));
  LFR_CUDA(cudaFuncSetAttribute(lfr::solve_warp_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                kMaxSmemPerBlock));
  LFR_CUDA(cudaFuncSetAttribute(lfr::solve_warp2_kernel<4, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                kMaxSmemPerBlock));
  LFR_CUDA(cudaFuncSetAttribute(lfr::solve_warp2_kernel<4, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                kMaxSmemPerBlock));
  LFR_CUDA(cudaFuncSetAttribute(lfr::solve_warp2_kernel<4, 24>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                kMaxSmemPerBlock));
  LFR_CUDA(cudaFuncSetAttribute(lfr::solve_warp2_kernel<4, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                kMaxSmemPerBlock));
  LFR_CUDA(cudaFuncSetAttribute(lfr::solve_warp2_kernel<1, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                kMaxSmemPerBlock));
  LFR_CUDA(cudaFuncSetAttribute(lfr::solve_tile_kernel<64, 48>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                kMaxSmemPerBlock));
  LFR_CUDA(cudaFuncSetAttribute(lfr::solve_tile_kernel<64, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                kMaxSmemPerBlock));
  LFR_CUDA(cudaFuncSetAttribute(lfr::solve_tile_kernel<128, 80>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                kMaxSmemPerBlock));
  if (dev >= 0 && dev < 16) done_for_device[dev] = true;
  return LFR_OK;
}

int launch_solve(lfr_plan* pl, cudaStream_t s) {
  LFR_TRY(set_kernel_attrs());
  if (pl->N && !pl->pos_is_staged)
    LFR_CUDA(cudaMemcpyAsync(pl->pos.p, pl->pos_init.p, sizeof(double) * 2 * (size_t)pl->N,
                             cudaMemcpyDeviceToDevice, s));
  pl->pos_is_staged = false;  // a second launch on the same plan needs the reset again
  const lfr::DevProblem P_hbm = pl->dev();  // edges read from the HBM copy by global index
  lfr::DevProblem P_stage = P_hbm;          // edges pulled once into shared memory, possibly from the caller's pinned buffer
  if (pl->zc_edges) {
    P_stage.edges = pl->zc_edges;
    P_stage.pull_window = kZeroCopyPullWindow;
  }
  const bool hbm_edges_on_copy_stream = pl->zc_edges && pl->edges_in_hbm;
  const int nb = (int)pl->buckets.size();
  const int n_cta_launches = pl->n_large ? (int)pl->cta_groups.size() : 0;
  const int n_side = std::max(0, nb + n_cta_launches - 1);
  if (n_side > 0) LFR_CUDA(cudaEventRecord(pl->ev_fork, s));
  int side = 0;
  if (pl->n_large) {  // the CTA tier first: its components are the longest
    const lfr::CtaArrays A = pl->cta_arrays();
    for (const CtaGroup& g : pl->cta_groups) {
      cudaStream_t bs = s;
      if (n_side > 0) {
        bs = pl->streams[side++ % pl->n_streams];
        LFR_CUDA(cudaStreamWaitEvent(bs, pl->ev_fork, 0));
      }
      if (pl->zc_edges && pl->cta_from_hbm) LFR_CUDA(cudaStreamWaitEvent(bs, pl->ev_edges, 0));
      // dynamic shared memory for the CG vectors of the group's largest component: p, w, r, z, y
      // (2 doubles per free node each) and the preconditioner (3); solve_cta_kernel keeps in HBM
      // whatever does not fit under the 200 KB cap
      const size_t cg_bytes = std::min<size_t>(200 * 1024, (size_t)g.max_free * 13 * sizeof(double));
      const lfr::CtaComp* comps = pl->L_comps.as<lfr::CtaComp>() + g.first;
      const unsigned smem_doubles = (unsigned)(cg_bytes / sizeof(double));
      // (512-thread CTAs were measured too — profiles/r02_cta_tier_tuning.txt: slower at every size class)
      if (g.minb >= 4)
        lfr::solve_cta_kernel<256, 4><<<g.n, 256, cg_bytes, bs>>>(P_hbm, pl->K, A, comps, smem_doubles);
      else if (g.minb == 3)
        lfr::solve_cta_kernel<256, 3><<<g.n, 256, cg_bytes, bs>>>(P_hbm, pl->K, A, comps, smem_doubles);
      else
        lfr::solve_cta_kernel<256, 2><<<g.n, 256, cg_bytes, bs>>>(P_hbm, pl->K, A, comps, smem_doubles);
      LFR_CUDA(cudaGetLastError());
    }
  }
  for (int i = 0; i < nb; ++i) {
    const Bucket& b = pl->buckets[i];
    // bucket 0 runs on the caller's stream, the others on side streams forked from it
    cudaStream_t bs = s;
    if (i > 0) {
      bs = pl->streams[side++ % pl->n_streams];
      LFR_CUDA(cudaStreamWaitEvent(bs, pl->ev_fork, 0));
    }
    lfr::WarpBucket wb;
    wb.list = pl->lists.as<uint32_t>() + b.offset;
    wb.n = b.n;
    wb.emax = b.emax;
    wb.ncmax = b.ncmax;
    wb.n2max = b.n2max;
    wb.smem_per_warp = b.smem_per_warp;
    const size_t smem = (size_t)b.smem_per_warp * b.warps;
    const unsigned grid = (b.n + b.warps - 1) / b.warps;
    const lfr::DevProblem& P = b.stages_edges() ? P_stage : P_hbm;
    if (!b.stages_edges() && hbm_edges_on_copy_stream) LFR_CUDA(cudaStreamWaitEvent(bs, pl->ev_edges, 0));
    if (b.variant == 48)
      lfr::solve_tile_kernel<64, 48><<<b.n, 64, smem, bs>>>(P, pl->K, wb);
    else if (b.variant == 64)
      lfr::solve_tile_kernel<64, 64><<<b.n, 64, smem, bs>>>(P, pl->K, wb);
    else if (b.variant == 80)
      lfr::solve_tile_kernel<128, 80><<<b.n, 128, smem, bs>>>(P, pl->K, wb);
    else if (b.variant == 8)
      lfr::solve_warp2_kernel<4, 8><<<grid, 128, smem, bs>>>(P, pl->K, wb);
    else if (b.variant == 16)
      lfr::solve_warp2_kernel<4, 16><<<grid, 128, smem, bs>>>(P, pl->K, wb);
    else if (b.variant == 24 && b.warps == 4)
      lfr::solve_warp2_kernel<4, 24><<<grid, 128, smem, bs>>>(P, pl->K, wb);
    else if (b.variant == 32 && b.warps == 4)
      lfr::solve_warp2_kernel<4, 32><<<grid, 128, smem, bs>>>(P, pl->K, wb);
    else if (b.variant == 32)
      lfr::solve_warp2_kernel<1, 32><<<grid, 32, smem, bs>>>(P, pl->K, wb);
    else if (b.warps == 4)
      lfr::solve_warp_kernel<4><<<grid, 128, smem, bs>>>(P, pl->K, wb);
    else
      lfr::solve_warp_kernel<1><<<grid, 32, smem, bs>>>(P, pl->K, wb);
    LFR_CUDA(cudaGetLastError());
  }
  for (int k = 0; k < std::min(side, pl->n_streams); ++k) {  // join the side streams
    LFR_CUDA(cudaEventRecord(pl->ev_join[k], pl->streams[k]));
    LFR_CUDA(cudaStreamWaitEvent(s, pl->ev_join[k], 0));
  }
  return LFR_OK;
}

int download(lfr_plan* pl, cudaStream_t s, double* positions, lfr_stats* st) {
  const size_t nb = pl->stats_bytes();
  if (pl->h_stage_cap < nb) {
    if (pl->h_stage) cudaFreeHost(pl->h_stage);
    pl->h_stage = nullptr;
    pl->h_stage_cap = 0;
    LFR_CUDA(cudaMallocHost(&pl->h_stage, nb + nb / 4));
    pl->h_stage_cap = nb + nb / 4;
  }
  LFR_CUDA(cudaMemcpyAsync(pl->h_stage, pl->stats.p, nb, cudaMemcpyDeviceToHost, s));
  LFR_CUDA(cudaStreamSynchronize(s));
  const size_t Cp = pl->Cp;
  const double* h_cost0 = static_cast<const double*>(pl->h_stage);
  const double* h_cost1 = h_cost0 + Cp;
  const int32_t* h_iter = reinterpret_cast<const int32_t*>(h_cost1 + Cp);
  const int32_t* h_term = h_iter + Cp;
  const uint32_t* h_ls = reinterpret_cast<const uint32_t*>(h_term + Cp);
  const uint32_t* h_kept = h_ls + Cp;
  const int err = *reinterpret_cast<const int*>(h_kept + Cp);
  // the error flag is checked BEFORE anything is copied into the caller's position array (with
  // zero-copy write-back the components that did solve have already been written: on LFR_EINVAL
  // the array holds a mixture of start values and results)
  if (err) return fail(LFR_EINVAL, "edge with dst out of range or a self edge (found while staging edges on the device)");
  if (positions && pl->N && !pl->zc_positions) {
    LFR_CUDA(cudaMemcpyAsync(positions, pl->pos.p, sizeof(double) * 2 * (size_t)pl->N, cudaMemcpyDeviceToHost, s));
    LFR_CUDA(cudaStreamSynchronize(s));
  }
  if (st) {
    uint64_t ti = 0, tl = 0;
    for (uint32_t c = 0; c < pl->C; ++c) {
      ti += (uint64_t)h_iter[c];
      tl += h_ls[c];
    }
    if (pl->C) {
      if (st->iterations) std::memcpy(st->iterations, h_iter, sizeof(int32_t) * pl->C);
      if (st->termination) std::memcpy(st->termination, h_term, sizeof(int32_t) * pl->C);
      if (st->initial_cost) std::memcpy(st->initial_cost, h_cost0, sizeof(double) * pl->C);
      if (st->final_cost) std::memcpy(st->final_cost, h_cost1, sizeof(double) * pl->C);
    }
    st->total_iterations = ti;
    st->total_line_search_steps = tl;
    st->n_solved = pl->n_solved;
    st->n_kernel_launches = (uint32_t)pl->buckets.size() + (uint32_t)pl->cta_groups.size();
  }
  return LFR_OK;
}

int select_device(const lfr_options& o) {
  int n_dev = 0;
  LFR_CUDA(cudaGetDeviceCount(&n_dev));
  if (n_dev == 0) return fail(LFR_ENODEV, "no CUDA device");
  if (o.device < 0 || o.device >= n_dev) return fail(LFR_ENODEV, "device ordinal out of range");
  LFR_CUDA(cudaSetDevice(o.device));
  return LFR_OK;
}

// lfr_solve()'s workspace: per device (shared by all host threads, guarded by g_ws_mutex), one cached
// plan (grow-only device buffers), one non-blocking stream and the events that time the call — all
// created with that device current.  Kept until lfr_shutdown() or process exit (no destructor calls
// into CUDA during teardown).
struct DeviceWorkspace {
  lfr_plan* plan = nullptr;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[4] = {};
  bool ready = false;
};
constexpr int kMaxDevices = 16;
DeviceWorkspace g_ws[kMaxDevices];
std::mutex g_ws_mutex[kMaxDevices];  // one solve at a time per device workspace; distinct devices run concurrently

int ensure_workspace(int device) {
  DeviceWorkspace& ws = g_ws[device];
  if (ws.ready) return LFR_OK;
  LFR_CUDA(cudaStreamCreateWithFlags(&ws.stream, cudaStreamNonBlocking));
  for (int i = 0; i < 4; ++i) LFR_CUDA(cudaEventCreate(&ws.ev[i]));
  ws.plan = new lfr_plan();
  ws.plan->device = device;
  ws.ready = true;
  return LFR_OK;
}

// One device's part of a solve: uploads, launches, results.  `slot_owner` / `owner_id` restrict the
// plan to the dispatch slots this device owns (nullptr = all).  Caller holds g_ws_mutex[device].
int solve_on_device(const lfr_problem* p, const lfr_options& o, double* positions, lfr_stats* st,
                    const uint8_t* slot_owner, uint8_t owner_id, double* pos_scratch) {
  LFR_TRY(select_device(o));
  LFR_TRY(ensure_workspace(o.device));
  DeviceWorkspace& ws = g_ws[o.device];
  lfr_plan* pl = ws.plan;
  cudaStream_t s = ws.stream;
  pl->slot_owner = slot_owner;
  pl->owner_id = owner_id;
  // page-locked caller buffers are used in place (see include/lfr.h); pageable ones go through HBM
  const bool zero_copy = !(o.debug_flags & LFR_DBG_NO_ZERO_COPY);
  const float4* zc_edges = (zero_copy && p->n_edges) ? static_cast<const float4*>(device_view_of_pinned(p->edges)) : nullptr;
  double* zc_positions = (zero_copy && p->n_nodes) ? static_cast<double*>(device_view_of_pinned(positions)) : nullptr;
  g_host_t0 = std::chrono::steady_clock::now();
  LFR_CUDA(cudaEventRecord(ws.ev[0], s));
  LFR_TRY(fill_plan(pl, p, o, positions, s, /*stage_positions_directly=*/true, zc_edges, zc_positions));
  host_mark(2);
  LFR_CUDA(cudaEventRecord(ws.ev[1], s));
  LFR_TRY(launch_solve(pl, s));
  LFR_CUDA(cudaEventRecord(ws.ev[2], s));
  host_mark(3);
  // several devices, pageable positions: each device returns its copy into its own scratch array
  // and the caller merges the entries of the components it owns
  int rc = download(pl, s, (slot_owner && !zc_positions) ? pos_scratch : positions, st);
  if (pl->copy_stream && pl->zc_edges && pl->edges_in_hbm) {
    // the bulk copy reads the caller's buffer: it must be over before the call returns
    cudaError_t e = cudaStreamSynchronize(pl->copy_stream);
    if (e != cudaSuccess && rc == LFR_OK) rc = fail(cuda_code(e), cudaGetErrorString(e));
  }
  host_mark(4);
  pl->slot_owner = nullptr;
  if (rc) return rc;
  LFR_CUDA(cudaEventRecord(ws.ev[3], s));
  LFR_CUDA(cudaEventSynchronize(ws.ev[3]));
  host_mark(5);
  if (st) {
    float a = 0, b = 0, c = 0;
    cudaEventElapsedTime(&a, ws.ev[0], ws.ev[1]);
    cudaEventElapsedTime(&b, ws.ev[1], ws.ev[2]);
    cudaEventElapsedTime(&c, ws.ev[2], ws.ev[3]);
    st->h2d_ms = a;     // uploads of the arrays that go through HBM (+ schedule)
    st->kernel_ms = b;  // the solve kernels (with zero-copy: including their PCIe pulls)
    st->d2h_ms = c;
    st->total_ms = (double)a + b + c;
  }
  return LFR_OK;
}

}  // namespace

extern "C" {

int lfr_abi_version(void) { return LFR_ABI_VERSION; }
const char* lfr_backend(void) { return "b200"; }
const char* lfr_last_error(void) { return g_last_error.c_str(); }

void lfr_options_default(lfr_options* o) {
  if (!o) return;
  std::memset(o, 0, sizeof *o);
  o->bound = 1.0;                 // solve.cc:89
  o->cauchy_a = 0.25;             // solve.cc:111
  o->tukey_a = 0.0625;            // solve.cc:120
  o->tukey_variant = 1;
  o->max_num_iterations = 100;    // solve.cc:149
  o->max_num_consecutive_invalid_steps = 10;  // solve.cc:151
  o->max_num_line_search_step_size_iterations = 20;
  o->function_tolerance = 1e-4;   // solve.cc:152
  o->gradient_tolerance = 1e-8;   // solve.cc:153
  o->parameter_tolerance = 1e-4;  // solve.cc:154
  o->initial_trust_region_radius = 1e4;
  o->max_trust_region_radius = 1e16;
  o->min_trust_region_radius = 1e-32;
  o->min_relative_decrease = 1e-3;
  o->min_lm_diagonal = 1e-6;
  o->max_lm_diagonal = 1e32;
  o->line_search_sufficient_function_decrease = 1e-4;
  o->max_line_search_step_contraction = 1e-3;
  o->min_line_search_step_contraction = 0.6;
  o->min_line_search_step_size = 1e-9;
  o->n_threads = 8;
  o->device = 0;
  o->linear_solver = 0;
}

int lfr_plan_create(const lfr_problem* p, const lfr_options* opt, const double* initial_positions,
                    lfr_plan** out) {
  if (!out) return fail(LFR_EINVAL, "out is NULL");
  *out = nullptr;
  LFR_TRY(validate(p));
  lfr_options o;
  if (opt) o = *opt; else lfr_options_default(&o);
  LFR_TRY(select_device(o));
  lfr_plan* pl = new lfr_plan();
  pl->device = o.device;
  int rc = fill_plan(pl, p, o, initial_positions, 0);
  if (rc == LFR_OK) {
    cudaError_t e = cudaStreamSynchronize(0);
    if (e != cudaSuccess) rc = fail(cuda_code(e), cudaGetErrorString(e));
  }
  if (rc) {
    free_plan(pl);
    return rc;
  }
  *out = pl;
  return LFR_OK;
}

int lfr_plan_solve(lfr_plan* pl, void* stream) {
  if (!pl) return fail(LFR_EINVAL, "plan is NULL");
  LFR_CUDA(cudaSetDevice(pl->device));
  return launch_solve(pl, (cudaStream_t)stream);
}

int lfr_plan_num_launches(const lfr_plan* pl) {
  // kernels only: the device-to-device reset of `positions` is a copy, not a kernel
  return pl ? (int)pl->buckets.size() + (int)pl->cta_groups.size() : 0;
}

int lfr_plan_download(lfr_plan* pl, void* stream, double* positions, lfr_stats* st) {
  if (!pl) return fail(LFR_EINVAL, "plan is NULL");
  LFR_CUDA(cudaSetDevice(pl->device));
  return download(pl, (cudaStream_t)stream, positions, st);
}

int lfr_plan_traffic(lfr_plan* pl, void* stream, uint64_t* algorithmic_bytes, uint64_t* one_pass_bytes) {
  if (!pl) return fail(LFR_EINVAL, "plan is NULL");
  LFR_CUDA(cudaSetDevice(pl->device));
  cudaStream_t s = (cudaStream_t)stream;
  std::vector<unsigned char> blk(pl->stats_bytes());
  LFR_CUDA(cudaMemcpyAsync(blk.data(), pl->stats.p, blk.size(), cudaMemcpyDeviceToHost, s));
  LFR_CUDA(cudaStreamSynchronize(s));
  const int32_t* it = reinterpret_cast<const int32_t*>(blk.data() + 16 * (size_t)pl->Cp);
  const uint32_t* kept = reinterpret_cast<const uint32_t*>(blk.data() + 16 * (size_t)pl->Cp + 12 * (size_t)pl->Cp);
  uint64_t alg = 0, one = 0;
  for (uint32_t c = 0; c < pl->C; ++c) {
    if (pl->comp_size[c] <= 1) continue;
    const uint64_t pass = 80ull * kept[c] + 36ull * pl->comp_size[c];  // SURVEY 8d
    one += pass;
    alg += pass * (uint64_t)std::max(it[c], 1);
  }
  if (algorithmic_bytes) *algorithmic_bytes = alg;
  if (one_pass_bytes) *one_pass_bytes = one;
  return LFR_OK;
}

/* debug (LFR_DBG_PROFILE): per-slot cycle counters, 8 x uint64 each */
int lfr_debug_plan_cycles(lfr_plan* pl, unsigned long long* out) {
  if (!pl || !pl->profile) return fail(LFR_EINVAL, "plan was not created with LFR_DBG_PROFILE");
  LFR_CUDA(cudaSetDevice(pl->device));
  LFR_CUDA(cudaMemcpy(out, pl->cycles.p, sizeof(unsigned long long) * 8 * (size_t)pl->C, cudaMemcpyDeviceToHost));
  return LFR_OK;
}

int lfr_debug_plan_times(lfr_plan* pl, unsigned long long* out) {
  if (!pl || !pl->profile) return fail(LFR_EINVAL, "plan was not created with LFR_DBG_PROFILE");
  LFR_CUDA(cudaSetDevice(pl->device));
  LFR_CUDA(cudaMemcpy(out, pl->times.p, sizeof(unsigned long long) * 2 * (size_t)pl->C, cudaMemcpyDeviceToHost));
  return LFR_OK;
}

/* debug (LFR_DBG_PROFILE): counters of the last lfr_solve() of this thread on `device`:
   cycles [8 per slot], times [2 per slot] = %globaltimer ns at start / end of each component */
int lfr_debug_last_solve_profile(int device, unsigned long long* cycles, unsigned long long* times) {
  if (device < 0 || device >= kMaxDevices || !g_ws[device].ready || !g_ws[device].plan->profile)
    return fail(LFR_EINVAL, "no profiled lfr_solve() on this device / thread");
  lfr_plan* pl = g_ws[device].plan;
  LFR_CUDA(cudaSetDevice(device));
  if (cycles) LFR_CUDA(cudaMemcpy(cycles, pl->cycles.p, sizeof(unsigned long long) * 8 * (size_t)pl->C, cudaMemcpyDeviceToHost));
  if (times) LFR_CUDA(cudaMemcpy(times, pl->times.p, sizeof(unsigned long long) * 2 * (size_t)pl->C, cudaMemcpyDeviceToHost));
  return LFR_OK;
}

// host-only: best-of-`reps` time of the schedule construction (build_buckets), no device needed
int lfr_debug_time_schedule(const lfr_problem* p, const lfr_options* opt, int reps, double* best_us, int* n_launches,
                            uint64_t* digest) {
  if (!p || !best_us) return fail(LFR_EINVAL, "null argument");
  LFR_TRY(validate(p));
  lfr_plan pl;
  if (opt) pl.opt = *opt; else lfr_options_default(&pl.opt);
  pl.N = p->n_nodes;
  pl.C = p->n_components;
  pl.total_slots = p->n_components ? p->comp_ptr[p->n_components] : 0;
  double best = 1e300;
  for (int r = 0; r < std::max(reps, 1); ++r) {
    const auto t0 = std::chrono::steady_clock::now();
    LFR_TRY(build_buckets(&pl, p));
    best = std::min(best, std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t0).count());
  }
  if (digest) {  // FNV-1a over everything the launches depend on: the schedule must not depend on the thread count
    uint64_t h = 1469598103934665603ull;
    auto mix = [&](uint64_t v) {
      for (int i = 0; i < 8; ++i) {
        h ^= (v >> (8 * i)) & 0xff;
        h *= 1099511628211ull;
      }
    };
    mix(pl.n_solved);
    for (const Bucket& b : pl.buckets) {
      mix(b.offset); mix(b.n); mix((uint64_t)b.emax); mix((uint64_t)b.ncmax); mix((uint64_t)b.n2max);
      mix((uint64_t)b.smem_per_warp); mix((uint64_t)b.warps); mix((uint64_t)b.variant);
    }
    for (uint32_t c : pl.list_host) mix(c);
    for (size_t i = 0; i < pl.large_slots.size(); ++i) {
      mix(pl.large_slots[i]); mix(pl.large_cand[i]); mix(pl.large_free[i]); mix(pl.large_ell[i]);
    }
    *digest = h;
  }
  *best_us = best;
  if (n_launches) *n_launches = (int)pl.buckets.size() + (pl.large_slots.empty() ? 0 : 1);  // (CTA tier counted once here)
  return LFR_OK;
}

int lfr_debug_last_host_marks(double* out6) {
  for (int i = 0; i < 6; ++i) out6[i] = g_host_marks[i];
  return LFR_OK;
}

void lfr_plan_destroy(lfr_plan* pl) {
  if (!pl) return;
  cudaSetDevice(pl->device);
  free_plan(pl);
}

int lfr_solve(const lfr_problem* p, const lfr_options* opt, double* positions, lfr_stats* st) {
  LFR_TRY(validate(p));
  if (p->n_nodes && !positions) return fail(LFR_EINVAL, "positions is NULL");
  lfr_options o;
  if (opt) o = *opt; else lfr_options_default(&o);
  if (o.device < 0 || o.device >= kMaxDevices) return fail(LFR_EUNSUPPORTED, "device ordinal out of [0, 16)");
  std::lock_guard<std::mutex> lock(g_ws_mutex[o.device]);
  return solve_on_device(p, o, positions, st, nullptr, 0, nullptr);
}

void* lfr_host_alloc(uint64_t bytes) {
  void* p = nullptr;
  if (cudaHostAlloc(&p, bytes ? (size_t)bytes : 1, cudaHostAllocPortable) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return p;
}

void lfr_host_free(void* p) {
  if (p) cudaFreeHost(p);
}

void lfr_shutdown(void) {
  // release the cached per-device workspaces of lfr_solve() / lfr_solve_multi() (device buffers,
  // pinned staging, streams, events); the next call re-creates what it needs
  for (int d = 0; d < kMaxDevices; ++d) {
    std::lock_guard<std::mutex> lock(g_ws_mutex[d]);
    DeviceWorkspace& ws = g_ws[d];
    if (!ws.ready) continue;
    if (cudaSetDevice(d) == cudaSuccess) {
      free_plan(ws.plan);
      for (int i = 0; i < 4; ++i)
        if (ws.ev[i]) cudaEventDestroy(ws.ev[i]);
      if (ws.stream) cudaStreamDestroy(ws.stream);
    }
    ws = DeviceWorkspace();
  }
}

int lfr_solve_multi(const lfr_problem* p, const lfr_options* opt, const int32_t* devices, int32_t n_devices,
                    double* positions, lfr_stats* st, lfr_multi_info* info) {
  LFR_TRY(validate(p));
  if (p->n_nodes && !positions) return fail(LFR_EINVAL, "positions is NULL");
  if (!devices || n_devices < 1 || n_devices > kMaxDevices) return fail(LFR_EINVAL, "devices: need 1..16 device ordinals");
  for (int d = 0; d < n_devices; ++d) {
    if (devices[d] < 0 || devices[d] >= kMaxDevices) return fail(LFR_EUNSUPPORTED, "device ordinal out of [0, 16)");
    for (int e = 0; e < d; ++e)
      if (devices[e] == devices[d]) return fail(LFR_EINVAL, "devices: duplicate ordinal");
  }
  lfr_options o0;
  if (opt) o0 = *opt; else lfr_options_default(&o0);
  const uint32_t C = p->n_components;
  // ---- LPT packing of the dispatch slots by directed-edge count, largest first (the reference's
  // largest-first queue, solve.cc:599-604, spread over devices); deterministic
  std::vector<uint64_t> weight(C, 0);
  const uint32_t total_slots = C ? p->comp_ptr[C] : 0;
  for (uint32_t c = 0; c < C; ++c) {
    const uint32_t beg = p->comp_ptr[c], end = p->comp_ptr[c + 1];
    if (end < beg || end > total_slots) return fail(LFR_EINVAL, "comp_ptr not monotone");
    if (end - beg <= 1) continue;
    for (uint32_t i = beg; i < end; ++i) {
      const uint32_t v = p->comp_nodes[i];
      if (v >= p->n_nodes) return fail(LFR_EINVAL, "comp_nodes out of range");
      weight[c] += p->row_ptr[v + 1] - p->row_ptr[v];
    }
  }
  std::vector<uint32_t> order(C);
  for (uint32_t c = 0; c < C; ++c) order[c] = c;
  std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return weight[a] > weight[b]; });
  std::vector<uint8_t> owner(C, 0);
  std::vector<uint64_t> load(n_devices, 0);
  std::vector<uint32_t> n_slots(n_devices, 0);
  for (uint32_t c : order) {
    int best = 0;
    for (int d = 1; d < n_devices; ++d)
      if (load[d] < load[best]) best = d;
    owner[c] = (uint8_t)best;
    load[best] += weight[c];
    if (weight[c]) ++n_slots[best];
  }
  // ---- one host thread per device: upload the (small) per-node arrays, launch, collect.  With
  // page-locked caller buffers every device pulls only ITS components' edge records from the shared
  // host array and writes its results straight into `positions` (disjoint entries): the edge data is
  // partitioned without ever being copied, and no collective is needed.
  std::vector<lfr_stats> dst(n_devices);
  std::vector<std::vector<int32_t>> d_iter(n_devices), d_term(n_devices);
  std::vector<std::vector<double>> d_c0(n_devices), d_c1(n_devices), d_pos(n_devices);
  std::vector<int> rcs(n_devices, LFR_OK);
  std::vector<std::string> errs(n_devices);
  const bool pos_pinned = !(o0.debug_flags & LFR_DBG_NO_ZERO_COPY) && p->n_nodes && device_view_of_pinned(positions) != nullptr;
  auto work = [&](int d) {
    lfr_options o = o0;
    o.device = devices[d];
    std::memset(&dst[d], 0, sizeof(lfr_stats));
    d_iter[d].assign(C, 0);
    d_term[d].assign(C, 0);
    d_c0[d].assign(C, 0.0);
    d_c1[d].assign(C, 0.0);
    dst[d].iterations = d_iter[d].data();
    dst[d].termination = d_term[d].data();
    dst[d].initial_cost = d_c0[d].data();
    dst[d].final_cost = d_c1[d].data();
    if (!pos_pinned) d_pos[d].assign(2 * (size_t)p->n_nodes, 0.0);
    std::lock_guard<std::mutex> lock(g_ws_mutex[o.device]);
    rcs[d] = solve_on_device(p, o, positions, &dst[d], owner.data(), (uint8_t)d, pos_pinned ? nullptr : d_pos[d].data());
    if (rcs[d]) errs[d] = g_last_error;
  };
  if (n_devices == 1) {
    work(0);
  } else {
    std::vector<std::thread> threads;
    for (int d = 0; d < n_devices; ++d) threads.emplace_back(work, d);
    for (auto& t : threads) t.join();
  }
  for (int d = 0; d < n_devices; ++d)
    if (rcs[d]) return fail(rcs[d], "device " + std::to_string(devices[d]) + ": " + errs[d]);
  // ---- merge by owner
  if (!pos_pinned) {
    for (uint32_t c = 0; c < C; ++c) {
      const uint32_t beg = p->comp_ptr[c], end = p->comp_ptr[c + 1];
      if (end - beg <= 1) continue;
      const double* src = d_pos[owner[c]].data();
      for (uint32_t i = beg; i < end; ++i) {
        const size_t v = p->comp_nodes[i];
        positions[2 * v] = src[2 * v];
        positions[2 * v + 1] = src[2 * v + 1];
      }
    }
  }
  if (st) {
    uint64_t ti = 0, tl = 0;
    uint32_t ns = 0, nk = 0;
    double h = 0, k = 0, dd = 0, tt = 0;
    for (int d = 0; d < n_devices; ++d) {
      ti += dst[d].total_iterations;
      tl += dst[d].total_line_search_steps;
      ns += dst[d].n_solved;
      nk += dst[d].n_kernel_launches;
      h = std::max(h, dst[d].h2d_ms);
      k = std::max(k, dst[d].kernel_ms);
      dd = std::max(dd, dst[d].d2h_ms);
      tt = std::max(tt, dst[d].total_ms);
    }
    for (uint32_t c = 0; c < C; ++c) {
      const int d = owner[c];
      if (st->iterations) st->iterations[c] = d_iter[d][c];
      if (st->termination) st->termination[c] = d_term[d][c];
      if (st->initial_cost) st->initial_cost[c] = d_c0[d][c];
      if (st->final_cost) st->final_cost[c] = d_c1[d][c];
    }
    st->total_iterations = ti;
    st->total_line_search_steps = tl;
    st->n_solved = ns;
    st->n_kernel_launches = nk;
    st->h2d_ms = h;       // maxima over the devices (they run concurrently)
    st->kernel_ms = k;
    st->d2h_ms = dd;
    st->total_ms = tt;
  }
  if (info) {
    for (int d = 0; d < n_devices && d < 16; ++d) {
      info->kernel_ms[d] = dst[d].kernel_ms;
      info->total_ms[d] = dst[d].total_ms;
      info->n_slots[d] = n_slots[d];
      info->n_edges[d] = load[d];
    }
    info->zero_copy = (pos_pinned && p->n_edges && device_view_of_pinned(p->edges) != nullptr) ? 1 : 0;
  }
  return LFR_OK;
}

int lfr_debug_edge_eval(const lfr_edge* edges, const uint8_t* kind, uint64_t n, const double* xs,
                        const double* xd, const lfr_options* opt, double* r, double* jac, double* rho) {
  lfr_options o;
  if (opt) o = *opt; else lfr_options_default(&o);
  LFR_TRY(select_device(o));
  if (n == 0) return LFR_OK;
  DevBuf d_e, d_k, d_xs, d_xd, d_r, d_j, d_rho;
  int rc = LFR_OK;
  auto run = [&]() -> int {
    LFR_TRY(upload(&d_e, edges, n, 0));
    LFR_TRY(upload(&d_k, kind, n, 0));
    LFR_TRY(upload(&d_xs, xs, 2 * n, 0));
    LFR_TRY(upload(&d_xd, xd, 2 * n, 0));
    LFR_TRY(d_r.reserve(n * 16));
    LFR_TRY(d_j.reserve(n * 32));
    LFR_TRY(d_rho.reserve(n * 24));
    lfr::edge_eval_kernel<<<(unsigned)((n + 127) / 128), 128>>>(d_e.as<float4>(), d_k.as<uint8_t>(), n,
                                                               d_xs.as<double>(), d_xd.as<double>(),
                                                               make_consts(o), d_r.as<double>(), d_j.as<double>(),
                                                               d_rho.as<double>());
    LFR_CUDA(cudaGetLastError());
    LFR_CUDA(cudaMemcpy(r, d_r.p, n * 16, cudaMemcpyDeviceToHost));
    LFR_CUDA(cudaMemcpy(jac, d_j.p, n * 32, cudaMemcpyDeviceToHost));
    LFR_CUDA(cudaMemcpy(rho, d_rho.p, n * 24, cudaMemcpyDeviceToHost));
    return LFR_OK;
  };
  rc = run();
  d_e.release(); d_k.release(); d_xs.release(); d_xd.release(); d_r.release(); d_j.release(); d_rho.release();
  return rc;
}

/* test hook: real roots in [lo, hi] of n quartics (5 coefficients each, highest degree first,
   leading coefficient != 0) by the line search's root finders; use_grid = 1 -> Budan-Fourier grid
   isolation (the production route), 0 -> derivative recursion */
int lfr_debug_quartic_roots(const double* coef, const double* lohi, uint64_t n, int use_grid, double* roots,
                            int* counts) {
  lfr_options o;
  lfr_options_default(&o);
  LFR_TRY(select_device(o));
  if (n == 0) return LFR_OK;
  DevBuf d_c, d_l, d_r, d_n;
  auto run = [&]() -> int {
    LFR_TRY(upload(&d_c, coef, 5 * n, 0));
    LFR_TRY(upload(&d_l, lohi, 2 * n, 0));
    LFR_TRY(d_r.reserve(n * 32));
    LFR_TRY(d_n.reserve(n * 4));
    lfr::quartic_roots_kernel<<<(unsigned)((n + 3) / 4), 128>>>(d_c.as<double>(), d_l.as<double>(), (int)n, use_grid,
                                                                d_r.as<double>(), d_n.as<int>());
    LFR_CUDA(cudaGetLastError());
    LFR_CUDA(cudaMemcpy(roots, d_r.p, n * 32, cudaMemcpyDeviceToHost));
    LFR_CUDA(cudaMemcpy(counts, d_n.p, n * 4, cudaMemcpyDeviceToHost));
    return LFR_OK;
  };
  const int rc = run();
  d_c.release(); d_l.release(); d_r.release(); d_n.release();
  return rc;
}

/* test hook: the line search's interpolating-polynomial minimiser on n cases of 11 doubles
   {f0, g0, x1, f1, g1, three, x2, f2, g2, lo, hi}; out[n] = selected step size */
int lfr_debug_ls_minimizer(const double* cases, uint64_t n, double* out) {
  lfr_options o;
  lfr_options_default(&o);
  LFR_TRY(select_device(o));
  if (n == 0) return LFR_OK;
  DevBuf d_i, d_o;
  auto run = [&]() -> int {
    LFR_TRY(upload(&d_i, cases, 11 * n, 0));
    LFR_TRY(d_o.reserve(n * 8));
    lfr::ls_minimizer_kernel<<<(unsigned)((n + 3) / 4), 128>>>(d_i.as<double>(), (int)n, d_o.as<double>());
    LFR_CUDA(cudaGetLastError());
    LFR_CUDA(cudaMemcpy(out, d_o.p, n * 8, cudaMemcpyDeviceToHost));
    return LFR_OK;
  };
  const int rc = run();
  d_i.release(); d_o.release();
  return rc;
}

}  // extern "C"
