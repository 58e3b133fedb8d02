// ba_solver.cu — host side of HP2: problem flattening/tiling, the Levenberg-Marquardt
// trust-region loop (Ceres 2.0.0 TrustRegionMinimizer + LevenbergMarquardtStrategy
// semantics, SURVEY.md Appendix A.1/A.2), PCG on the reduced camera system, and the
// C ABI of include/psfm_b200.h.
//
// Drop-in target: colmap::BundleAdjuster::Solve
//   (reference sfm/gmapper/src/optim/bundle_adjustment.cc:259-320), problem assembly
//   rules from :326-447 / :500-544, solver selection rule :276-286, option policy
//   controllers/global_mapper.cc:41-71.
// There is no CPU path: every numeric step below is a kernel launch.
#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cmath>
#include <mutex>
#include <thread>
#include <vector>

#include "ba_small_kernels.cuh"
#include "ba_structure.cuh"
#include "ba_schur_explicit.cuh"
#include "ba_band_chol.cuh"
#include "ba_refine.cuh"
#include "dist.cuh"

namespace psfm {
namespace ba {

struct EventPool {
  std::vector<cudaEvent_t> ev;
  size_t used = 0;
  cudaEvent_t get() {
    if (used == ev.size()) {
      cudaEvent_t e;
      PSFM_CUDA(cudaEventCreate(&e));
      ev.push_back(e);
    }
    return ev[used++];
  }
  void reset() { used = 0; }
  ~EventPool() {
    for (auto e : ev) cudaEventDestroy(e);
  }
};

struct HostScalars {   // pinned
  double lin_cost;
  double gmax;
  double prep_fail;
  double step[4];      // sum m(r+m/2), |dX|^2, |Xc|^2, candidate cost
  double rep[2];       // |dcam|^2, |cam_c|^2   (must follow step: one copy of six doubles, compute_step)
  double x2;
  PcgState pcg;
  int chol_fail;
  int pad;
};

}  // namespace ba
}  // namespace psfm

using namespace psfm;
using namespace psfm::ba;

// Pinned host staging is expensive to allocate (cudaMallocHost of 12 MB costs ~10 ms): buffers
// are recycled across solver instances through a small process-wide free list.
namespace {
struct PinnedPool {
  std::mutex mu;
  std::vector<std::pair<void*, size_t>> free_list;
  void* acquire(size_t bytes, size_t* got) {
    {
      std::lock_guard<std::mutex> lk(mu);
      int best = -1;
      for (int i = 0; i < (int)free_list.size(); ++i)
        if (free_list[i].second >= bytes && (best < 0 || free_list[i].second < free_list[best].second)) best = i;
      if (best >= 0) {
        void* p = free_list[best].first;
        *got = free_list[best].second;
        free_list.erase(free_list.begin() + best);
        return p;
      }
    }
    void* p = nullptr;
    if (cudaMallocHost(&p, bytes) != cudaSuccess) return nullptr;
    *got = bytes;
    return p;
  }
  void release(void* p, size_t bytes) {
    if (!p) return;
    std::lock_guard<std::mutex> lk(mu);
    if (free_list.size() < 8) { free_list.push_back({p, bytes}); return; }
    cudaFreeHost(p);
  }
};
PinnedPool g_pinned;
}  // namespace

struct StreamHolder {   // declared first in the solver => destroyed last (after every DBuf)
  cudaStream_t s = nullptr;
  cudaStream_t copy = nullptr;      // second H2D queue: the coordinates travel while the index arrays are being sorted
  cudaEvent_t ev_idx = nullptr, ev_xy = nullptr;
  ~StreamHolder() {
    if (copy) { cudaStreamSynchronize(copy); cudaStreamDestroy(copy); }
    if (s) { cudaStreamSynchronize(s); cudaStreamDestroy(s); }
    if (ev_idx) cudaEventDestroy(ev_idx);
    if (ev_xy) cudaEventDestroy(ev_xy);
  }
};

struct psfm_ba_solver {
  StreamHolder sh;
  int F = 0, P_total = 0, P = 0, M = 0, C = 0, NS = 0, NB = 0, T = 0, nseg = 0, tile = 256, maxL = 0;
  int cap_ns = 1, cap_np = 1;
  // the caller's observations stay on the device for the life of the solver; `alive` marks the ones
  // still in the problem (the filters of the refinement loop clear bits, rebuild_structure re-packs)
  int M0 = 0;
  long long num_alive = 0;
  bool structure_dirty = false;
  DBuf<int> d_in_img, d_in_pt;
  DBuf<double2> d_in_xy;
  DBuf<unsigned char> d_alive;
  DBuf<double> d_pt_error;       // [P_total] Point3D::Error of the last point filter (NaN: not set)
  DBuf<unsigned long long> d_count;
  // host structure / config
  std::vector<int> pt_orig;      // internal point -> caller's point id
  std::vector<int> obs_orig;     // sorted observation -> caller's observation index
  std::vector<int> image_camera;
  std::vector<unsigned char> pose_constant, tvec_mask, camera_constant, img_has_obs, cam_has_obs;
  int flags_world = 1;           // world size for which img_has_obs / cam_has_obs have been made global
  // host state (caller layout)
  std::vector<double> h_qvec, h_tvec, h_K;   // the points' state of record is pin_state's X part (tile order, own points only)
  // device structure
  DBuf<int> d_tile_start, d_tile_pt, d_pt_ptr, d_obs_img, d_obs_pt, d_cseg_ptr, d_cseg_img, d_img_cam;
  DBuf<unsigned short> d_tile_perm, d_cseg_off, d_obs_lseg, d_obs_lpt;
  DBuf<int> d_obs_orig;
  DBuf<double2> d_obs_xy;
  // pipeline form of the structure (ba_tile_pipe.cuh)
  bool pipe = false;
  int sm_count = 0;
  DBuf<int4> d_tile_hdr;
  DBuf<int> d_pstart_rel, d_cseg_off32;
  DBuf<double> d_seg_pose;
  DBuf<unsigned char> d_active;
  // device state
  DBuf<double> d_pose[2], d_X[2], d_K[2];
  int cur = 0;
  // linearisation
  DBuf<double> d_r, d_a, d_pose16, d_xs, d_hpp, d_gp, d_wk, d_hinv, d_w, d_scale_c, d_scale_p;
  // reduced system / PCG
  DBuf<double> d_lin, d_prep, d_step, d_rep, d_gmax, d_x2, d_Dc2, d_Minv, d_rhs, d_x, d_rv, d_p, d_z, d_y, d_zero;
  DBuf<double> d_camrep, d_yrep;   // [NREP] replicas of the per-image accumulators (see ba_kernels.cuh)
  // explicit Schur complement (exact mode, ba_schur_explicit.cuh)
  bool pairs_ready = false;
  // k_point_blocks of the current linearisation at this radius is already in d_hinv / d_w / d_prep (rank-local,
  // not yet all-reduced): linearize_and_measure computes it for gradient_max_norm, compute_step reuses it
  bool pb_fresh = false;
  double pb_radius = 0.0;
  int nblocks = 0, nchunks = 0, bw = 0;
  long long npairs = 0;
  DBuf<unsigned long long> d_entries;
  DBuf<int> d_blk_key, d_chunk_blk, d_cholfail;
  DBuf<unsigned long long> d_cholprof;
  DBuf<unsigned int> d_cholbar;
  DBuf<double> d_cholLp, d_cholLd;
  DBuf<long long> d_chunk_beg;
  DBuf<double> d_W, d_WH, d_xcam, d_xcamrep, d_Sblk, d_S;
  // fused tile path (k_schur_tile): tile-local pair tasks and the band-block accumulator
  bool fused = false;
  int span = 0, ntasks = 0, band_nrep = 1;
  size_t band_n = 0;
  DBuf<unsigned int> d_tentries;
  DBuf<int> d_task_slot, d_tile_task;
  DBuf<int2> d_task_rng;
  DBuf<double> d_xband, d_bandrep;      // d_xband = [xcam F*NVX2 | Sband band_n] (one all-reduce)
  // single-CTA sliding-window band Cholesky (ba_band_chol.cuh): compact band matrix, factor, scratch
  bool band_chol = false;
  BandWork bwk;             // plan + buffers of k_band_chol
  DBuf<PcgState> d_pcg;
  HostScalars* hs = nullptr;
  double* pin_state = nullptr;     // pinned staging of the state: pose (8F) | X (3P) | K (3C)
  size_t pin_state_bytes = 0, hs_bytes = 0;
  cudaStream_t stream = nullptr;
  EventPool events;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev_lin, ev_sp, ev_sw, ev_pairs, ev_chol;

  TileCtx tc() const {
    TileCtx t;
    t.tile_start = d_tile_start.p; t.tile_pt = d_tile_pt.p; t.pt_ptr = d_pt_ptr.p;
    t.obs_img = d_obs_img.p; t.obs_pt = d_obs_pt.p; t.obs_xy = d_obs_xy.p;
    t.obs_lseg = d_obs_lseg.p; t.obs_lpt = d_obs_lpt.p; t.cap_ns = cap_ns; t.cap_np = cap_np;
    t.tile_perm = d_tile_perm.p; t.cseg_ptr = d_cseg_ptr.p; t.cseg_img = d_cseg_img.p;
    t.cseg_off = d_cseg_off.p; t.img_cam = d_img_cam.p;
    t.F = F; t.P = P; t.M = M; t.C = C; t.T = T;
    return t;
  }
  ~psfm_ba_solver() {
    if (stream) cudaStreamSynchronize(stream);
    g_pinned.release(hs, hs_bytes);
    g_pinned.release(pin_state, pin_state_bytes);
  }
};

namespace {

double now_s() {
  return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// ---------------------------------------------------------------- structure

struct PhaseTimer {
  bool on;
  double t;
  explicit PhaseTimer() : on(getenv("PSFM_TIMING") != nullptr), t(now_s()) {}
  void mark(const char* what) {
    if (!on) return;
    const double n = now_s();
    fprintf(stderr, "[psfm timing] %-28s %8.2f ms\n", what, 1e3 * (n - t));
    t = n;
  }
};

template <typename T>
void d2h_sync(cudaStream_t st, T* dst, const T* src, size_t n) {
  if (n) PSFM_CUDA(cudaMemcpyAsync(dst, src, n * sizeof(T), cudaMemcpyDeviceToHost, st));
  PSFM_CUDA(cudaStreamSynchronize(st));
}

inline unsigned grid_for(size_t n, int block = 256) { return (unsigned)((n + block - 1) / block); }

// Configuration and the caller's observations -> device (once per solver).
int upload_problem(psfm_ba_solver* S, const psfm_ba_problem* pb) {
  const int F = pb->num_images, Pt = pb->num_points, M = pb->num_observations, C = pb->num_cameras;
  if (F <= 0 || C <= 0 || Pt < 0 || M < 0) { set_error("psfm_ba_create: bad sizes"); return PSFM_ERR_INVALID; }
  S->F = F; S->P_total = Pt; S->M = M; S->M0 = M; S->num_alive = M; S->C = C; S->NS = 6 * F + 3 * C; S->NB = 2 * F + C;
  S->image_camera.assign(pb->image_camera, pb->image_camera + F);
  for (int i = 0; i < F; ++i)
    if (S->image_camera[i] < 0 || S->image_camera[i] >= C) { set_error("image_camera out of range"); return PSFM_ERR_INVALID; }
  S->pose_constant.assign(F, 0); S->tvec_mask.assign(F, 0); S->camera_constant.assign(C, 0);
  if (pb->pose_constant) S->pose_constant.assign(pb->pose_constant, pb->pose_constant + F);
  if (pb->tvec_constant_mask) S->tvec_mask.assign(pb->tvec_constant_mask, pb->tvec_constant_mask + F);
  if (pb->camera_constant) S->camera_constant.assign(pb->camera_constant, pb->camera_constant + C);
  cudaStream_t st = S->stream;
  S->d_img_cam.alloc(F, st); S->d_img_cam.upload(S->image_camera.data(), F, st);
  S->d_in_img.alloc(M, st); S->d_in_pt.alloc(M, st); S->d_in_xy.alloc(M, st); S->d_alive.alloc(M, st);
  S->d_in_img.upload(pb->obs_image, M, st); S->d_in_pt.upload(pb->obs_point, M, st);
  // the coordinates (half of the bytes) follow on the copy queue: counting, ordering and sorting need the
  // indices only, k_st_gather waits for ev_xy
  PSFM_CUDA(cudaEventRecord(S->sh.ev_idx, st));
  PSFM_CUDA(cudaStreamWaitEvent(S->sh.copy, S->sh.ev_idx, 0));
  S->d_in_xy.upload(reinterpret_cast<const double2*>(pb->obs_xy), M, S->sh.copy);
  PSFM_CUDA(cudaEventRecord(S->sh.ev_xy, S->sh.copy));
  PSFM_CUDA(cudaMemsetAsync(S->d_alive.p, 1, (size_t)(M ? M : 1), st));
  S->d_count.alloc(1, st);
  return PSFM_OK;
}

// Device-side flattening of the ALIVE observations into tiles (ba_structure.cuh).  Called at
// creation and again whenever a filter removed observations: the observations are re-packed
// from the resident arrays, nothing is uploaded again.
int build_structure(psfm_ba_solver* S) {
  PhaseTimer tm;
  const int F = S->F, Pt = S->P_total, C = S->C;
  cudaStream_t st = S->stream;
  S->img_has_obs.assign(F, 0); S->cam_has_obs.assign(C, 0);
  S->flags_world = 1;
  DBuf<int> c_img, c_pt, sel, cnt, min_img, order, keys32, keys32_out, pt_new, cnt_sorted, idx, idx_out, tile_ns, bad;
  DBuf<double2> c_xy;
  DBuf<unsigned long long> keys, keys_out;
  DBuf<unsigned char> has_obs, tmp;
  int M = S->M0;
  const int* in_img_p = S->d_in_img.p;
  const int* in_pt_p = S->d_in_pt.p;
  const double2* in_xy_p = S->d_in_xy.p;
  if (S->num_alive != S->M0) {
    PSFM_CUDA(cudaStreamWaitEvent(st, S->sh.ev_xy, 0));
    // stream compaction of the alive observations (index select + gather)
    DBuf<int> iota, nsel;
    iota.alloc(S->M0, st); sel.alloc(S->M0, st); nsel.alloc(1, st);
    k_st_iota<<<grid_for(S->M0), 256, 0, st>>>(iota.p, S->M0); PSFM_LAUNCH_CHECK();
    size_t need = 0;
    cub::DeviceSelect::Flagged(nullptr, need, iota.p, S->d_alive.p, sel.p, nsel.p, S->M0, st);
    DBuf<unsigned char> t2; t2.alloc(need + 256, st);
    cub::DeviceSelect::Flagged(t2.p, need, iota.p, S->d_alive.p, sel.p, nsel.p, S->M0, st);
    int h_n = 0;
    PSFM_CUDA(cudaMemcpyAsync(&h_n, nsel.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    PSFM_CUDA(cudaStreamSynchronize(st));
    M = h_n;
    c_img.alloc(M, st); c_pt.alloc(M, st); c_xy.alloc(M, st);
    if (M) { k_gather_alive<<<grid_for(M), 256, 0, st>>>(sel.p, M, S->d_in_img.p, S->d_in_pt.p, S->d_in_xy.p, c_img.p, c_pt.p, c_xy.p); PSFM_LAUNCH_CHECK(); }
    in_img_p = c_img.p; in_pt_p = c_pt.p; in_xy_p = c_xy.p;
    S->num_alive = M;
  }
  S->M = M;
  cnt.alloc(Pt, st); min_img.alloc(Pt, st); has_obs.alloc(F, st); bad.alloc(1, st);
  has_obs.zero(st); bad.zero(st);
  if (Pt) { k_st_init<<<grid_for(Pt), 256, 0, st>>>(cnt.p, min_img.p, Pt, F); PSFM_LAUNCH_CHECK(); }
  if (M) { k_st_count<<<grid_for(M), 256, 0, st>>>(in_img_p, in_pt_p, M, F, Pt, cnt.p, min_img.p, has_obs.p, bad.p); PSFM_LAUNCH_CHECK(); }
  // internal point order: observed points by (first image, id); unobserved (key F) last
  order.alloc(Pt, st); keys32.alloc(Pt, st); keys32_out.alloc(Pt, st); idx.alloc(std::max(Pt, M), st); idx_out.alloc(std::max(Pt, M), st);
  pt_new.alloc(Pt, st); cnt_sorted.alloc((size_t)Pt + 1, st);
  int fbits = 1; while ((1 << fbits) <= F) ++fbits;
  size_t tmp_bytes = 0, need = 0;
  if (Pt) {
    k_st_iota<<<grid_for(Pt), 256, 0, st>>>(idx.p, Pt); PSFM_LAUNCH_CHECK();
    cub::DeviceRadixSort::SortPairs(nullptr, need, min_img.p, keys32_out.p, idx.p, order.p, Pt, 0, fbits, st);
    tmp_bytes = std::max(tmp_bytes, need);
    cub::DeviceScan::ExclusiveSum(nullptr, need, cnt_sorted.p, cnt_sorted.p, Pt + 1, st);
    tmp_bytes = std::max(tmp_bytes, need);
  }
  int pbits = 1; while ((1ll << pbits) <= (long long)Pt) ++pbits;
  keys.alloc(M, st); keys_out.alloc(M, st);
  if (M) {
    cub::DeviceRadixSort::SortPairs(nullptr, need, keys.p, keys_out.p, idx.p, idx_out.p, M, 0, 32 + pbits, st);
    tmp_bytes = std::max(tmp_bytes, need);
  }
  tmp.alloc(tmp_bytes + 256, st);
  std::vector<int> h_cnt(Pt);
  if (Pt) {
    need = tmp_bytes + 256;
    cub::DeviceRadixSort::SortPairs(tmp.p, need, min_img.p, keys32_out.p, idx.p, order.p, Pt, 0, fbits, st);
    k_st_rank<<<grid_for(Pt), 256, 0, st>>>(order.p, cnt.p, Pt, pt_new.p, cnt_sorted.p); PSFM_LAUNCH_CHECK();
  }
  PSFM_CUDA(cudaMemsetAsync(cnt_sorted.p + Pt, 0, sizeof(int), st));
  // host needs: validity, observed flags, point order, counts
  int h_bad = 0;
  std::vector<unsigned char> h_has(F);
  std::vector<int> h_order(Pt), h_cs(Pt);
  PSFM_CUDA(cudaMemcpyAsync(&h_bad, bad.p, sizeof(int), cudaMemcpyDeviceToHost, st));
  PSFM_CUDA(cudaMemcpyAsync(h_has.data(), has_obs.p, F, cudaMemcpyDeviceToHost, st));
  if (Pt) {
    PSFM_CUDA(cudaMemcpyAsync(h_order.data(), order.p, sizeof(int) * Pt, cudaMemcpyDeviceToHost, st));
    PSFM_CUDA(cudaMemcpyAsync(h_cs.data(), cnt_sorted.p, sizeof(int) * Pt, cudaMemcpyDeviceToHost, st));
  }
  PSFM_CUDA(cudaStreamSynchronize(st));
  if (h_bad) { set_error("observation index out of range"); return PSFM_ERR_INVALID; }
  tm.mark("upload + count + order points");
  // sort observations by (internal point, image) NOW: it only needs the point ranks, and runs on
  // the device while the host packs the tiles below (radix sort is stable => ties keep input order)
  S->d_obs_img.alloc(M, st); S->d_obs_pt.alloc(M, st); S->d_obs_xy.alloc(M, st); S->d_obs_orig.alloc(M, st);
  if (M) {
    k_st_keys<<<grid_for(M), 256, 0, st>>>(in_img_p, in_pt_p, pt_new.p, M, keys.p, idx.p); PSFM_LAUNCH_CHECK();
    need = tmp_bytes + 256;
    cub::DeviceRadixSort::SortPairs(tmp.p, need, keys.p, keys_out.p, idx.p, S->d_obs_orig.p, M, 0, 32 + pbits, st);
    PSFM_CUDA(cudaStreamWaitEvent(st, S->sh.ev_xy, 0));
    k_st_gather<<<grid_for(M), 256, 0, st>>>(keys_out.p, S->d_obs_orig.p, in_xy_p, M, S->d_obs_img.p, S->d_obs_pt.p, S->d_obs_xy.p);
    PSFM_LAUNCH_CHECK();
    if (sel.n) { k_compose_index<<<grid_for(M), 256, 0, st>>>(S->d_obs_orig.p, sel.p, M); PSFM_LAUNCH_CHECK(); }   // -> caller's index
  }
  for (int i = 0; i < F; ++i) if (h_has[i]) { S->img_has_obs[i] = 1; S->cam_has_obs[S->image_camera[i]] = 1; }
  int P = 0, maxL = 0;
  while (P < Pt && h_cs[P] > 0) ++P;           // observed points come first
  for (int j = 0; j < P; ++j) maxL = std::max(maxL, h_cs[j]);
  if (dist::world_size() > 1) {   // every rank takes the same code paths: the longest track of ANY shard decides
    DBuf<double> mx; mx.alloc(1, st);
    k_fill<<<1, 32, 0, st>>>(mx.p, (double)maxL, 1); PSFM_LAUNCH_CHECK();
    dist::allreduce_max(mx.p, 1, st);
    double h = 0.0;
    PSFM_CUDA(cudaMemcpyAsync(&h, mx.p, sizeof(double), cudaMemcpyDeviceToHost, st));
    PSFM_CUDA(cudaStreamSynchronize(st));
    maxL = (int)(h + 0.5);
  }
  S->P = P; S->maxL = maxL;
  S->pt_orig.assign(h_order.begin(), h_order.begin() + P);
  // A track lives in one tile and a tile's per-image staging grows with the images it spans: beyond
  // 512 observations the shared memory of an SM (227 KB) no longer holds a tile.
  if (maxL > 512) { set_error("a track with more than 512 observations is not supported"); return PSFM_ERR_UNSUPPORTED; }
  S->tile = (maxL <= 256 && !getenv("PSFM_TILE512")) ? 256 : 512;
  // tiles: whole points, <= tile observations (greedy, host: P iterations)
  const int TILE = S->tile;
  std::vector<int> pt_ptr(P + 1, 0), tile_start, tile_pt;
  tile_start.push_back(0); tile_pt.push_back(0);
  {
    int cur = 0, np_cur = 0, cap_np = 1;
    for (int id = 0; id < P; ++id) {
      const int L = h_cs[id];
      pt_ptr[id + 1] = pt_ptr[id] + L;
      if (cur + L > TILE) { tile_start.push_back(pt_ptr[id]); tile_pt.push_back(id); cap_np = std::max(cap_np, np_cur); cur = 0; np_cur = 0; }
      cur += L; ++np_cur;
    }
    cap_np = std::max(cap_np, np_cur);
    if (P > 0) { tile_start.push_back(M); tile_pt.push_back(P); }
    S->cap_np = cap_np;
  }
  const int T = (int)tile_start.size() - 1;
  S->T = T;
  S->d_tile_start.alloc(T + 1, st); S->d_tile_start.upload(tile_start.data(), T + 1, st);
  S->d_tile_pt.alloc(T + 1, st); S->d_tile_pt.upload(tile_pt.data(), T + 1, st);
  S->d_pt_ptr.alloc(P + 1, st); S->d_pt_ptr.upload(pt_ptr.data(), P + 1, st);
  tm.mark("tiles (host greedy)");
  S->d_tile_perm.alloc((size_t)M + 2, st); S->d_obs_lseg.alloc((size_t)M + 2, st); S->d_obs_lpt.alloc((size_t)M + 2, st);
  S->d_cseg_ptr.alloc((size_t)T + 1, st);
  // per tile: image order, local indices, segments
  tile_ns.alloc((size_t)T + 1, st);
  PSFM_CUDA(cudaMemsetAsync(tile_ns.p, 0, sizeof(int) * ((size_t)T + 1), st));
  if (T) {
    if (TILE == 256) k_st_tile_order<256><<<T, 256, 0, st>>>(S->d_tile_start.p, S->d_tile_pt.p, S->d_obs_img.p, S->d_obs_pt.p, S->d_tile_perm.p, S->d_obs_lseg.p, S->d_obs_lpt.p, tile_ns.p);
    else k_st_tile_order<512><<<T, 512, 0, st>>>(S->d_tile_start.p, S->d_tile_pt.p, S->d_obs_img.p, S->d_obs_pt.p, S->d_tile_perm.p, S->d_obs_lseg.p, S->d_obs_lpt.p, tile_ns.p);
    PSFM_LAUNCH_CHECK();
  }
  {
    need = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, need, tile_ns.p, S->d_cseg_ptr.p, T + 1, st);
    DBuf<unsigned char> tmp2; tmp2.alloc(need + 256, st);
    cub::DeviceScan::ExclusiveSum(tmp2.p, need, tile_ns.p, S->d_cseg_ptr.p, T + 1, st);
    DBuf<int> mx; mx.alloc(1, st);
    size_t need2 = 0;
    cub::DeviceReduce::Max(nullptr, need2, tile_ns.p, mx.p, T + 1, st);
    DBuf<unsigned char> tmp3; tmp3.alloc(need2 + 256, st);
    cub::DeviceReduce::Max(tmp3.p, need2, tile_ns.p, mx.p, T + 1, st);
    int h_nseg = 0, h_mx = 1;
    PSFM_CUDA(cudaMemcpyAsync(&h_nseg, S->d_cseg_ptr.p + T, sizeof(int), cudaMemcpyDeviceToHost, st));
    PSFM_CUDA(cudaMemcpyAsync(&h_mx, mx.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    PSFM_CUDA(cudaStreamSynchronize(st));
    S->nseg = h_nseg; S->cap_ns = std::max(1, h_mx);
  }
  S->d_cseg_img.alloc(S->nseg, st); S->d_cseg_off.alloc(S->nseg, st);
  if (T) {
    if (TILE == 256) k_st_tile_segments<256><<<T, 256, 0, st>>>(S->d_tile_start.p, S->d_obs_img.p, S->d_tile_perm.p, S->d_obs_lseg.p, S->d_cseg_ptr.p, S->d_cseg_img.p, S->d_cseg_off.p);
    else k_st_tile_segments<512><<<T, 512, 0, st>>>(S->d_tile_start.p, S->d_obs_img.p, S->d_tile_perm.p, S->d_obs_lseg.p, S->d_cseg_ptr.p, S->d_cseg_img.p, S->d_cseg_off.p);
    PSFM_LAUNCH_CHECK();
  }
  // pipeline form: packed tile headers, tile-relative point starts, 32-bit segment offsets
  S->pipe = T > 0 && !getenv("PSFM_NO_PIPE");
  if (S->pipe) {
    int dev = 0;
    PSFM_CUDA(cudaGetDevice(&dev));
    PSFM_CUDA(cudaDeviceGetAttribute(&S->sm_count, cudaDevAttrMultiProcessorCount, dev));
    S->d_tile_hdr.alloc(2 * (size_t)T, st); S->d_pstart_rel.alloc((size_t)P + 1, st);
    S->d_cseg_off32.alloc((size_t)S->nseg + 1, st); S->d_seg_pose.alloc(PSFM_SPS * (size_t)S->nseg + 2, st); S->d_seg_pose.zero(st);
    k_pipe_headers<<<grid_for(T), 256, 0, st>>>(S->d_tile_start.p, S->d_tile_pt.p, S->d_cseg_ptr.p, T, S->d_tile_hdr.p);
    PSFM_LAUNCH_CHECK();
    k_pipe_pstart<<<T, 128, 0, st>>>(S->d_tile_start.p, S->d_tile_pt.p, S->d_pt_ptr.p, T, S->d_pstart_rel.p);
    PSFM_LAUNCH_CHECK();
    k_pipe_off32<<<grid_for(S->nseg), 256, 0, st>>>(S->d_cseg_off.p, S->nseg, S->d_cseg_off32.p);
    PSFM_LAUNCH_CHECK();
  }
  PSFM_CUDA(cudaStreamSynchronize(st));
  tm.mark("sort + tile order (device)");
  return PSFM_OK;
}

void alloc_work(psfm_ba_solver* S) {
  const size_t M = S->M, P = S->P, F = S->F, C = S->C, NS = S->NS;
  if (S->hs) { g_pinned.release(S->hs, S->hs_bytes); S->hs = nullptr; }
  if (S->pin_state) { g_pinned.release(S->pin_state, S->pin_state_bytes); S->pin_state = nullptr; }
  S->d_active.alloc(NS, S->stream);
  for (int k = 0; k < 2; ++k) { S->d_pose[k].alloc(8 * F, S->stream); S->d_X[k].alloc(3 * P, S->stream); S->d_K[k].alloc(3 * C, S->stream); }
  S->d_r.alloc(2 * M, S->stream); S->d_a.alloc(3 * M, S->stream);
  S->d_pose16.alloc(16 * F, S->stream); S->d_xs.alloc(NS, S->stream);
  S->d_hpp.alloc(6 * P, S->stream); S->d_gp.alloc(3 * P, S->stream); S->d_wk.alloc(9 * P, S->stream); S->d_hinv.alloc(6 * P, S->stream); S->d_w.alloc(3 * P, S->stream);
  S->d_scale_c.alloc(NS, S->stream); S->d_scale_p.alloc(3 * P, S->stream);
  S->d_lin.alloc(F * NVL + C * NVI + 1, S->stream);
  S->d_prep.alloc(F * NVL + C * NVI + 1, S->stream);
  S->d_step.alloc(8, S->stream); S->d_rep.alloc(2, S->stream); S->d_gmax.alloc(1, S->stream); S->d_x2.alloc(1, S->stream);
  S->d_Dc2.alloc(NS, S->stream); S->d_Minv.alloc(9 * (size_t)S->NB, S->stream); S->d_rhs.alloc(NS, S->stream);
  S->d_x.alloc(NS, S->stream); S->d_rv.alloc(NS, S->stream); S->d_p.alloc(NS, S->stream); S->d_z.alloc(NS, S->stream); S->d_y.alloc(NS, S->stream); S->d_zero.alloc(NS, S->stream);
  S->d_zero.zero(S->stream);
  S->d_camrep.alloc((size_t)NREP * F * NVL, S->stream); S->d_camrep.zero(S->stream);
  S->d_yrep.alloc((size_t)NREP * NS, S->stream); S->d_yrep.zero(S->stream);
  S->d_pcg.alloc(1, S->stream);
  S->hs = (HostScalars*)g_pinned.acquire(sizeof(HostScalars), &S->hs_bytes);
  S->pin_state = (double*)g_pinned.acquire(sizeof(double) * (8 * F + 3 * P + 3 * C + 1), &S->pin_state_bytes);
  if (!S->hs || !S->pin_state) { set_error("cudaMallocHost failed"); throw CudaFail{PSFM_ERR_CUDA}; }
  memset(S->hs, 0, sizeof(HostScalars));
}

// ---------------------------------------------------------------- kernel dispatch

#define PSFM_TILE_LAUNCH(KERNEL, NV, NPT, S, ROT, ARGS)                                                    \
  do {                                                                                                     \
    const TileCtx _tc = (S)->tc();                                                                         \
    if ((S)->T > 0) {                                                                                      \
      auto _go = [&](auto tile_c, auto rot_c) {                                                            \
        constexpr int TL = decltype(tile_c)::value;                                                        \
        constexpr bool RT = decltype(rot_c)::value;                                                        \
        const size_t smem = TileSmem<TL>::bytes(NV, NPT, (S)->cap_ns, (S)->cap_np);                        \
        static size_t attr_bytes = 0;                                                                      \
        if (smem > attr_bytes) {                                                                           \
          PSFM_CUDA(cudaFuncSetAttribute(KERNEL<TL, RT>, cudaFuncAttributeMaxDynamicSharedMemorySize,      \
                                         (int)smem));                                                      \
          attr_bytes = smem;                                                                               \
        }                                                                                                  \
        KERNEL<TL, RT><<<(S)->T, TL, smem, (S)->stream>>>(_tc, ARGS);                                       \
      };                                                                                                   \
      using std::integral_constant;                                                                        \
      if ((S)->tile == 256) { if (ROT) _go(integral_constant<int, 256>{}, std::true_type{}); else _go(integral_constant<int, 256>{}, std::false_type{}); } \
      else { if (ROT) _go(integral_constant<int, 512>{}, std::true_type{}); else _go(integral_constant<int, 512>{}, std::false_type{}); } \
      PSFM_LAUNCH_CHECK();                                                                                 \
    }                                                                                                      \
  } while (0)

// persistent pipelined tile kernels: grid = SMs x resident CTAs (capped by the tile count)
#define PSFM_PIPE_LAUNCH(KERNEL, SMEM_FN, S, ROT, PS, ARGS)                                                 \
  do {                                                                                                     \
    const TileCtx _tc = (S)->tc();                                                                         \
    auto _go = [&](auto tile_c, auto rot_c) {                                                              \
      constexpr int TL = decltype(tile_c)::value;                                                          \
      constexpr bool RT = decltype(rot_c)::value;                                                          \
      const size_t smem = SMEM_FN<TL>((S)->cap_ns, (S)->cap_np);                                           \
      static size_t attr_bytes = 0;                                                                        \
      static int occ = 0;                                                                                  \
      if (smem > attr_bytes || occ == 0) {                                                                 \
        PSFM_CUDA(cudaFuncSetAttribute(KERNEL<TL, RT>, cudaFuncAttributeMaxDynamicSharedMemorySize,        \
                                       (int)smem));                                                        \
        PSFM_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, KERNEL<TL, RT>, TL, smem));          \
        if (occ < 1) occ = 1;                                                                              \
        attr_bytes = smem;                                                                                 \
      }                                                                                                    \
      const int grid = std::min((S)->T, (S)->sm_count * occ);                                              \
      KERNEL<TL, RT><<<grid, TL, smem, (S)->stream>>>(_tc, PS, ARGS);                                      \
    };                                                                                                     \
    using std::integral_constant;                                                                          \
    if ((S)->tile == 256) { if (ROT) _go(integral_constant<int, 256>{}, std::true_type{}); else _go(integral_constant<int, 256>{}, std::false_type{}); } \
    else { if (ROT) _go(integral_constant<int, 512>{}, std::true_type{}); else _go(integral_constant<int, 512>{}, std::false_type{}); } \
    PSFM_LAUNCH_CHECK();                                                                                   \
  } while (0)

struct RunCfg {
  psfm_ba_options o;
  bool rot = false;
  int intr = 0;
  int solver = 0;
  std::vector<unsigned char> active;
  int num_effective_parameters = 0;
};

int resolve_cfg(psfm_ba_solver* S, const psfm_ba_options* opts, RunCfg& c) {
  if (opts) c.o = *opts; else psfm_ba_default_options(&c.o);
  const psfm_ba_options& o = c.o;
  const int F = S->F, C = S->C;
  c.active.assign(S->NS, 0);
  bool any_rot = false;
  for (int i = 0; i < F; ++i) {
    const bool constant_pose = !o.refine_extrinsics || S->pose_constant[i];   // bundle_adjustment.cc:361-362
    if (!S->img_has_obs[i] || constant_pose) continue;
    for (int k = 0; k < 3; ++k) {
      c.active[6 * i + k] = o.refine_rotation ? 1 : 0;                        // :429-431
      c.active[6 * i + 3 + k] = ((S->tvec_mask[i] >> k) & 1) ? 0 : 1;         // :432-444
    }
    any_rot |= o.refine_rotation != 0;
  }
  // ParameterizeCameras (:500-544); SIMPLE_PINHOLE: focal {0}, principal point {1,2}, no extra
  const bool constant_camera = !o.refine_focal_length && !o.refine_principal_point && !o.refine_extra_params;
  bool any_f = false, any_pp = false;
  for (int cc = 0; cc < C; ++cc) {
    if (!S->cam_has_obs[cc] || constant_camera || S->camera_constant[cc]) continue;
    c.active[6 * F + 3 * cc] = o.refine_focal_length ? 1 : 0;
    c.active[6 * F + 3 * cc + 1] = c.active[6 * F + 3 * cc + 2] = o.refine_principal_point ? 1 : 0;
    any_f |= o.refine_focal_length != 0;
    any_pp |= o.refine_principal_point != 0;
  }
  c.rot = any_rot;
  c.intr = any_pp ? 3 : (any_f ? 1 : 0);
  if (c.intr > 0 && C > 1) {
    set_error("refining intrinsics is supported for a single shared camera (the pipeline's single_camera=1)");
    return PSFM_ERR_UNSUPPORTED;
  }
  c.solver = o.linear_solver;
  if (c.solver == PSFM_BA_SOLVER_AUTO)   // bundle_adjustment.cc:276-286
    c.solver = (F <= 1000) ? PSFM_BA_SOLVER_EXACT_SCHUR : PSFM_BA_SOLVER_ITERATIVE_SCHUR;
  int np = 0;
  for (unsigned char a : c.active) np += a;
  c.num_effective_parameters = np;   // + 3 per observed point, added by the caller (all ranks)
  return PSFM_OK;
}

// split [0, n) over a few host threads (the permuted copies below move 12 MB per call at 500 k points: ~1 ms on one core)
template <typename Fn>
void host_parallel_for(size_t n, Fn fn) {
  const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
  const size_t nt = n < (size_t)1 << 16 ? 1 : std::min<size_t>({(size_t)8, (size_t)hw, n >> 15});
  if (nt <= 1) { fn((size_t)0, n); return; }
  std::vector<std::thread> th;
  const size_t chunk = (n + nt - 1) / nt;
  for (size_t t = 1; t < nt; ++t) th.emplace_back([=] { fn(std::min(n, t * chunk), std::min(n, (t + 1) * chunk)); });
  fn((size_t)0, std::min(n, chunk));
  for (auto& x : th) x.join();
}

// caller's xyz [3 * P_total] <-> the pinned X staging (tile order, this solver's observed points)
void gather_points(psfm_ba_solver* S, const double* xyz) {
  double* X = S->pin_state + 8 * (size_t)S->F;
  const int* po = S->pt_orig.data();
  host_parallel_for((size_t)S->P, [=](size_t i0, size_t i1) {
    for (size_t id = i0; id < i1; ++id) {
      const double* src = xyz + 3 * (size_t)po[id];
      X[3 * id] = src[0]; X[3 * id + 1] = src[1]; X[3 * id + 2] = src[2];
    }
  });
}
void scatter_points(const psfm_ba_solver* S, double* xyz) {
  const double* X = S->pin_state + 8 * (size_t)S->F;
  const int* po = S->pt_orig.data();
  host_parallel_for((size_t)S->P, [=](size_t i0, size_t i1) {
    for (size_t id = i0; id < i1; ++id) {
      double* dst = xyz + 3 * (size_t)po[id];
      dst[0] = X[3 * id]; dst[1] = X[3 * id + 1]; dst[2] = X[3 * id + 2];
    }
  });
}

void upload_state(psfm_ba_solver* S) {
  const int F = S->F, P = S->P, C = S->C;
  double* pose = S->pin_state;
  double* X = pose + 8 * (size_t)F;
  double* K = X + 3 * (size_t)P;
  for (int i = 0; i < F; ++i) {
    // image.NormalizeQvec() — bundle_adjustment.cc:355
    double* q = &S->h_qvec[4 * (size_t)i];
    const double n = std::sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
    if (n == 0.0) { q[0] = 1.0; q[1] = q[2] = q[3] = 0.0; }
    else for (int k = 0; k < 4; ++k) q[k] /= n;
    for (int k = 0; k < 4; ++k) pose[8 * (size_t)i + k] = q[k];
    for (int k = 0; k < 3; ++k) pose[8 * (size_t)i + 4 + k] = S->h_tvec[3 * (size_t)i + k];
    pose[8 * (size_t)i + 7] = 0.0;
  }
  for (int k = 0; k < 3 * C; ++k) K[k] = S->h_K[k];
  S->cur = 0;
  S->d_pose[0].upload(pose, 8 * (size_t)F, S->stream);
  S->d_X[0].upload(X, 3 * (size_t)P, S->stream);
  S->d_K[0].upload(K, 3 * (size_t)C, S->stream);
  PSFM_CUDA(cudaStreamSynchronize(S->stream));
}

void download_state(psfm_ba_solver* S) {
  const int F = S->F, P = S->P, C = S->C;
  double* pose = S->pin_state;
  double* X = pose + 8 * (size_t)F;
  double* K = X + 3 * (size_t)P;
  PSFM_CUDA(cudaMemcpyAsync(pose, S->d_pose[S->cur].p, 8 * (size_t)F * sizeof(double), cudaMemcpyDeviceToHost, S->stream));
  if (P) PSFM_CUDA(cudaMemcpyAsync(X, S->d_X[S->cur].p, 3 * (size_t)P * sizeof(double), cudaMemcpyDeviceToHost, S->stream));
  PSFM_CUDA(cudaMemcpyAsync(K, S->d_K[S->cur].p, 3 * (size_t)C * sizeof(double), cudaMemcpyDeviceToHost, S->stream));
  PSFM_CUDA(cudaStreamSynchronize(S->stream));
  for (int k = 0; k < 3 * C; ++k) S->h_K[k] = K[k];
  for (int i = 0; i < F; ++i) {
    for (int k = 0; k < 4; ++k) S->h_qvec[4 * (size_t)i + k] = pose[8 * (size_t)i + k];
    for (int k = 0; k < 3; ++k) S->h_tvec[3 * (size_t)i + k] = pose[8 * (size_t)i + 4 + k];
  }
}

Lin lin_of(psfm_ba_solver* S) {
  Lin L;
  L.r = S->d_r.p; L.a = S->d_a.p;
  return L;
}

template <typename T>
void d2h(psfm_ba_solver* S, T* dst, const T* src, size_t n) {
  PSFM_CUDA(cudaMemcpyAsync(dst, src, n * sizeof(T), cudaMemcpyDeviceToHost, S->stream));
}

void fold_replicas(psfm_ba_solver* S, double* dst, double* rep, size_t n, const double* scale, const int* skip_flag) {
  k_fold_replicas<<<(unsigned)((n + 255) / 256), 256, 0, S->stream>>>(dst, rep, n, n, NREP, scale, skip_flag);
  PSFM_LAUNCH_CHECK();
}

PipeSrc pipe_src(psfm_ba_solver* S) {
  PipeSrc ps;
  memset(&ps, 0, sizeof(ps));
  ps.tile_hdr = S->d_tile_hdr.p; ps.obs_lseg = S->d_obs_lseg.p; ps.obs_lpt = S->d_obs_lpt.p; ps.tile_perm = S->d_tile_perm.p;
  ps.pstart_rel = S->d_pstart_rel.p; ps.cseg_img = S->d_cseg_img.p; ps.cseg_off32 = S->d_cseg_off32.p;
  ps.seg_pose = S->d_seg_pose.p; ps.X = S->d_X[S->cur].p;
  return ps;
}

// the pipelined kernels need the tile inputs to fit twice in shared memory
// The 227 KB opt-in limit covers static + dynamic shared memory.  Every k_*_p kernel declares the same static part
// (header ring, barriers, descriptors: 1936 bytes): a dynamic size within that much of the limit makes
// cudaFuncSetAttribute fail (seen with PSFM_FUSED_COST on 512-wide tiles and a 320-image pose table).
size_t pipe_static_smem() {
  static const size_t bytes = [] {
    cudaFuncAttributes a{};
    PSFM_CUDA(cudaFuncGetAttributes(&a, k_back_substitute_p<256, false>));
    return a.sharedSizeBytes;
  }();
  return bytes;
}

bool pipe_ok(psfm_ba_solver* S, size_t smem) { return S->pipe && smem + pipe_static_smem() <= (size_t)227 * 1024; }

// Jacobian sweep at the current state (r, J, E'E, E'r, F'F blocks, F'r, cost)
void do_linearize(psfm_ba_solver* S, const RunCfg& c, bool timed) {
  S->d_lin.zero(S->stream);
  k_pose_table<<<(S->F + 127) / 128, 128, 0, S->stream>>>(S->d_pose[S->cur].p, S->F, S->d_pose16.p);
  PSFM_LAUNCH_CHECK();
  LinArgs a;
  a.pose16 = S->d_pose16.p; a.X = S->d_X[S->cur].p; a.K = S->d_K[S->cur].p;
  a.loss.type = c.o.loss_function_type; a.loss.a = c.o.loss_function_scale;
  a.intr = c.intr;
  a.L = lin_of(S);
  a.hpp = S->d_hpp.p; a.gp = S->d_gp.p; a.wk = S->d_wk.p;
  a.acc_cam = S->d_camrep.p; a.rep_stride = (size_t)S->F * NVL; a.acc_intr = S->d_lin.p + (size_t)S->F * NVL;
  a.acc_cost = S->d_lin.p + (size_t)S->F * NVL + (size_t)S->C * NVI;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  const size_t pipe_smem = S->tile == 256 ? pipe_smem_linearize<256>(S->cap_ns, S->cap_np) : pipe_smem_linearize<512>(S->cap_ns, S->cap_np);
  if (pipe_ok(S, pipe_smem)) {
    k_seg_pose<<<grid_for(12 * (size_t)S->nseg), 256, 0, S->stream>>>(S->d_cseg_img.p, S->d_pose16.p, S->nseg, S->d_seg_pose.p);
    PSFM_LAUNCH_CHECK();
  }
  if (timed) { e0 = S->events.get(); e1 = S->events.get(); PSFM_CUDA(cudaEventRecord(e0, S->stream)); }
  if (pipe_ok(S, pipe_smem)) {
    PipeSrc ps = pipe_src(S);
    ps.obs_xy = S->d_obs_xy.p;
    PSFM_PIPE_LAUNCH(k_linearize_p, pipe_smem_linearize, S, c.rot, ps, a);
  } else {
    PSFM_TILE_LAUNCH(k_linearize, 18, 3, S, c.rot, a);
  }
  if (timed) { PSFM_CUDA(cudaEventRecord(e1, S->stream)); S->ev_lin.push_back({e0, e1}); }
  fold_replicas(S, S->d_lin.p, S->d_camrep.p, (size_t)S->F * NVL, nullptr, nullptr);
  dist::allreduce_sum(S->d_lin.p, S->d_lin.n, S->stream);
}

// per-point (E'E + D^2)^-1, its product with E'r, the points' share of gradient_max_norm
void do_point_blocks(psfm_ba_solver* S, const RunCfg& c, double radius) {
  if (S->P == 0) return;
  PtsArgs a;
  a.hpp = S->d_hpp.p; a.gp = S->d_gp.p; a.wk = S->d_wk.p; a.scale_p = S->d_scale_p.p;
  a.radius = radius; a.min_diag = c.o.min_lm_diagonal; a.max_diag = c.o.max_lm_diagonal;
  a.intr = c.intr; a.P = S->P;
  a.ht = S->d_hinv.p; a.wt = S->d_w.p;
  a.acc_intr = S->d_prep.p + (size_t)S->F * NVL;
  a.acc_fail = S->d_prep.p + (size_t)S->F * NVL + (size_t)S->C * NVI;
  a.gmax = S->d_gmax.p;
  k_point_blocks<<<(S->P + 255) / 256, 256, 0, S->stream>>>(a);
  PSFM_LAUNCH_CHECK();
}

void do_cam_gmax(psfm_ba_solver* S) {
  const int n = S->F + S->C;
  k_cam_gmax<<<(n + 127) / 128, 128, 0, S->stream>>>(S->d_lin.p, S->d_lin.p + (size_t)S->F * NVL,
                                                     S->d_active.p, S->d_pose[S->cur].p, S->F, S->C, S->d_gmax.p);
  PSFM_LAUNCH_CHECK();
}

// reduced system: Schur-Jacobi blocks, rhs, LM diagonal
void cam_finalize(psfm_ba_solver* S, const RunCfg& c, double radius, bool fused) {
  CamFinArgs f;
  f.lin_cam = S->d_lin.p; f.lin_intr = S->d_lin.p + (size_t)S->F * NVL;
  if (fused) { f.prep_cam = S->d_xband.p; f.prep_stride = NVX2; f.prep_goff = 21; f.prep_blocks = 0; }
  else { f.prep_cam = S->d_prep.p; f.prep_stride = NVL; f.prep_goff = 12; f.prep_blocks = 1; }
  f.prep_intr = S->d_prep.p + (size_t)S->F * NVL;
  f.active = S->d_active.p; f.scale_c = S->d_scale_c.p; f.radius = radius; f.min_diag = c.o.min_lm_diagonal; f.max_diag = c.o.max_lm_diagonal;
  f.F = S->F; f.C = S->C; f.Dc2 = S->d_Dc2.p; f.Minv = S->d_Minv.p; f.rhs = S->d_rhs.p;
  k_cam_finalize<<<(S->NB + 127) / 128, 128, 0, S->stream>>>(f);
  PSFM_LAUNCH_CHECK();
}

// fused_explicit: the rhs correction comes out of k_schur_tile (do_explicit_solve_fused), the
// Schur-Jacobi blocks are not needed; only the point blocks and the intrinsics sums are made here
void do_reduced_setup(psfm_ba_solver* S, const RunCfg& c, double radius, bool fused_explicit = false) {
  if (!(S->pb_fresh && S->pb_radius == radius)) {
    S->d_prep.zero(S->stream);
    do_point_blocks(S, c, radius);
  }
  S->pb_fresh = false;           // d_prep is all-reduced in place below
  if (fused_explicit) {
    dist::allreduce_sum(S->d_prep.p, S->d_prep.n, S->stream);
    return;
  }
  PrepArgs a;
  a.L = lin_of(S); a.pose16 = S->d_pose16.p; a.X = S->d_X[S->cur].p; a.ht = S->d_hinv.p; a.wt = S->d_w.p;
  a.acc_cam = S->d_camrep.p; a.rep_stride = (size_t)S->F * NVL;
  PSFM_TILE_LAUNCH(k_schur_prep, 18, 12, S, c.rot, a);
  fold_replicas(S, S->d_prep.p, S->d_camrep.p, (size_t)S->F * NVL, nullptr, nullptr);
  dist::allreduce_sum(S->d_prep.p, S->d_prep.n, S->stream);
  cam_finalize(S, c, radius, false);
}

void scale_vec(psfm_ba_solver* S, const double* x, const int* skip_flag) {
  k_scale_vec<<<(S->NS + 255) / 256, 256, 0, S->stream>>>(x, S->d_scale_c.p, (size_t)S->NS, S->d_xs.p, skip_flag);
  PSFM_LAUNCH_CHECK();
}

void do_schur_product(psfm_ba_solver* S, const RunCfg& c, const double* x, bool timed) {
  const int* flag = &S->d_pcg.p->flag;
  scale_vec(S, x, flag);
  SpArgs a;
  a.L = lin_of(S); a.pose16 = S->d_pose16.p; a.X = S->d_X[S->cur].p; a.ht = S->d_hinv.p; a.xs = S->d_xs.p;
  a.y = S->d_yrep.p; a.rep_stride = (size_t)S->NS; a.flag = flag; a.K = S->d_K[S->cur].p; a.intr = c.intr;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  if (timed) { e0 = S->events.get(); e1 = S->events.get(); PSFM_CUDA(cudaEventRecord(e0, S->stream)); }
  PSFM_TILE_LAUNCH(k_schur_product, 6, 9, S, c.rot, a);
  if (timed) { PSFM_CUDA(cudaEventRecord(e1, S->stream)); S->ev_sp.push_back({e0, e1}); }
  fold_replicas(S, S->d_y.p, S->d_yrep.p, (size_t)S->NS, S->d_scale_c.p, flag);
  dist::allreduce_sum(S->d_y.p, S->d_y.n, S->stream);
}

// ConjugateGradientsSolver::Solve on the implicit Schur complement; returns PcgFlag
int do_pcg(psfm_ba_solver* S, const RunCfg& c, double q_tol, double r_tol, int max_it, int* iters, int* nprod) {
  PcgArgs a;
  a.st = S->d_pcg.p; a.b = S->d_rhs.p; a.Minv = S->d_Minv.p; a.Dc2 = S->d_Dc2.p;
  a.x = S->d_x.p; a.r = S->d_rv.p; a.p = S->d_p.p; a.z = S->d_z.p; a.y = S->d_y.p;
  a.NS = S->NS; a.NB = S->NB; a.F = S->F;
  a.q_tol = q_tol; a.r_tol = r_tol; a.max_it = max_it; a.min_it = 0;
  k_pcg_init<<<1, 1024, 0, S->stream>>>(a);
  PSFM_LAUNCH_CHECK();
  const int period = c.o.pcg_check_period > 0 ? c.o.pcg_check_period : 4;
  PcgState st;
  st.flag = PCG_RUNNING; st.it = 1;
  for (int it = 1; it <= max_it; ++it) {
    do_schur_product(S, c, S->d_p.p, true);
    ++*nprod;
    if (it % 10 != 0) {   // residual_reset_period = 10
      k_pcg_update<<<1, 1024, 0, S->stream>>>(a, 0);
      PSFM_LAUNCH_CHECK();
    } else {
      k_pcg_update<<<1, 1024, 0, S->stream>>>(a, 1);
      PSFM_LAUNCH_CHECK();
      do_schur_product(S, c, S->d_x.p, true);
      ++*nprod;
      k_pcg_update<<<1, 1024, 0, S->stream>>>(a, 2);
      PSFM_LAUNCH_CHECK();
    }
    if (it % period == 0 || it == max_it) {
      d2h(S, &S->hs->pcg, S->d_pcg.p, 1);
      PSFM_CUDA(cudaStreamSynchronize(S->stream));
      st = S->hs->pcg;
      if (st.flag != PCG_RUNNING) break;
    }
  }
  if (st.flag == PCG_RUNNING) {   // max_it == 0 corner
    d2h(S, &S->hs->pcg, S->d_pcg.p, 1);
    PSFM_CUDA(cudaStreamSynchronize(S->stream));
    st = S->hs->pcg;
  }
  *iters = st.it;
  return st.flag;
}

void set_masks_and_unit_scale(psfm_ba_solver* S, const RunCfg& c) {
  S->d_active.upload(c.active.data(), c.active.size(), S->stream);
  std::vector<double> sc(S->NS);
  for (int k = 0; k < S->NS; ++k) sc[k] = c.active[k] ? 1.0 : 0.0;
  S->d_scale_c.upload(sc.data(), sc.size(), S->stream);
  PSFM_CUDA(cudaStreamSynchronize(S->stream));
  if (S->P) {
    const size_t n = 3 * (size_t)S->P;
    k_fill<<<(unsigned)((n + 255) / 256), 256, 0, S->stream>>>(S->d_scale_p.p, 1.0, n);
    PSFM_LAUNCH_CHECK();
  }
}

void compute_jacobi_scaling(psfm_ba_solver* S) {
  k_scale_cams<<<(S->NS + 127) / 128, 128, 0, S->stream>>>(S->d_lin.p, S->d_lin.p + (size_t)S->F * NVL, S->d_active.p,
                                                         S->F, S->C, S->d_scale_c.p);
  PSFM_LAUNCH_CHECK();
  if (S->P) {
    k_scale_points<<<(S->P + 255) / 256, 256, 0, S->stream>>>(S->d_hpp.p, S->P, S->d_scale_p.p);
    PSFM_LAUNCH_CHECK();
  }
}

// |x|^2 over the reduced program's parameter blocks at the current state
double current_x_sqnorm(psfm_ba_solver* S) {
  S->d_x2.zero(S->stream);
  S->d_rep.zero(S->stream);
  if (S->P) {
    const size_t n = 3 * (size_t)S->P;
    const unsigned g = (unsigned)std::min<size_t>((n + 255) / 256, 1184);
    k_sqnorm<<<g, 256, 0, S->stream>>>(S->d_X[S->cur].p, n, S->d_x2.p);
    PSFM_LAUNCH_CHECK();
  }
  dist::allreduce_sum(S->d_x2.p, 1, S->stream);
  ApplyArgs a;
  a.yc = S->d_zero.p; a.scale_c = S->d_scale_c.p; a.active = S->d_active.p;
  a.pose = S->d_pose[S->cur].p; a.K = S->d_K[S->cur].p;
  a.pose_c = S->d_pose[1 - S->cur].p; a.K_c = S->d_K[1 - S->cur].p;
  a.F = S->F; a.C = S->C; a.acc = S->d_rep.p;
  const int n = S->F + S->C;
  k_apply_cams<<<(n + 255) / 256, 256, 0, S->stream>>>(a);
  PSFM_LAUNCH_CHECK();
  d2h(S, &S->hs->x2, S->d_x2.p, 1);
  d2h(S, S->hs->rep, S->d_rep.p, 2);
  PSFM_CUDA(cudaStreamSynchronize(S->stream));
  return S->hs->x2 + S->hs->rep[1];
}

struct LinOut { double cost, gmax; };

// EvaluateGradientAndJacobian + the quantities the loop head needs
LinOut linearize_and_measure(psfm_ba_solver* S, const RunCfg& c, double radius, bool timed, bool first = false) {
  do_linearize(S, c, timed);
  // the sweep accumulates with the unscaled Jacobian, so the iteration-0 column norms that
  // define Ceres' jacobi scaling come from the same sweep (no second linearisation)
  if (first && c.o.jacobi_scaling) compute_jacobi_scaling(S);
  S->d_gmax.zero(S->stream);
  S->d_prep.zero(S->stream);
  do_point_blocks(S, c, radius);
  S->pb_fresh = true; S->pb_radius = radius;
  dist::allreduce_max(S->d_gmax.p, 1, S->stream);
  do_cam_gmax(S);
  d2h(S, &S->hs->lin_cost, S->d_lin.p + (size_t)S->F * NVL + (size_t)S->C * NVI, 1);
  d2h(S, &S->hs->gmax, S->d_gmax.p, 1);
  PSFM_CUDA(cudaStreamSynchronize(S->stream));
  LinOut o;
  o.cost = S->hs->lin_cost;
  o.gmax = S->hs->gmax;
  return o;
}

struct StepOut {
  bool linear_ok;
  int pcg_flag, pcg_iters;
  double mcc, step_sq, cand_x2, cand_cost;
};

__global__ void k_point_span(const int* pt_ptr, const int* obs_img, int P, int* span_max) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  const int b = pt_ptr[p], e = pt_ptr[p + 1];
  if (e > b) atomicMax(span_max, obs_img[e - 1] - obs_img[b]);
}

// The fused path ends in Sband: when the band is narrow enough for the register window of
// k_band_chol, the reduced system never exists as a dense matrix.
void setup_band_chol(psfm_ba_solver* S) {
  const BandPlan pl = band_chol_plan(6 * S->F, S->bw, S->span);
  S->band_chol = S->fused && pl.W > 0 && !getenv("PSFM_OLD_CHOL");
  if (!S->band_chol) {
    S->d_S.alloc((size_t)(S->NS + 1) * (S->NS + 1), S->stream);
    return;
  }
  S->bwk.alloc(pl, S->stream);
}

// (i, j) observation pairs of every point grouped by image pair — built once per problem
void ensure_pairs(psfm_ba_solver* S) {
  if (S->pairs_ready) return;
  PhaseTimer tm;
  cudaStream_t st = S->stream;
  const int M = S->M, F = S->F;
  DBuf<int> cnt, span;
  DBuf<unsigned int> keys, keys_out, ukeys;
  DBuf<unsigned long long> vals;
  DBuf<int> ucount, nruns;
  cnt.alloc((size_t)M + 1, st); span.alloc(1, st); span.zero(st);
  PSFM_CUDA(cudaMemsetAsync(cnt.p + M, 0, sizeof(int), st));
  if (M) {   // a rank of a sharded problem may own no observation at all
    k_pair_count<<<grid_for(M), 256, 0, st>>>(S->d_pt_ptr.p, S->d_obs_pt.p, S->d_obs_img.p, M, cnt.p);
    PSFM_LAUNCH_CHECK();
    k_point_span<<<grid_for(S->P), 256, 0, st>>>(S->d_pt_ptr.p, S->d_obs_img.p, S->P, span.p);
    PSFM_LAUNCH_CHECK();
  }
  // exclusive scan of the per-observation entry counts (64-bit total)
  DBuf<long long> ptr64;
  ptr64.alloc((size_t)M + 1, st);
  {
    size_t need = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, need, cnt.p, ptr64.p, M + 1, st);
    DBuf<unsigned char> tmp; tmp.alloc(need + 256, st);
    cub::DeviceScan::ExclusiveSum(tmp.p, need, cnt.p, ptr64.p, M + 1, st);
    long long total = 0; int h_span = 0;
    PSFM_CUDA(cudaMemcpyAsync(&total, ptr64.p + M, sizeof(long long), cudaMemcpyDeviceToHost, st));
    PSFM_CUDA(cudaMemcpyAsync(&h_span, span.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    PSFM_CUDA(cudaStreamSynchronize(st));
    S->npairs = total;
    if (dist::world_size() > 1) {   // every rank must use the same band: max span over all shards
      DBuf<double> sp; sp.alloc(1, st);
      k_fill<<<1, 32, 0, st>>>(sp.p, (double)h_span, 1); PSFM_LAUNCH_CHECK();
      dist::allreduce_max(sp.p, 1, st);
      double hs = 0.0;
      PSFM_CUDA(cudaMemcpyAsync(&hs, sp.p, sizeof(double), cudaMemcpyDeviceToHost, st));
      PSFM_CUDA(cudaStreamSynchronize(st));
      h_span = (int)(hs + 0.5);
    }
    S->bw = 6 * h_span + 5;
  }
  {
    // an error on one rank is an error on all of them (nobody is left waiting in an all-reduce)
    double too_many = S->npairs >= (1ll << 31) ? 1.0 : 0.0;
    if (dist::world_size() > 1) {
      DBuf<double> fl; fl.alloc(1, st);
      k_fill<<<1, 32, 0, st>>>(fl.p, too_many, 1); PSFM_LAUNCH_CHECK();
      dist::allreduce_max(fl.p, 1, st);
      PSFM_CUDA(cudaMemcpyAsync(&too_many, fl.p, sizeof(double), cudaMemcpyDeviceToHost, st));
      PSFM_CUDA(cudaStreamSynchronize(st));
    }
    if (too_many > 0.5) { set_error("too many observation pairs for the explicit Schur complement"); throw CudaFail{PSFM_ERR_UNSUPPORTED}; }
  }
  S->span = (S->bw - 5) / 6;
  {
    const size_t smem256 = TileSmem<256>::bytes(NVX2, 15, S->cap_ns, S->cap_np), smem512 = TileSmem<512>::bytes(NVX2, 15, S->cap_ns, S->cap_np);
    const size_t smem = S->tile == 256 ? smem256 : smem512;
    S->fused = smem <= 227 * 1024 && !getenv("PSFM_SCHUR_UNFUSED");
  }
  if (dist::world_size() > 1) {   // fused and unfused paths all-reduce different buffers: one decision for all ranks
    DBuf<double> fl; fl.alloc(1, st);
    k_fill<<<1, 32, 0, st>>>(fl.p, S->fused ? 0.0 : 1.0, 1); PSFM_LAUNCH_CHECK();
    dist::allreduce_max(fl.p, 1, st);
    double h = 0.0;
    PSFM_CUDA(cudaMemcpyAsync(&h, fl.p, sizeof(double), cudaMemcpyDeviceToHost, st));
    PSFM_CUDA(cudaStreamSynchronize(st));
    S->fused = h < 0.5;
  }
  if (M == 0 && S->fused) {   // nothing to contribute: zero accumulators that still take part in the all-reduces
    S->ntasks = 0;
    S->band_n = (size_t)F * (S->span + 1) * 36; S->band_nrep = 1;
    S->d_xband.alloc((size_t)F * NVX2 + S->band_n, st);
    S->d_bandrep.alloc(S->band_n, st); S->d_bandrep.zero(st);
    S->d_xcamrep.alloc((size_t)NREP * F * NVX2, st); S->d_xcamrep.zero(st);
    S->d_cholfail.alloc(1, st);
    setup_band_chol(S);
    PSFM_CUDA(cudaStreamSynchronize(st));
    S->pairs_ready = true;
    return;
  }
  const size_t NPr = (size_t)S->npairs;
  // 32-bit offsets for the fill kernel
  DBuf<int> ptr32; ptr32.alloc((size_t)M + 1, st);
  {
    size_t need = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, need, cnt.p, ptr32.p, M + 1, st);
    DBuf<unsigned char> tmp; tmp.alloc(need + 256, st);
    cub::DeviceScan::ExclusiveSum(tmp.p, need, cnt.p, ptr32.p, M + 1, st);
  }
  if (S->fused) {
    // ---- tile-local tasks for k_schur_tile
    const int T = S->T;
    int fb = 1; while ((1 << fb) < F) ++fb;
    int tb = 1; while ((1ll << tb) < (long long)T + 1) ++tb;
    DBuf<unsigned long long> k64, k64_out, uk64;
    DBuf<unsigned int> v32;
    k64.alloc(NPr, st); k64_out.alloc(NPr, st); v32.alloc(NPr, st); S->d_tentries.alloc(NPr, st);
    k_pair_fill_tile<<<grid_for(M), 256, 0, st>>>(S->d_pt_ptr.p, S->d_obs_pt.p, S->d_obs_img.p, ptr32.p, M,
                                                   S->d_tile_start.p, T, fb, k64.p, v32.p);
    PSFM_LAUNCH_CHECK();
    {
      // k_pair_fill_tile writes the entries in observation order, i.e. already tile by tile: what is left is a
      // sort of each tile's ~1.6 k entries by their image pair (the low 2 fb bits) — one pass through shared
      // memory per tile instead of four passes of a global 64-bit radix sort over 39 M pairs
      DBuf<int> seg; seg.alloc((size_t)T + 1, st);
      k_tile_entry_offsets<<<grid_for((size_t)T + 1), 256, 0, st>>>(S->d_tile_start.p, ptr32.p, T, seg.p); PSFM_LAUNCH_CHECK();
      size_t need = 0;
      cub::DeviceSegmentedRadixSort::SortPairs(nullptr, need, k64.p, k64_out.p, v32.p, S->d_tentries.p, (int)NPr, T, seg.p, seg.p + 1, 0, 2 * fb, st);
      DBuf<unsigned char> tmp; tmp.alloc(need + 256, st);
      cub::DeviceSegmentedRadixSort::SortPairs(tmp.p, need, k64.p, k64_out.p, v32.p, S->d_tentries.p, (int)NPr, T, seg.p, seg.p + 1, 0, 2 * fb, st);
    }
    k64.release(); v32.release();
    uk64.alloc(NPr, st); ucount.alloc(NPr + 1, st); nruns.alloc(1, st);
    {
      size_t need = 0;
      cub::DeviceRunLengthEncode::Encode(nullptr, need, k64_out.p, uk64.p, ucount.p, nruns.p, (int)NPr, st);
      DBuf<unsigned char> tmp; tmp.alloc(need + 256, st);
      cub::DeviceRunLengthEncode::Encode(tmp.p, need, k64_out.p, uk64.p, ucount.p, nruns.p, (int)NPr, st);
    }
    int nr = 0;
    PSFM_CUDA(cudaMemcpyAsync(&nr, nruns.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    PSFM_CUDA(cudaStreamSynchronize(st));
    // runs -> units of <= chunk entries (k_unit_count / k_unit_fill)
    int chunk = 1 << 30;
    if (const char* e = getenv("PSFM_TASK_CHUNK")) chunk = std::max(1, atoi(e));
    const int by_pair = getenv("PSFM_TASK_BY_LENGTH") ? 0 : 1;
    DBuf<int> beg0, nun, ubeg;
    beg0.alloc((size_t)nr + 1, st); nun.alloc((size_t)nr + 1, st); ubeg.alloc((size_t)nr + 1, st);
    PSFM_CUDA(cudaMemsetAsync(ucount.p + nr, 0, sizeof(int), st));
    k_unit_count<<<grid_for((size_t)nr + 1), 256, 0, st>>>(ucount.p, nr, chunk, nun.p); PSFM_LAUNCH_CHECK();
    {
      size_t need = 0, need2 = 0;
      cub::DeviceScan::ExclusiveSum(nullptr, need, ucount.p, beg0.p, nr + 1, st);
      cub::DeviceScan::ExclusiveSum(nullptr, need2, nun.p, ubeg.p, nr + 1, st);
      DBuf<unsigned char> tmp; tmp.alloc(std::max(need, need2) + 256, st);
      cub::DeviceScan::ExclusiveSum(tmp.p, need, ucount.p, beg0.p, nr + 1, st);
      cub::DeviceScan::ExclusiveSum(tmp.p, need2, nun.p, ubeg.p, nr + 1, st);
    }
    int nt = 0;
    PSFM_CUDA(cudaMemcpyAsync(&nt, ubeg.p + nr, sizeof(int), cudaMemcpyDeviceToHost, st));
    PSFM_CUDA(cudaStreamSynchronize(st));
    S->ntasks = nt;
    S->d_task_slot.alloc(nt, st); S->d_task_rng.alloc(nt, st); S->d_tile_task.alloc((size_t)T + 1, st);
    DBuf<int> slot0, idx0, order;
    DBuf<int2> rng0;
    DBuf<unsigned long long> key2, key2_out;
    slot0.alloc(nt, st); rng0.alloc(nt, st); idx0.alloc(nt, st); order.alloc(nt, st); key2.alloc(nt, st); key2_out.alloc(nt, st);
    if (nt) {
      k_unit_fill<<<grid_for(nr), 256, 0, st>>>(uk64.p, ucount.p, beg0.p, ubeg.p, nr, fb, S->span, by_pair, key2.p, idx0.p, slot0.p, rng0.p);
      PSFM_LAUNCH_CHECK();
      size_t need = 0;
      cub::DeviceRadixSort::SortPairs(nullptr, need, key2.p, key2_out.p, idx0.p, order.p, nt, 0, 32 + tb, st);
      DBuf<unsigned char> tmp; tmp.alloc(need + 256, st);
      cub::DeviceRadixSort::SortPairs(tmp.p, need, key2.p, key2_out.p, idx0.p, order.p, nt, 0, 32 + tb, st);
      k_task_gather<<<grid_for(nt), 256, 0, st>>>(order.p, slot0.p, rng0.p, nt, S->d_task_slot.p, S->d_task_rng.p); PSFM_LAUNCH_CHECK();
    }
    k_tile_tasks<<<grid_for((size_t)T + 1), 256, 0, st>>>(key2_out.p, nt, T, S->d_tile_task.p);
    PSFM_LAUNCH_CHECK();
    S->band_n = (size_t)F * (S->span + 1) * 36;
    int nrep = 8;   // the pair-task REDs are spread over many band blocks: few replicas suffice (fold cost grows with them)
    while (nrep > 1 && S->band_n * nrep * sizeof(double) > ((size_t)256 << 20)) nrep >>= 1;
    S->band_nrep = nrep;
    S->d_xband.alloc((size_t)F * NVX2 + S->band_n, st);
    S->d_bandrep.alloc(S->band_n * nrep, st); S->d_bandrep.zero(st);
    S->d_xcamrep.alloc((size_t)NREP * F * NVX2, st); S->d_xcamrep.zero(st);
    S->d_cholfail.alloc(1, st);
    setup_band_chol(S);
    PSFM_CUDA(cudaStreamSynchronize(st));
    S->pairs_ready = true;
    tm.mark("tile pair tasks (explicit Schur, fused)");
    return;
  }
  keys.alloc(NPr, st); keys_out.alloc(NPr, st); vals.alloc(NPr, st); S->d_entries.alloc(NPr, st);
  k_pair_fill<<<grid_for(M), 256, 0, st>>>(S->d_pt_ptr.p, S->d_obs_pt.p, S->d_obs_img.p, ptr32.p, M, F, keys.p, vals.p);
  PSFM_LAUNCH_CHECK();
  int kbits = 1; while ((1ull << kbits) < (unsigned long long)F * F) ++kbits;
  {
    size_t need = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, need, keys.p, keys_out.p, vals.p, S->d_entries.p, (int)NPr, 0, kbits, st);
    DBuf<unsigned char> tmp; tmp.alloc(need + 256, st);
    cub::DeviceRadixSort::SortPairs(tmp.p, need, keys.p, keys_out.p, vals.p, S->d_entries.p, (int)NPr, 0, kbits, st);
  }
  // run-length encode -> image-pair blocks
  ukeys.alloc(NPr, st); ucount.alloc(NPr, st); nruns.alloc(1, st);
  {
    size_t need = 0;
    cub::DeviceRunLengthEncode::Encode(nullptr, need, keys_out.p, ukeys.p, ucount.p, nruns.p, (int)NPr, st);
    DBuf<unsigned char> tmp; tmp.alloc(need + 256, st);
    cub::DeviceRunLengthEncode::Encode(tmp.p, need, keys_out.p, ukeys.p, ucount.p, nruns.p, (int)NPr, st);
  }
  int nb = 0;
  PSFM_CUDA(cudaMemcpyAsync(&nb, nruns.p, sizeof(int), cudaMemcpyDeviceToHost, st));
  PSFM_CUDA(cudaStreamSynchronize(st));
  S->nblocks = nb;
  std::vector<unsigned int> h_keys(nb);
  std::vector<int> h_cnt(nb);
  PSFM_CUDA(cudaMemcpyAsync(h_keys.data(), ukeys.p, sizeof(unsigned) * nb, cudaMemcpyDeviceToHost, st));
  PSFM_CUDA(cudaMemcpyAsync(h_cnt.data(), ucount.p, sizeof(int) * nb, cudaMemcpyDeviceToHost, st));
  PSFM_CUDA(cudaStreamSynchronize(st));
  // chunks of <= 4096 entries of one block
  const int CH = 4096;
  std::vector<int> chunk_blk, blk_key(nb);
  std::vector<long long> chunk_beg;
  long long off = 0;
  for (int b = 0; b < nb; ++b) {
    blk_key[b] = (int)h_keys[b];
    for (int c0 = 0; c0 < h_cnt[b]; c0 += CH) { chunk_blk.push_back(b); chunk_beg.push_back(off + c0); }
    off += h_cnt[b];
  }
  chunk_beg.push_back(off);
  // a chunk ends where the next begins, except at block boundaries: store explicit ends by
  // making chunk_beg[k+1] the end of chunk k (chunks are consecutive in entry order)
  S->nchunks = (int)chunk_blk.size();
  S->d_blk_key.alloc(nb, st); S->d_blk_key.upload(blk_key.data(), nb, st);
  S->d_chunk_blk.alloc(S->nchunks, st); S->d_chunk_blk.upload(chunk_blk.data(), S->nchunks, st);
  S->d_chunk_beg.alloc((size_t)S->nchunks + 1, st); S->d_chunk_beg.upload(chunk_beg.data(), (size_t)S->nchunks + 1, st);
  S->d_W.alloc(18 * (size_t)M, st); S->d_WH.alloc(18 * (size_t)M, st);
  S->d_xcam.alloc((size_t)F * NVX, st); S->d_xcamrep.alloc((size_t)NREP * F * NVX, st); S->d_xcamrep.zero(st);
  S->d_Sblk.alloc((size_t)nb * 36, st); S->d_S.alloc((size_t)(S->NS + 1) * (S->NS + 1), st); S->d_cholfail.alloc(1, st);
  PSFM_CUDA(cudaStreamSynchronize(st));
  S->pairs_ready = true;
  tm.mark("pair structure (explicit Schur)");
}

// blocked band(+arrow) Cholesky of d_S (rhs carried as the extra row) -> d_x; d_cholfail[0] = 1 on a
// bad pivot (read back with the step scalars at the end of compute_step: no host sync here)
void launch_cholesky(psfm_ba_solver* S) {
  cudaStream_t st = S->stream;
  const int nbnd = 6 * S->F;
  const int bw = std::min(S->bw, nbnd);
  {
    int dev = 0;
    PSFM_CUDA(cudaGetDevice(&dev));
    static std::mutex mu;
    static std::vector<int> grid_limit_by_dev;
    int grid_limit = 0;
    {
      std::lock_guard<std::mutex> lk(mu);
      if ((int)grid_limit_by_dev.size() <= dev) grid_limit_by_dev.resize(dev + 1, 0);
      if (grid_limit_by_dev[dev] == 0) {
        int sms = 0, per_sm = 0;
        PSFM_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        PSFM_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_chol_blocked, 256, 0));
        grid_limit_by_dev[dev] = std::max(1, sms * std::min(per_sm, 1));
      }
      grid_limit = grid_limit_by_dev[dev];
    }
    CholArgs ca;
    ca.A = S->d_S.p; ca.ns = S->NS; ca.lda = S->NS + 1; ca.nb = nbnd; ca.bw = bw + 1; ca.x = S->d_x.p; ca.fail = S->d_cholfail.p;
    if (S->d_cholbar.n == 0) S->d_cholbar.alloc(1, st);
    S->d_cholbar.zero(st);
    ca.bar = S->d_cholbar.p;
    {
      const int npanel = (S->NS + CB - 1) / CB;
      const int rmax = std::min(bw + 1, nbnd) + (S->NS + 1 - nbnd) + 1;
      if (S->d_cholLp.n < (size_t)npanel * rmax * CB) S->d_cholLp.alloc((size_t)npanel * rmax * CB, st);
      if (S->d_cholLd.n < (size_t)npanel * CB * CB) S->d_cholLd.alloc((size_t)npanel * CB * CB, st);
      ca.Lp = S->d_cholLp.p; ca.Ld = S->d_cholLd.p; ca.rmax = rmax;
    }
    static const bool want_prof = getenv("PSFM_CHOL_PROFILE") != nullptr;
    if (want_prof && S->d_cholprof.n == 0) { S->d_cholprof.alloc(8, st); S->d_cholprof.zero(st); }
    ca.prof = want_prof ? S->d_cholprof.p : nullptr;
    void* kargs[] = {(void*)&ca};
    // few CTAs when the band is narrow (cheaper grid barriers), all SMs for a dense system
    const int tiles = (std::min(bw + 2, nbnd) + (S->NS + 1 - nbnd) + CB - 1) / CB;
    const int grid = std::max(1, std::min(grid_limit, tiles * (tiles + 1) / 2));
    PSFM_CUDA(cudaLaunchCooperativeKernel((void*)k_chol_blocked, dim3(grid), dim3(256), kargs, 0, st));
    PSFM_LAUNCH_CHECK();
  }
  { cudaEvent_t e = S->events.get(); PSFM_CUDA(cudaEventRecord(e, st)); S->ev_chol.back().second = e; }
  if (S->d_cholprof.n) {   // debugging aid: cumulative SM cycles of CTA 0 per phase
    unsigned long long h[8];
    PSFM_CUDA(cudaStreamSynchronize(st));
    PSFM_CUDA(cudaMemcpy(h, S->d_cholprof.p, sizeof(h), cudaMemcpyDeviceToHost));
    fprintf(stderr, "[psfm chol cycles] diag %llu rows %llu sync %llu trail %llu sync %llu backsub %llu\n",
            h[0], h[1], h[2], h[3], h[4], h[5]);
  }
}

// single-CTA register-window band Cholesky (ba_band_chol.cuh): assemble the compact band matrix,
// factor, solve -> d_x; d_cholfail[0] = 1 on a bad pivot
void launch_band_cholesky(psfm_ba_solver* S) {
  cudaStream_t st = S->stream;
  const BandPlan& pl = S->bwk.pl;
  BandAsmArgs2 b;
  b.Sband = S->d_xband.p + (size_t)S->F * NVX2;
  b.lin_cam = S->d_lin.p; b.lin_intr = S->d_lin.p + (size_t)S->F * NVL;
  b.prep_intr = S->d_prep.p + (size_t)S->F * NVL;
  b.xcam = S->d_xband.p; b.xstride = NVX2;
  b.scale_c = S->d_scale_c.p; b.Dc2 = S->d_Dc2.p; b.rhs = S->d_rhs.p; b.active = S->d_active.p;
  b.F = S->F; b.span = S->span; b.pl = pl;
  b.Ab = S->bwk.ab(0); b.Ab1 = S->bwk.ab(1); b.C4 = S->bwk.C4.p; b.fail = S->d_cholfail.p;
  k_band_assemble<<<grid_for((size_t)(pl.rows[0] + pl.rows[1]) * pl.RS), 256, 0, st>>>(b);
  PSFM_LAUNCH_CHECK();
  BandCholArgs c = S->bwk.args(S->d_x.p, S->NS, S->d_cholfail.p);
  static const bool want_prof = getenv("PSFM_CHOL_PROFILE") != nullptr;
  if (want_prof && S->d_cholprof.n < 16) { S->d_cholprof.alloc(16, st); S->d_cholprof.zero(st); }
  c.prof = want_prof ? reinterpret_cast<long long*>(S->d_cholprof.p) : nullptr;
  band_chol_launch(c, st);
  if (want_prof) {
    long long h[16];
    PSFM_CUDA(cudaStreamSynchronize(st));
    PSFM_CUDA(cudaMemcpy(h, S->d_cholprof.p, sizeof(h), cudaMemcpyDeviceToHost));
    if (c.blk6) fprintf(stderr, "[psfm chol6 cycles/step] worker0 update %.0f recycle %.0f publish %.0f | panel pbar %.0f chol+solve %.0f out %.0f (steps %lld)\n",
                        h[8] / (h[3] / 6.0), h[9] / (h[3] / 6.0), h[10] / (h[3] / 6.0), h[11] / (h[3] / 6.0), h[12] / (h[3] / 6.0), h[13] / (h[3] / 6.0), h[3] / 6);
    const double np_ = (double)std::max(1ll, h[3]);
    fprintf(stderr, "[psfm band chol cycles] factor %lld (%lld pivots, %.0f / pivot) corner+stage %lld backsub %lld | per pivot own/wait: helper %.0f/%.0f worker0 %.0f/%.0f\n",
            h[0], h[3], (double)h[0] / np_, h[1], h[2], h[4] / np_, h[5] / np_, h[6] / np_, h[7] / np_);
  }
  { cudaEvent_t e = S->events.get(); PSFM_CUDA(cudaEventRecord(e, st)); S->ev_chol.back().second = e; }
}


// exact reduced-system solve, fused tile path: k_schur_tile -> band blocks -> (band matrix | dense S) -> Cholesky
void do_explicit_solve_fused(psfm_ba_solver* S, const RunCfg& c, double radius) {
  cudaStream_t st = S->stream;
  const size_t nx = (size_t)S->F * NVX2;
  StArgs w;
  w.L = lin_of(S); w.pose16 = S->d_pose16.p; w.X = S->d_X[S->cur].p; w.ht = S->d_hinv.p; w.wt = S->d_w.p; w.wk = S->d_wk.p;
  w.K = S->d_K[S->cur].p; w.acc_cam = S->d_xcamrep.p; w.rep_stride = nx; w.intr = c.intr;
  w.entries = S->d_tentries.p; w.task_slot = S->d_task_slot.p; w.task_rng = S->d_task_rng.p; w.tile_task = S->d_tile_task.p;
  w.Sband = S->d_bandrep.p; w.band_stride = S->band_n; w.nrep_mask = S->band_nrep - 1;
  { static const int dbg = getenv("PSFM_SCHUR_FLAGS") ? atoi(getenv("PSFM_SCHUR_FLAGS")) : 0; w.dbg = dbg; }
  auto mark = [&](std::vector<std::pair<cudaEvent_t, cudaEvent_t>>& v, bool begin) {
    cudaEvent_t e = S->events.get();
    PSFM_CUDA(cudaEventRecord(e, st));
    if (begin) v.push_back({e, nullptr}); else v.back().second = e;
  };
  mark(S->ev_sw, true);
  const size_t pipe_smem = S->tile == 256 ? pipe_smem_schur_tile<256>(S->cap_ns, S->cap_np) : pipe_smem_schur_tile<512>(S->cap_ns, S->cap_np);
  if (pipe_ok(S, pipe_smem) && !getenv("PSFM_NO_PIPE_SCHUR")) {
    PipeSrc ps = pipe_src(S);
    ps.obs_a = S->d_a.p; ps.p6 = S->d_hinv.p; ps.p3a = S->d_wk.p; ps.p3b = S->d_w.p;
    PSFM_PIPE_LAUNCH(k_schur_tile_p, pipe_smem_schur_tile, S, c.rot, ps, w);
  } else {
    PSFM_TILE_LAUNCH(k_schur_tile, NVX2, 15, S, c.rot, w);
  }
  mark(S->ev_sw, false);
  mark(S->ev_chol, true);
  k_fold_replicas2<<<grid_for(nx + S->band_n), 256, 0, st>>>(S->d_xband.p, S->d_xcamrep.p, nx, NREP, S->d_bandrep.p, S->band_n, S->band_nrep);
  PSFM_LAUNCH_CHECK();
  dist::allreduce_sum(S->d_xband.p, S->d_xband.n, st);
  cam_finalize(S, c, radius, true);
  if (S->band_chol) { launch_band_cholesky(S); return; }
  S->d_S.zero(st);
  BandAsmArgs ba_;
  ba_.Sband = S->d_xband.p + nx; ba_.scale_c = S->d_scale_c.p; ba_.F = S->F; ba_.span = S->span; ba_.lda = S->NS + 1; ba_.S = S->d_S.p;
  k_schur_assemble_band<<<grid_for(S->band_n), 256, 0, st>>>(ba_); PSFM_LAUNCH_CHECK();
  AsmArgs a;
  a.Sblk = nullptr; a.blk_key = nullptr; a.nblocks = 0;
  a.lin_cam = S->d_lin.p; a.lin_intr = S->d_lin.p + (size_t)S->F * NVL;
  a.prep_intr = S->d_prep.p + (size_t)S->F * NVL; a.xcam = S->d_xband.p; a.xstride = NVX2;
  a.scale_c = S->d_scale_c.p; a.Dc2 = S->d_Dc2.p; a.active = S->d_active.p;
  a.rhs = S->d_rhs.p;
  a.F = S->F; a.C = S->C; a.NS = S->NS; a.lda = S->NS + 1; a.S = S->d_S.p;
  k_schur_assemble_local<<<grid_for(S->F, 128), 128, 0, st>>>(a); PSFM_LAUNCH_CHECK();
  k_schur_assemble_global<<<grid_for(S->F + S->C, 128), 128, 0, st>>>(a); PSFM_LAUNCH_CHECK();
  k_schur_assemble_finish<<<grid_for(S->NS, 128), 128, 0, st>>>(a); PSFM_LAUNCH_CHECK();
  launch_cholesky(S);
}

// exact reduced-system solve: explicit S, banded Cholesky; solution in d_x (d_cholfail on failure)
void do_explicit_solve(psfm_ba_solver* S, const RunCfg& c) {
  ensure_pairs(S);
  cudaStream_t st = S->stream;
  SwArgs w;
  w.L = lin_of(S); w.pose16 = S->d_pose16.p; w.X = S->d_X[S->cur].p; w.ht = S->d_hinv.p; w.wk = S->d_wk.p;
  w.K = S->d_K[S->cur].p; w.W = S->d_W.p; w.WH = S->d_WH.p; w.acc_cam = S->d_xcamrep.p;
  w.rep_stride = (size_t)S->F * NVX; w.intr = c.intr;
  auto mark = [&](std::vector<std::pair<cudaEvent_t, cudaEvent_t>>& v, bool begin) {
    cudaEvent_t e = S->events.get();
    PSFM_CUDA(cudaEventRecord(e, st));
    if (begin) v.push_back({e, nullptr}); else v.back().second = e;
  };
  mark(S->ev_sw, true);
  PSFM_TILE_LAUNCH(k_schur_w, NVX, 12, S, c.rot, w);
  mark(S->ev_sw, false);
  fold_replicas(S, S->d_xcam.p, S->d_xcamrep.p, (size_t)S->F * NVX, nullptr, nullptr);
  S->d_Sblk.zero(st);
  PairArgs pa;
  pa.entries = S->d_entries.p; pa.chunk_blk = S->d_chunk_blk.p; pa.chunk_beg = S->d_chunk_beg.p;
  pa.W = S->d_W.p; pa.WH = S->d_WH.p; pa.Sblk = S->d_Sblk.p;
  mark(S->ev_pairs, true);
  if (S->nchunks) { k_schur_pairs<<<S->nchunks, 128, 0, st>>>(pa); PSFM_LAUNCH_CHECK(); }
  mark(S->ev_pairs, false);
  mark(S->ev_chol, true);
  S->d_S.zero(st);
  AsmArgs a;
  a.Sblk = S->d_Sblk.p; a.blk_key = S->d_blk_key.p; a.nblocks = S->nblocks;
  a.lin_cam = S->d_lin.p; a.lin_intr = S->d_lin.p + (size_t)S->F * NVL;
  a.prep_intr = S->d_prep.p + (size_t)S->F * NVL; a.xcam = S->d_xcam.p; a.xstride = NVX;
  a.scale_c = S->d_scale_c.p; a.Dc2 = S->d_Dc2.p; a.active = S->d_active.p;
  a.rhs = S->d_rhs.p;
  a.F = S->F; a.C = S->C; a.NS = S->NS; a.lda = S->NS + 1; a.S = S->d_S.p;
  if (S->nblocks) { k_schur_assemble_blocks<<<grid_for((size_t)S->nblocks * 36), 256, 0, st>>>(a); PSFM_LAUNCH_CHECK(); }
  k_schur_assemble_local<<<grid_for(S->F, 128), 128, 0, st>>>(a); PSFM_LAUNCH_CHECK();
  dist::allreduce_sum(S->d_S.p, S->d_S.n, st);
  k_schur_assemble_global<<<grid_for(S->F + S->C, 128), 128, 0, st>>>(a); PSFM_LAUNCH_CHECK();
  k_schur_assemble_finish<<<grid_for(S->NS, 128), 128, 0, st>>>(a); PSFM_LAUNCH_CHECK();
  launch_cholesky(S);
}

// LevenbergMarquardtStrategy::ComputeStep + ComputeCandidatePointAndEvaluateCost
StepOut compute_step(psfm_ba_solver* S, const RunCfg& c, double radius, int* nprod) {
  StepOut so;
  memset(&so, 0, sizeof(so));
  int max_it, iters = 0;
  double q_tol, r_tol;
  if (c.solver == PSFM_BA_SOLVER_ITERATIVE_SCHUR) {
    q_tol = c.o.eta; r_tol = -1.0; max_it = c.o.max_linear_solver_iterations;
  } else {
    q_tol = 0.0; r_tol = c.o.exact_r_tolerance;
    max_it = c.o.exact_max_iterations > 0 ? c.o.exact_max_iterations
                                          : std::min(20000, std::max(1000, 5 * S->NS));
  }
  const bool explicit_ok = c.solver == PSFM_BA_SOLVER_EXACT_SCHUR && c.intr <= 1 && !getenv("PSFM_EXACT_PCG") &&
                           (size_t)S->NS * S->NS * sizeof(double) <= ((size_t)4 << 30);
  if (explicit_ok) ensure_pairs(S);
  const bool fused = explicit_ok && S->fused;
  do_reduced_setup(S, c, radius, fused);
  if (explicit_ok) {
    if (fused) do_explicit_solve_fused(S, c, radius); else do_explicit_solve(S, c);
    so.pcg_flag = PCG_SUCCESS;     // the factorisation's verdict comes back with the step scalars below
    iters = 1;
  } else {
    so.pcg_flag = do_pcg(S, c, q_tol, r_tol, max_it, &iters, nprod);
  }
  so.pcg_iters = iters;
  // candidate: points (inside the back-substitution), poses/intrinsics, cost
  S->d_step.zero(S->stream);          // [0..3] step scalars, [4..5] the camera share (k_apply_cams): one memset
  scale_vec(S, S->d_x.p, nullptr);
  // candidate poses / intrinsics first: they only need the reduced-system solution, and the pipelined
  // back-substitution can then evaluate the candidate cost in the same sweep (no k_cost pass over the observations)
  ApplyArgs a;
  a.yc = S->d_x.p; a.scale_c = S->d_scale_c.p; a.active = S->d_active.p;
  a.pose = S->d_pose[S->cur].p; a.K = S->d_K[S->cur].p;
  a.pose_c = S->d_pose[1 - S->cur].p; a.K_c = S->d_K[1 - S->cur].p;
  a.F = S->F; a.C = S->C; a.acc = S->d_step.p + 4;
  const int n = S->F + S->C;
  k_apply_cams<<<(n + 255) / 256, 256, 0, S->stream>>>(a);
  PSFM_LAUNCH_CHECK();
  BackArgs b;
  b.L = lin_of(S); b.pose16 = S->d_pose16.p; b.X = S->d_X[S->cur].p; b.ht = S->d_hinv.p; b.wt = S->d_w.p;
  b.xs = S->d_xs.p; b.K = S->d_K[S->cur].p; b.Xc = S->d_X[1 - S->cur].p; b.acc = S->d_step.p; b.intr = c.intr;
  b.pose_c = nullptr; b.K_c = S->d_K[1 - S->cur].p;
  b.loss.type = c.o.loss_function_type; b.loss.a = c.o.loss_function_scale;
  bool cost_fused = false;
  {
    g_bs_nxs = S->NS;
    static const bool no_pipe = getenv("PSFM_NO_PIPE_BACK") != nullptr, no_fuse = getenv("PSFM_FUSED_COST") == nullptr;
    const size_t lin_smem = S->tile == 256 ? pipe_smem_linearize<256>(S->cap_ns, S->cap_np) : pipe_smem_linearize<512>(S->cap_ns, S->cap_np);
    auto bs_bytes = [&]() { return S->tile == 256 ? pipe_smem_back_substitute<256>(S->cap_ns, S->cap_np) : pipe_smem_back_substitute<512>(S->cap_ns, S->cap_np); };
    // fused cost (opt-in, PSFM_FUSED_COST=1): the candidate pose table (8 F doubles) lives in shared memory; at least
    // two CTAs per SM must fit.  Measured on the bench workload: 16.61 ms per solve fused against 16.57 ms with the
    // separate k_cost pass — the table and the second 16-byte stage cost the third resident CTA, which cancels the
    // 0.085 ms of k_cost.  Kept for problems with few images; off by default.
    g_bs_fuse_F = no_fuse ? 0 : S->F;
    if (g_bs_fuse_F && !(pipe_ok(S, bs_bytes()) && (S->tile != 256 || 2 * (bs_bytes() + 1024) <= (size_t)227 * 1024))) g_bs_fuse_F = 0;
    const size_t bs_smem = bs_bytes();
    if (!no_pipe && pipe_ok(S, lin_smem) && pipe_ok(S, bs_smem)) {     // seg_pose exists iff the sweep was pipelined
      PipeSrc ps = pipe_src(S);
      ps.obs_xy = reinterpret_cast<const double2*>(S->d_r.p); ps.obs_a = S->d_a.p; ps.p6 = S->d_hinv.p; ps.p3a = S->d_w.p;
      if (g_bs_fuse_F) { ps.obs_xy2 = S->d_obs_xy.p; b.pose_c = S->d_pose[1 - S->cur].p; cost_fused = true; }
      PSFM_PIPE_LAUNCH(k_back_substitute_p, pipe_smem_back_substitute, S, c.rot, ps, b);
    } else {
      g_bs_fuse_F = 0;
      PSFM_TILE_LAUNCH(k_back_substitute, 3, 12, S, c.rot, b);
    }
  }
  if (S->M && !cost_fused) {
    CostArgs ca;
    ca.pose = S->d_pose[1 - S->cur].p; ca.X = S->d_X[1 - S->cur].p; ca.K = S->d_K[1 - S->cur].p;
    ca.loss.type = c.o.loss_function_type; ca.loss.a = c.o.loss_function_scale;
    ca.acc_cost = S->d_step.p + 3;
    const unsigned g = (unsigned)std::min<size_t>(((size_t)S->M + 255) / 256, 148 * 8);
    k_cost<<<g, 256, 0, S->stream>>>(S->tc(), ca);
    PSFM_LAUNCH_CHECK();
  }
  dist::allreduce_sum(S->d_step.p, 4, S->stream);
  d2h(S, S->hs->step, S->d_step.p, 6);          // step[4] | rep[2]: adjacent in HostScalars and in d_step
  d2h(S, &S->hs->prep_fail, S->d_prep.p + (size_t)S->F * NVL + (size_t)S->C * NVI, 1);
  if (explicit_ok) d2h(S, &S->hs->chol_fail, S->d_cholfail.p, 1);
  PSFM_CUDA(cudaStreamSynchronize(S->stream));
  if (explicit_ok && S->hs->chol_fail) so.pcg_flag = PCG_FAILURE;
  so.linear_ok = (so.pcg_flag != PCG_FAILURE) && !(S->hs->prep_fail > 0.0);
  so.mcc = -S->hs->step[0];
  so.step_sq = S->hs->step[1] + S->hs->rep[0];
  so.cand_x2 = S->hs->step[2] + S->hs->rep[1];
  so.cand_cost = S->hs->step[3];
  if (!std::isfinite(so.mcc) || !std::isfinite(so.step_sq) || !std::isfinite(so.cand_cost)) {
    // IsArrayValid(step) failed somewhere -> LINEAR_SOLVER_FAILURE
    if (!std::isfinite(so.mcc) || !std::isfinite(so.step_sq)) so.linear_ok = false;
  }
  return so;
}

int count_observed_points_all_ranks(psfm_ba_solver* S) {
  // every point lives on exactly one rank
  if (dist::world_size() == 1) return S->P;
  S->d_x2.zero(S->stream);
  k_fill<<<1, 32, 0, S->stream>>>(S->d_x2.p, (double)S->P, 1);
  PSFM_LAUNCH_CHECK();
  dist::allreduce_sum(S->d_x2.p, 1, S->stream);
  d2h(S, &S->hs->x2, S->d_x2.p, 1);
  PSFM_CUDA(cudaStreamSynchronize(S->stream));
  return (int)(S->hs->x2 + 0.5);
}

// Sharded problems: whether an image / a camera has observations — i.e. whether Ceres would add
// its parameter block at all (bundle_adjustment.cc:348-366) — is a property of the WHOLE problem.
// A shard that happens not to see an image must still treat its pose as variable, otherwise the
// ranks disagree on the active unknowns.  Max all-reduce of the per-rank flags, once per world.
void sync_observed_flags(psfm_ba_solver* S) {
  const int world = dist::world_size();
  if (world <= 1 || S->flags_world == world) return;
  const int n = S->F + S->C;
  std::vector<double> h((size_t)n);
  for (int i = 0; i < S->F; ++i) h[i] = S->img_has_obs[i] ? 1.0 : 0.0;
  for (int c = 0; c < S->C; ++c) h[(size_t)S->F + c] = S->cam_has_obs[c] ? 1.0 : 0.0;
  DBuf<double> d;
  d.alloc((size_t)n, S->stream);
  d.upload(h.data(), (size_t)n, S->stream);
  dist::allreduce_max(d.p, (size_t)n, S->stream);
  PSFM_CUDA(cudaMemcpyAsync(h.data(), d.p, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, S->stream));
  PSFM_CUDA(cudaStreamSynchronize(S->stream));
  for (int i = 0; i < S->F; ++i) S->img_has_obs[i] = h[i] > 0.5 ? 1 : 0;
  for (int c = 0; c < S->C; ++c) S->cam_has_obs[c] = h[(size_t)S->F + c] > 0.5 ? 1 : 0;
  S->flags_world = world;
}

int total_observations_all_ranks(psfm_ba_solver* S) {
  if (dist::world_size() == 1) return S->M;
  k_fill<<<1, 32, 0, S->stream>>>(S->d_x2.p, (double)S->M, 1);
  PSFM_LAUNCH_CHECK();
  dist::allreduce_sum(S->d_x2.p, 1, S->stream);
  d2h(S, &S->hs->x2, S->d_x2.p, 1);
  PSFM_CUDA(cudaStreamSynchronize(S->stream));
  return (int)(S->hs->x2 + 0.5);
}

void print_summary(const psfm_ba_summary& s) {
  // PrintSolverSummary, bundle_adjustment.cc:560-614
  static const char* tn[] = {"Convergence", "Convergence", "Convergence", "No convergence", "Failure", "Convergence"};
  printf("    Residuals : %d\n   Parameters : %d\n   Iterations : %d\n         Time : %g [s]\n"
         " Initial cost : %.6g [px]\n   Final cost : %.6g [px]\n  Termination : %s\n\n",
         s.num_residuals_reduced, s.num_effective_parameters_reduced, s.num_successful_steps + s.num_unsuccessful_steps,
         s.total_time_in_seconds, std::sqrt(s.initial_cost / s.num_residuals_reduced),
         std::sqrt(s.final_cost / s.num_residuals_reduced), tn[s.termination]);
}

// Re-pack the surviving observations (after a filter) on the device: new tiles, new pair structure;
// the state of record moves through the caller-order scratch (a point keeps its id, its slot changes).
void rebuild_structure(psfm_ba_solver* S) {
  PSFM_CUDA(cudaStreamSynchronize(S->stream));
  std::vector<double> xyz(3 * (size_t)S->P_total, 0.0);
  scatter_points(S, xyz.data());
  S->num_alive = -1;                       // unknown until the compaction has counted
  const int rc = build_structure(S);
  if (rc != PSFM_OK) throw CudaFail{rc};
  S->pairs_ready = false; S->fused = false; S->band_chol = false;
  alloc_work(S);
  gather_points(S, xyz.data());
  PSFM_CUDA(cudaStreamSynchronize(S->stream));
  S->structure_dirty = false;
}

inline void ensure_structure(psfm_ba_solver* S) {
  if (S->structure_dirty) rebuild_structure(S);
}

int run_impl(psfm_ba_solver* S, const psfm_ba_options* opts, psfm_ba_summary* out) {
  RunCfg c;
  ensure_structure(S);
  sync_observed_flags(S);
  int rc = resolve_cfg(S, opts, c);
  if (rc != PSFM_OK) return rc;
  const psfm_ba_options& o = c.o;
  psfm_ba_summary s;
  memset(&s, 0, sizeof(s));
  s.world_size = dist::world_size();
  s.linear_solver_used = c.solver;
  const int M_all = total_observations_all_ranks(S);
  if (M_all == 0) {
    if (o.print_summary) printf("Zero residual for BA\n");
    if (out) *out = s;
    return PSFM_ZERO_RESIDUALS;
  }
  const double t0 = now_s();
  S->events.reset(); S->ev_lin.clear(); S->ev_sp.clear(); S->ev_sw.clear(); S->ev_pairs.clear(); S->ev_chol.clear();
  upload_state(S);
  S->pb_fresh = false;
  set_masks_and_unit_scale(S, c);
  s.num_residuals_reduced = 2 * M_all;
  s.num_effective_parameters_reduced = c.num_effective_parameters + 3 * count_observed_points_all_ranks(S);

  cudaEvent_t ev_begin = S->events.get(), ev_end = S->events.get();
  PSFM_CUDA(cudaEventRecord(ev_begin, S->stream));

  // ---- TrustRegionMinimizer::Minimize ----
  double radius = o.initial_trust_region_radius;
  double decrease_factor = 2.0;
  int num_invalid = 0, iteration = 0, nprod = 0;
  // iteration 0: evaluate; jacobi scaling from the unscaled Jacobian, then re-linearise scaled
  LinOut lo;
  lo = linearize_and_measure(S, c, radius, true, true);
  s.num_linearize = 1;
  double x_cost = lo.cost, gmax = lo.gmax;
  double x_norm = std::sqrt(current_x_sqnorm(S));
  s.initial_cost = x_cost;
  int term = PSFM_TERM_NO_CONVERGENCE;
  bool step_ok_prev = true;
  if (o.minimizer_progress_to_stdout)
    printf("iter      cost      cost_change  |gradient|   |step|    tr_ratio  tr_radius  ls_iter\n%4d % .6e  % .3e  % .3e\n",
           0, x_cost, 0.0, gmax);
  for (;;) {
    if (step_ok_prev && iteration > 0) s.num_successful_steps++;
    if (iteration >= o.max_num_iterations) { term = PSFM_TERM_NO_CONVERGENCE; break; }
    if (gmax <= o.gradient_tolerance) { term = PSFM_TERM_CONVERGENCE_GRADIENT; break; }
    if (radius <= o.min_trust_region_radius) { term = PSFM_TERM_MIN_RADIUS; break; }
    ++iteration;
    step_ok_prev = false;
    const StepOut so = compute_step(S, c, radius, &nprod);
    s.num_linear_iterations += so.pcg_iters;
    const bool valid = so.linear_ok && so.mcc > 0.0;
    if (!valid) {
      // HandleInvalidStep -> LevenbergMarquardtStrategy::StepIsInvalid == StepRejected(0)
      s.num_unsuccessful_steps++;
      if (++num_invalid >= o.max_num_consecutive_invalid_steps) { term = PSFM_TERM_FAILURE; break; }
      radius = radius / decrease_factor;
      decrease_factor *= 2.0;
      continue;
    }
    num_invalid = 0;
    const double step_norm = std::sqrt(so.step_sq);
    if (step_norm <= o.parameter_tolerance * (x_norm + o.parameter_tolerance)) { term = PSFM_TERM_CONVERGENCE_PARAMETER; break; }
    const double cost_change = x_cost - so.cand_cost;
    if (std::fabs(cost_change) <= o.function_tolerance * x_cost) { term = PSFM_TERM_CONVERGENCE_FUNCTION; break; }
    const double rho = cost_change / so.mcc;
    if (rho > o.min_relative_decrease) {
      S->cur = 1 - S->cur;   // x = candidate
      x_norm = std::sqrt(so.cand_x2);
      const double t = 2.0 * rho - 1.0;
      radius = radius / std::max(1.0 / 3.0, 1.0 - t * t * t);
      radius = std::min(o.max_trust_region_radius, radius);
      decrease_factor = 2.0;
      lo = linearize_and_measure(S, c, radius, true);
      s.num_linearize++;
      x_cost = lo.cost;
      gmax = lo.gmax;
      step_ok_prev = true;
    } else {
      s.num_unsuccessful_steps++;
      radius = radius / decrease_factor;
      decrease_factor *= 2.0;
    }
    if (o.minimizer_progress_to_stdout)
      printf("%4d % .6e  % .3e  % .3e  % .3e  % .3e  % .3e  %d\n", iteration, step_ok_prev ? x_cost : so.cand_cost,
             cost_change, gmax, step_norm, rho, radius, so.pcg_iters);
  }
  PSFM_CUDA(cudaEventRecord(ev_end, S->stream));
  PSFM_CUDA(cudaStreamSynchronize(S->stream));
  float ms = 0.f;
  PSFM_CUDA(cudaEventElapsedTime(&ms, ev_begin, ev_end));
  s.device_ms = ms;
  for (auto& e : S->ev_lin) { PSFM_CUDA(cudaEventElapsedTime(&ms, e.first, e.second)); s.linearize_ms += ms; }
  for (auto& e : S->ev_sp) { PSFM_CUDA(cudaEventElapsedTime(&ms, e.first, e.second)); s.schur_product_ms += ms; }
  for (auto& e : S->ev_sw) { PSFM_CUDA(cudaEventElapsedTime(&ms, e.first, e.second)); s.schur_w_ms += ms; }
  for (auto& e : S->ev_pairs) { PSFM_CUDA(cudaEventElapsedTime(&ms, e.first, e.second)); s.schur_pairs_ms += ms; }
  for (auto& e : S->ev_chol) { PSFM_CUDA(cudaEventElapsedTime(&ms, e.first, e.second)); s.cholesky_ms += ms; }
  s.num_explicit_solves = (int)S->ev_chol.size();
  s.num_pair_entries = S->npairs; s.num_pair_tasks = S->ntasks; s.explicit_fused = S->fused ? 1 : 0;
  s.num_linearize = (int)S->ev_lin.size();
  s.num_schur_products = (int)S->ev_sp.size();
  s.num_iterations = iteration;
  s.termination = term;
  s.final_cost = x_cost;
  download_state(S);
  s.total_time_in_seconds = now_s() - t0;
  if (o.print_summary && dist::rank() == 0) print_summary(s);
  if (out) *out = s;
  return PSFM_OK;
}

int check_device() {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
    cudaGetLastError();
    set_error("no CUDA device available (this library has no CPU path)");
    return PSFM_ERR_NO_DEVICE;
  }
  return PSFM_OK;
}

}  // namespace

// ---------------------------------------------------------------- C ABI

extern "C" void psfm_ba_default_options(psfm_ba_options* o) {
  memset(o, 0, sizeof(*o));
  o->loss_function_type = PSFM_LOSS_TRIVIAL;   // bundle_adjustment.h:51
  o->loss_function_scale = 1.0;                // :54
  o->refine_focal_length = 1;                  // :57
  o->refine_principal_point = 0;               // :60
  o->refine_extra_params = 1;                  // :63
  o->refine_extrinsics = 1;                    // :66
  o->refine_rotation = 1;                      // :69
  o->print_summary = 1;                        // :72
  o->minimizer_progress_to_stdout = 0;         // :86
  o->function_tolerance = 0.0;                 // :83
  o->gradient_tolerance = 0.0;                 // :84
  o->parameter_tolerance = 0.0;                // :85
  o->max_num_iterations = 100;                 // :87
  o->max_linear_solver_iterations = 200;       // :88
  o->max_num_consecutive_invalid_steps = 10;   // :89
  o->linear_solver = PSFM_BA_SOLVER_AUTO;
  o->eta = 1e-1;                               // Ceres default
  o->exact_r_tolerance = 1e-10;
  o->exact_max_iterations = 0;
  o->initial_trust_region_radius = 1e4;        // Ceres defaults
  o->max_trust_region_radius = 1e16;
  o->min_trust_region_radius = 1e-32;
  o->min_relative_decrease = 1e-3;
  o->min_lm_diagonal = 1e-6;
  o->max_lm_diagonal = 1e32;
  o->jacobi_scaling = 1;
  o->pcg_check_period = 0;
}

extern "C" void psfm_ba_global_options(psfm_ba_options* o) {
  // GlobalMapperOptions::GlobalBundleAdjustment, controllers/global_mapper.cc:41-71
  psfm_ba_default_options(o);
  o->function_tolerance = 1e-6;
  o->gradient_tolerance = 1.0;
  o->parameter_tolerance = 1e-8;
  o->max_num_iterations = 50;
  o->max_linear_solver_iterations = 100;
  o->minimizer_progress_to_stdout = 1;
  o->print_summary = 1;
  o->refine_rotation = 0;
  o->refine_focal_length = 0;
  o->refine_principal_point = 0;
  o->refine_extra_params = 0;
  o->loss_function_type = PSFM_LOSS_SOFT_L1;
}

extern "C" int psfm_ba_create(const psfm_ba_problem* pb, psfm_ba_solver** out) {
  if (!pb || !out) { set_error("psfm_ba_create: null argument"); return PSFM_ERR_INVALID; }
  *out = nullptr;
  int rc = check_device();
  if (rc != PSFM_OK) return rc;
  psfm_ba_solver* S = new psfm_ba_solver();
  try {
    PSFM_CUDA(cudaStreamCreateWithFlags(&S->sh.s, cudaStreamNonBlocking));
    PSFM_CUDA(cudaStreamCreateWithFlags(&S->sh.copy, cudaStreamNonBlocking));
    PSFM_CUDA(cudaEventCreateWithFlags(&S->sh.ev_idx, cudaEventDisableTiming));
    PSFM_CUDA(cudaEventCreateWithFlags(&S->sh.ev_xy, cudaEventDisableTiming));
    S->stream = S->sh.s;
    rc = upload_problem(S, pb);
    if (rc == PSFM_OK) rc = build_structure(S);
    if (rc != PSFM_OK) { delete S; return rc; }
    S->h_qvec.assign(pb->qvec, pb->qvec + 4 * (size_t)S->F);
    S->h_tvec.assign(pb->tvec, pb->tvec + 3 * (size_t)S->F);
    S->h_K.assign(pb->cam_params, pb->cam_params + 3 * (size_t)S->C);
    PhaseTimer tm;
    alloc_work(S);
    gather_points(S, pb->xyz);
    PSFM_CUDA(cudaStreamSynchronize(S->stream));
    tm.mark("allocate work buffers");
  } catch (const CudaFail& f) {
    delete S;
    return f.code;
  }
  *out = S;
  return PSFM_OK;
}

extern "C" int psfm_ba_set_state(psfm_ba_solver* S, const double* qvec, const double* tvec, const double* xyz,
                                 const double* cam_params) {
  if (!S) return PSFM_ERR_INVALID;
  if (qvec) S->h_qvec.assign(qvec, qvec + 4 * (size_t)S->F);
  if (tvec) S->h_tvec.assign(tvec, tvec + 3 * (size_t)S->F);
  if (xyz) gather_points(S, xyz);
  if (cam_params) S->h_K.assign(cam_params, cam_params + 3 * (size_t)S->C);
  return PSFM_OK;
}

extern "C" int psfm_ba_get_state(psfm_ba_solver* S, double* qvec, double* tvec, double* xyz, double* cam_params) {
  if (!S) return PSFM_ERR_INVALID;
  if (qvec) memcpy(qvec, S->h_qvec.data(), sizeof(double) * S->h_qvec.size());
  if (tvec) memcpy(tvec, S->h_tvec.data(), sizeof(double) * S->h_tvec.size());
  if (xyz) scatter_points(S, xyz);   // points this solver does not observe are left untouched
  if (cam_params) memcpy(cam_params, S->h_K.data(), sizeof(double) * S->h_K.size());
  return PSFM_OK;
}

extern "C" int psfm_ba_run(psfm_ba_solver* S, const psfm_ba_options* opts, psfm_ba_summary* summary) {
  if (!S) return PSFM_ERR_INVALID;
  try {
    return run_impl(S, opts, summary);
  } catch (const CudaFail& f) {
    return f.code;
  }
}

extern "C" void psfm_ba_destroy(psfm_ba_solver* S) { delete S; }

extern "C" int psfm_ba_solve(psfm_ba_problem* pb, const psfm_ba_options* opts, psfm_ba_summary* summary) {
  if (!pb) return PSFM_ERR_INVALID;
  if (pb->num_observations == 0 && dist::world_size() == 1) {
    psfm_ba_options o;
    if (opts) o = *opts; else psfm_ba_default_options(&o);
    if (o.print_summary) printf("Zero residual for BA\n");
    if (summary) memset(summary, 0, sizeof(*summary));
    return PSFM_ZERO_RESIDUALS;
  }
  psfm_ba_solver* S = nullptr;
  int rc = psfm_ba_create(pb, &S);
  if (rc != PSFM_OK) return rc;
  rc = psfm_ba_run(S, opts, summary);
  if (rc == PSFM_OK) psfm_ba_get_state(S, pb->qvec, pb->tvec, pb->xyz, pb->cam_params);
  psfm_ba_destroy(S);
  return rc;
}

extern "C" int psfm_ba_evaluate(psfm_ba_solver* S, const psfm_ba_options* opts, double* cost, double* residuals,
                                double* gradient_cam, double* gradient_pts) {
  if (!S) return PSFM_ERR_INVALID;
  try {
    RunCfg c;
    ensure_structure(S);
    sync_observed_flags(S);
    int rc = resolve_cfg(S, opts, c);
    if (rc != PSFM_OK) return rc;
    upload_state(S);
    set_masks_and_unit_scale(S, c);
    do_linearize(S, c, false);
    const size_t F = S->F, C = S->C, M = S->M, P = S->P;
    std::vector<double> lin(S->d_lin.n), r(2 * M), gp(3 * P);
    std::vector<int> obs_orig(M);
    if (M) d2h(S, obs_orig.data(), S->d_obs_orig.p, M);
    d2h(S, lin.data(), S->d_lin.p, lin.size());
    if (M) d2h(S, r.data(), S->d_r.p, 2 * M);
    if (P) d2h(S, gp.data(), S->d_gp.p, 3 * P);
    PSFM_CUDA(cudaStreamSynchronize(S->stream));
    if (cost) *cost = lin[F * NVL + C * NVI];
    if (residuals) memset(residuals, 0, sizeof(double) * 2 * (size_t)S->M0);      // filtered observations: 0
    if (residuals)
      for (size_t j = 0; j < M; ++j) {
        residuals[2 * (size_t)obs_orig[j]] = r[2 * j];
        residuals[2 * (size_t)obs_orig[j] + 1] = r[2 * j + 1];
      }
    if (gradient_cam) {
      for (size_t i = 0; i < F; ++i)
        for (int k = 0; k < 6; ++k) gradient_cam[6 * i + k] = c.active[6 * i + k] ? lin[i * NVL + 12 + k] : 0.0;
      for (size_t cc = 0; cc < C; ++cc)
        for (int k = 0; k < 3; ++k)
          gradient_cam[6 * F + 3 * cc + k] = c.active[6 * F + 3 * cc + k] ? lin[F * NVL + cc * NVI + 6 + k] : 0.0;
    }
    if (gradient_pts) {
      memset(gradient_pts, 0, sizeof(double) * 3 * (size_t)S->P_total);
      for (size_t id = 0; id < P; ++id)
        for (int k = 0; k < 3; ++k) gradient_pts[3 * (size_t)S->pt_orig[id] + k] = gp[k * P + id];
    }
    return PSFM_OK;
  } catch (const CudaFail& f) {
    return f.code;
  }
}

// ---------------------------------------------------------------- refinement loop around the BA

namespace {

FilterCtx filter_ctx(psfm_ba_solver* S) {
  FilterCtx c;
  c.pt_ptr = S->d_pt_ptr.p; c.obs_img = S->d_obs_img.p; c.obs_xy = S->d_obs_xy.p; c.obs_orig = S->d_obs_orig.p;
  c.pt_orig = nullptr; c.img_cam = S->d_img_cam.p;
  c.pose = S->d_pose[S->cur].p; c.X = S->d_X[S->cur].p; c.K = S->d_K[S->cur].p;
  c.P = S->P; c.alive = S->d_alive.p; c.count = S->d_count.p;
  return c;
}

// the reference's num_filtered, summed over the ranks
long long read_filter_count(psfm_ba_solver* S) {
  unsigned long long h = 0;
  PSFM_CUDA(cudaMemcpyAsync(&h, S->d_count.p, sizeof(h), cudaMemcpyDeviceToHost, S->stream));
  PSFM_CUDA(cudaStreamSynchronize(S->stream));
  if (dist::world_size() > 1) {
    k_fill<<<1, 32, 0, S->stream>>>(S->d_x2.p, (double)h, 1);
    PSFM_LAUNCH_CHECK();
    dist::allreduce_sum(S->d_x2.p, 1, S->stream);
    d2h(S, &S->hs->x2, S->d_x2.p, 1);
    PSFM_CUDA(cudaStreamSynchronize(S->stream));
    h = (unsigned long long)(S->hs->x2 + 0.5);
  }
  return (long long)h;
}

long long filter_negative_depth_impl(psfm_ba_solver* S) {
  ensure_structure(S);
  upload_state(S);
  S->d_count.zero(S->stream);
  if (S->P) {
    k_filter_negative_depth<<<grid_for(S->P, 128), 128, 0, S->stream>>>(filter_ctx(S));
    PSFM_LAUNCH_CHECK();
  }
  const long long n = read_filter_count(S);
  if (n > 0) S->structure_dirty = true;
  return n;
}

long long filter_points_impl(psfm_ba_solver* S, double max_reproj_error, double min_tri_angle_deg) {
  ensure_structure(S);
  upload_state(S);
  cudaStream_t st = S->stream;
  if (S->d_pt_error.n != (size_t)S->P_total) {
    S->d_pt_error.alloc(S->P_total, st);
    if (S->P_total) { k_fill<<<grid_for(S->P_total), 256, 0, st>>>(S->d_pt_error.p, nan(""), (size_t)S->P_total); PSFM_LAUNCH_CHECK(); }
  }
  DBuf<double> centres;
  DBuf<int> pt_orig;
  centres.alloc(3 * (size_t)S->F, st);
  pt_orig.alloc(S->P, st);
  pt_orig.upload(S->pt_orig.data(), S->P, st);
  k_proj_centres<<<grid_for(S->F, 128), 128, 0, st>>>(S->d_pose[S->cur].p, S->F, centres.p);
  PSFM_LAUNCH_CHECK();
  S->d_count.zero(st);
  if (S->P) {
    FilterCtx c = filter_ctx(S);
    c.pt_orig = pt_orig.p;
    k_filter_points<<<grid_for(S->P, 128), 128, 0, st>>>(c, centres.p, max_reproj_error * max_reproj_error,
                                                        min_tri_angle_deg * 0.017453292519943295, S->d_pt_error.p);
    PSFM_LAUNCH_CHECK();
  }
  const long long n = read_filter_count(S);
  if (n > 0) S->structure_dirty = true;
  return n;
}

// Reconstruction::Normalize(extent, p0, p1, use_images = true), base/reconstruction.cc:373-468, on
// the state of record (host; every run uploads it): per-axis independently sorted FLOAT coordinates
// of the projection centres, robust box [P0, P1], translation = mean of the sorted coordinates in
// that range, scale = extent / |box diagonal|.
void normalize_impl(psfm_ba_solver* S, double extent, double p0, double p1, double* translation, double* scale_out) {
  ensure_structure(S);
  const int F = S->F;
  double mean[3] = {0, 0, 0}, scale = 1.0;
  if (F >= 2) {
    std::vector<double> cen(3 * (size_t)F), R(9 * (size_t)F);
    std::vector<float> cx(F), cy(F), cz(F);
    for (int i = 0; i < F; ++i) {
      double* q = &S->h_qvec[4 * (size_t)i];
      const double n = std::sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
      if (n == 0.0) { q[0] = 1.0; q[1] = q[2] = q[3] = 0.0; } else for (int k = 0; k < 4; ++k) q[k] /= n;
      double* r = &R[9 * (size_t)i];
      const double q0 = q[0], q1 = q[1], q2 = q[2], q3 = q[3];
      r[0] = 1.0 - 2.0 * (q2 * q2 + q3 * q3); r[1] = 2.0 * (q1 * q2 - q0 * q3); r[2] = 2.0 * (q1 * q3 + q0 * q2);
      r[3] = 2.0 * (q1 * q2 + q0 * q3); r[4] = 1.0 - 2.0 * (q1 * q1 + q3 * q3); r[5] = 2.0 * (q2 * q3 - q0 * q1);
      r[6] = 2.0 * (q1 * q3 - q0 * q2); r[7] = 2.0 * (q2 * q3 + q0 * q1); r[8] = 1.0 - 2.0 * (q1 * q1 + q2 * q2);
      const double* t = &S->h_tvec[3 * (size_t)i];
      for (int k = 0; k < 3; ++k) cen[3 * (size_t)i + k] = -(r[k] * t[0] + r[3 + k] * t[1] + r[6 + k] * t[2]);
      cx[i] = (float)cen[3 * (size_t)i]; cy[i] = (float)cen[3 * (size_t)i + 1]; cz[i] = (float)cen[3 * (size_t)i + 2];
    }
    std::sort(cx.begin(), cx.end()); std::sort(cy.begin(), cy.end()); std::sort(cz.begin(), cz.end());
    const size_t n = (size_t)F;
    const size_t P0 = (size_t)((n > 3) ? p0 * (double)(n - 1) : 0.0);
    const size_t P1 = (size_t)((n > 3) ? p1 * (double)(n - 1) : (double)(n - 1));
    for (size_t i = P0; i <= P1; ++i) { mean[0] += cx[i]; mean[1] += cy[i]; mean[2] += cz[i]; }
    for (int k = 0; k < 3; ++k) mean[k] /= (double)(P1 - P0 + 1);
    const double dx = (double)cx[P1] - (double)cx[P0], dy = (double)cy[P1] - (double)cy[P0], dz = (double)cz[P1] - (double)cz[P0];
    const double old_extent = std::sqrt(dx * dx + dy * dy + dz * dz);
    scale = (old_extent < 2.220446049250313e-16) ? 1.0 : extent / old_extent;
    for (int i = 0; i < F; ++i) {
      const double* r = &R[9 * (size_t)i];
      double c[3];
      for (int k = 0; k < 3; ++k) c[k] = -((cen[3 * (size_t)i + k] - mean[k]) * scale);
      double* t = &S->h_tvec[3 * (size_t)i];
      for (int k = 0; k < 3; ++k) t[k] = r[3 * k] * c[0] + r[3 * k + 1] * c[1] + r[3 * k + 2] * c[2];
    }
    double* X = S->pin_state + 8 * (size_t)F;
    for (size_t id = 0; id < (size_t)S->P; ++id)
      for (int k = 0; k < 3; ++k) X[3 * id + k] = (X[3 * id + k] - mean[k]) * scale;
  }
  if (translation) for (int k = 0; k < 3; ++k) translation[k] = mean[k];
  if (scale_out) *scale_out = scale;
}

}  // namespace

extern "C" void psfm_ba_default_refine_options(psfm_ba_refine_options* r) {
  r->max_refinements = 5;                 // ba_global_max_refinements, controllers/global_mapper.h:68
  r->max_refinement_change = 0.0005;      // ba_global_max_refinement_change, :69
  r->filter_max_reproj_error = 4.0;       // sfm/global_mapper.h:53
  r->filter_min_tri_angle = 1.5;          // :56
  r->normalize_extent = 10.0;             // Reconstruction::Normalize defaults, base/reconstruction.h
  r->normalize_p0 = 0.1;
  r->normalize_p1 = 0.9;
}

extern "C" int psfm_ba_filter_negative_depth(psfm_ba_solver* S, int64_t* num_filtered) {
  if (!S) return PSFM_ERR_INVALID;
  try {
    const long long n = filter_negative_depth_impl(S);
    if (num_filtered) *num_filtered = n;
    return PSFM_OK;
  } catch (const CudaFail& f) { return f.code; }
}

extern "C" int psfm_ba_filter_points(psfm_ba_solver* S, double max_reproj_error, double min_tri_angle_deg, int64_t* num_filtered) {
  if (!S || !(max_reproj_error >= 0.0) || !(min_tri_angle_deg >= 0.0)) return PSFM_ERR_INVALID;
  try {
    const long long n = filter_points_impl(S, max_reproj_error, min_tri_angle_deg);
    if (num_filtered) *num_filtered = n;
    return PSFM_OK;
  } catch (const CudaFail& f) { return f.code; }
}

extern "C" int psfm_ba_normalize(psfm_ba_solver* S, double extent, double p0, double p1, double* translation, double* scale) {
  if (!S || !(extent > 0.0) || !(p0 >= 0.0 && p0 <= p1 && p1 <= 1.0)) return PSFM_ERR_INVALID;   // CHECKs :375-380
  try {
    normalize_impl(S, extent, p0, p1, translation, scale);
    return PSFM_OK;
  } catch (const CudaFail& f) { return f.code; }
}

extern "C" int psfm_ba_num_observations(psfm_ba_solver* S, int64_t* num_alive) {
  if (!S) return PSFM_ERR_INVALID;
  try {
    ensure_structure(S);
    if (num_alive) *num_alive = total_observations_all_ranks(S);
    return PSFM_OK;
  } catch (const CudaFail& f) { return f.code; }
}

extern "C" int psfm_ba_get_observation_mask(psfm_ba_solver* S, uint8_t* alive) {
  if (!S || !alive) return PSFM_ERR_INVALID;
  try {
    if (S->M0) PSFM_CUDA(cudaMemcpyAsync(alive, S->d_alive.p, (size_t)S->M0, cudaMemcpyDeviceToHost, S->stream));
    PSFM_CUDA(cudaStreamSynchronize(S->stream));
    return PSFM_OK;
  } catch (const CudaFail& f) { return f.code; }
}

extern "C" int psfm_ba_get_point_errors(psfm_ba_solver* S, double* error) {
  if (!S || !error) return PSFM_ERR_INVALID;
  try {
    if (S->d_pt_error.n != (size_t)S->P_total) {
      for (int k = 0; k < S->P_total; ++k) error[k] = nan("");
      return PSFM_OK;
    }
    if (S->P_total) PSFM_CUDA(cudaMemcpyAsync(error, S->d_pt_error.p, sizeof(double) * (size_t)S->P_total, cudaMemcpyDeviceToHost, S->stream));
    PSFM_CUDA(cudaStreamSynchronize(S->stream));
    return PSFM_OK;
  } catch (const CudaFail& f) { return f.code; }
}

// IterativeGlobalRefinement (controllers/global_mapper.cc:245-271) on the resident problem, minus the
// IncrementalTriangulator calls (CompleteAndMergeTracks / Retriangulate: out of scope, 0 changes):
// <= max_refinements rounds of { AdjustGlobalBundle = negative-depth filter, BA, Normalize ;
// FilterAllPoints3D }, until the changed fraction drops below max_refinement_change.
extern "C" int psfm_ba_iterative_refinement(psfm_ba_solver* S, const psfm_ba_options* opts, const psfm_ba_refine_options* ropts,
                                            psfm_ba_refine_report* report) {
  if (!S) return PSFM_ERR_INVALID;
  psfm_ba_refine_options r;
  if (ropts) r = *ropts; else psfm_ba_default_refine_options(&r);
  psfm_ba_options o;
  if (opts) o = *opts; else psfm_ba_global_options(&o);
  if (r.max_refinements <= 0 || r.max_refinements > PSFM_BA_MAX_REFINEMENTS || r.max_refinement_change < 0.0) {   // CHECK_OPTION :84-85
    set_error("psfm_ba_iterative_refinement: bad refinement options");
    return PSFM_ERR_INVALID;
  }
  if (S->F < 10) {   // kMinNumRegImagesForFastBA, controllers/global_mapper.cc:226-235
    o.function_tolerance /= 10; o.gradient_tolerance /= 10; o.parameter_tolerance /= 10;
    o.max_num_iterations *= 2; o.max_linear_solver_iterations = 200;
  }
  psfm_ba_refine_report rep;
  memset(&rep, 0, sizeof(rep));
  const double t0 = now_s();
  try {
    for (int i = 0; i < r.max_refinements; ++i) {
      ensure_structure(S);
      const long long num_obs = total_observations_all_ranks(S);
      rep.num_observations[i] = num_obs;
      rep.num_negative_depth[i] = filter_negative_depth_impl(S);
      psfm_ba_summary sum;
      const int rc = run_impl(S, &o, &sum);
      if (rc < 0) return rc;
      rep.ba_iterations[i] = sum.num_iterations;
      rep.ba_final_cost[i] = sum.final_cost;
      rep.ba_termination[i] = sum.termination;
      if (rc == PSFM_OK) normalize_impl(S, r.normalize_extent, r.normalize_p0, r.normalize_p1, nullptr, nullptr);
      const long long changed = filter_points_impl(S, r.filter_max_reproj_error, r.filter_min_tri_angle);
      rep.num_changed[i] = changed;
      rep.changed[i] = num_obs > 0 ? (double)changed / (double)num_obs : 0.0;
      rep.num_rounds = i + 1;
      if (rep.changed[i] < r.max_refinement_change) break;
    }
    ensure_structure(S);
    rep.final_num_observations = total_observations_all_ranks(S);
    rep.total_time_in_seconds = now_s() - t0;
    if (report) *report = rep;
    return PSFM_OK;
  } catch (const CudaFail& f) { return f.code; }
}

extern "C" int psfm_ba_band_solve(const double* A, const double* b, int32_t nb, int32_t bw, double* x) {
  if (!A || !b || !x || nb < 1 || bw < 0) return PSFM_ERR_INVALID;
  int rc = check_device();
  if (rc != PSFM_OK) return rc;
  bw = std::min(bw, nb - 1);
  const BandPlan pl = band_chol_plan(nb, bw);
  const int W = pl.W, RS = pl.RS, n = nb + 3;
  if (W == 0) { set_error("psfm_ba_band_solve: band too wide for the register window"); return PSFM_ERR_UNSUPPORTED; }
  bw = pl.bw;
  // the layout k_band_assemble writes, from the dense input (both sides of the two-sided form)
  auto entry = [&](int R, int e) -> double {            // A[R][R - e], identity below nb
    if (R >= nb) return e == 0 ? 1.0 : 0.0;
    return A[(size_t)R * n + (R - e)];
  };
  auto arrow = [&](int R, int aa) -> double {
    if (R >= nb) return 0.0;
    return aa < 3 ? A[(size_t)(nb + aa) * n + R] : b[R];
  };
  std::vector<double> Ab((size_t)(pl.rows[0] + pl.rows[1]) * RS, 0.0), C4(32, 0.0);
  for (int r = 0; r < pl.rows[0]; ++r) {
    double* row = &Ab[(size_t)r * RS];
    if (r >= std::min((int)nb, pl.nbs[0])) { row[0] = 1.0; continue; }
    for (int k = 0; k <= std::min((int)bw, r); ++k) row[k] = entry(r, k);
    for (int a = 0; a < 4; ++a) row[W + a] = arrow(r, a);
  }
  for (int r = 0; r < pl.rows[1]; ++r) {
    double* row = &Ab[(size_t)(pl.rows[0] + r) * RS];
    if (r >= pl.nbs[1]) { row[0] = 1.0; continue; }
    for (int k = 0; k <= std::min((int)bw, r); ++k)
      if (!(r >= pl.n1 && r - k >= pl.n1)) row[k] = entry(pl.nbp - 1 - (r - k), k);
    if (r < pl.n1)
      for (int a = 0; a < 4; ++a) row[W + a] = arrow(pl.nbp - 1 - r, a);
  }
  for (int a = 0; a < 3; ++a) {
    for (int c = 0; c < 3; ++c) C4[4 * a + c] = A[(size_t)(nb + a) * n + nb + c];
    C4[12 + a] = C4[4 * a + 3] = b[nb + a];
  }
  try {
    cudaStream_t st = nullptr;
    BandWork wk;
    DBuf<double> dx;
    DBuf<int> dfail;
    wk.alloc(pl, st); dx.alloc(n); dfail.alloc(1); dfail.zero(st);
    wk.Ab.upload(Ab.data(), Ab.size(), st); wk.C4.upload(C4.data(), 32, st);
    BandCholArgs c = wk.args(dx.p, n, dfail.p);
    band_chol_launch(c, st);
    int fail = 0;
    PSFM_CUDA(cudaMemcpy(&fail, dfail.p, sizeof(int), cudaMemcpyDeviceToHost));
    if (fail) { set_error("psfm_ba_band_solve: matrix is not positive definite"); return PSFM_ERR_INVALID; }
    PSFM_CUDA(cudaMemcpy(x, dx.p, sizeof(double) * n, cudaMemcpyDeviceToHost));
    return PSFM_OK;
  } catch (const CudaFail& f) {
    return f.code;
  }
}

extern "C" int psfm_ba_linear_step(psfm_ba_solver* S, const psfm_ba_options* opts, double radius, double* step_cam,
                                   double* step_pts, int32_t* num_linear_iterations) {
  if (!S) return PSFM_ERR_INVALID;
  try {
    RunCfg c;
    ensure_structure(S);
    sync_observed_flags(S);
    int rc = resolve_cfg(S, opts, c);
    if (rc != PSFM_OK) return rc;
    S->events.reset(); S->ev_lin.clear(); S->ev_sp.clear(); S->ev_sw.clear(); S->ev_pairs.clear(); S->ev_chol.clear();
    upload_state(S);
    set_masks_and_unit_scale(S, c);
    linearize_and_measure(S, c, radius, false, true);
    int nprod = 0;
    const StepOut so = compute_step(S, c, radius, &nprod);
    const size_t NS = S->NS, P = S->P;
    std::vector<double> yc(NS), X(3 * P), Xc(3 * P), sp(3 * P);
    d2h(S, yc.data(), S->d_x.p, NS);
    if (P) {
      d2h(S, X.data(), S->d_X[S->cur].p, 3 * P);
      d2h(S, Xc.data(), S->d_X[1 - S->cur].p, 3 * P);
      d2h(S, sp.data(), S->d_scale_p.p, 3 * P);
    }
    PSFM_CUDA(cudaStreamSynchronize(S->stream));
    if (step_cam) for (size_t k = 0; k < NS; ++k) step_cam[k] = -yc[k];
    if (step_pts) {
      memset(step_pts, 0, sizeof(double) * 3 * (size_t)S->P_total);
      for (size_t id = 0; id < P; ++id)
        for (int k = 0; k < 3; ++k)
          step_pts[3 * (size_t)S->pt_orig[id] + k] = (Xc[3 * id + k] - X[3 * id + k]) / sp[3 * id + k];
    }
    if (num_linear_iterations) *num_linear_iterations = so.pcg_iters;
    return so.linear_ok ? PSFM_OK : PSFM_ERR_INVALID;
  } catch (const CudaFail& f) {
    return f.code;
  }
}
