// pipeline.cu — handle, device memory plan, stream orchestration and the C ABI of
// libconesgpu.so (include/conesgpu.h).  No CPU fallback: every compute entry point needs
// a CUDA device; without one cp_create fails with CP_E_CUDA.
#include "../../include/conesgpu.h"

#include <math.h>
#include <stdio.h>
#include <string.h>
#include <time.h>

#include <algorithm>
#include <memory>
#include <new>
#include <string>
#include <vector>

#include "cluster_front.cuh"
#include "cluster_kernels.cuh"
#include "color_kernels.cuh"
#include "color_net.cuh"
#include "common.cuh"
#include "copy_pool.hpp"
#include "frame_kernels.cuh"
#include "plane_kernels.cuh"
#include "radix_sort.cuh"
#include "single_frame.cuh"
#include "stream_kernels.cuh"
#include "tflite_reader.hpp"
#include "track_kernels.cuh"
#include "voxel_kernels.cuh"

using namespace cp;

namespace {

constexpr u32 kAbiVersion = 2;  // 2: colour classifier (cp_color_net_*, cp_cone_colors, cp_classify_images), cp_last_pairs
constexpr size_t kStageChunk = 32ull << 20;  // pinned staging buffers for pageable host clouds (two of them)
constexpr size_t kStageMinChunk = 256ull << 10;

struct HostGeom {
  std::vector<u32> frame_n;
  std::vector<u64> frame_off;
  std::vector<u32> frame_tile0;
  std::vector<u32> tile_frame;
  u32 uniform_n = 0, tpf = 0, n_tiles = 0, n_frames = 0;
  u64 n_points = 0;
};

}  // namespace

// parameters of the run in flight (kept so cp_sync can re-run the back half in another mode)
struct RunParams {
  cp_detect_params d;
  VoxelK vk;
  ClusterK ck;
  GroundK gk;
  CropK crop;
  u32 csort_bits, osort_bits;
};

struct cp_handle {
  cp_config cfg{};
  int sms = 148;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_stage[2] = {nullptr, nullptr};
  cudaEvent_t ev_k[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};  // around pass 1, pass 2, per-frame kernel
  bool stage_timing = false;
  std::string err = "";
  u32 launches = 0;
  bool batch_ready = false, ran = false;
  bool taps = false, counted_ground = false, ran_ground = false;
  // back half: 0..2 = shared-memory frame kernel with growing budgets (1024/512 survivors/voxels at
  // 4 CTAs per SM, 2048/1024 at 2, 4096/2048 at 1), 3 = general global-memory path
  int back_mode = 0;
  RunParams rp{};
  u64* d_desc_fv = nullptr;  // frame descriptors of the voxel-offset look-back (parity taps only)
  u32* d_frame_ticket = nullptr;
  u32* d_done = nullptr;  // pass-1 tiles finished per frame (fused front kernel)
  u32 fused_grid = 0;
  bool use_cluster = false, ran_cluster = false;  // single-pass cluster front end (cluster_front.cuh)
  size_t cluster_smem = 0;
  u32 cluster_max = 0;
  bool use_fused = false, ran_fused = false;  // measured slower than two kernels (DESIGN.md §4): opt-in
  u32* d_fc = nullptr;      // [F][8] cp_frame_counters, written on the device
  u32* h_fc = nullptr;      // pinned mirror
  u32* h_result = nullptr;  // pinned mirror of the head of the result block
  u64 prefetch_cap = 0, prefetched = 0;
  bool fetched = false;  // the pinned mirrors hold the results of the run in flight
  // CUDA-graph replay of repeated identical runs
  bool use_graph = true, capturing = false, key_valid = false, graph_key_valid = false;
  cudaGraphExec_t graph_exec = nullptr;
  u32 graph_launches = 0;
  bool graph_plane_run = false;  // the captured run was the plane chain (replays restore the run state below)
  alignas(8) unsigned char last_key[224], graph_key[224];
  // peer-memory gather of the result block (multi-GPU result path)
  struct {
    bool open = false, owner = false;
    u32* base = nullptr;       // owner: own allocation; others: cudaIpcOpenMemHandle mapping
    u32 world = 0, rank = 0, slot_words = 0, seq = 0;
    u32* d_done = nullptr;     // local CTA-completion counter of the publish kernel
    u32* d_seq = nullptr;      // local run number (device-resident: graph replays need no parameter update)
    u32* h_flags = nullptr;    // pinned (owner)
  } gather;
  size_t off_words = 0;
  u32* d_ncrop_f = nullptr;
  u32* d_nvox_f = nullptr;
  ClusterRec* d_slots = nullptr;  // [max_frames][2048] per-frame result slots of the fast back half
  bool gathered = false;  // the global scan + gather of the current run has been enqueued
  bool masked = false;    // keep_mask_kernel of the current run has been enqueued (global keep mask + tile counts)
  // per-frame kernel evaluates pass 2 itself (CONESGPU_FUSED_MASK=0: separate keep_mask_kernel; 2: fused even for a
  // few frames without ground removal, where the default prefers the streaming kernel)
  bool fuse_mask = true, fuse_mask_always = false;
  bool run_fused_mask = false;
  bool ran_frame_kernel = false;

  u64 cap_c = 0, cap_v = 0;
  u32 tiles_cap = 0, sort_tiles_cap = 0, hash_cap = 0;

  // device memory
  Ctl* d_ctl = nullptr;
  uint8_t* d_in = nullptr;  // staged input (host batches)
  size_t d_in_bytes = 0;
  uint8_t* d_out32 = nullptr;   // the ground node's messages (max_points x 32 B), allocated on first use
  u64 ground_points = 0;        // points of the messages cp_batch_ground_remove left in d_out32 ...
  bool ground_out = false;      // ... valid until the next staging, run or ground call
  u32* h_ground = nullptr;      // pinned readback of cp_batch_ground_remove: G_f, then the sector minima
  // colour path (color_kernels.cuh): allocated on first use, grown on demand
  struct ColorBufs {
    u32 *mask = nullptr, *tcount = nullptr, *texcl = nullptr, *off = nullptr, *flags = nullptr;
    float4* pts = nullptr;
    uint8_t* img = nullptr;
    size_t mask_n = 0, tile_n = 0, texcl_n = 0, off_n = 0, flags_n = 0, pts_n = 0, img_n = 0;
    void* pin = nullptr;
    size_t pin_bytes = 0;
    // classifier (color_net.cuh): weights in one device block, per-cone outputs
    float* net_w = nullptr;
    size_t net_w_n = 0;
    ColorNetDev net{};
    bool net_loaded = false;
    uint8_t* colors = nullptr;
    float* probs = nullptr;     // [n][classes] probabilities, then [n][classes] logits
    u32* net_flags = nullptr;
    size_t colors_n = 0, probs_n = 0, net_flags_n = 0;
    // every cluster of a run (cp_batch_cone_colors): boxes, frames, per-cluster counts, (cluster, row, ballot)
    // triples and their sort; the triple buffers are as long as the crop buffer (a triple holds >= 1 crop point)
    float4* box = nullptr;
    u32 *kframe = nullptr, *cnt = nullptr, *tcnt = nullptr, *toff = nullptr, *bctl = nullptr;
    u64 *keys_a = nullptr, *keys_b = nullptr;
    u32 *vals_a = nullptr, *vals_b = nullptr, *sort_hdr = nullptr, *sort_state = nullptr;
    size_t box_n = 0, kframe_n = 0, cnt_n = 0, tcnt_n = 0, toff_n = 0, bctl_n = 0;
    size_t keys_a_n = 0, keys_b_n = 0, vals_a_n = 0, vals_b_n = 0, sort_hdr_n = 0, sort_state_n = 0;
  } color;
  // frame sequences (cp_batch_track, track_kernels.cuh): the slot state is double-buffered (the call writes the other
  // buffer and the host swaps only when the call succeeds); scratch is grown on demand
  struct TrackBufs {
    TrackCone* st[2] = {nullptr, nullptr};
    size_t st_n[2] = {0, 0};
    int cur = 0;
    std::vector<u32> st_off, st_prev;  // layout of st[cur]: slot s = [st_off[s], st_off[s+1]); st_prev[s]: seen a frame
    std::vector<u32> par, coff;        // per-call parameter block (one upload), cloud offsets read back
    u32 *par_d = nullptr, *kframe = nullptr, *bits = nullptr, *rank = nullptr, *cnt = nullptr, *coff_d = nullptr;
    float2* ext = nullptr;
    uint8_t *info = nullptr, *fcol = nullptr, *ans = nullptr;
    TrackCone* out = nullptr;
    ClusterRec* rec = nullptr;  // cp_debug_track inputs
    u32 *rec_off = nullptr, *flags = nullptr;
    uint8_t* colors = nullptr;
    size_t par_n = 0, kframe_n = 0, bits_n = 0, rank_n = 0, cnt_n = 0, coff_n = 0, ext_n = 0, info_n = 0, fcol_n = 0,
           ans_n = 0, out_n = 0, rec_n = 0, rec_off_n = 0, flags_n = 0, colors_n = 0;
  } track;
  bool tracked = false;  // the current run's frames have advanced the slot state
  int32_t color_cloud = CP_COLOR_CLOUD_STAGED;  // cp_set_color_cloud: what colour crops are cut from
  const uint8_t* in_ptr = nullptr;  // current batch input (d_in or caller memory)
  Layout layout{};
  // what the run (or ground call) in flight reads: the staged input, or under the plane model the plane ground node's
  // messages in d_out32 (the colour paths always read the staged input)
  const uint8_t* run_in = nullptr;
  Layout run_layout{};
  // plane ground model (cp_set_ground_plane, plane_kernels.cuh)
  bool plane_on = false;
  cp_plane_params plane{};
  double plane_cos = 0.0;
  bool plane_run = false;    // the last run was the plane chain
  bool plane_valid = false;  // the last run or ground call used the plane model: the plane buffers describe it
  u32 plane_frames = 0, plane_h = 0;
  PlaneBufs pb{};
  HostGeom hg;
  u32 *d_frame_n = nullptr, *d_frame_tile0 = nullptr, *d_tile_frame = nullptr;
  u64* d_frame_off = nullptr;
  u32 *d_low_key = nullptr, *d_bbox = nullptr, *d_c_off = nullptr, *d_gcount = nullptr, *d_v_off = nullptr;
  u32 *d_ncomp_f = nullptr, *d_kcount_f = nullptr, *d_k_off = nullptr;
  VoxelFrame* d_vf = nullptr;
  float4* d_pts = nullptr;
  u32 *d_src = nullptr, *d_frame = nullptr;
  u64 *d_keys_a = nullptr, *d_keys_b = nullptr, *d_okeys_a = nullptr, *d_okeys_b = nullptr;
  u32 *d_vals_a = nullptr, *d_vals_b = nullptr, *d_ovals_a = nullptr, *d_ovals_b = nullptr;
  u32 *d_sort_hdr = nullptr, *d_sort_state = nullptr;   // radix_sort.cuh: tickets + digit totals, look-back words
  u32 *d_vstart = nullptr, *d_cstart = nullptr, *d_comp_start = nullptr;
  float4* d_vox = nullptr;
  u32 *d_vox_frame = nullptr, *d_parent = nullptr, *d_label = nullptr;
  u64* d_hkeys = nullptr;
  u32* d_hvals = nullptr;
  ClusterRec* d_clusters = nullptr;
  u32 *d_mask = nullptr, *d_tile_count = nullptr, *d_tile_excl = nullptr;
  float* d_thr_f = nullptr;    // [F][32] ground thresholds per sector, slot 31 = their minimum
  u32* d_rowmax = nullptr;     // highest z (ordered key) of every 32-point row, written by pass 1
  bool rowmax_valid = false;   // pass 1 of the current run filled d_rowmax
  bool use_rowskip = true;     // CONESGPU_ROWSKIP=0 disables the skip (A/B measurements)
  bool use_single = true;      // CONESGPU_SINGLE=0: a single frame takes the multi-launch path (A/B, tests)
  bool self_published = false; // the last run stored its results into the pinned mirrors itself (single_frame.cuh)
  bool graph_self_published = false;
  // survivor / voxel counts of the last synchronised run: the general back half sizes its grids for about twice
  // these instead of the handle's capacity (every kernel is a grid-stride loop over device-resident bounds, so
  // any grid is correct; a grid sized for millions of slots costs microseconds per launch in empty CTAs)
  u64 hint_c = 0, hint_v = 0;
  cp_ground_params rp_ground{};   // ground parameters of the last run (valid when rp_has_ground)
  bool rp_has_ground = false;
  bool tail_priority = false;  // CONESGPU_PRIO=1: greatest-priority stream, pass 1 demoted
  int prio_low = 0;
  int k1_ctas_per_sm = 0;  // CONESGPU_K1_CTAS: separate grid cap for pass 1 (0 = stream_ctas_per_sm)
  int frame_ctas_per_sm = 0;  // CONESGPU_FRAME_CTAS: grid cap of the per-frame kernel (0 = what fits)
  // one CTA per tile in the sort passes and the tile scan (kernels that end a tile with a decoupled look-back on
  // the spot): a persistent CTA cannot publish its next tile's counts before its current look-back has resolved.
  // Measured equal to persistent grids (DESIGN.md §4.3); mask_compact and the segment heads defer their look-back
  // instead and are always persistent.  CONESGPU_TILE_CTAS=0 restores the persistent grids.
  bool tile_ctas = true;
  u32 run_sgrid = 0;  // grid of the streaming kernels of the current run
  int stream_ctas_per_sm = 8;  // grid cap of the streaming kernels (CONESGPU_STREAM_CTAS: leave room for a second handle)
  u64 *d_desc_a = nullptr, *d_desc_b = nullptr, *d_desc_c = nullptr, *d_desc_d = nullptr;
  u32 *d_tap_keys = nullptr, *d_tap_order = nullptr;
  i32* d_tap_labels = nullptr;
  // pinned host mirrors
  uint8_t* h_stage[2] = {nullptr, nullptr};
  bool stage_streaming = true;  // non-temporal stores into the pinned staging buffer (CONESGPU_STAGE_NT=0: memcpy)
  int stage_threads = 1;  // threads (caller included) that copy a pageable cloud into the pinned staging buffer
  std::unique_ptr<CopyPool> copy_pool;
  Ctl* h_ctl = nullptr;
  u32* h_frame_u32 = nullptr;  // scratch for per-frame readback
  std::vector<void*> dev_allocs, pin_allocs;
};

namespace {

#define CK(call)                                                                              \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess) {                                                                  \
      char buf_[512];                                                                         \
      snprintf(buf_, sizeof(buf_), "%s:%d %s -> %s", __FILE__, __LINE__, #call,               \
               cudaGetErrorString(e_));                                                       \
      h->err = buf_;                                                                          \
      return CP_E_CUDA;                                                                       \
    }                                                                                         \
  } while (0)

template <typename T>
cp_status dalloc(cp_handle* h, T** p, size_t count) {
  void* q = nullptr;
  if (count == 0) count = 1;
  cudaError_t e = cudaMalloc(&q, count * sizeof(T));
  if (e != cudaSuccess) {
    h->err = std::string("cudaMalloc failed: ") + cudaGetErrorString(e);
    return e == cudaErrorMemoryAllocation ? CP_E_NOMEM : CP_E_CUDA;
  }
  h->dev_allocs.push_back(q);
  *p = static_cast<T*>(q);
  return CP_OK;
}
template <typename T>
cp_status palloc(cp_handle* h, T** p, size_t count) {
  void* q = nullptr;
  if (count == 0) count = 1;
  cudaError_t e = cudaMallocHost(&q, count * sizeof(T));
  if (e != cudaSuccess) {
    h->err = std::string("cudaMallocHost failed: ") + cudaGetErrorString(e);
    return CP_E_NOMEM;
  }
  h->pin_allocs.push_back(q);
  *p = static_cast<T*>(q);
  return CP_OK;
}

u32 ceil_log2_host(u64 v) {
  u32 b = 0;
  while ((1ull << b) < v && b < 63) ++b;
  return b;
}

// ---- exact threshold solving (SURVEY A.3): the reference compares (double)(float)sqrt(s)
// against double parameters; since that is monotone in s, find the switching point once.
double bits_to_double(u64 b) {
  double d;
  memcpy(&d, &b, 8);
  return d;
}
// smallest non-negative double s (by bit pattern, up to +inf) with pred(s) true; pred monotone
template <typename F>
double first_true(F pred) {
  const u64 inf_bits = 0x7FF0000000000000ull;
  if (pred(0.0)) return 0.0;
  if (!pred(bits_to_double(inf_bits))) return bits_to_double(0x7FF8000000000000ull);  // NaN: never
  u64 lo = 0, hi = inf_bits;  // pred(lo) false, pred(hi) true
  while (hi - lo > 1) {
    const u64 mid = lo + (hi - lo) / 2;
    if (pred(bits_to_double(mid))) hi = mid; else lo = mid;
  }
  return bits_to_double(hi);
}
float round_up_to_float(double t) {  // smallest float >= t
  if (t != t) return -INFINITY;      // NaN threshold: the reference's compare is always false
  float f = (float)t;
  if ((double)f < t) f = nextafterf(f, INFINITY);
  return f;
}

cp_status make_crop(cp_handle* h, const cp_detect_params* d, CropK* c) {
  memset(c, 0, sizeof(*c));
  c->do_crop = 1;
  const double dmax = d->distance_treshold_max, dmin = d->distance_treshold_min;
  // src/cone_detection.cpp:195  p.z < level_threshold  (float promoted to double)
  c->zthr = round_up_to_float(d->level_threshold);
  // :196-197 via utils.cpp:32-34:  d = (float)sqrt(s);  drop iff d > dmax or d < dmin
  auto dist = [](double s) { return (double)(float)sqrt(s); };
  c->smax = first_true([&](double s) { return dist(s) > dmax; });          // drop iff s >= smax
  c->smin = first_true([&](double s) { return !(dist(s) < dmin); });       // drop iff s <  smin
  if (c->smax != c->smax) c->smax = INFINITY;  // never dropped by dmax (inf >= inf only for s = inf,
                                               // where (float)sqrt(inf)=inf > dmax is false iff dmax=inf)
  if (c->smin != c->smin) c->smin = INFINITY;  // always dropped by dmin
  const double g = 2e-6;
  c->smax_lo = (float)(c->smax * (1.0 - g));
  c->smax_hi = (float)(c->smax * (1.0 + g));
  c->smin_lo = (float)(c->smin * (1.0 - g));
  c->smin_hi = (float)(c->smin * (1.0 + g));
  if (c->smax == 0.0) c->smax_lo = -1.0f, c->smax_hi = 0.0f;  // everything dropped: sf >= 0 >= smax_hi
  if (c->smin == 0.0) c->smin_lo = -1.0f, c->smin_hi = -1.0f; // nothing dropped by dmin
  // :200-201  -theta >= a  or  a >= theta  <=>  !(|a| < F), F = smallest float >= theta
  const double theta = d->angle_threshold * M_PI / 180;
  c->f_hi = (theta != theta) ? INFINITY : round_up_to_float(theta);
  c->f_lo_guard = c->f_hi - 4e-6f;
  c->f_hi_guard = c->f_hi + 4e-6f;
  (void)h;
  return CP_OK;
}

// does the ground node's zero filler point (0,0,0) survive the crop?  (host restatement of
// the predicate for this single constant point; needed to honour src/ground_removal.cpp:79)
bool zero_point_survives(const cp_detect_params* d) {
  if (0.0 < d->level_threshold) return false;
  const double dist = 0.0;
  if (dist > d->distance_treshold_max) return false;
  if (dist < d->distance_treshold_min) return false;
  const double a = 0.0, theta = d->angle_threshold * M_PI / 180;
  if (-theta >= a) return false;
  if (a >= theta) return false;
  return true;
}

// host upper bound on the voxel key width, from the crop's extents (only used to decide
// how many sort passes to enqueue; the live width is computed on the device)
u32 voxel_bits_bound(const cp_detect_params* d, const VoxelK& vk, u64 cap_c) {
  const double dmax = fabs(d->distance_treshold_max);
  const double zlo = std::max(-dmax, d->level_threshold);
  const double ex = 2.0 * dmax * vk.inv[0] + 3.0, ey = 2.0 * dmax * vk.inv[1] + 3.0;
  const double ez = std::max(0.0, dmax - zlo) * vk.inv[2] + 3.0;
  const double cells = ex * ey * ez;
  u32 b = 32;
  if (cells == cells && cells < 2147483648.0) b = ceil_log2_host((u64)cells + 1);
  // passthrough frames key by position: up to ceil(log2(cap_c)) bits
  return std::max(b, std::min<u32>(32u, ceil_log2_host(cap_c)));
}

cp_status make_cluster(cp_handle* h, const cp_detect_params* d, u32 n_frames, ClusterK* k, u32* csort_bits,
                       u32* osort_bits) {
  // src/cone_detection.cpp:212  sqrt(pow(CONE_HEIGHT,2)+pow(CONE_WIDTH,2)) in double;
  // PCL extract(): static_cast<float>(tolerance); KdTreeFLANN::radiusSearch: (float)(r*r) in double
  const double tol = sqrt((double)d->cone_height * (double)d->cone_height +
                          (double)d->cone_width * (double)d->cone_width);
  const float tol_f = (float)tol;
  k->r2 = (float)((double)tol_f * (double)tol_f);
  if (!(tol_f > 0.0f) || !isfinite(tol_f)) {
    h->err = "cone_width/cone_height give a non-positive or non-finite cluster tolerance";
    return CP_E_PARAM;
  }
  const double edge = (double)tol_f * 0.505;   // general path's grid: cell diagonal < tolerance (cell_union_kernel)
  double reach = fabs(d->distance_treshold_max);
  if (!(reach < 1e6)) {
    h->err = "distance_treshold_max must be finite and below 1e6 m";
    return CP_E_PARAM;
  }
  reach += 4 * edge;
  const u64 nx = (u64)ceil(2.0 * reach / edge) + 2;
  k->inv_h = (float)(1.0 / ((double)tol_f * 1.01));   // sweep cells of the per-frame kernel
  k->inv_g = (float)(1.0 / edge);
  k->origin = (float)reach;
  k->nx = (u32)nx;
  const u64 cells = (u64)n_frames * nx * nx * nx;
  if (nx > (1u << 20) || ceil_log2_host(cells) > 60) {
    h->err = "neighbour grid too large for 64-bit cell keys";
    return CP_E_PARAM;
  }
  *csort_bits = ceil_log2_host(cells);
  if (*csort_bits == 0) *csort_bits = 1;
  k->min_size = d->min_cluster_size < 0 ? 0u : (u32)d->min_cluster_size;
  k->max_size = d->max_cluster_size < 0 ? 0u : (u32)d->max_cluster_size;
  k->frame_bits = ceil_log2_host(n_frames);
  k->size_bits = ceil_log2_host((u64)k->max_size + 1);
  *osort_bits = k->frame_bits + k->size_bits + 1;
  return CP_OK;
}

__global__ void init_kernel(Ctl* ctl, u32 n_frames, float default_low, u32* low_key, u32* bbox, u32* c_off,
                            u32* gcount, u32* ncomp_f, u32* kcount_f, u64* desc_a, u32 na, u64* desc_b,
                            u64* desc_c, u64* desc_d, u32 nb) {
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x, stride = gridDim.x * blockDim.x;
  if (t == 0) {
    Ctl z;
    memset(&z, 0, sizeof(z));
    *ctl = z;
    c_off[0] = 0;
  }
  const u32 lk = f2ord(default_low);
  for (u32 i = t; i < n_frames * kSectStride; i += stride) low_key[i] = lk;
  for (u32 i = t; i < n_frames * 8; i += stride) bbox[i] = ((i & 7u) < 4u) ? 0xFFFFFFFFu : 0u;
  for (u32 i = t; i < n_frames; i += stride) {
    gcount[i] = 0;
    ncomp_f[i] = 0;
    kcount_f[i] = 0;
    c_off[i + 1] = 0;
  }
  for (u32 i = t; i < na; i += stride) desc_a[i] = 0;
  for (u32 i = t; i < nb; i += stride) {
    desc_b[i] = 0;
    desc_c[i] = 0;
    desc_d[i] = 0;
  }
}

__global__ void tap_voxel_kernel(const Ctl* ctl, const u64* keys_a, const u64* keys_b, const u32* vals_a,
                                 const u32* vals_b, u32* tap_keys, u32* tap_order) {
  const u32 n = ctl->n_surv;
  const bool inb = sorted_in_b(ctl->vsort_bits);
  const u64* keys = inb ? keys_b : keys_a;
  const u32* vals = inb ? vals_b : vals_a;
  const u64 mask = (ctl->voxel_key_bits >= 64) ? ~0ull : ((1ull << ctl->voxel_key_bits) - 1ull);
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    tap_keys[i] = (u32)(keys[i] & mask);
    tap_order[i] = vals[i];
  }
}

cp_status check_view(cp_handle* h, const cp_cloud_view* v) {
  if (!v) {
    h->err = "NULL cloud view";
    return CP_E_PARAM;
  }
  const u64 n = (u64)v->width * v->height;
  if (n && !v->data) {
    h->err = "cloud view has points but a NULL data pointer";
    return CP_E_PARAM;
  }
  if (v->is_bigendian) {
    h->err = "big-endian PointCloud2 data is not supported (pcl::fromROSMsg does not swap either)";
    return CP_E_BADFIELD;
  }
  if (v->off_x < 0 || v->off_y < 0 || v->off_z < 0) {
    h->err = "x/y/z FLOAT32 fields are required";
    return CP_E_BADFIELD;
  }
  const i32 mx = std::max(std::max(v->off_x, v->off_y), std::max(v->off_z, v->off_intensity));
  if ((u32)mx + 4 > v->point_step) {
    h->err = "field offset + 4 exceeds point_step";
    return CP_E_BADFIELD;
  }
  if (v->height > 1 && v->row_step < v->width * v->point_step) {
    h->err = "row_step smaller than width * point_step";
    return CP_E_BADFIELD;
  }
  return CP_OK;
}

Layout make_layout(u32 step, i32 ox, i32 oy, i32 oz, i32 oi) {
  Layout L;
  L.step = step;
  L.ox = ox;
  L.oy = oy;
  L.oz = oz;
  L.oi = oi;
  if (step == 16 && ox == 0 && oy == 4 && oz == 8 && oi == 12)
    L.mode = 0;
  else if (step % 4 == 0 && ox % 4 == 0 && oy % 4 == 0 && oz % 4 == 0 && (oi < 0 || oi % 4 == 0))
    L.mode = 1;
  else
    L.mode = 2;
  return L;
}

cp_status set_geometry(cp_handle* h, const u32* frame_points, u32 n_frames) {
  HostGeom& g = h->hg;
  if (n_frames == 0 || n_frames > h->cfg.max_frames) {
    h->err = "n_frames is 0 or exceeds cp_config.max_frames";
    return n_frames ? CP_E_CAPACITY : CP_E_PARAM;
  }
  // unchanged batch shape (the usual case for a node or a replay loop): nothing to rebuild or upload
  if (g.n_frames == n_frames && g.frame_n.size() == n_frames &&
      memcmp(g.frame_n.data(), frame_points, sizeof(u32) * n_frames) == 0)
    return CP_OK;
  g.n_frames = 0;  // invalid until the new geometry is fully set
  g.frame_n.assign(frame_points, frame_points + n_frames);
  g.frame_off.resize(n_frames);
  g.frame_tile0.resize(n_frames);
  u64 off = 0;
  u64 tiles = 0;
  bool uniform = true;
  for (u32 f = 0; f < n_frames; ++f) {
    g.frame_off[f] = off;
    g.frame_tile0[f] = (u32)tiles;
    off += frame_points[f];
    u64 t = ((u64)frame_points[f] + kStreamTile - 1) / kStreamTile;
    if (t == 0) t = 1;  // empty frames still own one (empty) tile so their offsets get written
    tiles += t;
    if (frame_points[f] != frame_points[0]) uniform = false;
  }
  if (off > h->cfg.max_points || off >= (1ull << 31)) {
    h->err = "batch holds more points than cp_config.max_points (or >= 2^31)";
    return CP_E_CAPACITY;
  }
  if (tiles > h->tiles_cap) {
    h->err = "batch needs more stream tiles than the handle was sized for";
    return CP_E_CAPACITY;
  }
  g.n_points = off;
  g.n_tiles = (u32)tiles;
  g.uniform_n = (uniform && frame_points[0] > 0) ? frame_points[0] : 0;
  g.tpf = g.uniform_n ? (g.uniform_n + kStreamTile - 1) / kStreamTile : 0;
  CK(cudaMemcpyAsync(h->d_frame_n, g.frame_n.data(), sizeof(u32) * n_frames, cudaMemcpyHostToDevice, h->stream));
  if (!g.uniform_n) {
    g.tile_frame.resize(g.n_tiles);
    for (u32 f = 0; f < n_frames; ++f) {
      const u32 t1 = (f + 1 < n_frames) ? g.frame_tile0[f + 1] : g.n_tiles;
      for (u32 t = g.frame_tile0[f]; t < t1; ++t) g.tile_frame[t] = f;
    }
    // pageable sources: the copies below are staged by the runtime before returning
    CK(cudaMemcpyAsync(h->d_frame_off, g.frame_off.data(), sizeof(u64) * n_frames, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_frame_tile0, g.frame_tile0.data(), sizeof(u32) * n_frames, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_tile_frame, g.tile_frame.data(), sizeof(u32) * g.n_tiles, cudaMemcpyHostToDevice, h->stream));
  }
  g.n_frames = n_frames;
  return CP_OK;
}

Geom device_geom(const cp_handle* h) {
  Geom g;
  g.n_frames = h->hg.n_frames;
  g.uniform_n = h->hg.uniform_n;
  g.tpf = h->hg.tpf;
  g.n_tiles = h->hg.n_tiles;
  g.frame_n = h->d_frame_n;
  g.frame_off = h->d_frame_off;
  g.tile_frame = h->d_tile_frame;
  g.frame_tile0 = h->d_frame_tile0;
  return g;
}

u64 hinted(u64 cap, u64 hint) { return hint ? std::min<u64>(cap, 2 * hint + 8192) : cap; }

u32 grid_for(u64 work, u32 block, int sms, int per_sm) {
  u64 b = (work + block - 1) / block;
  if (b == 0) b = 1;
  const u64 cap = (u64)sms * per_sm;
  return (u32)(b < cap ? b : cap);
}

// pass 2 of the front end, part 1: keep mask + survivors per tile
void launch_keep_mask(cp_handle* h, const Geom& g, const CropK& c, const GroundK& gk, u32 grid) {
  MaskOut mo;
  mo.mask = h->d_mask;
  mo.tile_count = h->d_tile_count;
  mo.gcount = h->d_gcount;
  mo.rows_loaded = &h->d_ctl->rows_loaded;
  if (gk.do_ground) {
    ground_thresholds_kernel<<<(g.n_frames + 127) / 128, 128, 0, h->stream>>>(g.n_frames, h->d_low_key, h->d_thr_f);
    h->launches++;
  }
  // skipped units write nothing: the keep mask and the tile counts start from zero
  cudaMemsetAsync(h->d_mask, 0, sizeof(u32) * (size_t)g.n_tiles * kTileWords, h->stream);
  cudaMemsetAsync(h->d_tile_count, 0, sizeof(u32) * g.n_tiles, h->stream);
  if (h->stage_timing) cudaEventRecord(h->ev_k[2], h->stream);
  // few frames: share each 32-row group between up to 8 warps so the whole GPU works on the batch
  const u32 total_warps = (u32)h->sms * 4u * kStreamWarps;
  u32 split_log2 = 0;
  while (split_log2 < 3 && (((u64)g.n_tiles * 2u) << (split_log2 + 1)) <= total_warps) ++split_log2;
  if (split_log2) grid = grid_for((((u64)g.n_tiles * 2u) << split_log2) * 32u, kStreamThreads, h->sms, h->stream_ctas_per_sm);
  const u32* rm = h->rowmax_valid ? h->d_rowmax : nullptr;
  switch (h->run_layout.mode) {
    case 0: keep_mask_kernel<0><<<grid, kStreamThreads, 0, h->stream>>>(h->run_in, h->run_layout, g, c, gk, h->d_thr_f, rm, mo, split_log2); break;
    case 1: keep_mask_kernel<1><<<grid, kStreamThreads, 0, h->stream>>>(h->run_in, h->run_layout, g, c, gk, h->d_thr_f, rm, mo, split_log2); break;
    default: keep_mask_kernel<2><<<grid, kStreamThreads, 0, h->stream>>>(h->run_in, h->run_layout, g, c, gk, h->d_thr_f, rm, mo, split_log2); break;
  }
  if (h->stage_timing) cudaEventRecord(h->ev_k[3], h->stream);
  h->launches++;
  h->masked = true;
}

// part 2: tile scan -> ordered gather (+bbox) into the global survivor arrays
// (general back half, parity taps)
void launch_scan_gather(cp_handle* h, const Geom& g, const GroundK& gk, u32 cap) {
  GatherOut go;
  go.pts = h->d_pts;
  go.src = h->d_src;
  go.frame = h->d_frame;
  go.cap = cap;
  go.bbox_key = h->d_bbox;
  go.out32 = nullptr;
  const u32 stiles = (g.n_tiles + kScanTile - 1) / kScanTile;
  tile_scan_kernel<<<(h->tile_ctas || stiles < (u32)h->sms * 4) ? stiles : (u32)h->sms * 4, kScanThreads, 0, h->stream>>>(
      g, h->d_tile_count, h->d_tile_excl, h->d_c_off, h->d_desc_a, h->d_ctl, cap);
  const u32 ggrid = grid_for((u64)g.n_tiles * 32, 256, h->sms, 8);
  switch (h->run_layout.mode) {
    case 0: gather_survivors_kernel<0><<<ggrid, 256, 0, h->stream>>>(h->run_in, h->run_layout, g, gk, h->d_mask, h->d_tile_count, h->d_tile_excl, go); break;
    case 1: gather_survivors_kernel<1><<<ggrid, 256, 0, h->stream>>>(h->run_in, h->run_layout, g, gk, h->d_mask, h->d_tile_count, h->d_tile_excl, go); break;
    default: gather_survivors_kernel<2><<<ggrid, 256, 0, h->stream>>>(h->run_in, h->run_layout, g, gk, h->d_mask, h->d_tile_count, h->d_tile_excl, go); break;
  }
  h->launches += 2;
  h->gathered = true;
}
// pass 2 + ordered compaction in one pass over the scan (mask_compact_kernel): the general back half's and the
// ground node's front end when no keep mask exists yet
template <bool OUT32>
void launch_mask_compact(cp_handle* h, const Geom& g, const CropK& c, const GroundK& gk, u32 cap, uint8_t* out32) {
  GatherOut go;
  go.pts = h->d_pts;
  go.src = h->d_src;
  go.frame = h->d_frame;
  go.cap = cap;
  go.bbox_key = h->d_bbox;
  go.out32 = out32;
  if (gk.do_ground) {
    ground_thresholds_kernel<<<(g.n_frames + 127) / 128, 128, 0, h->stream>>>(g.n_frames, h->d_low_key, h->d_thr_f);
    h->launches++;
  }
  const u32* rm = h->rowmax_valid ? h->d_rowmax : nullptr;
  // persistent CTAs: a tile's look-back is resolved while the CTA's next tile is already judged
  const u32 grid = std::min<u32>(g.n_tiles ? g.n_tiles : 1u, (u32)h->sms * 4u);
  u32* ticket = &h->d_ctl->ticket[0];
#define CP_MC(M) mask_compact_kernel<M, OUT32><<<grid, kStreamThreads, 0, h->stream>>>(                         \
      h->run_in, h->run_layout, g, c, gk, h->d_thr_f, rm, h->d_desc_a, ticket, go, h->d_c_off, h->d_gcount, h->d_ctl)
  switch (h->run_layout.mode) {
    case 0: CP_MC(0); break;
    case 1: CP_MC(1); break;
    default: CP_MC(2); break;
  }
#undef CP_MC
  h->launches++;
  h->gathered = true;
}
// single HBM pass: one 16-CTA cluster per frame, points stashed in shared memory (cluster_front.cuh)
bool cluster_front_eligible(const cp_handle* h, const Geom& g, bool ground) {
  return h->use_cluster && ground && g.uniform_n && h->run_layout.mode == 0 &&
         g.uniform_n <= (u32)kClusterSize * kClMaxPtsPerCta;
}

bool launch_front_cluster(cp_handle* h, const Geom& g, const CropK& c, const GroundK& gk, float default_low) {
  ClusterArgs a;
  a.in = reinterpret_cast<const float4*>(h->run_in);
  a.n_frames = g.n_frames;
  a.n = g.uniform_n;
  const u32 per = (g.uniform_n + kClusterSize - 1) / kClusterSize;
  a.pts_per_cta = (per + kStreamTile - 1) / kStreamTile * kStreamTile;
  a.tpf = g.tpf;
  a.default_low = default_low;
  a.c = c;
  a.gk = gk;
  a.low_key = h->d_low_key;
  a.o.mask = h->d_mask;
  a.o.tile_count = h->d_tile_count;
  a.o.gcount = h->d_gcount;
  a.o.rows_loaded = &h->d_ctl->rows_loaded;
  const size_t smem = (size_t)a.pts_per_cta * 3 * sizeof(float);  // x, y, z stash
  if (h->cluster_smem != smem) {
    if (cudaFuncSetAttribute(front_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess ||
        cudaFuncSetAttribute(front_cluster_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess) {
      cudaGetLastError();
      return false;
    }
    h->cluster_smem = smem;
    h->cluster_max = 0;
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = kClusterSize;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.blockDim = dim3(kClThreads, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = h->stream;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (h->cluster_max == 0) {
    cfg.gridDim = dim3(kClusterSize, 1, 1);
    int nmax = 0;
    if (cudaOccupancyMaxActiveClusters(&nmax, front_cluster_kernel, &cfg) != cudaSuccess || nmax < 1) {
      cudaGetLastError();
      return false;
    }
    h->cluster_max = (u32)nmax;
  }
  const u32 ncl = std::min<u32>(h->cluster_max, g.n_frames);
  cfg.gridDim = dim3(ncl * kClusterSize, 1, 1);
  if (h->stage_timing && !h->capturing) cudaEventRecord(h->ev_k[0], h->stream);
  if (cudaLaunchKernelEx(&cfg, front_cluster_kernel, a) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  if (h->stage_timing && !h->capturing) cudaEventRecord(h->ev_k[1], h->stream);
  h->launches++;
  return true;
}

// both streaming passes in one persistent kernel (uniform batches with ground removal)
void launch_front_fused(cp_handle* h, const Geom& g, const CropK& c, const GroundK& gk) {
  MaskOut mo;
  mo.mask = h->d_mask;
  mo.tile_count = h->d_tile_count;
  mo.gcount = h->d_gcount;
  mo.rows_loaded = &h->d_ctl->rows_loaded;
  if (h->fused_grid == 0) {
    int occ = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, front_fused_kernel<0>, kStreamThreads, 0);
    if (occ < 1) occ = 1;
    h->fused_grid = (u32)(h->sms * occ);
  }
  FusedArgs fa;
  const u32 gf = (h->fused_grid + g.tpf - 1) / g.tpf;  // frames per group: one resident wave of tiles
  fa.group_tiles = gf * g.tpf;
  fa.n_groups = (g.n_frames + gf - 1) / gf;
  fa.done = h->d_done;
  fa.ticket = h->d_frame_ticket + 1;
  cudaMemsetAsync(h->d_done, 0, sizeof(u32) * g.n_frames, h->stream);
  cudaMemsetAsync(h->d_frame_ticket + 1, 0, sizeof(u32), h->stream);
  const u32 items = fa.n_groups * fa.group_tiles * 2u;
  const u32 grid = items < h->fused_grid ? items : h->fused_grid;
  if (h->stage_timing) cudaEventRecord(h->ev_k[0], h->stream);
  switch (h->run_layout.mode) {
    case 0: front_fused_kernel<0><<<grid, kStreamThreads, 0, h->stream>>>(h->run_in, h->run_layout, g, c, gk, h->d_low_key, mo, fa); break;
    case 1: front_fused_kernel<1><<<grid, kStreamThreads, 0, h->stream>>>(h->run_in, h->run_layout, g, c, gk, h->d_low_key, mo, fa); break;
    default: front_fused_kernel<2><<<grid, kStreamThreads, 0, h->stream>>>(h->run_in, h->run_layout, g, c, gk, h->d_low_key, mo, fa); break;
  }
  if (h->stage_timing) cudaEventRecord(h->ev_k[1], h->stream);
  h->launches++;
}

template <int MODE>
void launch_sector_min_mode(cp_handle* h, const Geom& g, u32 grid) {
  if (!h->tail_priority) {
    ground_sector_min_kernel<MODE><<<grid, kStreamThreads, 0, h->stream>>>(h->run_in, h->run_layout, g, h->d_low_key, h->d_rowmax);
    return;
  }
  // the stream runs at the greatest priority; pass 1 alone is demoted, so that the short kernels behind
  // it (another handle's pass 2 / per-frame kernel) take the SM slots pass 1 frees, not the other way round
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kStreamThreads);
  cfg.stream = h->stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributePriority;
  at[0].val.priority = h->prio_low;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, ground_sector_min_kernel<MODE>, h->run_in, h->run_layout, g, h->d_low_key, h->d_rowmax);
}
void launch_sector_min(cp_handle* h, const Geom& g, u32 grid) {
  if (h->k1_ctas_per_sm)
    grid = grid_for((u64)g.n_tiles * kStreamThreads, kStreamThreads, h->sms, h->k1_ctas_per_sm);
  switch (h->run_layout.mode) {
    case 0: launch_sector_min_mode<0>(h, g, grid); break;
    case 1: launch_sector_min_mode<1>(h, g, grid); break;
    default: launch_sector_min_mode<2>(h, g, grid); break;
  }
}

void launch_init(cp_handle* h, float default_low) {
  const u32 nb = (u32)(h->cap_c / kHeadTile + 2);
  init_kernel<<<h->sms * 2, 256, 0, h->stream>>>(h->d_ctl, h->hg.n_frames, default_low, h->d_low_key, h->d_bbox,
                                                 h->d_c_off, h->d_gcount, h->d_ncomp_f, h->d_kcount_f,
                                                 h->d_desc_a, h->hg.n_tiles, h->d_desc_b, h->d_desc_c, h->d_desc_d, nb);
  cudaMemsetAsync(h->d_desc_fv, 0, sizeof(u64) * h->hg.n_frames, h->stream);
  h->launches++;
}

SortArgs sort_args(cp_handle* h, bool order_sort, const u32* d_n, const u32* d_bits) {
  SortArgs a;
  a.keys_a = order_sort ? h->d_okeys_a : h->d_keys_a;
  a.keys_b = order_sort ? h->d_okeys_b : h->d_keys_b;
  a.vals_a = order_sort ? h->d_ovals_a : h->d_vals_a;
  a.vals_b = order_sort ? h->d_ovals_b : h->d_vals_b;
  a.d_n = d_n;
  a.d_bits = d_bits;
  a.hdr = h->d_sort_hdr;
  a.state = h->d_sort_state;
  a.tiles_cap = h->sort_tiles_cap;
  return a;
}

__global__ void back_reset_kernel(Ctl* ctl, u32 n_frames, u32* ncomp_f, u32* kcount_f) {
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t == 0) {
    ctl->n_vox = ctl->n_cells = ctl->n_comp = ctl->n_clusters = 0;
    ctl->voxel_key_bits = 0;
    ctl->fast_overflow = 0;
    ctl->pairs_visited = ctl->pairs_tested = 0;   // a retried back half counts its own pairs only
    ctl->error &= kErrSurvivors;
  }
  for (u32 i = t; i < n_frames; i += gridDim.x * blockDim.x) {
    ncomp_f[i] = 0;
    kcount_f[i] = 0;
  }
}

// general back half: global-memory kernels, any frame size.  Every sort's keys are produced by a kernel of this
// sequence, which also counts their digits (sort_feed_*), so a sort is its passes and nothing else; the one-thread
// bookkeeping steps live inside their neighbours.
void enqueue_back_general(cp_handle* h, const RunParams& rp) {
  const cp_detect_params* d = &rp.d;
  const VoxelK& vk = rp.vk;
  const ClusterK& ck = rp.ck;
  const u32 csort_bits = rp.csort_bits, osort_bits = rp.osort_bits;
  const u32 F = h->hg.n_frames;
  const bool persistent = !h->tile_ctas;
  // the four sorts (voxel, cell, label, order) have a header each: one memset in front of all of them
  cudaMemsetAsync(h->d_sort_hdr, 0, sizeof(u32) * kSortHdrWords * 4, h->stream);
  auto sort_of = [&](int which, bool order_sort, const u32* d_n, const u32* d_bits) {
    SortArgs a = sort_args(h, order_sort, d_n, d_bits);
    a.hdr = h->d_sort_hdr + (size_t)which * kSortHdrWords;
    return a;
  };
  // ---- VoxelGrid
  const u32 fgrid = (F + 255) / 256;
  voxel_setup_kernel<<<fgrid, 256, 0, h->stream>>>(F, vk, h->d_bbox, h->d_c_off, h->d_vf, h->d_ctl);
  const u64 work_c = hinted(h->cap_c, h->hint_c), work_v = hinted(h->cap_v, h->hint_v);
  const u32 cgrid = grid_for(work_c, 256, h->sms, 8);
  {
    SortArgs sa = sort_of(0, false, &h->d_ctl->n_surv, &h->d_ctl->vsort_bits);
    voxel_key_kernel<<<cgrid, 256, 0, h->stream>>>(h->d_ctl, vk, h->d_pts, h->d_frame, h->d_c_off, h->d_vf,
                                                   h->d_keys_a, h->d_vals_a, sa.hdr, sa.state);
    h->launches += 2;
    h->launches += radix_sort_passes(h->stream, sa, voxel_bits_bound(d, vk, h->cap_c) + vk.frame_bits, (u32)work_c,
                                     h->sms, persistent);
  }
  if (h->taps) {
    tap_voxel_kernel<<<cgrid, 256, 0, h->stream>>>(h->d_ctl, h->d_keys_a, h->d_keys_b, h->d_vals_a, h->d_vals_b,
                                                   h->d_tap_keys, h->d_tap_order);
    h->launches++;
  }
  const u32 hgrid = grid_for(work_c, kHeadTile, h->sms, 4);   // persistent: look-backs are resolved one tile later
  {
    HeadArgs ha = {};
    ha.keys_a = h->d_keys_a;
    ha.keys_b = h->d_keys_b;
    ha.d_bits = &h->d_ctl->vsort_bits;
    ha.d_n = &h->d_ctl->n_surv;
    ha.starts = h->d_vstart;
    ha.starts_cap = (u32)h->cap_v;
    ha.d_total = &h->d_ctl->n_vox;
    ha.desc = h->d_desc_b;
    ha.ticket = &h->d_ctl->ticket[1];
    ha.error = &h->d_ctl->error;
    ha.err_bit = kErrVoxels;
    segment_heads_kernel<<<hgrid, kHeadThreads, 0, h->stream>>>(ha);
  }
  const u32 vgrid = grid_for(work_v, 256, h->sms, 8);
  VoxelOut vo;
  vo.vox = h->d_vox;
  vo.vox_frame = h->d_vox_frame;
  vo.v_off = h->d_v_off;
  voxel_mean_kernel<<<grid_for(work_v * 32ull, 256, h->sms, 8), 256, 0, h->stream>>>(
      h->d_ctl, h->d_keys_a, h->d_keys_b, h->d_vals_a, h->d_vals_b, h->d_vstart, h->d_pts, h->d_src, h->d_frame_n,
      h->hg.uniform_n, h->d_gcount, rp.gk.pad_survives, F, vo);
  h->launches += 2;

  // ---- Euclidean clustering
  {
    SortArgs sa = sort_of(1, false, &h->d_ctl->n_vox, &h->d_ctl->csort_bits);
    cell_key_kernel<<<vgrid, 256, 0, h->stream>>>(h->d_ctl, ck, h->d_vox, h->d_vox_frame, h->d_keys_a, h->d_vals_a,
                                                  h->d_parent, csort_bits, osort_bits, h->hash_cap, h->d_hkeys,
                                                  sa.hdr, sa.state);
    h->launches++;
    h->launches += radix_sort_passes(h->stream, sa, csort_bits, (u32)work_v, h->sms, persistent);
  }
  const u32 hvgrid = grid_for(work_v, kHeadTile, h->sms, 4);
  {
    HeadArgs ha = {};
    ha.keys_a = h->d_keys_a;
    ha.keys_b = h->d_keys_b;
    ha.d_bits = &h->d_ctl->csort_bits;
    ha.d_n = &h->d_ctl->n_vox;
    ha.starts = h->d_cstart;
    ha.starts_cap = (u32)h->cap_v;
    ha.d_total = &h->d_ctl->n_cells;
    ha.desc = h->d_desc_c;
    ha.ticket = &h->d_ctl->ticket[2];
    ha.error = &h->d_ctl->error;
    ha.err_bit = kErrInternal;
    ha.hkeys = h->d_hkeys;       // cell key -> cell id, entered as the heads are found
    ha.hvals = h->d_hvals;
    ha.d_hash_mask = &h->d_ctl->hash_mask;
    segment_heads_kernel<<<hvgrid, kHeadThreads, 0, h->stream>>>(ha);
  }
  cell_union_kernel<<<grid_for(work_v * 32ull, 256, h->sms, 8), 256, 0, h->stream>>>(
      h->d_ctl, ck, h->d_keys_a, h->d_keys_b, h->d_vals_a, h->d_vals_b, h->d_cstart, h->d_hkeys, h->d_hvals,
      h->d_vox, h->d_parent, h->d_ctl);
  h->launches += 2;
  {
    SortArgs sa = sort_of(2, false, &h->d_ctl->n_vox, &h->d_ctl->lsort_bits);
    flatten_kernel<<<vgrid, 256, 0, h->stream>>>(h->d_ctl, h->d_parent, h->d_label, h->d_keys_a, h->d_vals_a, sa.hdr,
                                                 sa.state);
    h->launches++;
    h->launches += radix_sort_passes(h->stream, sa, ceil_log2_host(h->cap_v) + 1, (u32)work_v, h->sms, persistent);
  }
  {
    HeadArgs ha = {};
    ha.keys_a = h->d_keys_a;
    ha.keys_b = h->d_keys_b;
    ha.d_bits = &h->d_ctl->lsort_bits;
    ha.d_n = &h->d_ctl->n_vox;
    ha.starts = h->d_comp_start;
    ha.starts_cap = (u32)h->cap_v;
    ha.d_total = &h->d_ctl->n_comp;
    ha.desc = h->d_desc_d;
    ha.ticket = &h->d_ctl->ticket[3];
    ha.error = &h->d_ctl->error;
    ha.err_bit = kErrInternal;
    segment_heads_kernel<<<hvgrid, kHeadThreads, 0, h->stream>>>(ha);
  }
  {
    SortArgs sa = sort_of(3, true, &h->d_ctl->n_comp, &h->d_ctl->osort_bits);
    component_kernel<<<vgrid, 256, 0, h->stream>>>(h->d_ctl, ck, h->d_keys_a, h->d_keys_b, h->d_comp_start,
                                                   h->d_vox_frame, h->d_ncomp_f, h->d_kcount_f, h->d_okeys_a,
                                                   h->d_ovals_a, h->d_ctl, sa.hdr, sa.state);
    h->launches += 2;
    h->launches += radix_sort_passes(h->stream, sa, osort_bits, (u32)work_v, h->sms, persistent);
  }
  FinishArgs fin;
  fin.n_frames = F;
  fin.frame_n = h->d_frame_n;
  fin.uniform_n = h->hg.uniform_n;
  fin.c_off = h->d_c_off;
  fin.ncomp_f = h->d_ncomp_f;
  fin.kcount_f = h->d_kcount_f;
  fin.vf = h->d_vf;
  fin.gcount = h->d_gcount;
  fin.counted_ground = h->counted_ground ? 1 : 0;
  fin.k_off = h->d_k_off;
  fin.fc = h->d_fc;
  emit_clusters_kernel<<<vgrid, 256, 0, h->stream>>>(h->d_ctl, h->d_ovals_a, h->d_ovals_b, h->d_keys_a, h->d_keys_b,
                                                     h->d_vals_a, h->d_vals_b, h->d_comp_start, h->d_vox,
                                                     h->d_vox_frame, h->d_v_off, h->d_clusters, (u32)h->cap_v,
                                                     h->d_ctl, fin);
  h->launches++;
  if (h->taps) {
    local_labels_kernel<<<vgrid, 256, 0, h->stream>>>(h->d_ctl, h->d_label, h->d_vox_frame, h->d_v_off,
                                                      h->d_tap_labels);
    h->launches++;
  }
}

// fast back half: one CTA per frame in shared memory (frame_kernels.cuh)
template <int CMAX, int VMAX, int MODE, int T>
void launch_frame_kernel(cp_handle* h, const FrameArgs& fa) {
  const size_t smem = sizeof(FrameSmem<CMAX, VMAX, T>);
  // function attributes are per device: a process may hold handles on several GPUs
  constexpr int kMaxDevices = 64;
  static int per_sm_dev[kMaxDevices] = {0};  // 0 = not set up on that device yet
  const int dev = (h->cfg.device >= 0 && h->cfg.device < kMaxDevices) ? h->cfg.device : 0;
  if (per_sm_dev[dev] == 0) {
    int per_sm = 1;
    cudaFuncSetAttribute(frame_backend_kernel<CMAX, VMAX, MODE, T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         (int)smem);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, frame_backend_kernel<CMAX, VMAX, MODE, T>, T, smem) !=
            cudaSuccess || per_sm < 1)
      per_sm = 1;
    per_sm_dev[dev] = per_sm;
  }
  const int per_sm = h->frame_ctas_per_sm ? std::min(h->frame_ctas_per_sm, per_sm_dev[dev]) : per_sm_dev[dev];
  const u32 grid = std::min<u32>(fa.n_frames, (u32)h->sms * (u32)per_sm);
  if (h->stage_timing && !h->capturing) cudaEventRecord(h->ev_k[4], h->stream);
  frame_backend_kernel<CMAX, VMAX, MODE, T><<<grid, T, smem, h->stream>>>(fa);
  if (h->stage_timing && !h->capturing) cudaEventRecord(h->ev_k[5], h->stream);
  h->ran_frame_kernel = true;
  h->launches++;
}

// arguments of the per-frame back half (frame_kernels.cuh) for the current run
FrameArgs frame_args(cp_handle* h, const RunParams& rp) {
  FrameArgs fa;
  fa.n_frames = h->hg.n_frames;
  fa.in = h->run_in;
  fa.layout = h->run_layout;
  fa.geom = device_geom(h);
  fa.mask = h->run_fused_mask ? nullptr : h->d_mask;
  fa.rowmax = h->rowmax_valid ? h->d_rowmax : nullptr;
  fa.low_key = h->d_low_key;
  fa.crop = rp.crop;
  fa.gk = rp.gk;
  fa.rows_loaded = &h->d_ctl->rows_loaded;
  fa.c_off = h->taps ? h->d_c_off : nullptr;
  fa.gcount = h->d_gcount;
  fa.pad_survives = rp.gk.pad_survives;
  fa.vk = rp.vk;
  fa.ck = rp.ck;
  fa.vf = h->d_vf;
  fa.v_off = h->d_v_off;
  fa.k_off = h->d_k_off;
  fa.ncomp_f = h->d_ncomp_f;
  fa.kcount_f = h->d_kcount_f;
  fa.ncrop_f = h->d_ncrop_f;
  fa.slots = h->d_slots;
  const bool direct = fa.n_frames == 1;  // a node's single frame: the frame kernel writes the result list itself
  fa.direct_out = direct ? reinterpret_cast<ClusterRec*>(h->d_clusters) : nullptr;
  fa.direct_cap = (u32)std::min<u64>(h->cap_v, 0xFFFFFFFFu);
  fa.fc = h->d_fc;
  fa.counted_ground = h->counted_ground ? 1 : 0;
  fa.nvox_f = h->d_nvox_f;
  fa.desc_v = h->d_desc_fv;
  fa.ctl = h->d_ctl;
  fa.ticket = h->d_frame_ticket;
  fa.tap_vox = h->taps ? h->d_vox : nullptr;
  fa.tap_vox_cap = (u32)h->cap_v;
  fa.tap_keys = h->taps ? h->d_tap_keys : nullptr;
  fa.tap_order = h->taps ? h->d_tap_order : nullptr;
  fa.tap_labels = h->taps ? h->d_tap_labels : nullptr;
  return fa;
}

// ---- a single frame in ONE launch (single_frame.cuh): 16-CTA cluster front end, back half and result publish
template <int CMAX, int VMAX, int MODE>
bool launch_single_frame_t(cp_handle* h, const SingleArgs& a, size_t smem) {
  static bool ready[64] = {};                // per device: attributes set and a cluster of 16 fits
  static bool usable[64] = {};
  const int dev = h->cfg.device & 63;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = kSfCluster;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.gridDim = dim3(kSfCluster, 1, 1);
  cfg.blockDim = dim3(kSfThreads, 1, 1);
  cfg.dynamicSmemBytes = kSfMaxPtsPerCta * 3 * sizeof(float);   // attributes are set for the largest stash
  cfg.stream = h->stream;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  auto kern = single_frame_kernel<CMAX, VMAX, MODE>;
  if (!ready[dev]) {
    ready[dev] = true;
    const size_t max_smem = std::max<size_t>(cfg.dynamicSmemBytes, sizeof(FrameSmem<CMAX, VMAX, kSfThreads>));
    int n = 0;
    cfg.dynamicSmemBytes = max_smem;
    usable[dev] = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)max_smem) == cudaSuccess &&
                  cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess &&
                  cudaOccupancyMaxActiveClusters(&n, kern, &cfg) == cudaSuccess && n >= 1;
    cudaGetLastError();
  }
  if (!usable[dev]) return false;
  cfg.dynamicSmemBytes = smem;
  if (cudaLaunchKernelEx(&cfg, kern, a) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return true;
}

bool single_frame_eligible(const cp_handle* h, const Geom& g) {
  return h->use_single && !h->plane_run && g.n_frames == 1 && g.uniform_n != 0 && h->run_layout.mode <= 1 && !h->taps && !h->stage_timing &&
         h->back_mode < 3 && !h->gather.open && g.uniform_n <= (u32)kSfCluster * kSfMaxPtsPerCta;
}

bool launch_single_frame(cp_handle* h, const RunParams& rp, float default_low) {
  SingleArgs a;
  h->run_fused_mask = false;   // the back half reads the keep mask the front end of the same kernel wrote
  h->rowmax_valid = false;
  a.fa = frame_args(h, rp);
  a.n = h->hg.uniform_n;
  const u32 per = (a.n + kSfCluster - 1) / kSfCluster;
  a.pts_per_cta = (per + kSfSub - 1) / kSfSub * kSfSub;
  a.default_low = default_low;
  a.o.mask = h->d_mask;
  a.o.tile_count = h->d_tile_count;
  a.o.gcount = h->d_gcount;
  a.o.rows_loaded = &h->d_ctl->rows_loaded;
  a.low_key = h->d_low_key;
  a.h_ctl = reinterpret_cast<u32*>(h->h_ctl);
  a.h_fc = h->h_fc;
  a.h_res = h->h_result;
  a.off_words = (u32)h->off_words;
  a.max_records = (u32)std::min<u64>(h->prefetch_cap, 0xFFFFFFFFu);
  const size_t stash = (size_t)a.pts_per_cta * 3 * sizeof(float);
  bool ok;
#define CP_SF(CM, VM)                                                                                         \
  do {                                                                                                        \
    const size_t smem = std::max(stash, sizeof(FrameSmem<CM, VM, kSfThreads>));                               \
    ok = h->run_layout.mode == 0 ? launch_single_frame_t<CM, VM, 0>(h, a, smem) : launch_single_frame_t<CM, VM, 1>(h, a, smem); \
  } while (0)
  if (h->back_mode == 0) CP_SF(1024, 512);
  else if (h->back_mode == 1) CP_SF(2048, 1024);
  else CP_SF(4096, 2048);
#undef CP_SF
  return ok;
}

// fast back half: one CTA per frame in shared memory (frame_kernels.cuh)
template <int CMAX, int VMAX, int T>
void enqueue_back_fast(cp_handle* h, const RunParams& rp) {
  FrameArgs fa = frame_args(h, rp);
  const bool direct = fa.n_frames == 1;
  cudaMemsetAsync(h->d_frame_ticket, 0, sizeof(u32), h->stream);
  fa.tap_vox = h->taps ? h->d_vox : nullptr;
  fa.tap_vox_cap = (u32)h->cap_v;
  fa.tap_keys = h->taps ? h->d_tap_keys : nullptr;
  fa.tap_order = h->taps ? h->d_tap_order : nullptr;
  fa.tap_labels = h->taps ? h->d_tap_labels : nullptr;
  // the crop taps (survivor arrays, offsets) come from the global keep mask + gather
  if (h->taps && !h->masked) launch_keep_mask(h, fa.geom, rp.crop, rp.gk, h->run_sgrid);
  if (h->taps && !h->gathered) launch_scan_gather(h, fa.geom, rp.gk, (u32)h->cap_c);
  switch (h->run_layout.mode) {
    case 0: launch_frame_kernel<CMAX, VMAX, 0, T>(h, fa); break;
    case 1: launch_frame_kernel<CMAX, VMAX, 1, T>(h, fa); break;
    default: launch_frame_kernel<CMAX, VMAX, 2, T>(h, fa); break;
  }
  if (!direct) {
    pack_clusters_kernel<<<fa.n_frames, 256, 0, h->stream>>>(fa.n_frames, VMAX, h->d_kcount_f, h->d_slots, h->d_k_off,
                                                             h->d_clusters, (u32)h->cap_v, h->d_ctl);
    h->launches++;
  }
}

// ---- result path over peer memory (NVLink): every rank's publish kernel stores its packed cone
// list (offsets + records) straight into the gathering rank's buffer and then raises a sequence
// flag there.  No collective kernel has to be co-scheduled with the grid-filling compute kernels.
// buffer layout (u32 words): [flags: 2 x world, padded to 64] [parity 0: world slots] [parity 1: world slots]
constexpr u32 kGatherFlagWords = 64;

// The run number lives on the device (d_seq) so that a CUDA-graph replay publishes under a fresh
// number without any kernel parameter changing: every CTA reads it on entry, the last one to finish
// advances it.  `advance` = 0 re-publishes under the current number (back-half retry by cp_sync).
constexpr u32 kGatherOverflowBit = 0x80000000u;  // flag bit: the rank had more cones than its slot holds

__global__ void __launch_bounds__(256) gather_publish_kernel(const u32* __restrict__ src, u32 words, u32* base,
                                                             u32 world, u32 rank, u32 slot_words, u32 off_words,
                                                             u32* d_seq, u32 advance, u32* done, Ctl* ctl) {
  const u32 seq = *((volatile u32*)d_seq) + advance;
  const u32 parity = seq & 1u;
  u32* dst = base + kGatherFlagWords + ((size_t)parity * world + rank) * slot_words;
  const uint4* s4 = reinterpret_cast<const uint4*>(src);
  uint4* d4 = reinterpret_cast<uint4*>(dst);
  // only the live part travels: the offsets and the K records of this run
  const u64 live = (u64)off_words + 4ull * ctl->n_clusters;
  const bool overflow = live > (u64)words;
  const u32 n4 = (u32)((overflow ? (u64)words : live) / 4);
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += gridDim.x * blockDim.x) d4[i] = s4[i];
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    const u32 t = atomicAdd(done, 1u);
    if (t == gridDim.x - 1) {
      *done = 0;
      *d_seq = seq;
      // never silently truncated: the publishing rank's cp_sync fails with CP_E_CAPACITY and the gathering
      // rank's cp_gather_wait sees the overflow bit in the flag
      if (overflow) atomicOr(&ctl->error, kErrGather);
      __threadfence_system();
      // a run whose shared-memory back half overflowed is re-run (and re-published) by cp_sync
      if (ctl->fast_overflow == 0)
        *((volatile u32*)(base + parity * world + rank)) = (seq & ~kGatherOverflowBit) | (overflow ? kGatherOverflowBit : 0u);
    }
  }
}

void enqueue_gather_publish(cp_handle* h, bool retry) {
  auto& g = h->gather;
  const u32 words = (u32)std::min<size_t>(g.slot_words, h->off_words + 4 * (size_t)h->cap_v) / 4 * 4;
  const u32 grid = std::max<u32>(1, std::min<u32>(64, words / 4 / 256));
  gather_publish_kernel<<<grid, 256, 0, h->stream>>>(h->d_k_off, words, g.base, g.world, g.rank, g.slot_words,
                                                     (u32)h->off_words, g.d_seq, retry ? 0u : 1u, g.d_done, h->d_ctl);
  h->launches++;
}

cp_status enqueue_back(cp_handle* h, bool retry) {
  const RunParams& rp = h->rp;
  if (retry) {
    back_reset_kernel<<<h->sms, 256, 0, h->stream>>>(h->d_ctl, h->hg.n_frames, h->d_ncomp_f, h->d_kcount_f);
    CK(cudaMemsetAsync(h->d_desc_fv, 0, sizeof(u64) * h->hg.n_frames, h->stream));
    h->launches++;
  }
  // smallest budget: 256-thread CTAs (4 per SM) keep a whole big batch resident in one wave; for a few
  // frames latency matters instead, so they get 512 threads each
  if (h->back_mode == 0 && h->hg.n_frames > (u32)h->sms * 2) enqueue_back_fast<1024, 512, 256>(h, rp);
  else if (h->back_mode == 0) enqueue_back_fast<1024, 512, 512>(h, rp);
  else if (h->back_mode == 1) enqueue_back_fast<2048, 1024, 512>(h, rp);
  else if (h->back_mode == 2) enqueue_back_fast<4096, 2048, 512>(h, rp);
  else {
    // the pass over the scan below counts the ground survivors again (atomically); a per-frame kernel that evaluated
    // pass 2 itself has already stored them
    if (retry && !h->masked) CK(cudaMemsetAsync(h->d_gcount, 0, sizeof(u32) * h->hg.n_frames, h->stream));
    if (!h->masked && !h->gathered) {
      launch_mask_compact<false>(h, device_geom(h), rp.crop, rp.gk, (u32)h->cap_c, nullptr);
    } else {   // a keep mask exists already (single-pass front ends, a retried one-launch frame)
      if (!h->masked) launch_keep_mask(h, device_geom(h), rp.crop, rp.gk, h->run_sgrid);
      if (!h->gathered) launch_scan_gather(h, device_geom(h), rp.gk, (u32)h->cap_c);
    }
    enqueue_back_general(h, rp);
  }
  if (h->plane_run) {
    plane_counters_kernel<<<(h->hg.n_frames + 255) / 256, 256, 0, h->stream>>>(h->hg.n_frames, h->pb.kept, h->d_fc);
    h->launches++;
  }
  if (h->gather.open) enqueue_gather_publish(h, retry);
  if (!h->capturing) cudaEventRecord(h->ev1, h->stream);
  h->fetched = false;
  CK(cudaGetLastError());
  return CP_OK;
}

// One batch of device-to-host copies behind the kernels: control block, per-frame counters and the
// head of the result block (offsets + the first records) go to pinned mirrors, so reading results
// costs ONE stream synchronisation.  Issued when the host asks for results (cp_sync), not per run:
// a caller that keeps results on the device (multi-GPU gather) pays no PCIe traffic per step.
// Small batches (a ROS node's single frame): one kernel stores the control block, the per-frame counters,
// the offsets and the K cluster records straight into the pinned host mirrors (zero-copy writes over PCIe)
// instead of three DMA copies with their per-copy latency, and only K records travel, not a fixed prefix.
__global__ void __launch_bounds__(256) result_publish_kernel(const Ctl* __restrict__ ctl, u32* __restrict__ h_ctl,
                                                             const u32* __restrict__ fc, u32* __restrict__ h_fc,
                                                             u32 fc_words, const u32* __restrict__ k_off,
                                                             u32* __restrict__ h_res, u32 off_words, u32 max_records) {
  const u32 tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
  const u32 K = ctl->n_clusters < max_records ? ctl->n_clusters : max_records;
  for (u32 i = tid; i < sizeof(Ctl) / 4; i += nth) h_ctl[i] = reinterpret_cast<const u32*>(ctl)[i];
  for (u32 i = tid; i < fc_words; i += nth) h_fc[i] = fc[i];
  const u32 res_words = off_words + 4u * K;
  for (u32 i = tid; i < res_words; i += nth) h_res[i] = k_off[i];
}
constexpr u32 kPublishMaxFrames = 64;

cp_status enqueue_result_fetch(cp_handle* h) {
  if (h->hg.n_frames <= kPublishMaxFrames) {
    h->prefetched = h->prefetch_cap;
    result_publish_kernel<<<4, 256, 0, h->stream>>>(h->d_ctl, reinterpret_cast<u32*>(h->h_ctl), h->d_fc, h->h_fc,
                                                    8u * h->hg.n_frames, h->d_k_off, h->h_result, (u32)h->off_words,
                                                    (u32)std::min<u64>(h->prefetch_cap, 0xFFFFFFFFu));
    CK(cudaGetLastError());
    h->fetched = true;
    return CP_OK;
  }
  CK(cudaMemcpyAsync(h->h_ctl, h->d_ctl, sizeof(Ctl), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(h->h_fc, h->d_fc, sizeof(u32) * 8 * h->hg.n_frames, cudaMemcpyDeviceToHost, h->stream));
  h->prefetched = std::min<u64>(h->prefetch_cap, std::max<u64>(4096, 64ull * h->hg.n_frames));
  CK(cudaMemcpyAsync(h->h_result, h->d_k_off, sizeof(u32) * (h->off_words + 4 * h->prefetched),
                     cudaMemcpyDeviceToHost, h->stream));
  h->fetched = true;
  return CP_OK;
}

cp_status ensure_out32(cp_handle* h) {
  if (h->d_out32) return CP_OK;
  cudaError_t e = cudaMalloc(&h->d_out32, (size_t)h->cfg.max_points * 32);
  if (e != cudaSuccess) {
    cudaGetLastError();
    h->err = "cudaMalloc of the 32-byte output cloud failed";
    return CP_E_NOMEM;
  }
  return CP_OK;
}

// The plane ground node over the staged input (plane_kernels.cuh): every frame's message into d_out32, G_f into
// pb.kept, the chosen planes into pb.sel / pb.info.  Five launches.  count_rows: add every row to rows_loaded (the
// ground calls; in a run the detector's own pass over the messages counts them).
template <int MODE>
void launch_plane_node_t(cp_handle* h, const Geom& g, const PlaneK& k, u32 hgrid, Ctl* ctl) {
  plane_hyp_kernel<MODE><<<hgrid, 256, 0, h->stream>>>(h->in_ptr, h->layout, g, k, h->pb);
  plane_score_kernel<MODE><<<g.n_tiles, kStreamThreads, 0, h->stream>>>(h->in_ptr, h->layout, g, k, h->pb);
  plane_select_kernel<<<(g.n_frames + 3) / 4, 128, 0, h->stream>>>(g.n_frames, k, h->pb);
  plane_count_kernel<MODE><<<g.n_tiles, kStreamThreads, 0, h->stream>>>(h->in_ptr, h->layout, g, k, h->pb);
  plane_write_kernel<MODE><<<g.n_tiles, kStreamThreads, 0, h->stream>>>(h->in_ptr, h->layout, g, k, h->pb, h->d_out32,
                                                                        ctl);
}
cp_status enqueue_plane_node(cp_handle* h, bool count_rows) {
  const Geom g = device_geom(h);
  PlaneK k;
  k.seed = h->plane.seed;
  k.H = h->plane.n_hypotheses;
  k.inlier = h->plane.inlier_distance;
  k.height = h->plane.ground_height;
  k.cos_tilt = h->plane_cos;
  const u32 hgrid = grid_for((u64)g.n_frames * k.H, 256, h->sms, 8);
  Ctl* ctl = count_rows ? h->d_ctl : nullptr;
  switch (h->layout.mode) {
    case 0: launch_plane_node_t<0>(h, g, k, hgrid, ctl); break;
    case 1: launch_plane_node_t<1>(h, g, k, hgrid, ctl); break;
    default: launch_plane_node_t<2>(h, g, k, hgrid, ctl); break;
  }
  h->launches += 5;
  h->plane_valid = true;
  h->plane_frames = g.n_frames;
  h->plane_h = k.H;
  CK(cudaGetLastError());
  return CP_OK;
}

cp_status enqueue_pipeline(cp_handle* h, const cp_detect_params* d, const cp_ground_params* ground) {
  // the plane model (cp_set_ground_plane): the plane ground node's messages, then the detector without ground
  // removal on them — the two-node chain, on the device
  const bool plane = ground && h->plane_on;
  if (plane) ground = nullptr;
  if (!d) {
    h->err = "NULL detect params";
    return CP_E_PARAM;
  }
  if (!h->batch_ready) {
    h->err = "no batch input set";
    return CP_E_STATE;
  }
  const float leaf[3] = {(float)d->voxel_filter_leaf_size_x, (float)d->voxel_filter_leaf_size_y,
                         (float)d->voxel_filter_leaf_size_z};
  for (int a = 0; a < 3; ++a)
    if (!(leaf[a] > 0.0f) || !isfinite(leaf[a])) {
      h->err = "voxel_filter_leaf_size_* must be positive and finite";
      return CP_E_PARAM;
    }
  CropK crop;
  cp_status st = make_crop(h, d, &crop);
  if (st) return st;
  ClusterK ck;
  u32 csort_bits = 0, osort_bits = 0;
  st = make_cluster(h, d, h->hg.n_frames, &ck, &csort_bits, &osort_bits);
  if (st) return st;
  GroundK gk;
  gk.do_ground = ground ? 1 : 0;
  gk.pad_survives = (ground && zero_point_survives(d)) ? 1 : 0;
  gk.want_count = gk.do_ground;   // ground survivors are always counted (n_ground_kept); skipped rows hold none
  h->counted_ground = gk.do_ground != 0;
  VoxelK vk;
  for (int a = 0; a < 3; ++a) vk.inv[a] = 1.0f / leaf[a];
  vk.frame_bits = ceil_log2_host(h->hg.n_frames);

  const Geom g = device_geom(h);
  h->launches = 0;
  h->plane_run = plane;
  if (!plane) h->plane_valid = false;
  h->run_in = plane ? h->d_out32 : h->in_ptr;
  h->run_layout = plane ? make_layout(32, 0, 4, 8, 16) : h->layout;
  h->rp.d = *d;
  h->rp.vk = vk;
  h->rp.ck = ck;
  h->rp.gk = gk;
  h->rp.crop = crop;
  h->rp.csort_bits = csort_bits;
  h->rp.osort_bits = osort_bits;
  h->rp_has_ground = ground != nullptr;
  if (ground) h->rp_ground = *ground;
  h->self_published = false;
  if (single_frame_eligible(h, g)) {
    // a node's single frame: front end, back half and result publish in one launch (single_frame.cuh)
    h->ran_cluster = h->ran_fused = false;
    if (launch_single_frame(h, h->rp, ground ? ground->default_lowest_point : 0.0f)) {
      h->masked = true;           // keep mask and tile counts are in place for a back-half retry
      h->gathered = false;
      h->ran_ground = ground != nullptr;
      h->ran_frame_kernel = true;
      h->launches = 1;
      h->self_published = true;
      h->fetched = true;
      h->prefetched = h->prefetch_cap;
      h->ran = true;
      return CP_OK;
    }
  }
  if (!h->capturing) cudaEventRecord(h->ev0, h->stream);
  launch_init(h, ground ? ground->default_lowest_point : 0.0f);
  if (plane) {
    st = enqueue_plane_node(h, false);
    if (st) return st;
  }
  h->masked = false;
  h->run_fused_mask = false;
  h->ran_frame_kernel = false;
  const u32 sgrid = grid_for((u64)g.n_tiles * kStreamThreads, kStreamThreads, h->sms, h->stream_ctas_per_sm);
  h->run_sgrid = sgrid;
  h->ran_cluster = cluster_front_eligible(h, g, ground != nullptr) &&
                   launch_front_cluster(h, g, crop, gk, ground->default_lowest_point);
  h->ran_fused = !h->ran_cluster && ground && g.uniform_n && h->use_fused;
  if (h->ran_cluster) {
    h->masked = true;  // front end done in one launch
  } else if (h->ran_fused) {
    launch_front_fused(h, g, crop, gk);
    h->masked = true;
  } else {
    h->rowmax_valid = false;
    if (ground) {
      if (h->stage_timing) cudaEventRecord(h->ev_k[0], h->stream);
      launch_sector_min(h, g, sgrid);
      if (h->stage_timing) cudaEventRecord(h->ev_k[1], h->stream);
      h->launches++;
      h->rowmax_valid = h->use_rowskip;
    }
    // pass 2 (ground verdicts + crop) normally runs inside the per-frame kernel; the separate streaming kernel
    // serves the general back half and — a few frames without ground removal, where every row is live and one
    // CTA per frame would be too few — small unskippable batches
    // (the plane chain too, so that its launch count does not depend on the number of frames)
    h->run_fused_mask = h->fuse_mask && h->back_mode < 3 &&
                        (ground != nullptr || plane || g.n_frames >= (u32)h->sms || h->fuse_mask_always);
    // (the general back half judges and compacts the points in one pass of its own: no keep mask for it)
    if (!h->run_fused_mask && h->back_mode < 3) launch_keep_mask(h, g, crop, gk, sgrid);
  }
  h->gathered = false;
  h->ran_ground = ground != nullptr;
  if (h->gather.open) h->gather.seq++;
  st = enqueue_back(h, false);
  if (st) return st;
  h->ran = true;
  return CP_OK;
}

// A pageable cloud of a megabyte or more: one core's memcpy into pinned memory (about 10 GB/s) costs more than
// the DMA and the kernels together.  Helper threads share the copy in 64 KB pieces; the calling thread copies too
// and issues one DMA per group of pieces as soon as the group is complete, so copies and DMAs overlap.
constexpr size_t kParallelStageMin = 512ull << 10;
constexpr size_t kStagePiece = 64ull << 10;
cp_status stage_parallel(cp_handle* h, const uint8_t* src, size_t total, size_t dst_off, int* ring) {
  if (!h->copy_pool) {
    try {
      h->copy_pool.reset(new CopyPool(h->stage_threads - 1));
    } catch (...) {  // no helper threads to be had: nothing may cross the C ABI, copy on the calling thread instead
      h->stage_threads = 1;
      return CP_E_STATE;
    }
  }
  size_t done = 0;
  while (done < total) {
    const size_t chunk = std::min(kStageChunk, total - done);
    const int r = *ring;
    CK(cudaEventSynchronize(h->ev_stage[r]));
    // 4+ DMAs per cloud, each 256 KB .. 2 MB
    const size_t group_bytes = std::min<size_t>(2ull << 20, std::max<size_t>(256ull << 10, (chunk / 4 + kStagePiece - 1) / kStagePiece * kStagePiece));
    const u32 ppg = (u32)(group_bytes / kStagePiece);
    std::shared_ptr<CopyPool::Batch> b = h->copy_pool->start(h->h_stage[r], src + done, chunk, kStagePiece, ppg, h->stage_streaming);
    u32 issued = 0;
    cudaError_t err = cudaSuccess;
    auto issue_ready = [&](bool block) {
      while (issued < b->n_groups) {
        if (!b->group_done(issued)) {
          if (!block) return;
          std::this_thread::yield();
          continue;
        }
        const size_t off = (size_t)issued * group_bytes;
        const size_t len = std::min(group_bytes, chunk - off);
        if (err == cudaSuccess)
          err = cudaMemcpyAsync(h->d_in + dst_off + done + off, h->h_stage[r] + off, len, cudaMemcpyHostToDevice, h->stream);
        ++issued;
      }
    };
    while (b->take_one()) issue_ready(false);
    issue_ready(true);  // every piece is copied when this returns: no helper touches the buffers afterwards
    CK(err);
    CK(cudaEventRecord(h->ev_stage[r], h->stream));
    *ring = r ^ 1;
    done += chunk;
  }
  return CP_OK;
}

// copy a host cloud into the device input buffer at byte offset `dst_off`
cp_status stage_view(cp_handle* h, const cp_cloud_view* v, size_t dst_off, int* ring) {
  const u64 n = (u64)v->width * v->height;
  if (n == 0) return CP_OK;
  const size_t row_bytes = (size_t)v->width * v->point_step;
  const bool contiguous = (v->height <= 1) || (v->row_step == row_bytes);
  cudaPointerAttributes attr;
  bool pinned = false;
  if (cudaPointerGetAttributes(&attr, v->data) == cudaSuccess)
    pinned = (attr.type == cudaMemoryTypeHost);
  else
    cudaGetLastError();
  if (pinned && contiguous) {
    CK(cudaMemcpyAsync(h->d_in + dst_off, v->data, row_bytes * v->height, cudaMemcpyHostToDevice, h->stream));
    return CP_OK;
  }
  // pageable (or row-padded) source: pack through the pinned ring, chunk by chunk
  const size_t total = row_bytes * v->height;
  if (contiguous && h->stage_threads > 1 && total >= kParallelStageMin) {
    const cp_status sp = stage_parallel(h, v->data, total, dst_off, ring);
    if (sp != CP_E_STATE) return sp;  // CP_E_STATE: the helper pool could not be created; fall through
  }
  size_t done = 0;
  while (done < total) {
    // a cloud is cut into at least 4 pieces so the host memcpy of piece k+1 overlaps the DMA of piece k
    const size_t piece = std::min(kStageChunk, std::max(kStageMinChunk, (total / 4 + 255) / 256 * 256));
    const size_t chunk = std::min(piece, total - done);
    const int r = *ring;
    CK(cudaEventSynchronize(h->ev_stage[r]));
    if (contiguous) {
      if (h->stage_streaming) copy_streaming(h->h_stage[r], v->data + done, chunk);
      else memcpy(h->h_stage[r], v->data + done, chunk);
    } else {
      size_t w = 0;
      while (w < chunk) {  // row-wise pack (rows are row_step apart in the source)
        const size_t pos = done + w;
        const size_t row = pos / row_bytes, col = pos % row_bytes;
        const size_t take = std::min(row_bytes - col, chunk - w);
        memcpy(h->h_stage[r] + w, v->data + row * v->row_step + col, take);
        w += take;
      }
    }
    CK(cudaMemcpyAsync(h->d_in + dst_off + done, h->h_stage[r], chunk, cudaMemcpyHostToDevice, h->stream));
    CK(cudaEventRecord(h->ev_stage[r], h->stream));
    *ring = r ^ 1;
    done += chunk;
  }
  return CP_OK;
}

cp_status device_errors(cp_handle* h) {
  const u32 e = h->h_ctl->error;
  if (!e) return CP_OK;
  if (e & kErrSurvivors) h->err = "more crop survivors than cp_config.max_survivors";
  else if (e & kErrVoxels) h->err = "more voxels / clusters than cp_config.max_voxels";
  else if (e & kErrHash) h->err = "neighbour-grid hash table too small for this batch";
  else if (e & kErrGather) h->err = "this rank found more cones than its slot of the gather buffer holds (slot_words)";
  else h->err = "internal capacity error";
  return CP_E_CAPACITY;
}

}  // namespace

// ======================================================================== C ABI
// ---- colour path inputs (color_kernels.cuh) ----------------------------------------------
constexpr size_t kColorPrefetch = 16384;  // crop points copied back speculatively with the offsets
template <typename T>
cp_status grow(cp_handle* h, T** p, size_t* have, size_t need) {
  if (need <= *have && *p) return CP_OK;
  if (*p) {
    cudaStreamSynchronize(h->stream);
    cudaFree(*p);
    *p = nullptr;
    *have = 0;
  }
  void* q = nullptr;
  const size_t n = std::max<size_t>(need, 1);
  cudaError_t e = cudaMalloc(&q, n * sizeof(T));
  if (e != cudaSuccess) {
    cudaGetLastError();
    h->err = std::string("cudaMalloc failed (colour path): ") + cudaGetErrorString(e);
    return e == cudaErrorMemoryAllocation ? CP_E_NOMEM : CP_E_CUDA;
  }
  *p = static_cast<T*>(q);
  *have = n;
  return CP_OK;
}

// Whether a colour-path call on the staged input (cloud NULL) crops from the ground node's message: the handle is
// set to CP_COLOR_CLOUD_GROUNDLESS and the last run fused ground removal.  The crops then need that run's sector
// minima and final counters (cp_sync: the back half may be re-run), so the input must not have been staged since.
static cp_status groundless_crops(cp_handle* h, const cp_cloud_view* cloud, bool* groundless) {
  *groundless = false;
  if (cloud || h->color_cloud != CP_COLOR_CLOUD_GROUNDLESS) return CP_OK;
  if (!h->ran) {
    h->err = "groundless colour crops need a run on the staged input (none since it was staged)";
    return CP_E_STATE;
  }
  if (h->plane_run) {
    h->err = "groundless colour crops re-derive the sector model's verdict: not available after a plane-model run";
    return CP_E_STATE;
  }
  if (!h->rp_has_ground) return CP_OK;
  *groundless = true;
  return cp_sync(h);
}

// Resolves the cloud a colour-path call works on and enqueues the box gather of all centres.
// On return crop offsets are in h->color.off (device) and the packed crops in h->color.pts.
// groundless: crop frame `frame` of the staged input as the ground node's message of the last run (color_kernels.cuh).
cp_status enqueue_cone_crops(cp_handle* h, const cp_cloud_view* cloud, u32 frame, const cp_cone_center* centers,
                             u32 n_centers, float cone_width, size_t want_cap, bool groundless) {
  if (n_centers && !centers) {
    h->err = "NULL centers";
    return CP_E_PARAM;
  }
  if (cloud) {
    cp_status st = cp_batch_set_host_input(h, cloud, 1);
    if (st) return st;
    frame = 0;
  } else if (!h->batch_ready) {
    h->err = "cloud is NULL and no input has been staged on this handle";
    return CP_E_STATE;
  }
  if (frame >= h->hg.n_frames) {
    h->err = "frame index outside the staged batch";
    return CP_E_PARAM;
  }
  const u32 n_points = h->hg.frame_n[frame];
  const u64 first_point = h->hg.frame_off[frame];
  const u32 n_rows = (n_points + 31) / 32;
  const u32 n_tiles = std::max<u32>(1, (n_rows + kTileWords - 1) / kTileWords);
  cp_handle::ColorBufs& cb = h->color;
  cp_status st;
  if ((st = grow(h, &cb.mask, &cb.mask_n, (size_t)kConeChunk * std::max<u32>(n_rows, 1)))) return st;
  if ((st = grow(h, &cb.tcount, &cb.tile_n, (size_t)kConeChunk * n_tiles))) return st;
  if ((st = grow(h, &cb.texcl, &cb.texcl_n, (size_t)kConeChunk * n_tiles))) return st;
  if ((st = grow(h, &cb.off, &cb.off_n, (size_t)n_centers + 1))) return st;
  if ((st = grow(h, &cb.flags, &cb.flags_n, (size_t)n_centers + 1))) return st;
  if ((st = grow(h, &cb.pts, &cb.pts_n, std::max<size_t>(want_cap, 1u << 16)))) return st;
  const u32 cap = (u32)std::min<size_t>(cb.pts_n, 0xFFFFFFFFu);
  CK(cudaMemsetAsync(cb.off, 0, sizeof(u32), h->stream));
  const double hw = (double)cone_width / 1.5;  // CONE_WIDTH / 1.5: float / double literal
  const u32* low_key = groundless ? h->d_low_key + (size_t)frame * kSectStride : nullptr;
  const u32* fc = groundless ? h->d_fc : nullptr;
  for (u32 k0 = 0; k0 < n_centers; k0 += kConeChunk) {
    ConeBoxes B;
    memset(&B, 0, sizeof(B));
    B.n = std::min<u32>(kConeChunk, n_centers - k0);
    u64 origin = 0;  // boxes that hold the ground node's zero padding points
    for (u32 k = 0; k < B.n; ++k) {
      box_bounds(centers[k0 + k].x, hw, &B.xlo[k], &B.xhi[k]);
      box_bounds(centers[k0 + k].y, hw, &B.ylo[k], &B.yhi[k]);
      if (groundless && B.xlo[k] <= 0.0f && B.xhi[k] >= 0.0f && B.ylo[k] <= 0.0f && B.yhi[k] >= 0.0f)
        origin |= 1ull << k;
    }
    CK(cudaMemsetAsync(cb.mask, 0, sizeof(u32) * (size_t)B.n * std::max<u32>(n_rows, 1), h->stream));
    CK(cudaMemsetAsync(cb.tcount, 0, sizeof(u32) * (size_t)B.n * n_tiles, h->stream));
    const u32 mgrid = (n_rows + kStreamWarps - 1) / kStreamWarps;
    if (n_points) {
      switch (h->layout.mode) {
        case 0: cone_box_mask_kernel<0><<<mgrid, kStreamThreads, 0, h->stream>>>(h->in_ptr, h->layout, first_point, n_points, B, low_key, n_rows, n_tiles, cb.mask, cb.tcount); break;
        case 1: cone_box_mask_kernel<1><<<mgrid, kStreamThreads, 0, h->stream>>>(h->in_ptr, h->layout, first_point, n_points, B, low_key, n_rows, n_tiles, cb.mask, cb.tcount); break;
        default: cone_box_mask_kernel<2><<<mgrid, kStreamThreads, 0, h->stream>>>(h->in_ptr, h->layout, first_point, n_points, B, low_key, n_rows, n_tiles, cb.mask, cb.tcount); break;
      }
    }
    cone_box_scan_kernel<<<1, 1024, 0, h->stream>>>(B.n, k0, n_tiles, origin, fc, frame, cb.tcount, cb.texcl, cb.off);
    if (n_points) {
      switch (h->layout.mode) {
        case 0: cone_box_gather_kernel<0><<<n_tiles, kStreamThreads, 0, h->stream>>>(h->in_ptr, h->layout, first_point, B.n, k0, n_rows, n_tiles, origin, fc, frame, cb.mask, cb.tcount, cb.texcl, cb.off, cap, cb.pts); break;
        case 1: cone_box_gather_kernel<1><<<n_tiles, kStreamThreads, 0, h->stream>>>(h->in_ptr, h->layout, first_point, B.n, k0, n_rows, n_tiles, origin, fc, frame, cb.mask, cb.tcount, cb.texcl, cb.off, cap, cb.pts); break;
        default: cone_box_gather_kernel<2><<<n_tiles, kStreamThreads, 0, h->stream>>>(h->in_ptr, h->layout, first_point, B.n, k0, n_rows, n_tiles, origin, fc, frame, cb.mask, cb.tcount, cb.texcl, cb.off, cap, cb.pts); break;
      }
    }
  }
  CK(cudaGetLastError());
  return CP_OK;
}

cp_status enqueue_raster(cp_handle* h, u32 n_cones) {
  cp_handle::ColorBufs& cb = h->color;
  cp_status st = grow(h, &cb.img, &cb.img_n, (size_t)std::max<u32>(n_cones, 1) * kImgPix);
  if (st) return st;
  if (n_cones)
    cone_raster_kernel<<<n_cones, kRasterThreads, 0, h->stream>>>(cb.pts, cb.off, (u32)std::min<size_t>(cb.pts_n, 0xFFFFFFFFu),
                                                                 cb.img, cb.flags);
  CK(cudaGetLastError());
  return CP_OK;
}

// ---- colour classifier (color_net.cuh) ------------------------------------------------------
static cp_status load_color_net(cp_handle* h, const cp_color_net* n) {
  if (!n || !n->conv1_w || !n->conv1_b || !n->conv2_w || !n->conv2_b || !n->bn_scale || !n->bn_shift || !n->dense_w ||
      !n->dense_b) {
    h->err = "NULL colour-net tensor";
    return CP_E_PARAM;
  }
  if (n->c1 < 1 || n->c1 > (u32)kNetMaxC1 || n->c2 < 1 || n->c2 > (u32)kNetMaxC2 || n->n_classes < 1 ||
      n->n_classes > (u32)kNetMaxClasses || n->n_classes > 3 || !(n->threshold >= 0.f && n->threshold <= 1.f)) {
    h->err = "colour net out of range: c1 <= 16, c2 <= 32, classes <= 3 (yellow, blue, orange), threshold in [0, 1]";
    return CP_E_PARAM;
  }
  const u32 C1 = n->c1, C2 = n->c2, NC = n->n_classes, K = kPool2H * kPool2W * C2;
  // device layout: w1t[9][C1] b1 w2t[9*C1][C2] b2 scale shift wd[NC][K] bd
  std::vector<float> w;
  w.reserve(9 * C1 + C1 + 9 * C1 * C2 + 3 * C2 + NC * K + NC);
  const size_t o_w1 = w.size();
  for (u32 k = 0; k < 9; ++k)
    for (u32 c = 0; c < C1; ++c) w.push_back(n->conv1_w[c * 9 + k]);                 // [c][ky][kx][1] -> [k][c]
  const size_t o_b1 = w.size();
  w.insert(w.end(), n->conv1_b, n->conv1_b + C1);
  const size_t o_w2 = w.size();
  for (u32 k = 0; k < 9; ++k)
    for (u32 ci = 0; ci < C1; ++ci)
      for (u32 c = 0; c < C2; ++c) w.push_back(n->conv2_w[((size_t)c * 9 + k) * C1 + ci]);   // [c][k][ci] -> [k][ci][c]
  const size_t o_b2 = w.size();
  w.insert(w.end(), n->conv2_b, n->conv2_b + C2);
  const size_t o_sc = w.size();
  w.insert(w.end(), n->bn_scale, n->bn_scale + C2);
  const size_t o_sh = w.size();
  w.insert(w.end(), n->bn_shift, n->bn_shift + C2);
  const size_t o_wd = w.size();
  w.insert(w.end(), n->dense_w, n->dense_w + (size_t)NC * K);
  const size_t o_bd = w.size();
  w.insert(w.end(), n->dense_b, n->dense_b + NC);
  cp_handle::ColorBufs& cb = h->color;
  CK(cudaSetDevice(h->cfg.device));
  cp_status st = grow(h, &cb.net_w, &cb.net_w_n, w.size());
  if (st) return st;
  CK(cudaStreamSynchronize(h->stream));
  CK(cudaMemcpy(cb.net_w, w.data(), sizeof(float) * w.size(), cudaMemcpyHostToDevice));
  cb.net = ColorNetDev{cb.net_w + o_w1, cb.net_w + o_b1, cb.net_w + o_w2, cb.net_w + o_b2, cb.net_w + o_sc,
                       cb.net_w + o_sh, cb.net_w + o_wd, cb.net_w + o_bd, C1, C2, NC, n->threshold};
  cb.net_loaded = true;
  return CP_OK;
}

// cone_color_kernel over n images already on the device (cb.img or `images_dev`); outputs stay in cb.colors/probs
static cp_status enqueue_color_net(cp_handle* h, const uint8_t* images_dev, const u32* raster_flags, u32 n) {
  cp_handle::ColorBufs& cb = h->color;
  if (!cb.net_loaded) {
    h->err = "no colour net loaded (cp_color_net_load / cp_color_net_load_tflite)";
    return CP_E_STATE;
  }
  cp_status st;
  if ((st = grow(h, &cb.colors, &cb.colors_n, (size_t)std::max<u32>(n, 1)))) return st;
  if ((st = grow(h, &cb.probs, &cb.probs_n, (size_t)std::max<u32>(n, 1) * 2 * kNetMaxClasses))) return st;
  if ((st = grow(h, &cb.net_flags, &cb.net_flags_n, (size_t)std::max<u32>(n, 1)))) return st;
  if (n)
    cone_color_kernel<<<n, kNetThreads, 0, h->stream>>>(images_dev, raster_flags, cb.net, cb.colors, cb.probs,
                                                        cb.probs + (size_t)n * cb.net.classes, cb.net_flags);
  CK(cudaGetLastError());
  h->launches += n ? 1 : 0;
  return CP_OK;
}

// cp_batch_cone_colors: crops of every cluster of the run, straight from the run's raw input (color_kernels.cuh),
// or from the ground node's messages of the run (groundless).
// Returns the kernel launches; on return the crop offsets are in color.off and the crops in color.pts.
template <int MODE>
static u32 enqueue_batch_crops(cp_handle* h, u32 K, double ext, double hw, u32 row_bits, u32 key_bits,
                               u32 max_key_bits, bool groundless) {
  cp_handle::ColorBufs& cb = h->color;
  const u32 cap = (u32)std::min<size_t>(cb.pts_n, 0xFFFFFFFFu);
  const Geom g = device_geom(h);
  batch_box_kernel<<<(K + 255) / 256, 256, 0, h->stream>>>(h->d_clusters, h->d_k_off, g.n_frames, K, ext, hw,
                                                           key_bits, groundless ? h->d_fc : nullptr, cb.box,
                                                           cb.kframe, cb.cnt, cb.tcnt, cb.bctl);
  const u32 mgrid = std::max<u32>(1, std::min<u32>(g.n_tiles, (u32)h->sms * (u32)h->stream_ctas_per_sm));
  batch_mark_kernel<MODE><<<mgrid, kStreamThreads, 0, h->stream>>>(h->in_ptr, h->layout, g, h->d_k_off, cb.box,
                                                                   groundless ? h->d_low_key : nullptr, row_bits, cap,
                                                                   cb.keys_a, cb.vals_a, cb.cnt, cb.tcnt, cb.bctl);
  batch_scan_kernel<<<1, kBatchScanThreads, 0, h->stream>>>(K, cb.cnt, cb.tcnt, cb.off, cb.toff, cap, cb.bctl);
  SortArgs sa;
  sa.keys_a = cb.keys_a;
  sa.keys_b = cb.keys_b;
  sa.vals_a = cb.vals_a;
  sa.vals_b = cb.vals_b;
  sa.d_n = cb.bctl + 2;
  sa.d_bits = cb.bctl + 1;
  sa.hdr = cb.sort_hdr;
  sa.state = cb.sort_state;
  sa.tiles_cap = (u32)(cb.sort_state_n / (2 * kRadix));
  // passes for the widest key this handle can produce, so that the launch count does not follow K
  const u32 sorts = (u32)radix_sort_enqueue(h->stream, sa, max_key_bits, cap, h->sms, !h->tile_ctas);
  const bool inb = sorted_in_b(key_bits);
  batch_gather_kernel<MODE><<<(K + 7) / 8, 256, 0, h->stream>>>(h->in_ptr, h->layout, g, K, cb.kframe,
                                                                inb ? cb.keys_b : cb.keys_a, inb ? cb.vals_b : cb.vals_a,
                                                                cb.toff, cb.off, row_bits, cap, cb.bctl, cb.pts);
  return 4 + sorts;
}

// Nothing may propagate through the C ABI: host-side allocation failures and the like become a status.
static cp_status abi_exception(cp_handle* h) noexcept {
  try {
    throw;
  } catch (const std::bad_alloc&) {
    try { if (h) h->err = "out of host memory"; } catch (...) {}
    return CP_E_NOMEM;
  } catch (const std::exception& e) {
    try { if (h) h->err = std::string("internal error: ") + e.what(); } catch (...) {}
    return CP_E_STATE;
  } catch (...) {
    return CP_E_STATE;
  }
}

extern "C" {

const char* cp_strerror(cp_status s) {
  switch (s) {
    case CP_OK: return "ok";
    case CP_E_PARAM: return "invalid parameter";
    case CP_E_BADFIELD: return "unsupported PointCloud2 field layout";
    case CP_E_CAPACITY: return "capacity exceeded";
    case CP_E_CUDA: return "CUDA error";
    case CP_E_NOMEM: return "out of memory";
    case CP_E_STATE: return "invalid call order";
  }
  return "unknown status";
}

const char* cp_last_error(const cp_handle* h) { return h ? h->err.c_str() : "NULL handle"; }
uint32_t cp_abi_version(void) { return kAbiVersion; }

static std::string g_create_error;
const char* cp_create_error(void) { return g_create_error.c_str(); }

cp_status cp_create(cp_handle** out, const cp_config* cfg) try {
  if (!out || !cfg) return CP_E_PARAM;
  *out = nullptr;
  if (cfg->max_points == 0 || cfg->max_frames == 0 || cfg->max_points >= (1ull << 31)) {
    g_create_error = "max_points must be in [1, 2^31) and max_frames >= 1";
    return CP_E_PARAM;
  }
  int ndev = 0;
  cudaError_t ce = cudaGetDeviceCount(&ndev);
  if (ce != cudaSuccess || ndev == 0) {
    g_create_error = std::string("no CUDA device: ") + cudaGetErrorString(ce) +
                     " (libconesgpu has no CPU fallback)";
    cudaGetLastError();
    return CP_E_CUDA;
  }
  if (cfg->device < 0 || cfg->device >= ndev) {
    g_create_error = "device ordinal out of range";
    return CP_E_PARAM;
  }
  cp_handle* h = new (std::nothrow) cp_handle();
  if (!h) return CP_E_NOMEM;
  h->cfg = *cfg;
  cp_status st = CP_OK;
  auto fail = [&](cp_status s) {
    g_create_error = h->err;
    cp_destroy(h);
    return s;
  };
  if (cudaSetDevice(cfg->device) != cudaSuccess) {
    h->err = "cudaSetDevice failed";
    return fail(CP_E_CUDA);
  }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, cfg->device) != cudaSuccess) {
    h->err = "cudaGetDeviceProperties failed";
    return fail(CP_E_CUDA);
  }
  if (prop.major < 10) {
    h->err = "libconesgpu is built for sm_100a only; device compute capability is too low";
    return fail(CP_E_CUDA);
  }
  h->sms = prop.multiProcessorCount;
  const char* prio_env = getenv("CONESGPU_PRIO");
  h->tail_priority = prio_env && prio_env[0] == '1';
  int prio_hi = 0;
  cudaDeviceGetStreamPriorityRange(&h->prio_low, &prio_hi);
  const char* k1_env = getenv("CONESGPU_K1_CTAS");
  if (k1_env && atoi(k1_env) >= 1 && atoi(k1_env) <= 256) h->k1_ctas_per_sm = atoi(k1_env);
  const char* tc_env = getenv("CONESGPU_TILE_CTAS");
  if (tc_env) h->tile_ctas = tc_env[0] != '0';
  const char* fc_env = getenv("CONESGPU_FRAME_CTAS");
  if (fc_env && atoi(fc_env) >= 1 && atoi(fc_env) <= 16) h->frame_ctas_per_sm = atoi(fc_env);
  if (cudaStreamCreateWithPriority(&h->stream, cudaStreamNonBlocking, h->tail_priority ? prio_hi : h->prio_low) != cudaSuccess ||
      cudaEventCreate(&h->ev0) != cudaSuccess || cudaEventCreate(&h->ev1) != cudaSuccess ||
      cudaEventCreateWithFlags(&h->ev_stage[0], cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&h->ev_stage[1], cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreate(&h->ev_k[0]) != cudaSuccess || cudaEventCreate(&h->ev_k[1]) != cudaSuccess ||
      cudaEventCreate(&h->ev_k[2]) != cudaSuccess || cudaEventCreate(&h->ev_k[3]) != cudaSuccess ||
      cudaEventCreate(&h->ev_k[4]) != cudaSuccess || cudaEventCreate(&h->ev_k[5]) != cudaSuccess) {
    h->err = "stream/event creation failed";
    return fail(CP_E_CUDA);
  }
  const char* tap_env = getenv("CONESGPU_TAPS");
  h->taps = tap_env && tap_env[0] == '1';
  const char* mode_env = getenv("CONESGPU_BACK_MODE");  // tests: force the back-half variant
  if (mode_env && mode_env[0] >= '0' && mode_env[0] <= '3') h->back_mode = mode_env[0] - '0';
  const char* sc_env = getenv("CONESGPU_STREAM_CTAS");
  if (sc_env && atoi(sc_env) >= 1 && atoi(sc_env) <= 8) h->stream_ctas_per_sm = atoi(sc_env);
  {
    const unsigned hw = std::thread::hardware_concurrency();
    h->stage_threads = hw >= 8 ? 4 : (hw >= 4 ? 2 : 1);
    const char* nt_env = getenv("CONESGPU_STAGE_NT");
    if (nt_env) h->stage_streaming = nt_env[0] != '0';
    const char* st_env = getenv("CONESGPU_STAGE_THREADS");
    if (st_env && atoi(st_env) >= 1 && atoi(st_env) <= 16) h->stage_threads = atoi(st_env);
  }
  const char* fm_env = getenv("CONESGPU_FUSED_MASK");  // "0": pass 2 as a separate streaming kernel
  if (fm_env) h->fuse_mask = fm_env[0] != '0', h->fuse_mask_always = fm_env[0] == '2';
  const char* rs_env = getenv("CONESGPU_ROWSKIP");
  if (rs_env) h->use_rowskip = rs_env[0] != '0';
  const char* sf_env = getenv("CONESGPU_SINGLE");
  if (sf_env) h->use_single = sf_env[0] != '0';
  const char* cl_env = getenv("CONESGPU_CLUSTER_FRONT");  // "1": single-pass 16-CTA-cluster front end
  if (cl_env) h->use_cluster = cl_env[0] == '1';
  const char* graph_env = getenv("CONESGPU_GRAPH");  // "0": never replay runs from a CUDA graph
  if (graph_env && graph_env[0] == '0') h->use_graph = false;
  const char* fused_env = getenv("CONESGPU_FUSED_FRONT");  // "1": both streaming passes in one persistent kernel
  if (fused_env) h->use_fused = fused_env[0] == '1';
  const u64 P = cfg->max_points;
  const u32 F = cfg->max_frames;
  h->cap_c = cfg->max_survivors ? std::min<u64>(cfg->max_survivors, P + F) : P + F;
  h->cap_v = cfg->max_voxels ? std::min<u64>(cfg->max_voxels, h->cap_c) : h->cap_c;
  h->tiles_cap = (u32)(P / kStreamTile + F + 1);
  h->sort_tiles_cap = (u32)(h->cap_c / kSortTile + 2);
  u64 hc = 64;
  while (hc < 2 * h->cap_v) hc <<= 1;
  h->hash_cap = (u32)std::min<u64>(hc, 1ull << 31);
  const u32 step = cfg->max_point_step ? cfg->max_point_step : 16;
  h->d_in_bytes = (size_t)P * step;
#define A(call)                \
  do {                         \
    st = (call);               \
    if (st) return fail(st);   \
  } while (0)
  A(dalloc(h, &h->d_ctl, 1));
  A(dalloc(h, &h->d_frame_n, F));
  A(dalloc(h, &h->d_frame_off, F));
  A(dalloc(h, &h->d_frame_tile0, F));
  A(dalloc(h, &h->d_tile_frame, h->tiles_cap));
  A(dalloc(h, &h->d_low_key, (size_t)F * kSectStride));
  A(dalloc(h, &h->d_bbox, (size_t)F * 8));
  A(dalloc(h, &h->d_c_off, F + 1));
  A(dalloc(h, &h->d_gcount, F));
  A(dalloc(h, &h->d_v_off, F + 1));
  A(dalloc(h, &h->d_ncomp_f, F));
  A(dalloc(h, &h->d_kcount_f, F));
  A(dalloc(h, &h->d_vf, F));
  A(dalloc(h, &h->d_pts, h->cap_c));
  A(dalloc(h, &h->d_src, h->cap_c));
  A(dalloc(h, &h->d_frame, h->cap_c));
  A(dalloc(h, &h->d_keys_a, h->cap_c));
  A(dalloc(h, &h->d_keys_b, h->cap_c));
  A(dalloc(h, &h->d_vals_a, h->cap_c));
  A(dalloc(h, &h->d_vals_b, h->cap_c));
  A(dalloc(h, &h->d_okeys_a, h->cap_v));
  A(dalloc(h, &h->d_okeys_b, h->cap_v));
  A(dalloc(h, &h->d_ovals_a, h->cap_v));
  A(dalloc(h, &h->d_ovals_b, h->cap_v));
  A(dalloc(h, &h->d_sort_state, (size_t)2 * kRadix * h->sort_tiles_cap));
  A(dalloc(h, &h->d_sort_hdr, kSortHdrWords * 4));   // one header per sort of the general back half
  A(dalloc(h, &h->d_vstart, h->cap_v));
  A(dalloc(h, &h->d_cstart, h->cap_v));
  A(dalloc(h, &h->d_comp_start, h->cap_v));
  A(dalloc(h, &h->d_vox, h->cap_v));
  A(dalloc(h, &h->d_vox_frame, h->cap_v));
  A(dalloc(h, &h->d_parent, h->cap_v));
  A(dalloc(h, &h->d_label, h->cap_v));
  A(dalloc(h, &h->d_hkeys, h->hash_cap));
  A(dalloc(h, &h->d_hvals, h->hash_cap));
  {
    // results live in ONE block — cluster offsets [round_up(F+1, 4) words] then the packed records —
    // so a multi-GPU caller can hand the whole cone list to a single collective
    const size_t off_words = ((size_t)F + 1 + 3) / 4 * 4;
    u32* block = nullptr;
    A(dalloc(h, &block, off_words + (size_t)h->cap_v * 4));
    h->d_k_off = block;
    h->d_clusters = reinterpret_cast<ClusterRec*>(block + off_words);
    h->off_words = off_words;
    h->prefetch_cap = std::min<u64>(h->cap_v, 1ull << 20);
    A(palloc(h, &h->h_result, off_words + 4 * (size_t)h->prefetch_cap));
    A(dalloc(h, &h->d_fc, (size_t)F * 8));
    A(palloc(h, &h->h_fc, (size_t)F * 8));
  }
  A(dalloc(h, &h->d_desc_a, h->tiles_cap));
  A(dalloc(h, &h->d_frame_ticket, 2));
  A(dalloc(h, &h->d_done, F));
  A(dalloc(h, &h->d_ncrop_f, F));
  A(dalloc(h, &h->d_nvox_f, F));
  A(dalloc(h, &h->d_slots, (size_t)F * 2048));
  A(dalloc(h, &h->d_desc_fv, F));
  A(dalloc(h, &h->d_mask, (size_t)h->tiles_cap * kTileWords));
  A(dalloc(h, &h->d_rowmax, (size_t)h->tiles_cap * kTileWords));
  A(dalloc(h, &h->d_thr_f, (size_t)F * kSectStride));
  A(dalloc(h, &h->d_tile_count, h->tiles_cap));
  A(dalloc(h, &h->d_tile_excl, h->tiles_cap));
  const size_t nb = h->cap_c / kHeadTile + 2;
  A(dalloc(h, &h->d_desc_b, nb));
  A(dalloc(h, &h->d_desc_c, nb));
  A(dalloc(h, &h->d_desc_d, nb));
  if (h->taps) {
    A(dalloc(h, &h->d_tap_keys, h->cap_c));
    A(dalloc(h, &h->d_tap_order, h->cap_c));
    A(dalloc(h, &h->d_tap_labels, h->cap_v));
  }
  A(palloc(h, &h->h_stage[0], kStageChunk));
  A(palloc(h, &h->h_stage[1], kStageChunk));
  A(palloc(h, &h->h_ctl, 1));
  // per-frame readback scratch; cp_ground_remove also parks one frame's kNSect sector minima in it
  A(palloc(h, &h->h_frame_u32, std::max<size_t>((size_t)(F + 1) * 8, (size_t)kSectStride)));
#undef A
  memset(h->h_ctl, 0, sizeof(Ctl));
  *out = h;
  return CP_OK;
} catch (...) {
  return abi_exception(nullptr);
}

void cp_destroy(cp_handle* h) {
  if (!h) return;
  cudaSetDevice(h->cfg.device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  if (h->gather.open && !h->gather.owner && h->gather.base) cudaIpcCloseMemHandle(h->gather.base);
  for (void* p : h->dev_allocs) cudaFree(p);
  for (void* p : h->pin_allocs) cudaFreeHost(p);
  if (h->d_out32) cudaFree(h->d_out32);
  for (void* q : {(void*)h->color.mask, (void*)h->color.tcount, (void*)h->color.texcl, (void*)h->color.off,
                  (void*)h->color.flags, (void*)h->color.pts, (void*)h->color.img, (void*)h->color.net_w,
                  (void*)h->color.colors, (void*)h->color.probs, (void*)h->color.net_flags, (void*)h->color.box,
                  (void*)h->color.kframe, (void*)h->color.cnt, (void*)h->color.tcnt, (void*)h->color.toff,
                  (void*)h->color.bctl, (void*)h->color.keys_a, (void*)h->color.keys_b, (void*)h->color.vals_a,
                  (void*)h->color.vals_b, (void*)h->color.sort_hdr, (void*)h->color.sort_state})
    if (q) cudaFree(q);
  if (h->color.pin) cudaFreeHost(h->color.pin);
  const cp_handle::TrackBufs& tb = h->track;
  for (void* q : {(void*)tb.st[0], (void*)tb.st[1], (void*)tb.par_d, (void*)tb.kframe, (void*)tb.bits, (void*)tb.rank,
                  (void*)tb.cnt, (void*)tb.coff_d, (void*)tb.ext, (void*)tb.info, (void*)tb.fcol, (void*)tb.ans,
                  (void*)tb.out, (void*)tb.rec, (void*)tb.rec_off, (void*)tb.flags, (void*)tb.colors})
    if (q) cudaFree(q);
  if (h->graph_exec) cudaGraphExecDestroy(h->graph_exec);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  for (int i = 0; i < 2; ++i)
    if (h->ev_stage[i]) cudaEventDestroy(h->ev_stage[i]);
  for (int i = 0; i < 6; ++i)
    if (h->ev_k[i]) cudaEventDestroy(h->ev_k[i]);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
}

cp_status cp_pinned_alloc(int32_t device, size_t bytes, int32_t write_combined, void** out) {
  if (!out || bytes == 0) return CP_E_PARAM;
  *out = nullptr;
  if (cudaSetDevice(device) != cudaSuccess) {
    cudaGetLastError();
    return CP_E_CUDA;
  }
  const unsigned flags = cudaHostAllocPortable | (write_combined ? cudaHostAllocWriteCombined : 0u);
  const cudaError_t e = cudaHostAlloc(out, bytes, flags);
  if (e != cudaSuccess) {
    cudaGetLastError();
    *out = nullptr;
    return e == cudaErrorMemoryAllocation ? CP_E_NOMEM : CP_E_CUDA;
  }
  return CP_OK;
}
void cp_pinned_free(void* p) {
  if (p) cudaFreeHost(p);
}

cp_status cp_batch_set_device_input(cp_handle* h, const void* d_points, uint32_t n_frames,
                                    const uint32_t* frame_points, uint32_t point_step, int32_t off_x,
                                    int32_t off_y, int32_t off_z, int32_t off_intensity) try {
  if (!h) return CP_E_PARAM;
  if (!d_points || !frame_points) {
    h->err = "NULL device pointer or frame_points";
    return CP_E_PARAM;
  }
  if (off_x < 0 || off_y < 0 || off_z < 0 ||
      (u32)std::max(std::max(off_x, off_y), std::max(off_z, off_intensity)) + 4 > point_step) {
    h->err = "x/y/z offsets missing or beyond point_step";
    return CP_E_BADFIELD;
  }
  CK(cudaSetDevice(h->cfg.device));
  h->batch_ready = false;
  h->ground_out = false;
  h->plane_valid = false;   // the planes belong to the previous input
  cp_status st = set_geometry(h, frame_points, n_frames);
  if (st) return st;
  h->layout = make_layout(point_step, off_x, off_y, off_z, off_intensity);
  if (h->layout.mode == 0 && ((uintptr_t)d_points & 15u)) h->layout.mode = 1;
  h->in_ptr = static_cast<const uint8_t*>(d_points);
  h->batch_ready = true;
  h->ran = false;
  return CP_OK;
} catch (...) {
  return abi_exception(h);
}

cp_status cp_batch_set_host_input(cp_handle* h, const cp_cloud_view* frames, uint32_t n_frames) try {
  if (!h) return CP_E_PARAM;
  if (!frames || n_frames == 0) {
    h->err = "NULL frames or n_frames == 0";
    return CP_E_PARAM;
  }
  CK(cudaSetDevice(h->cfg.device));
  h->batch_ready = false;
  h->ground_out = false;
  h->plane_valid = false;   // the planes belong to the previous input
  std::vector<u32> fp(n_frames);
  size_t bytes = 0;
  for (u32 f = 0; f < n_frames; ++f) {
    cp_status st = check_view(h, &frames[f]);
    if (st) return st;
    const cp_cloud_view& v = frames[f];
    if (v.point_step != frames[0].point_step || v.off_x != frames[0].off_x || v.off_y != frames[0].off_y ||
        v.off_z != frames[0].off_z || v.off_intensity != frames[0].off_intensity) {
      h->err = "all frames of a batch must share point_step and field offsets";
      return CP_E_BADFIELD;
    }
    const u64 n = (u64)v.width * v.height;
    if (n >= (1ull << 31)) {
      h->err = "frame too large";
      return CP_E_CAPACITY;
    }
    fp[f] = (u32)n;
    bytes += (size_t)n * v.point_step;
  }
  if (bytes > h->d_in_bytes) {
    h->err = "batch bytes exceed max_points * max_point_step of the handle";
    return CP_E_CAPACITY;
  }
  if (!h->d_in) {  // staged input buffer: only handles that take host clouds pay for it
    cp_status sa = dalloc(h, &h->d_in, h->d_in_bytes);
    if (sa) return sa;
  }
  cp_status st = set_geometry(h, fp.data(), n_frames);
  if (st) return st;
  size_t off = 0;
  int ring = 0;
  // frames that sit back to back in host memory (a replay buffer, a pinned batch tensor) are
  // copied as one run: few large cudaMemcpyAsync calls instead of one per frame
  for (u32 f = 0; f < n_frames;) {
    const cp_cloud_view& v0 = frames[f];
    const size_t step = v0.point_step;
    auto packed = [&](const cp_cloud_view& v) { return v.height <= 1 || v.row_step == (size_t)v.width * v.point_step; };
    size_t run_bytes = (size_t)fp[f] * step;
    u32 e = f + 1;
    if (packed(v0))
      while (e < n_frames && packed(frames[e]) && frames[e].data == v0.data + run_bytes) {
        run_bytes += (size_t)fp[e] * step;
        ++e;
      }
    if (e == f + 1) {
      st = stage_view(h, &v0, off, &ring);
    } else {
      cp_cloud_view run = v0;
      run.height = 1;
      run.width = (u32)(run_bytes / step);
      run.row_step = (u32)std::min<size_t>(run_bytes, 0xFFFFFFFFu);
      st = (run_bytes / step < (1ull << 32)) ? stage_view(h, &run, off, &ring) : CP_E_CAPACITY;
    }
    if (st) return st;
    off += run_bytes;
    f = e;
  }
  h->layout = make_layout(frames[0].point_step, frames[0].off_x, frames[0].off_y, frames[0].off_z,
                          frames[0].off_intensity);
  h->in_ptr = h->d_in;
  h->batch_ready = true;
  h->ran = false;
  return CP_OK;
} catch (...) {
  return abi_exception(h);
}

// A run is replayed from a CUDA graph when it repeats the previous one exactly (same batch
// shape, input pointer, parameters, back-half mode): a ROS node or a replay loop sees the same
// launch sequence every frame, and one graph launch replaces ~10 API calls.
struct RunKey {
  const void* in_ptr;
  u32 n_frames, uniform_n, n_tiles, layout_mode, layout_step;
  i32 ox, oy, oz, oi;
  int back_mode, has_ground;
  // the result publish over peer memory is part of the enqueued sequence: a graph captured before the gather
  // was wired has no publish node, so the gather state is part of the key
  u32 gather_open, gather_rank, gather_slot_words;
  const void* gather_base;
  cp_detect_params d;
  cp_ground_params g;
  // the ground model: a graph captured under one model is never replayed under the other
  u32 plane_on;
  cp_plane_params plane;
};

static RunKey make_key(const cp_handle* h, const cp_detect_params* d, const cp_ground_params* ground) {
  RunKey k;
  memset(&k, 0, sizeof(k));
  k.in_ptr = h->in_ptr;
  k.n_frames = h->hg.n_frames;
  k.uniform_n = h->hg.uniform_n;
  k.n_tiles = h->hg.n_tiles;
  k.layout_mode = h->layout.mode;
  k.layout_step = h->layout.step;
  k.ox = h->layout.ox; k.oy = h->layout.oy; k.oz = h->layout.oz; k.oi = h->layout.oi;
  k.back_mode = h->back_mode;
  k.has_ground = ground ? 1 : 0;
  k.gather_open = h->gather.open ? 1u : 0u;
  k.gather_rank = h->gather.rank;
  k.gather_slot_words = h->gather.slot_words;
  k.gather_base = h->gather.base;
  k.d = *d;
  if (ground) k.g = *ground;
  if (ground && h->plane_on) {
    k.plane_on = 1;
    k.plane = h->plane;
  }
  return k;
}

cp_status cp_batch_run(cp_handle* h, const cp_detect_params* d, const cp_ground_params* ground) try {
  if (!h) return CP_E_PARAM;
  h->tracked = false;
  h->ground_out = false;
  CK(cudaSetDevice(h->cfg.device));
  const bool eligible = h->use_graph && d && h->batch_ready && !h->taps && !h->stage_timing && h->hg.uniform_n != 0;
  if (!eligible) {
    h->key_valid = false;
    return enqueue_pipeline(h, d, ground);
  }
  const RunKey key = make_key(h, d, ground);
  static_assert(sizeof(RunKey) <= sizeof(h->last_key), "RunKey storage too small");
  const bool same = h->key_valid && memcmp(&key, h->last_key, sizeof(RunKey)) == 0;
  memcpy(h->last_key, &key, sizeof(RunKey));
  h->key_valid = true;
  if (same && h->graph_exec && h->graph_key_valid && memcmp(&key, h->graph_key, sizeof(RunKey)) == 0) {
    if (h->gather.open) h->gather.seq++;
    if (!h->graph_self_published) cudaEventRecord(h->ev0, h->stream);
    CK(cudaGraphLaunch(h->graph_exec, h->stream));
    if (!h->graph_self_published) cudaEventRecord(h->ev1, h->stream);
    // the host state the enqueue set, for cp_sync's back-half retry, the taps and the colour calls
    h->plane_run = h->graph_plane_run;
    h->run_in = h->plane_run ? h->d_out32 : h->in_ptr;
    h->run_layout = h->plane_run ? make_layout(32, 0, 4, 8, 16) : h->layout;
    if (h->plane_run) {
      h->plane_valid = true;
      h->plane_frames = h->hg.n_frames;
      h->plane_h = h->plane.n_hypotheses;
    } else {
      h->plane_valid = false;
    }
    h->launches = h->graph_launches;
    h->gathered = false;
    h->self_published = h->graph_self_published;
    h->fetched = h->graph_self_published;   // a single-frame run stores its results into the pinned mirrors itself
    h->ran = true;
    return CP_OK;
  }
  if (!same) return enqueue_pipeline(h, d, ground);  // first sighting: run directly (also warms one-time setup)
  // second identical run: capture it, instantiate, launch
  if (h->graph_exec) {
    cudaGraphExecDestroy(h->graph_exec);
    h->graph_exec = nullptr;
    h->graph_key_valid = false;
  }
  CK(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
  h->capturing = true;
  cp_status st = enqueue_pipeline(h, d, ground);
  h->capturing = false;
  cudaGraph_t graph = nullptr;
  cudaError_t ce = cudaStreamEndCapture(h->stream, &graph);
  if (st != CP_OK || ce != cudaSuccess || !graph) {
    if (graph) cudaGraphDestroy(graph);
    cudaGetLastError();
    h->use_graph = false;  // capture is not possible here: stay on direct launches
    if (h->gather.open && st == CP_OK) h->gather.seq--;  // the captured (never executed) run was counted
    return st != CP_OK ? st : enqueue_pipeline(h, d, ground);
  }
  ce = cudaGraphInstantiate(&h->graph_exec, graph, 0);
  cudaGraphDestroy(graph);
  if (ce != cudaSuccess) {
    cudaGetLastError();
    h->graph_exec = nullptr;
    h->use_graph = false;
    if (h->gather.open) h->gather.seq--;
    return enqueue_pipeline(h, d, ground);
  }
  memcpy(h->graph_key, &key, sizeof(RunKey));
  h->graph_key_valid = true;
  h->graph_launches = h->launches;
  h->graph_self_published = h->self_published;
  h->graph_plane_run = h->plane_run;
  if (!h->self_published) cudaEventRecord(h->ev0, h->stream);
  CK(cudaGraphLaunch(h->graph_exec, h->stream));
  if (!h->self_published) cudaEventRecord(h->ev1, h->stream);
  h->ran = true;
  return CP_OK;
} catch (...) {
  return abi_exception(h);
}

cp_status cp_sync(cp_handle* h) try {
  if (!h) return CP_E_PARAM;
  CK(cudaSetDevice(h->cfg.device));  // it may launch (result publish, back-half retry): be on the handle's device
  if (h->ran && !h->fetched) {
    cp_status sf = enqueue_result_fetch(h);
    if (sf) return sf;
  }
  CK(cudaStreamSynchronize(h->stream));
  CK(cudaGetLastError());
  if (!h->ran) return CP_OK;
  if (h->h_ctl->n_surv) h->hint_c = h->h_ctl->n_surv;   // (the per-frame back half leaves these at zero)
  if (h->h_ctl->n_vox) h->hint_v = h->h_ctl->n_vox;
  // the shared-memory back half reports frames it could not hold: pick the next variant
  // (bigger shared-memory budget, then the general global-memory path) and redo the back half
  while (h->back_mode < 3 && h->h_ctl->fast_overflow != 0 && !(h->h_ctl->error & kErrSurvivors)) {
    const u32 mc = h->h_ctl->fast_max_c, mv = h->h_ctl->fast_max_v;
    int next = 3;
    if (h->back_mode < 1 && mc <= 2048 && mv <= 1024) next = 1;
    else if (h->back_mode < 2 && mc <= 4096 && mv <= 2048) next = 2;
    h->back_mode = next;
    cp_status st;
    if (h->self_published) {
      // the one-launch path skips the resets the other back halves rely on (look-back descriptors, tickets):
      // the frame is run again through the multi-launch path, which the handle then keeps for this budget
      const bool saved = h->use_single;
      const cp_detect_params dd = h->rp.d;
      const cp_ground_params gg = h->rp_ground;
      h->use_single = false;
      st = enqueue_pipeline(h, &dd, h->rp_has_ground ? &gg : nullptr);
      h->use_single = saved;
    } else {
      st = enqueue_back(h, true);
    }
    if (st) return st;
    st = enqueue_result_fetch(h);
    if (st) return st;
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaGetLastError());
  }
  return device_errors(h);
} catch (...) {
  return abi_exception(h);
}

cp_status cp_batch_results(cp_handle* h, cp_frame_counters* counters, uint32_t* cluster_offsets, cp_cluster* out,
                           uint64_t cap, uint64_t* n_total) try {
  if (!h) return CP_E_PARAM;
  if (!h->ran) {
    h->err = "cp_batch_results before cp_batch_run";
    return CP_E_STATE;
  }
  CK(cudaSetDevice(h->cfg.device));
  cp_status st = cp_sync(h);
  if (st) return st;
  const u32 F = h->hg.n_frames;
  const u64 K = h->h_ctl->n_clusters;
  if (n_total) *n_total = K;
  static_assert(sizeof(cp_frame_counters) == 32, "cp_frame_counters is 8 x u32");
  if (cluster_offsets) memcpy(cluster_offsets, h->h_result, sizeof(u32) * (F + 1));
  if (counters) memcpy(counters, h->h_fc, sizeof(cp_frame_counters) * F);
  if (out) {
    if (K > cap) {
      h->err = "cluster output buffer too small";
      return CP_E_CAPACITY;
    }
    if (K <= h->prefetched) {
      memcpy(out, h->h_result + h->off_words, sizeof(cp_cluster) * K);
    } else {
      CK(cudaMemcpyAsync(out, h->d_clusters, sizeof(cp_cluster) * K, cudaMemcpyDeviceToHost, h->stream));
      CK(cudaStreamSynchronize(h->stream));
    }
  }
  return CP_OK;
} catch (...) {
  return abi_exception(h);
}

cp_status cp_detect_batch(cp_handle* h, const cp_cloud_view* frames, uint32_t n_frames, const cp_detect_params* d,
                          const cp_ground_params* ground, cp_frame_counters* counters, uint32_t* cluster_offsets,
                          cp_cluster* out, uint64_t cap, uint64_t* n_total) try {
  cp_status st = cp_batch_set_host_input(h, frames, n_frames);
  if (st) return st;
  st = cp_batch_run(h, d, ground);
  if (st) return st;
  return cp_batch_results(h, counters, cluster_offsets, out, cap, n_total);
} catch (...) {
  return abi_exception(h);
}

cp_status cp_detect(cp_handle* h, const cp_cloud_view* in, const cp_detect_params* d, const cp_ground_params* ground,
                    cp_cluster* out, uint32_t cap, uint32_t* n_clusters, cp_frame_counters* counters) try {
  if (!h) return CP_E_PARAM;
  if (!n_clusters) {
    h->err = "NULL n_clusters";
    return CP_E_PARAM;
  }
  uint64_t total = 0;
  cp_status st = cp_detect_batch(h, in, 1, d, ground, counters, nullptr, out, cap, &total);
  *n_clusters = (uint32_t)total;
  return st;
} catch (...) {
  return abi_exception(h);
}

namespace {
// The ground node over the staged batch (cp_ground_remove, cp_batch_ground_remove): pass 1 (sector minima), then
// every frame's complete message into d_out32 in one pass (mask_compact_kernel<*, true>).  Enqueued only.
cp_status enqueue_ground(cp_handle* h, const cp_ground_params* g) {
  cp_status st = ensure_out32(h);
  if (st) return st;
  const Geom geo = device_geom(h);
  h->launches = 0;
  h->key_valid = false;   // the run state below is the ground call's: the next run is enqueued, not replayed
  h->plane_run = false;
  h->run_in = h->in_ptr;
  h->run_layout = h->layout;
  launch_init(h, g->default_lowest_point);
  if (h->plane_on) return enqueue_plane_node(h, true);
  h->plane_valid = false;
  const u32 sgrid = grid_for((u64)geo.n_tiles * kStreamThreads, kStreamThreads, h->sms, 8);
  launch_sector_min(h, geo, sgrid);
  h->launches++;
  h->rowmax_valid = h->use_rowskip;
  CropK crop;
  memset(&crop, 0, sizeof(crop));
  GroundK gk;
  gk.do_ground = 1;
  gk.want_count = 1;
  gk.pad_survives = 0;
  launch_mask_compact<true>(h, geo, crop, gk, (u32)h->hg.n_points, h->d_out32);
  return CP_OK;
}

// Only the survivors cross PCIe.  The padding points the node appends (:79: value-initialised PointXYZI, 1.0f at
// offset 12) are the same 32 bytes over and over: the host writes them into the caller's buffer itself — in
// parallel, while the GPU is still working — instead of a device-to-host copy carrying them back (for one frame
// that copy was most of the call).  The survivors are copied over the fill afterwards.
void fill_pad_host(cp_handle* h, uint8_t* out8, size_t out_bytes) {
  if (h->stage_threads > 1 && out_bytes >= kParallelStageMin) {
    if (!h->copy_pool) {
      try {
        h->copy_pool.reset(new CopyPool(h->stage_threads - 1));
      } catch (...) {
        h->stage_threads = 1;
      }
    }
    if (h->copy_pool) {
      std::shared_ptr<CopyPool::Batch> b = h->copy_pool->start(out8, nullptr, out_bytes, kStagePiece, 1, true);
      b->work();
      for (u32 gi = 0; gi < b->n_groups; ++gi)
        while (!b->group_done(gi)) std::this_thread::yield();
      return;
    }
  }
  fill_pad_points(out8, out_bytes);
}
}  // namespace

cp_status cp_ground_remove(cp_handle* h, const cp_cloud_view* in, const cp_ground_params* g, void* out_xyzi32,
                           uint32_t* n_kept, float* low17) try {
  if (!h) return CP_E_PARAM;
  if (!g || !out_xyzi32) {
    h->err = "NULL ground params or output";
    return CP_E_PARAM;
  }
  if (low17 && h->plane_on) {
    h->err = "low17 (sector minima) requested under the plane ground model";
    return CP_E_PARAM;
  }
  cp_status st = cp_batch_set_host_input(h, in, 1);
  if (st) return st;
  const u32 n = h->hg.frame_n[0];
  st = enqueue_ground(h, g);
  if (st) return st;
  CK(cudaMemcpyAsync(h->h_ctl, h->d_ctl, sizeof(Ctl), cudaMemcpyDeviceToHost, h->stream));
  if (h->plane_on) CK(cudaMemcpyAsync(&h->h_ctl->n_surv, h->pb.kept, sizeof(u32), cudaMemcpyDeviceToHost, h->stream));
  static_assert(kNSect <= kSectStride, "h_frame_u32 holds at least kSectStride words");
  if (low17) CK(cudaMemcpyAsync(h->h_frame_u32, h->d_low_key, sizeof(u32) * kNSect, cudaMemcpyDeviceToHost, h->stream));
  uint8_t* out8 = static_cast<uint8_t*>(out_xyzi32);
  fill_pad_host(h, out8, (size_t)n * 32);
  CK(cudaStreamSynchronize(h->stream));
  CK(cudaGetLastError());
  const u32 kept = h->h_ctl->n_surv;
  if (kept) {
    CK(cudaMemcpyAsync(out8, h->d_out32, (size_t)std::min(kept, n) * 32, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
  }
  if (n_kept) *n_kept = h->h_ctl->n_surv;
  if (low17)
    for (int s = 0; s < kNSect; ++s) low17[s] = ord2f(h->h_frame_u32[s]);
  h->ran = false;
  return CP_OK;
} catch (...) {
  return abi_exception(h);
}

cp_status cp_batch_ground_remove(cp_handle* h, const cp_ground_params* g, void* out_xyzi32, uint64_t cap_points,
                                 uint32_t* n_kept, float* low17) try {
  if (!h) return CP_E_PARAM;
  h->ground_out = false;   // from here on d_out32 is being rewritten
  if (!g) {
    h->err = "NULL ground params";
    return CP_E_PARAM;
  }
  if (low17 && h->plane_on) {
    h->err = "low17 (sector minima) requested under the plane ground model";
    return CP_E_PARAM;
  }
  if (!h->batch_ready) {
    h->err = "cp_batch_ground_remove before cp_batch_set_device_input / cp_batch_set_host_input";
    return CP_E_STATE;
  }
  const u32 F = h->hg.n_frames;
  const u64 n = h->hg.n_points;
  if (out_xyzi32 && cap_points < n) {
    h->err = "output buffer holds fewer points than the staged batch";
    return CP_E_CAPACITY;
  }
  CK(cudaSetDevice(h->cfg.device));
  if (!h->h_ground) {
    cp_status sa = palloc(h, &h->h_ground, (size_t)h->cfg.max_frames * (1 + kSectStride));
    if (sa) return sa;
  }
  cp_status st = enqueue_ground(h, g);
  if (st) return st;
  h->ran = false;   // the run's intermediate buffers now hold the ground call's
  u32* h_kept = h->h_ground;
  u32* h_low = h->h_ground + F;
  CK(cudaMemcpyAsync(h->h_ctl, h->d_ctl, sizeof(Ctl), cudaMemcpyDeviceToHost, h->stream));   // cp_last_rows_loaded
  CK(cudaMemcpyAsync(h_kept, h->plane_on ? h->pb.kept : h->d_c_off + 1, sizeof(u32) * F, cudaMemcpyDeviceToHost,
                     h->stream));
  if (low17) CK(cudaMemcpyAsync(h_low, h->d_low_key, sizeof(u32) * kSectStride * F, cudaMemcpyDeviceToHost, h->stream));
  uint8_t* out8 = static_cast<uint8_t*>(out_xyzi32);
  if (out8) fill_pad_host(h, out8, (size_t)n * 32);
  CK(cudaStreamSynchronize(h->stream));
  CK(cudaGetLastError());
  if (out8) {
    // frame f's survivors lie at the start of its message; runs of frames that dropped nothing merge into one copy
    u64 lo = 0, hi = 0;   // pending copy [lo, hi) in points
    for (u32 f = 0; f < F; ++f) {
      const u64 p0 = h->hg.frame_off[f];
      if (p0 != hi) {
        if (hi > lo) CK(cudaMemcpyAsync(out8 + lo * 32, h->d_out32 + lo * 32, (hi - lo) * 32, cudaMemcpyDeviceToHost, h->stream));
        lo = p0;
      }
      hi = p0 + h_kept[f];
    }
    if (hi > lo) CK(cudaMemcpyAsync(out8 + lo * 32, h->d_out32 + lo * 32, (hi - lo) * 32, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
  }
  if (n_kept) memcpy(n_kept, h_kept, sizeof(u32) * F);
  if (low17)
    for (u32 f = 0; f < F; ++f)
      for (int s = 0; s < kNSect; ++s) low17[(size_t)f * kNSect + s] = ord2f(h_low[(size_t)f * kSectStride + s]);
  h->ground_points = n;
  h->ground_out = true;
  return CP_OK;
} catch (...) {
  return abi_exception(h);
}

cp_status cp_batch_ground_device_output(cp_handle* h, const void** d_out_xyzi32, uint64_t* n_points) try {
  if (!h) return CP_E_PARAM;
  if (!d_out_xyzi32 || !n_points) {
    h->err = "NULL d_out_xyzi32 or n_points";
    return CP_E_PARAM;
  }
  if (!h->ground_out) {
    h->err = "no cp_batch_ground_remove since the last staging or run";
    return CP_E_STATE;
  }
  *d_out_xyzi32 = h->d_out32;
  *n_points = h->ground_points;
  return CP_OK;
} catch (...) {
  return abi_exception(h);
}

cp_status cp_set_ground_plane(cp_handle* h, const cp_plane_params* p) try {
  if (!h) return CP_E_PARAM;
  if (!p) {
    h->plane_on = false;
    return CP_OK;
  }
  if (p->n_hypotheses < 1 || p->n_hypotheses > kPlaneMaxH || !std::isfinite(p->inlier_distance) ||
      !(p->inlier_distance > 0.0f) || !std::isfinite(p->ground_height) ||
      !(p->max_tilt_deg > 0.0f && p->max_tilt_deg <= 90.0f)) {
    h->err = "plane params: n_hypotheses 1..256, inlier_distance finite and > 0, ground_height finite, "
             "max_tilt_deg in (0, 90]";
    return CP_E_PARAM;
  }
  CK(cudaSetDevice(h->cfg.device));
  cp_status st = ensure_out32(h);
  if (st) return st;
  if (!h->pb.hyp) {
    const size_t F = h->cfg.max_frames;
    if ((st = dalloc(h, &h->pb.hyp, F * kPlaneMaxH))) return st;
    if ((st = dalloc(h, &h->pb.cnt, F * kPlaneMaxH))) return st;
    if ((st = dalloc(h, &h->pb.sel, F))) return st;
    if ((st = dalloc(h, &h->pb.info, 2 * F))) return st;
    if ((st = dalloc(h, &h->pb.tcount, (size_t)std::max<u32>(h->tiles_cap, 1)))) return st;
    if ((st = dalloc(h, &h->pb.kept, F))) return st;
  }
  h->plane = *p;
  h->plane_cos = cos((double)p->max_tilt_deg * (M_PI / 180.0));
  h->plane_on = true;
  return CP_OK;
} catch (...) {
  return abi_exception(h);
}

cp_status cp_ground_planes(cp_handle* h, float* planes, uint32_t* inliers, int32_t* hypothesis, uint32_t cap_frames) try {
  if (!h) return CP_E_PARAM;
  CK(cudaSetDevice(h->cfg.device));
  cp_status st = cp_sync(h);
  if (st) return st;
  if (!h->plane_valid) {
    h->err = "the last run or ground call did not use the plane ground model";
    return CP_E_STATE;
  }
  const u32 F = h->plane_frames;
  if (cap_frames < F) {
    h->err = "cap_frames is smaller than the number of frames";
    return CP_E_CAPACITY;
  }
  std::vector<float4> sel(F);
  std::vector<u32> info(2 * (size_t)F);
  CK(cudaMemcpy(sel.data(), h->pb.sel, sizeof(float4) * F, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(info.data(), h->pb.info, sizeof(u32) * 2 * F, cudaMemcpyDeviceToHost));
  for (u32 f = 0; f < F; ++f) {
    if (planes) {
      planes[4 * f] = sel[f].x;
      planes[4 * f + 1] = sel[f].y;
      planes[4 * f + 2] = sel[f].z;
      planes[4 * f + 3] = sel[f].w;
    }
    if (inliers) inliers[f] = info[2 * f];
    if (hypothesis) hypothesis[f] = (int32_t)info[2 * f + 1];
  }
  return CP_OK;
} catch (...) {
  return abi_exception(h);
}

cp_status cp_last_run_ms(cp_handle* h, float* ms) try {
  if (!h || !ms) return CP_E_PARAM;
  if (!h->ran) {
    h->err = "no batch has run";
    return CP_E_STATE;
  }
  if (h->self_published) {
    h->err = "single-frame runs are one launch and are not bracketed by events; cp_set_stage_timing(h, 1) times them";
    return CP_E_STATE;
  }
  CK(cudaEventSynchronize(h->ev1));
  CK(cudaEventElapsedTime(ms, h->ev0, h->ev1));
  return CP_OK;
} catch (...) {
  return abi_exception(h);
}

cp_status cp_set_stage_timing(cp_handle* h, int on) try {
  if (!h) return CP_E_PARAM;
  h->stage_timing = on != 0;
  return CP_OK;
} catch (...) {
  return abi_exception(h);
}

__global__ void debug_atan2f_kernel(const float* __restrict__ y, const float* __restrict__ x, u32 n, float* __restrict__ out) {
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) out[i] = atan2_exact(y[i], x[i]);
}

cp_status cp_debug_atan2f(cp_handle* h, const float* y, const float* x, uint32_t n, float* out) try {
  if (!h || !y || !x || !out) return CP_E_PARAM;
  if (n == 0) return CP_OK;
  CK(cudaSetDevice(h->cfg.device));
  float* d = nullptr;
  if (cudaMalloc(&d, sizeof(float) * 3 * (size_t)n) != cudaSuccess) {
    cudaGetLastError();
    h->err = "cudaMalloc failed (cp_debug_atan2f)";
    return CP_E_NOMEM;
  }
  cudaMemcpyAsync(d, y, sizeof(float) * n, cudaMemcpyHostToDevice, h->stream);
  cudaMemcpyAsync(d + n, x, sizeof(float) * n, cudaMemcpyHostToDevice, h->stream);
  debug_atan2f_kernel<<<grid_for(n, 256, h->sms, 8), 256, 0, h->stream>>>(d, d + n, n, d + 2 * (size_t)n);
  cudaMemcpyAsync(out, d + 2 * (size_t)n, sizeof(float) * n, cudaMemcpyDeviceToHost, h->stream);
  const cudaError_t e = cudaStreamSynchronize(h->stream);
  cudaFree(d);
  CK(e);
  CK(cudaGetLastError());
  return CP_OK;
} catch (...) {
  return abi_exception(h);
}

cp_status cp_debug_timeline(cp_handle* h, const cp_handle* base, float out_ms[6]) try {
  if (!h || !out_ms) return CP_E_PARAM;
  if (!h->ran || !h->stage_timing || !h->ran_ground || h->ran_fused || h->ran_cluster) {
    h->err = "cp_debug_timeline needs cp_set_stage_timing(1) and a two-kernel run with ground removal";
    return CP_E_STATE;
  }
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaEventSynchronize(h->ev1));
  const cudaEvent_t t0 = base ? base->ev0 : h->ev0;
  if (base) CK(cudaEventSynchronize(base->ev1));
  const cudaEvent_t ev[6] = {h->ev0, h->ev_k[0], h->ev_k[1], h->ev_k[2], h->ev_k[3], h->ev1};
  for (int i = 0; i < 6; ++i) CK(cudaEventElapsedTime(&out_ms[i], t0, ev[i]));
  return CP_OK;
} catch (...) {
  return abi_exception(h);
}

cp_status cp_stage_ms(cp_handle* h, cp_stage stage, float* ms) try {
  if (!h || !ms) return CP_E_PARAM;
  if (!h->ran || !h->stage_timing) {
    h->err = "cp_stage_ms needs cp_set_stage_timing(1) before the run";
    return CP_E_STATE;
  }
  if (stage == CP_STAGE_FRONT_CLUSTER) {
    if (!h->ran_cluster) {
      h->err = "the last run did not use the cluster front kernel";
      return CP_E_STATE;
    }
    CK(cudaEventSynchronize(h->ev_k[1]));
    CK(cudaEventElapsedTime(ms, h->ev_k[0], h->ev_k[1]));
  } else if (stage == CP_STAGE_FRONT_FUSED) {
    if (!h->ran_fused) {
      h->err = "the last run did not use the fused front kernel";
      return CP_E_STATE;
    }
    CK(cudaEventSynchronize(h->ev_k[1]));
    CK(cudaEventElapsedTime(ms, h->ev_k[0], h->ev_k[1]));
  } else if (stage == CP_STAGE_SECTOR_MIN) {
    if (!h->ran_ground || h->ran_fused || h->ran_cluster) {
      h->err = "the last run had no ground removal";
      return CP_E_STATE;
    }
    CK(cudaEventSynchronize(h->ev_k[1]));
    CK(cudaEventElapsedTime(ms, h->ev_k[0], h->ev_k[1]));
  } else if (stage == CP_STAGE_MASK_CROP_COMPACT) {
    if (h->ran_fused || h->ran_cluster) {
      h->err = "the last run used a single-kernel front end";
      return CP_E_STATE;
    }
    if (h->run_fused_mask && !h->masked) {
      h->err = "pass 2 ran inside the per-frame kernel (CP_STAGE_FRAME_BACKEND)";
      return CP_E_STATE;
    }
    CK(cudaEventSynchronize(h->ev_k[3]));
    CK(cudaEventElapsedTime(ms, h->ev_k[2], h->ev_k[3]));
  } else if (stage == CP_STAGE_FRAME_BACKEND) {
    if (!h->ran_frame_kernel) {
      h->err = "the last run used the general back half";
      return CP_E_STATE;
    }
    CK(cudaEventSynchronize(h->ev_k[5]));
    CK(cudaEventElapsedTime(ms, h->ev_k[4], h->ev_k[5]));
  } else {
    h->err = "unknown stage";
    return CP_E_PARAM;
  }
  return CP_OK;
} catch (...) {
  return abi_exception(h);
}

cp_status cp_device_results(cp_handle* h, const void** d_clusters, const uint32_t** d_cluster_offsets,
                            const uint32_t** d_n_clusters) try {
  if (!h) return CP_E_PARAM;
  if (!h->ran) {
    h->err = "cp_device_results before cp_batch_run";
    return CP_E_STATE;
  }
  if (d_clusters) *d_clusters = h->d_clusters;
  if (d_cluster_offsets) *d_cluster_offsets = h->d_k_off;
  if (d_n_clusters) *d_n_clusters = &h->d_ctl->n_clusters;
  return CP_OK;
} catch (...) {
  return abi_exception(h);
}

// the gather slot of a rank is laid out like the handle's own result block: round_up(max_frames + 1, 4) offset
// words, then the records.  A slot that cannot even hold the offsets is a caller error.
static cp_status gather_check(cp_handle* h, uint32_t slot_words) {
  if ((size_t)slot_words < h->off_words + 4) {
    h->err = "slot_words is smaller than round_up(max_frames + 1, 4) + 4: the slot cannot hold the offsets of this handle";
    return CP_E_PARAM;
  }
  // a graph captured before the gather was wired has no publish node
  if (h->graph_exec) {
    cudaGraphExecDestroy(h->graph_exec);
    h->graph_exec = nullptr;
  }
  h->graph_key_valid = false;
  h->key_valid = false;
  return CP_OK;
}

cp_status cp_gather_create(cp_handle* h, uint32_t world, uint32_t slot_words, uint8_t handle_out[64]) try {
  if (!h || !handle_out || world == 0 || slot_words == 0 || slot_words % 4) return CP_E_PARAM;
  CK(cudaSetDevice(h->cfg.device));
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handles are 64 bytes");
  auto& g = h->gather;
  if (g.open) {
    h->err = "gather already configured on this handle";
    return CP_E_STATE;
  }
  if (cp_status gs = gather_check(h, slot_words)) return gs;
  const size_t words = kGatherFlagWords + 2ull * world * slot_words;
  void* p = nullptr;
  CK(cudaMalloc(&p, words * sizeof(u32)));
  h->dev_allocs.push_back(p);
  CK(cudaMemset(p, 0, words * sizeof(u32)));
  cudaIpcMemHandle_t ih;
  CK(cudaIpcGetMemHandle(&ih, p));
  memcpy(handle_out, &ih, 64);
  g.base = static_cast<u32*>(p);
  g.owner = true;
  g.world = world;
  g.rank = 0;
  g.slot_words = slot_words;
  g.seq = 0;
  cp_status st = dalloc(h, &g.d_done, 1);
  if (st) return st;
  CK(cudaMemset(g.d_done, 0, sizeof(u32)));
  st = dalloc(h, &g.d_seq, 1);
  if (st) return st;
  CK(cudaMemset(g.d_seq, 0, sizeof(u32)));
  st = palloc(h, &g.h_flags, kGatherFlagWords);
  if (st) return st;
  g.open = true;
  return CP_OK;
} catch (...) {
  return abi_exception(h);
}

cp_status cp_gather_open(cp_handle* h, const uint8_t handle[64], uint32_t rank, uint32_t world, uint32_t slot_words) try {
  if (!h || !handle || rank == 0 || rank >= world || slot_words == 0 || slot_words % 4) return CP_E_PARAM;
  CK(cudaSetDevice(h->cfg.device));
  auto& g = h->gather;
  if (g.open) {
    h->err = "gather already configured on this handle";
    return CP_E_STATE;
  }
  if (cp_status gs = gather_check(h, slot_words)) return gs;
  cudaIpcMemHandle_t ih;
  memcpy(&ih, handle, 64);
  void* p = nullptr;
  CK(cudaIpcOpenMemHandle(&p, ih, cudaIpcMemLazyEnablePeerAccess));
  g.base = static_cast<u32*>(p);
  g.owner = false;
  g.world = world;
  g.rank = rank;
  g.slot_words = slot_words;
  g.seq = 0;
  cp_status st = dalloc(h, &g.d_done, 1);
  if (st) return st;
  CK(cudaMemset(g.d_done, 0, sizeof(u32)));
  st = dalloc(h, &g.d_seq, 1);
  if (st) return st;
  CK(cudaMemset(g.d_seq, 0, sizeof(u32)));
  g.open = true;
  return CP_OK;
} catch (...) {
  return abi_exception(h);
}

uint32_t cp_gather_seq(const cp_handle* h) { return h ? h->gather.seq : 0; }

// rows of 32 points the keep-mask pass read in the last synchronised run (others were skipped)
uint64_t cp_last_rows_loaded(const cp_handle* h) { return h ? h->h_ctl->rows_loaded : 0; }
void cp_last_pairs(const cp_handle* h, uint64_t* visited, uint64_t* tested) {
  if (visited) *visited = h ? h->h_ctl->pairs_visited : 0;
  if (tested) *tested = h ? h->h_ctl->pairs_tested : 0;
}

cp_status cp_gather_wait(cp_handle* h, uint32_t seq, uint32_t timeout_ms) try {
  if (!h) return CP_E_PARAM;
  auto& g = h->gather;
  if (!g.open || !g.owner) {
    h->err = "cp_gather_wait is for the handle that created the gather buffer";
    return CP_E_STATE;
  }
  CK(cudaSetDevice(h->cfg.device));
  const u32 parity = seq & 1u;
  for (u32 waited = 0;; ++waited) {
    CK(cudaMemcpy(g.h_flags, g.base, kGatherFlagWords * sizeof(u32), cudaMemcpyDeviceToHost));
    bool all = true;
    for (u32 r = 0; r < g.world; ++r)
      all = all && ((g.h_flags[parity * g.world + r] & ~kGatherOverflowBit) == (seq & ~kGatherOverflowBit));
    if (all) {
      for (u32 r = 0; r < g.world; ++r)
        if (g.h_flags[parity * g.world + r] & kGatherOverflowBit) {
          h->err = "rank " + std::to_string(r) + " published more cones than its gather slot holds";
          return CP_E_CAPACITY;
        }
      return CP_OK;
    }
    if (waited >= timeout_ms * 10) {
      h->err = "timed out waiting for the ranks to publish their cone lists";
      return CP_E_STATE;
    }
    struct timespec ts = {0, 100000};
    nanosleep(&ts, nullptr);
  }
} catch (...) {
  return abi_exception(h);
}

cp_status cp_gather_read(cp_handle* h, uint32_t seq, void* out_host, uint64_t cap_bytes) try {
  if (!h || !out_host) return CP_E_PARAM;
  auto& g = h->gather;
  if (!g.open || !g.owner) {
    h->err = "cp_gather_read is for the handle that created the gather buffer";
    return CP_E_STATE;
  }
  const size_t bytes = (size_t)g.world * g.slot_words * sizeof(u32);
  if (bytes > cap_bytes) {
    h->err = "gather output buffer too small";
    return CP_E_CAPACITY;
  }
  CK(cudaSetDevice(h->cfg.device));
  const u32 parity = seq & 1u;
  CK(cudaMemcpy(out_host, g.base + kGatherFlagWords + (size_t)parity * g.world * g.slot_words, bytes,
                cudaMemcpyDeviceToHost));
  return CP_OK;
} catch (...) {
  return abi_exception(h);
}

uint32_t cp_last_launch_count(const cp_handle* h) { return h ? h->launches : 0; }
void* cp_stream(cp_handle* h) { return h ? (void*)h->stream : nullptr; }

cp_status cp_debug_tap(cp_handle* h, cp_tap which, void* out, uint64_t cap_bytes, uint64_t* count) try {
  if (!h || !out || !count) return CP_E_PARAM;
  CK(cudaSetDevice(h->cfg.device));
  if (which == CP_TAP_PLANE_HYPOTHESES || which == CP_TAP_PLANE_COUNTS) {
    if (!h->plane_valid) {
      h->err = "the last run or ground call did not use the plane ground model";
      return CP_E_STATE;
    }
    cp_status st = cp_sync(h);
    if (st) return st;
    const u64 n = (u64)h->plane_frames * h->plane_h, esz = which == CP_TAP_PLANE_COUNTS ? 4 : 16;
    if (n * esz > cap_bytes) {
      h->err = "tap buffer too small";
      return CP_E_CAPACITY;
    }
    if (n) CK(cudaMemcpy(out, which == CP_TAP_PLANE_COUNTS ? (const void*)h->pb.cnt : (const void*)h->pb.hyp, n * esz,
                         cudaMemcpyDeviceToHost));
    *count = n;
    return CP_OK;
  }
  if (!h->ran) {
    h->err = "cp_debug_tap before a batch ran";
    return CP_E_STATE;
  }
  if (which == CP_TAP_SECTOR_LOW && h->plane_run) {
    h->err = "no sector minima: the last run used the plane ground model";
    return CP_E_STATE;
  }
  cp_status st = cp_sync(h);
  if (st) return st;
  const u32 F = h->hg.n_frames;
  const Ctl& c = *h->h_ctl;
  const void* src = nullptr;
  u64 n = 0, esz = 4;
  bool need_taps = false;
  switch (which) {
    case CP_TAP_SECTOR_LOW: src = h->d_low_key; n = (u64)F * kSectStride; break;
    case CP_TAP_CROP_INDEX: src = h->d_src; n = c.n_surv; break;
    case CP_TAP_CROP_POINTS: src = h->d_pts; n = c.n_surv; esz = 16; break;
    case CP_TAP_CROP_OFFSETS: src = h->d_c_off; n = F + 1; break;
    case CP_TAP_VOXEL_KEYS: src = h->d_tap_keys; n = c.n_surv; need_taps = true; break;
    case CP_TAP_VOXEL_ORDER: src = h->d_tap_order; n = c.n_surv; need_taps = true; break;
    case CP_TAP_VOXEL_CLOUD: src = h->d_vox; n = c.n_vox; esz = 16; break;
    case CP_TAP_VOXEL_OFFSETS: src = h->d_v_off; n = F + 1; break;
    case CP_TAP_LABELS: src = h->d_tap_labels; n = c.n_vox; need_taps = true; break;
    default: h->err = "unknown tap"; return CP_E_PARAM;
  }
  if (need_taps && !h->taps) {
    h->err = "this tap needs CONESGPU_TAPS=1 in the environment when the handle is created";
    return CP_E_STATE;
  }
  if (which == CP_TAP_SECTOR_LOW) {
    // decode the ordered-int minima into floats, 17 per frame
    if ((u64)F * kNSect * 4 > cap_bytes) {
      h->err = "tap buffer too small";
      return CP_E_CAPACITY;
    }
    std::vector<u32> tmp(n);
    CK(cudaMemcpy(tmp.data(), src, n * 4, cudaMemcpyDeviceToHost));
    float* o = static_cast<float*>(out);
    for (u32 f = 0; f < F; ++f)
      for (int s = 0; s < kNSect; ++s) o[f * kNSect + s] = ord2f(tmp[f * kSectStride + s]);
    *count = (u64)F * kNSect;
    return CP_OK;
  }
  if (n * esz > cap_bytes) {
    h->err = "tap buffer too small";
    return CP_E_CAPACITY;
  }
  if (n) CK(cudaMemcpy(out, src, n * esz, cudaMemcpyDeviceToHost));
  *count = n;
  return CP_OK;
} catch (...) {
  return abi_exception(h);
}

cp_status cp_debug_sort(cp_handle* h, uint64_t* keys, uint32_t* vals, uint32_t n, uint32_t bits) try {
  if (!h || !keys || !vals) return CP_E_PARAM;
  if (n > h->cap_v || bits > 64) {
    h->err = "cp_debug_sort: n exceeds max_voxels or bits > 64";
    return CP_E_CAPACITY;
  }
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaMemcpyAsync(h->d_okeys_a, keys, sizeof(u64) * n, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(h->d_ovals_a, vals, sizeof(u32) * n, cudaMemcpyHostToDevice, h->stream));
  Ctl z;
  memset(&z, 0, sizeof(z));
  z.n_comp = n;
  z.osort_bits = bits;
  CK(cudaMemcpyAsync(h->d_ctl, &z, sizeof(z), cudaMemcpyHostToDevice, h->stream));
  SortArgs sa = sort_args(h, true, &h->d_ctl->n_comp, &h->d_ctl->osort_bits);
  radix_sort_enqueue(h->stream, sa, bits, n, h->sms, !h->tile_ctas);
  const bool inb = sorted_in_b(bits);
  CK(cudaMemcpyAsync(keys, inb ? h->d_okeys_b : h->d_okeys_a, sizeof(u64) * n, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(vals, inb ? h->d_ovals_b : h->d_ovals_a, sizeof(u32) * n, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  CK(cudaGetLastError());
  return CP_OK;
} catch (...) {
  return abi_exception(h);
}

// pinned mirror of the colour-path results: [offsets n+1][flags n][images 180 n][first crop points], so that a
// call costs one stream synchronisation
static cp_status color_pin(cp_handle* h, u32 n_centers) {
  cp_handle::ColorBufs& cb = h->color;
  const size_t need = sizeof(u32) * (2 * (size_t)n_centers + 2) + (size_t)n_centers * kImgPix + 16 +
                      sizeof(float4) * kColorPrefetch;
  if (cb.pin && cb.pin_bytes >= need) return CP_OK;
  if (cb.pin) {
    cudaStreamSynchronize(h->stream);
    cudaFreeHost(cb.pin);
    cb.pin = nullptr;
  }
  if (cudaMallocHost(&cb.pin, need) != cudaSuccess) {
    cudaGetLastError();
    h->err = "cudaMallocHost failed (colour path)";
    return CP_E_NOMEM;
  }
  cb.pin_bytes = need;
  return CP_OK;
}
static u32* pin_off(cp_handle* h) { return reinterpret_cast<u32*>(h->color.pin); }
static u32* pin_flags(cp_handle* h, u32 n) { return pin_off(h) + n + 1; }
static uint8_t* pin_img(cp_handle* h, u32 n) { return reinterpret_cast<uint8_t*>(pin_flags(h, n) + n); }
static float4* pin_pts(cp_handle* h, u32 n) {
  uintptr_t p = reinterpret_cast<uintptr_t>(pin_img(h, n) + (size_t)n * kImgPix);
  return reinterpret_cast<float4*>((p + 15) & ~(uintptr_t)15);
}

cp_status cp_cone_crops(cp_handle* h, const cp_cloud_view* cloud, uint32_t frame, const cp_cone_center* centers,
                        uint32_t n_centers, float cone_width, uint32_t* crop_offsets, float* crop_xyzi,
                        uint32_t cap_points) try {
  if (!h) return CP_E_PARAM;
  if (!crop_offsets) {
    h->err = "NULL crop_offsets";
    return CP_E_PARAM;
  }
  CK(cudaSetDevice(h->cfg.device));
  bool groundless;
  cp_status st = groundless_crops(h, cloud, &groundless);
  if (st) return st;
  if ((st = color_pin(h, n_centers))) return st;
  st = enqueue_cone_crops(h, cloud, frame, centers, n_centers, cone_width, crop_xyzi ? cap_points : 0, groundless);
  if (st) return st;
  CK(cudaMemcpyAsync(pin_off(h), h->color.off, sizeof(u32) * ((size_t)n_centers + 1), cudaMemcpyDeviceToHost, h->stream));
  // the first crop points ride along speculatively: a typical frame's crops fit, so one synchronisation serves
  const u32 spec = crop_xyzi ? (u32)std::min<size_t>({(size_t)cap_points, (size_t)kColorPrefetch, h->color.pts_n}) : 0u;
  if (spec) CK(cudaMemcpyAsync(pin_pts(h, n_centers), h->color.pts, sizeof(float4) * spec, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  memcpy(crop_offsets, pin_off(h), sizeof(u32) * ((size_t)n_centers + 1));
  const u32 total = crop_offsets[n_centers];
  if (crop_xyzi) {
    if (total > cap_points) {
      h->err = "cone crops hold " + std::to_string(total) + " points, more than cap_points";
      return CP_E_CAPACITY;
    }
    memcpy(crop_xyzi, pin_pts(h, n_centers), sizeof(float4) * std::min(total, spec));
    if (total > spec) {
      CK(cudaMemcpyAsync(crop_xyzi + 4 * (size_t)spec, h->color.pts + spec, sizeof(float4) * (size_t)(total - spec),
                         cudaMemcpyDeviceToHost, h->stream));
      CK(cudaStreamSynchronize(h->stream));
    }
  }
  return CP_OK;
} catch (...) {
  return abi_exception(h);
}

cp_status cp_cone_images(cp_handle* h, const cp_cloud_view* cloud, uint32_t frame, const cp_cone_center* centers,
                         uint32_t n_centers, float cone_width, uint8_t* images, uint32_t* counts, uint32_t* flags) try {
  if (!h) return CP_E_PARAM;
  if (n_centers && !images) {
    h->err = "NULL images";
    return CP_E_PARAM;
  }
  CK(cudaSetDevice(h->cfg.device));
  bool groundless;
  cp_status st = groundless_crops(h, cloud, &groundless);
  if (st) return st;
  if ((st = color_pin(h, n_centers))) return st;
  size_t want = h->color.pts_n;
  for (int attempt = 0; attempt < 2; ++attempt) {
    // the cloud is staged by the first attempt only; a retry (crop buffer too small) reuses it.
    // Crops, raster and the copies go out back to back; the crop total is checked after the one sync.
    st = enqueue_cone_crops(h, attempt == 0 ? cloud : nullptr, attempt == 0 ? frame : (cloud ? 0 : frame), centers,
                            n_centers, cone_width, want, groundless);
    if (st) return st;
    if ((st = enqueue_raster(h, n_centers))) return st;
    CK(cudaMemcpyAsync(pin_off(h), h->color.off, sizeof(u32) * ((size_t)n_centers + 1), cudaMemcpyDeviceToHost, h->stream));
    if (n_centers) {
      CK(cudaMemcpyAsync(pin_flags(h, n_centers), h->color.flags, sizeof(u32) * n_centers, cudaMemcpyDeviceToHost, h->stream));
      CK(cudaMemcpyAsync(pin_img(h, n_centers), h->color.img, (size_t)n_centers * kImgPix, cudaMemcpyDeviceToHost, h->stream));
    }
    CK(cudaStreamSynchronize(h->stream));
    const u32 total = pin_off(h)[n_centers];
    if (total <= h->color.pts_n) break;
    if (total == 0xFFFFFFFFu || attempt == 1) {
      h->err = "cone crops exceed the addressable crop buffer";
      return CP_E_CAPACITY;
    }
    want = total;
  }
  if (n_centers) {
    memcpy(images, pin_img(h, n_centers), (size_t)n_centers * kImgPix);
    if (flags) memcpy(flags, pin_flags(h, n_centers), sizeof(u32) * n_centers);
  }
  if (counts)
    for (u32 c = 0; c < n_centers; ++c) counts[c] = pin_off(h)[c + 1] - pin_off(h)[c];
  return CP_OK;
} catch (...) {
  return abi_exception(h);
}

cp_status cp_rasterize_crops(cp_handle* h, const float* crop_xyzi, const uint32_t* crop_offsets, uint32_t n_crops,
                             uint8_t* images, uint32_t* flags) try {
  if (!h) return CP_E_PARAM;
  if (!crop_offsets || (n_crops && !images)) {
    h->err = "NULL crop_offsets or images";
    return CP_E_PARAM;
  }
  for (u32 c = 0; c < n_crops; ++c)
    if (crop_offsets[c + 1] < crop_offsets[c]) {
      h->err = "crop_offsets must be non-decreasing";
      return CP_E_PARAM;
    }
  const u32 total = crop_offsets[n_crops];
  if (total && !crop_xyzi) {
    h->err = "NULL crop_xyzi";
    return CP_E_PARAM;
  }
  CK(cudaSetDevice(h->cfg.device));
  cp_handle::ColorBufs& cb = h->color;
  cp_status st;
  if ((st = grow(h, &cb.off, &cb.off_n, (size_t)n_crops + 1))) return st;
  if ((st = grow(h, &cb.flags, &cb.flags_n, (size_t)n_crops + 1))) return st;
  if ((st = grow(h, &cb.pts, &cb.pts_n, std::max<size_t>(total, 1u << 16)))) return st;
  CK(cudaMemcpyAsync(cb.off, crop_offsets, sizeof(u32) * ((size_t)n_crops + 1), cudaMemcpyHostToDevice, h->stream));
  if (total) CK(cudaMemcpyAsync(cb.pts, crop_xyzi, sizeof(float4) * (size_t)total, cudaMemcpyHostToDevice, h->stream));
  if ((st = enqueue_raster(h, n_crops))) return st;
  if (n_crops) {
    CK(cudaMemcpyAsync(images, cb.img, (size_t)n_crops * kImgPix, cudaMemcpyDeviceToHost, h->stream));
    if (flags) CK(cudaMemcpyAsync(flags, cb.flags, sizeof(u32) * n_crops, cudaMemcpyDeviceToHost, h->stream));
  }
  CK(cudaStreamSynchronize(h->stream));
  return CP_OK;
} catch (...) {
  return abi_exception(h);
}

cp_status cp_color_net_load(cp_handle* h, const cp_color_net* net) try {
  if (!h) return CP_E_PARAM;
  return load_color_net(h, net);
} catch (...) {
  return abi_exception(h);
}

cp_status cp_color_net_load_tflite(cp_handle* h, const void* data, size_t bytes, float threshold) try {
  if (!h) return CP_E_PARAM;
  if (!data) {
    h->err = "NULL model data";
    return CP_E_PARAM;
  }
  cp_tflite::ColorNetWeights w;
  try {
    w = cp_tflite::read_color_net(static_cast<const uint8_t*>(data), bytes);
  } catch (const cp_tflite::Error& e) {
    h->err = "TFLite model refused: " + e.what;
    return CP_E_PARAM;
  }
  cp_color_net n{};
  n.c1 = w.c1;
  n.c2 = w.c2;
  n.n_classes = w.classes;
  n.conv1_w = w.conv1_w.data();
  n.conv1_b = w.conv1_b.data();
  n.conv2_w = w.conv2_w.data();
  n.conv2_b = w.conv2_b.data();
  n.bn_scale = w.bn_scale.data();
  n.bn_shift = w.bn_shift.data();
  n.dense_w = w.dense_w.data();
  n.dense_b = w.dense_b.data();
  n.threshold = threshold;
  return load_color_net(h, &n);
} catch (...) {
  return abi_exception(h);
}

static cp_status fetch_colors(cp_handle* h, u32 n, uint8_t* colors, float* probs, float* logits, uint32_t* flags) {
  cp_handle::ColorBufs& cb = h->color;
  const u32 NC = cb.net.classes;
  if (n) {
    CK(cudaMemcpyAsync(colors, cb.colors, n, cudaMemcpyDeviceToHost, h->stream));
    if (probs) CK(cudaMemcpyAsync(probs, cb.probs, sizeof(float) * n * NC, cudaMemcpyDeviceToHost, h->stream));
    if (logits) CK(cudaMemcpyAsync(logits, cb.probs + (size_t)n * NC, sizeof(float) * n * NC, cudaMemcpyDeviceToHost, h->stream));
    if (flags) CK(cudaMemcpyAsync(flags, cb.net_flags, sizeof(u32) * n, cudaMemcpyDeviceToHost, h->stream));
  }
  CK(cudaStreamSynchronize(h->stream));
  return CP_OK;
}

cp_status cp_classify_images(cp_handle* h, const uint8_t* images, uint32_t n_images, uint8_t* colors, float* probs,
                             float* logits) try {
  if (!h) return CP_E_PARAM;
  if (n_images && (!images || !colors)) {
    h->err = "NULL images or colors";
    return CP_E_PARAM;
  }
  CK(cudaSetDevice(h->cfg.device));
  cp_handle::ColorBufs& cb = h->color;
  cp_status st = grow(h, &cb.img, &cb.img_n, (size_t)std::max<u32>(n_images, 1) * kImgPix);
  if (st) return st;
  if (n_images) CK(cudaMemcpyAsync(cb.img, images, (size_t)n_images * kImgPix, cudaMemcpyHostToDevice, h->stream));
  h->launches = 0;
  if ((st = enqueue_color_net(h, cb.img, nullptr, n_images))) return st;
  return fetch_colors(h, n_images, colors, probs, logits, nullptr);
} catch (...) {
  return abi_exception(h);
}

cp_status cp_cone_colors(cp_handle* h, const cp_cloud_view* cloud, uint32_t frame, const cp_cone_center* centers,
                         uint32_t n_centers, float cone_width, uint8_t* colors, float* probs, uint32_t* flags) try {
  if (!h) return CP_E_PARAM;
  if (n_centers && !colors) {
    h->err = "NULL colors";
    return CP_E_PARAM;
  }
  if (!h->color.net_loaded) {
    h->err = "no colour net loaded (cp_color_net_load / cp_color_net_load_tflite)";
    return CP_E_STATE;
  }
  CK(cudaSetDevice(h->cfg.device));
  bool groundless;
  cp_status st = groundless_crops(h, cloud, &groundless);
  if (st) return st;
  if ((st = color_pin(h, n_centers))) return st;
  size_t want = h->color.pts_n;
  for (int attempt = 0; attempt < 2; ++attempt) {
    // crops -> range images -> classifier, back to back on the stream; one synchronisation, n_centers bytes back
    st = enqueue_cone_crops(h, attempt == 0 ? cloud : nullptr, attempt == 0 ? frame : (cloud ? 0 : frame), centers,
                            n_centers, cone_width, want, groundless);
    if (st) return st;
    if ((st = enqueue_raster(h, n_centers))) return st;
    if ((st = enqueue_color_net(h, h->color.img, h->color.flags, n_centers))) return st;
    CK(cudaMemcpyAsync(pin_off(h) + n_centers, h->color.off + n_centers, sizeof(u32), cudaMemcpyDeviceToHost, h->stream));
    if ((st = fetch_colors(h, n_centers, colors, probs, nullptr, flags))) return st;
    const u32 total = pin_off(h)[n_centers];
    if (total <= h->color.pts_n) break;
    if (total == 0xFFFFFFFFu || attempt == 1) {
      h->err = "cone crops exceed the addressable crop buffer";
      return CP_E_CAPACITY;
    }
    want = total;
  }
  return CP_OK;
} catch (...) {
  return abi_exception(h);
}

// The colour chain of cp_batch_cone_colors over the K > 0 records of the run.  Colours stay in cb.colors, flags in
// cb.net_flags, and the crop offsets come back to pin_off.  With colors NULL nothing else is copied back
// (cp_batch_track reads the per-cluster answers on the device).
static cp_status batch_colors(cp_handle* h, float cone_width, double extension_length, u32 K, uint8_t* colors,
                              float* probs, uint32_t* flags) {
  cp_status st;
  u32 max_rows = 0;
  // the ground node's messages of the run (cp_set_color_cloud); the caller has synchronised the run
  const bool groundless = h->color_cloud == CP_COLOR_CLOUD_GROUNDLESS && h->rp_has_ground;

  for (u32 n : h->hg.frame_n) max_rows = std::max(max_rows, (n + 31) / 32);
  const u32 row_bits = ceil_log2_host(max_rows);
  const u32 key_bits = ceil_log2_host(K) + row_bits;
  const u32 max_key_bits = ceil_log2_host(std::max<u64>(h->cap_v, K)) + row_bits;
  const double hw = (double)cone_width / 1.5;  // CONE_WIDTH / 1.5: float / double literal
  cp_handle::ColorBufs& cb = h->color;
  if ((st = color_pin(h, K))) return st;
  if ((st = grow(h, &cb.box, &cb.box_n, K))) return st;
  if ((st = grow(h, &cb.kframe, &cb.kframe_n, K))) return st;
  if ((st = grow(h, &cb.cnt, &cb.cnt_n, K))) return st;
  if ((st = grow(h, &cb.tcnt, &cb.tcnt_n, K))) return st;
  if ((st = grow(h, &cb.off, &cb.off_n, (size_t)K + 1))) return st;
  if ((st = grow(h, &cb.toff, &cb.toff_n, (size_t)K + 1))) return st;
  if ((st = grow(h, &cb.flags, &cb.flags_n, (size_t)K + 1))) return st;
  if ((st = grow(h, &cb.bctl, &cb.bctl_n, 4))) return st;
  if ((st = grow(h, &cb.sort_hdr, &cb.sort_hdr_n, kSortHdrWords))) return st;
  size_t want = std::max<size_t>(cb.pts_n, 1u << 16);
  for (int attempt = 0; attempt < 2; ++attempt) {
    if ((st = grow(h, &cb.pts, &cb.pts_n, want))) return st;
    if ((st = grow(h, &cb.keys_a, &cb.keys_a_n, cb.pts_n))) return st;
    if ((st = grow(h, &cb.keys_b, &cb.keys_b_n, cb.pts_n))) return st;
    if ((st = grow(h, &cb.vals_a, &cb.vals_a_n, cb.pts_n))) return st;
    if ((st = grow(h, &cb.vals_b, &cb.vals_b_n, cb.pts_n))) return st;
    if ((st = grow(h, &cb.sort_state, &cb.sort_state_n, 2 * kRadix * (cb.pts_n / kSortTile + 1)))) return st;
    switch (h->layout.mode) {
      case 0: h->launches += enqueue_batch_crops<0>(h, K, extension_length, hw, row_bits, key_bits, max_key_bits, groundless); break;
      case 1: h->launches += enqueue_batch_crops<1>(h, K, extension_length, hw, row_bits, key_bits, max_key_bits, groundless); break;
      default: h->launches += enqueue_batch_crops<2>(h, K, extension_length, hw, row_bits, key_bits, max_key_bits, groundless); break;
    }
    CK(cudaGetLastError());
    if ((st = enqueue_raster(h, K))) return st;
    h->launches += 1;
    if ((st = enqueue_color_net(h, cb.img, cb.flags, K))) return st;
    CK(cudaMemcpyAsync(pin_off(h), cb.off, sizeof(u32) * ((size_t)K + 1), cudaMemcpyDeviceToHost, h->stream));
    if (colors) {
      if ((st = fetch_colors(h, K, colors, probs, nullptr, flags))) return st;
    } else {
      CK(cudaStreamSynchronize(h->stream));
    }
    // every triple holds at least one crop point: crops that fit mean the triples fitted too
    const u32 total = pin_off(h)[K];
    if (total <= cb.pts_n) break;
    if (total == 0xFFFFFFFFu || attempt == 1) {
      h->err = "cone crops exceed the addressable crop buffer";
      return CP_E_CAPACITY;
    }
    want = total;
  }
  return CP_OK;
}

cp_status cp_set_color_cloud(cp_handle* h, int32_t cloud) try {
  if (!h) return CP_E_PARAM;
  if (cloud != CP_COLOR_CLOUD_STAGED && cloud != CP_COLOR_CLOUD_GROUNDLESS) {
    h->err = "cloud must be CP_COLOR_CLOUD_STAGED or CP_COLOR_CLOUD_GROUNDLESS";
    return CP_E_PARAM;
  }
  h->color_cloud = cloud;
  return CP_OK;
} catch (...) {
  return abi_exception(h);
}

cp_status cp_batch_cone_colors(cp_handle* h, float cone_width, double extension_length, uint8_t* colors, float* probs,
                               uint32_t* flags, uint32_t* counts, uint64_t cap) try {
  if (!h) return CP_E_PARAM;
  if (!std::isfinite(extension_length) || !std::isfinite(cone_width) || !(cone_width > 0.0f)) {
    h->err = "extension_length must be finite, cone_width positive and finite";
    return CP_E_PARAM;
  }
  if (!h->ran) {
    h->err = "no run on the staged input (cp_batch_run / cp_detect_batch / cp_detect), or input staged since";
    return CP_E_STATE;
  }
  if (!h->color.net_loaded) {
    h->err = "no colour net loaded (cp_color_net_load / cp_color_net_load_tflite)";
    return CP_E_STATE;
  }
  if (h->plane_run && h->color_cloud == CP_COLOR_CLOUD_GROUNDLESS) {
    h->err = "groundless colour crops re-derive the sector model's verdict: not available after a plane-model run";
    return CP_E_STATE;
  }
  cp_status st = cp_sync(h);  // the final records: cp_sync may re-run the back half
  if (st) return st;
  const u64 K64 = h->h_ctl->n_clusters;
  if (K64 > cap) {
    h->err = "colour outputs hold fewer entries than the run has clusters";
    return CP_E_CAPACITY;
  }
  if (K64 && !colors) {
    h->err = "NULL colors";
    return CP_E_PARAM;
  }
  h->launches = 0;
  if (K64 == 0) return CP_OK;
  const u32 K = (u32)K64;
  if ((st = batch_colors(h, cone_width, extension_length, K, colors, probs, flags))) return st;
  if (counts)
    for (u32 k = 0; k < K; ++k) counts[k] = pin_off(h)[k + 1] - pin_off(h)[k];
  return CP_OK;
} catch (...) {
  return abi_exception(h);
}

// ---- frame sequences (cp_batch_track, track_kernels.cuh) ----------------------------------------------
static_assert(sizeof(cp_tracked_cone) == sizeof(TrackCone), "cp_tracked_cone is TrackCone");
static_assert(sizeof(cp_cluster) == sizeof(ClusterRec), "cp_cluster is ClusterRec");

static cp_status track_check(cp_handle* h, const cp_track_params* t, const uint32_t* seq_offsets, uint32_t n_seqs,
                             u32 n_frames, const uint32_t* cloud_offsets, const uint64_t* n_out) {
  if (!t || !cloud_offsets || !n_out) {
    h->err = "NULL params, cloud_offsets or n_out";
    return CP_E_PARAM;
  }
  if (!std::isfinite(t->cones_matching_dist_theshold) || !std::isfinite(t->cone_position_extension_length) ||
      (t->classify_colors && !(std::isfinite(t->cone_width) && t->cone_width > 0.0f))) {
    h->err = "cones_matching_dist_theshold and cone_position_extension_length must be finite, cone_width positive "
             "and finite when classifying colours";
    return CP_E_PARAM;
  }
  if (n_seqs == 0 || n_seqs > h->cfg.max_frames || (!seq_offsets && n_seqs != 1)) {
    h->err = "n_seqs must be in [1, max_frames] (1 when seq_offsets is NULL)";
    return CP_E_PARAM;
  }
  if (seq_offsets) {
    bool ok = seq_offsets[0] == 0 && seq_offsets[n_seqs] == n_frames;
    for (u32 s = 0; ok && s < n_seqs; ++s) ok = seq_offsets[s] <= seq_offsets[s + 1];
    if (!ok) {
      h->err = "seq_offsets must be a non-decreasing partition of [0, n_frames]";
      return CP_E_PARAM;
    }
  }
  return CP_OK;
}

// The tracking kernels over K = k_off[F] records (rec, k_off_d on the device; k_off on the host) and, in colour mode,
// the per-record answers colors_d / flags_d of the service.  The new slot state goes to the other state buffer; the
// handle switches to it only when everything succeeded.
static cp_status track_run(cp_handle* h, const cp_track_params* t, const ClusterRec* rec, const u32* k_off_d,
                           const u32* k_off, u32 F, const uint8_t* colors_d, const u32* flags_d,
                           const uint32_t* seq_offsets, uint32_t n_seqs, cp_tracked_cone* out, uint32_t* cloud_offsets,
                           uint64_t cap, uint64_t* n_out) {
  cp_handle::TrackBufs& tb = h->track;
  const u32 M = h->cfg.max_frames, K = k_off[F];
  const bool classify = t->classify_colors != 0;
  if (tb.st_off.empty()) {
    tb.st_off.assign((size_t)M + 1, 0u);
    tb.st_prev.assign(M, 0u);
  }
  // parameter block: fslot[F] mbase[F+1] seq[n_seqs+1] new_off[M+1] new_src[M] old_off[M+1] old_prev[M]
  const size_t o_fslot = 0, o_mbase = o_fslot + F, o_seq = o_mbase + F + 1, o_noff = o_seq + n_seqs + 1,
               o_nsrc = o_noff + M + 1, o_ooff = o_nsrc + M, o_oprev = o_ooff + M + 1, n_par = o_oprev + M;
  std::vector<u32>& par = tb.par;
  par.assign(n_par, 0u);
  u32* so = par.data() + o_seq;
  for (u32 s = 0; s <= n_seqs; ++s) so[s] = seq_offsets ? seq_offsets[s] : (s ? F : 0u);
  for (u32 f = 0; f < F; ++f) par[o_fslot + f] = kTrackNoIndex;
  for (u32 s = 0; s < n_seqs; ++s)
    if (so[s] < so[s + 1]) par[o_fslot + so[s]] = s;
  u64 words = 0;  // match bit sets: every record of a later frame holds one bit per record of the frame before
  for (u32 f = 0; f < F; ++f) {
    par[o_mbase + f] = (u32)words;
    if (classify && par[o_fslot + f] == kTrackNoIndex)
      words += (u64)(k_off[f + 1] - k_off[f]) * ((k_off[f] - k_off[f - 1] + 31) / 32);
    if (words > 0xFFFFFFFFull) {
      h->err = "match sets of consecutive frames exceed 2^32 words";
      return CP_E_NOMEM;
    }
  }
  par[o_mbase + F] = (u32)words;
  std::vector<u32> new_prev(tb.st_prev);
  u64 total = 0;
  for (u32 s = 0; s < M; ++s) {
    const bool touched = s < n_seqs && so[s] < so[s + 1];
    const u32 last = touched ? so[s + 1] - 1 : 0u;
    par[o_noff + s] = (u32)total;
    par[o_nsrc + s] = touched ? last : kTrackNoIndex;
    total += touched ? k_off[last + 1] - k_off[last] : tb.st_off[s + 1] - tb.st_off[s];
    if (touched) new_prev[s] = 1u;
    if (total > 0xFFFFFFFFull) {
      h->err = "slot state exceeds 2^32 cones";
      return CP_E_NOMEM;
    }
  }
  par[o_noff + M] = (u32)total;
  std::copy(tb.st_off.begin(), tb.st_off.end(), par.begin() + o_ooff);
  std::copy(tb.st_prev.begin(), tb.st_prev.end(), par.begin() + o_oprev);
  const int nxt = 1 - tb.cur;
  cp_status st;
  if ((st = grow(h, &tb.par_d, &tb.par_n, n_par))) return st;
  if ((st = grow(h, &tb.ext, &tb.ext_n, K))) return st;
  if ((st = grow(h, &tb.kframe, &tb.kframe_n, K))) return st;
  if ((st = grow(h, &tb.info, &tb.info_n, K))) return st;
  if ((st = grow(h, &tb.fcol, &tb.fcol_n, K))) return st;
  if ((st = grow(h, &tb.ans, &tb.ans_n, K))) return st;
  if ((st = grow(h, &tb.rank, &tb.rank_n, K))) return st;
  if ((st = grow(h, &tb.out, &tb.out_n, K))) return st;
  if ((st = grow(h, &tb.bits, &tb.bits_n, words))) return st;
  if ((st = grow(h, &tb.cnt, &tb.cnt_n, 4 * (size_t)F))) return st;
  if ((st = grow(h, &tb.coff_d, &tb.coff_n, 4 * (size_t)F + 1))) return st;
  if ((st = grow(h, &tb.st[tb.cur], &tb.st_n[tb.cur], 1))) return st;
  if ((st = grow(h, &tb.st[nxt], &tb.st_n[nxt], total))) return st;
  CK(cudaMemcpyAsync(tb.par_d, par.data(), sizeof(u32) * n_par, cudaMemcpyHostToDevice, h->stream));
  const u32* pd = tb.par_d;
  const u32 grid = std::max<u32>(1, std::min<u32>((K + 255) / 256, (u32)h->sms * 8));
  track_ext_kernel<<<grid, 256, 0, h->stream>>>(rec, k_off_d, F, K, t->cone_position_extension_length, tb.ext,
                                                tb.kframe);
  track_match_kernel<<<grid, 256, 0, h->stream>>>(tb.ext, tb.kframe, k_off_d, K, pd + o_fslot, pd + o_mbase,
                                                  tb.st[tb.cur], pd + o_ooff, pd + o_oprev,
                                                  t->cones_matching_dist_theshold, t->use_points_buffer ? 1u : 0u,
                                                  classify ? 1u : 0u, tb.info, tb.bits);
  track_route_kernel<<<(n_seqs + 7) / 8, 256, 0, h->stream>>>(n_seqs, pd + o_seq, k_off_d, pd + o_mbase, tb.info,
                                                              tb.bits, classify ? 1u : 0u, colors_d, flags_d, tb.fcol,
                                                              tb.rank, tb.ans, tb.cnt);
  track_scan_kernel<<<1, kTrackScanThreads, 0, h->stream>>>(4 * F, tb.cnt, tb.coff_d);
  const u32 egrid = std::max<u32>(1, std::min<u64>((std::max<u64>(K, total) + 255) / 256, (u64)h->sms * 8));
  track_emit_kernel<<<egrid, 256, 0, h->stream>>>(K, tb.ext, tb.kframe, k_off_d, tb.fcol, tb.rank, tb.coff_d,
                                                  tb.out, M, (u32)total, pd + o_noff, pd + o_nsrc, pd + o_ooff,
                                                  tb.st[tb.cur], tb.st[nxt]);
  CK(cudaGetLastError());
  h->launches += 5;
  tb.coff.resize(4 * (size_t)F + 1);
  CK(cudaMemcpyAsync(tb.coff.data(), tb.coff_d, sizeof(u32) * tb.coff.size(), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  const u32 n = tb.coff[4 * (size_t)F];
  *n_out = n;
  if (n > cap) {
    h->err = "the published cones do not fit the output (cap < n_out)";
    return CP_E_CAPACITY;
  }
  if (n && !out) {
    h->err = "NULL out";
    return CP_E_PARAM;
  }
  if (n) {
    CK(cudaMemcpyAsync(out, tb.out, sizeof(TrackCone) * n, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
  }
  memcpy(cloud_offsets, tb.coff.data(), sizeof(u32) * tb.coff.size());
  tb.cur = nxt;
  tb.st_off.assign(par.begin() + o_noff, par.begin() + o_noff + M + 1);
  tb.st_prev.swap(new_prev);
  return CP_OK;
}

cp_status cp_batch_track(cp_handle* h, const cp_track_params* t, const uint32_t* seq_offsets, uint32_t n_seqs,
                         cp_tracked_cone* out, uint32_t* cloud_offsets, uint64_t cap, uint64_t* n_out) try {
  if (!h) return CP_E_PARAM;
  cp_status st = track_check(h, t, seq_offsets, n_seqs, h->ran ? h->hg.n_frames : 0u, cloud_offsets, n_out);
  if (st) return st;
  if (!h->ran) {
    h->err = "no run on the staged input (cp_batch_run / cp_detect_batch / cp_detect), or input staged since";
    return CP_E_STATE;
  }
  if (t->classify_colors && !h->color.net_loaded) {
    h->err = "no colour net loaded (cp_color_net_load / cp_color_net_load_tflite)";
    return CP_E_STATE;
  }
  if (t->classify_colors && h->plane_run && h->color_cloud == CP_COLOR_CLOUD_GROUNDLESS) {
    h->err = "groundless colour crops re-derive the sector model's verdict: not available after a plane-model run";
    return CP_E_STATE;
  }
  CK(cudaSetDevice(h->cfg.device));
  if ((st = cp_sync(h))) return st;  // the final records: cp_sync may re-run the back half
  if (h->tracked) {
    h->err = "this run's frames have already advanced the slot state (run again to track new frames)";
    return CP_E_STATE;
  }
  const u32 F = h->hg.n_frames;
  const u32* k_off = h->h_result;
  const u32 K = k_off[F];
  h->launches = 0;
  if (t->classify_colors && K)
    if ((st = batch_colors(h, t->cone_width, t->cone_position_extension_length, K, nullptr, nullptr, nullptr)))
      return st;
  st = track_run(h, t, h->d_clusters, h->d_k_off, k_off, F, h->color.colors, h->color.net_flags, seq_offsets, n_seqs,
                 out, cloud_offsets, cap, n_out);
  if (st == CP_OK) h->tracked = true;
  return st;
} catch (...) {
  return abi_exception(h);
}

cp_status cp_track_reset(cp_handle* h) try {
  if (!h) return CP_E_PARAM;
  h->track.st_off.assign((size_t)h->cfg.max_frames + 1, 0u);
  h->track.st_prev.assign(h->cfg.max_frames, 0u);
  return CP_OK;
} catch (...) {
  return abi_exception(h);
}

cp_status cp_debug_track(cp_handle* h, const cp_track_params* t, const cp_cluster* records,
                         const uint32_t* record_offsets, uint32_t n_frames, const uint8_t* colors,
                         const uint32_t* flags, const uint32_t* seq_offsets, uint32_t n_seqs, cp_tracked_cone* out,
                         uint32_t* cloud_offsets, uint64_t cap, uint64_t* n_out) try {
  if (!h) return CP_E_PARAM;
  cp_status st = track_check(h, t, seq_offsets, n_seqs, n_frames, cloud_offsets, n_out);
  if (st) return st;
  bool ok = record_offsets && record_offsets[0] == 0;
  for (u32 f = 0; ok && f < n_frames; ++f) ok = record_offsets[f] <= record_offsets[f + 1];
  const u32 K = ok ? record_offsets[n_frames] : 0u;
  if (!ok || (K && !records) || (t->classify_colors && K && (!colors || !flags))) {
    h->err = "record_offsets must be a non-decreasing partition starting at 0; records, colors and flags non-NULL";
    return CP_E_PARAM;
  }
  CK(cudaSetDevice(h->cfg.device));
  cp_handle::TrackBufs& tb = h->track;
  if ((st = grow(h, &tb.rec, &tb.rec_n, K))) return st;
  if ((st = grow(h, &tb.rec_off, &tb.rec_off_n, (size_t)n_frames + 1))) return st;
  if ((st = grow(h, &tb.colors, &tb.colors_n, K))) return st;
  if ((st = grow(h, &tb.flags, &tb.flags_n, K))) return st;
  CK(cudaMemcpyAsync(tb.rec_off, record_offsets, sizeof(u32) * ((size_t)n_frames + 1), cudaMemcpyHostToDevice,
                     h->stream));
  if (K) CK(cudaMemcpyAsync(tb.rec, records, sizeof(cp_cluster) * K, cudaMemcpyHostToDevice, h->stream));
  if (K && t->classify_colors) {
    CK(cudaMemcpyAsync(tb.colors, colors, K, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(tb.flags, flags, sizeof(u32) * K, cudaMemcpyHostToDevice, h->stream));
  }
  h->launches = 0;
  return track_run(h, t, tb.rec, tb.rec_off, record_offsets, n_frames, tb.colors, tb.flags, seq_offsets, n_seqs, out,
                   cloud_offsets, cap, n_out);
} catch (...) {
  return abi_exception(h);
}

}  // extern "C"
