// track_kernels.cuh — the stateful tail of ConeDetector::get_centroid_clouds (src/cone_detection.cpp:276-340) over
// many frame sequences at once (cp_batch_track): radial extension, temporal gate / points buffer, colour carry-over
// from the previous frame's colour clouds, the colour service's response rules, and the four published clouds.
//
//   track_ext_kernel     extended centre and frame of every record (thread per record)
//   track_match_kernel   gate verdict of every record against the previous frame (or the slot state for the first
//                        frame of a sequence) and, in colour mode, a bit set of the previous frame's records it
//                        matches (thread per record)
//   track_route_kernel   one warp per sequence, frames in order: carry-over from the previous frame's final colours,
//                        the need list, the response rule, per-(frame, cloud) counts and each cone's rank in its cloud
//   track_scan_kernel    cloud offsets (one CTA)
//   track_emit_kernel    scatter of the published cones, and the new slot state (into the second state buffer)
//
// Only the carry-over is sequential (a cone's colour depends on the final colours of the previous frame); every
// distance is evaluated in parallel beforehand.
#pragma once
#include "color_kernels.cuh"

namespace cp {

constexpr u32 kTrackNone = 0xFFu;  // final colour of a cone that is not published
constexpr u32 kTrackNeed = 0xFEu;  // route kernel, between its two passes: the cone waits for a service answer
constexpr u32 kTrackNoIndex = 0xFFFFFFFFu;  // no slot / no source frame
constexpr u32 kTrackScanThreads = 1024;

// cp_tracked_cone; also one entry of a slot's state (cluster unused, color = the cloud it was published in or
// kTrackNone)
struct TrackCone {
  float x, y;
  u32 cluster, color;
};

// (double)euclidan_dist(p, q) < thr, src/perception_handling/utils.cpp:32-34 with z = 0 on both sides (its term
// adds +0.0 to a sum of squares, which changes nothing): float differences, double squares and sum, double sqrt
// narrowed to float, compared in double.  Explicit _rn intrinsics: a contracted FMA would change the bits.
__device__ __forceinline__ bool cones_match(float px, float py, float qx, float qy, double thr) {
  const double dx = (double)__fsub_rn(px, qx), dy = (double)__fsub_rn(py, qy);
  const float d = __double2float_rn(__dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy))));
  return (double)d < thr;
}

// last frame f with k_off[f] <= k (empty frames share their offset with the next)
__device__ __forceinline__ u32 frame_of(const u32* __restrict__ k_off, u32 n_frames, u32 k) {
  u32 lo = 0, hi = n_frames;
  while (hi - lo > 1) {
    const u32 mid = (lo + hi) >> 1;
    if (k_off[mid] <= k) lo = mid; else hi = mid;
  }
  return lo;
}

__global__ void __launch_bounds__(256) track_ext_kernel(const ClusterRec* __restrict__ cl, const u32* __restrict__ k_off,
                                                        u32 n_frames, u32 K, double ext, float2* __restrict__ e,
                                                        u32* __restrict__ kframe) {
  for (u32 k = blockIdx.x * blockDim.x + threadIdx.x; k < K; k += gridDim.x * blockDim.x) {
    float ex, ey;
    extend_center(cl[k].x, cl[k].y, ext, &ex, &ey);
    e[k] = make_float2(ex, ey);
    kframe[k] = frame_of(k_off, n_frames, k);
  }
}

// info[k]: bit 0 = passes the gate (:282-286); bits 1-2 = for the first frame of a sequence, the colour carried from
// the slot state (0: none).  For later frames in colour mode, bits[mbase[f] + (k - k_off[f]) * w + j] holds the
// matches among records k_off[f-1] + 32 j .. (w = words per record of frame f).
// fslot[f]: the slot whose state precedes frame f when f opens a sequence, else kTrackNoIndex.
__global__ void __launch_bounds__(256) track_match_kernel(
    const float2* __restrict__ e, const u32* __restrict__ kframe, const u32* __restrict__ k_off, u32 K,
    const u32* __restrict__ fslot, const u32* __restrict__ mbase, const TrackCone* __restrict__ st,
    const u32* __restrict__ st_off, const u32* __restrict__ st_prev, double thr, u32 buffer, u32 classify,
    uint8_t* __restrict__ info, u32* __restrict__ bits) {
  for (u32 k = blockIdx.x * blockDim.x + threadIdx.x; k < K; k += gridDim.x * blockDim.x) {
    const u32 f = kframe[k], s = fslot[f];
    const float2 p = e[k];
    u32 out = 0;
    if (s != kTrackNoIndex) {
      const u32 q0 = st_off[s], q1 = st_off[s + 1];
      bool gate = st_prev[s] && q1 > q0, any = false;
      u32 carried = 0;
      for (u32 q = q0; q < q1; ++q) {
        const TrackCone c = st[q];
        if (!cones_match(p.x, p.y, c.x, c.y, thr)) continue;
        any = true;
        if (c.color >= 1 && c.color <= 3 && (carried == 0 || c.color < carried)) carried = c.color;
      }
      if (buffer) gate = gate && any;
      out = gate ? 1u | (classify ? carried << 1 : 0u) : 0u;
    } else {
      const u32 q0 = k_off[f - 1], q1 = k_off[f];
      const u32 w = (q1 - q0 + 31) / 32;
      u32* mb = bits + mbase[f] + (size_t)(k - k_off[f]) * w;
      bool any = false;
      for (u32 j = 0; j < w; ++j) {
        u32 word = 0;
        for (u32 b = 0; b < 32 && q0 + 32 * j + b < q1; ++b) {
          const float2 q = e[q0 + 32 * j + b];
          if (cones_match(p.x, p.y, q.x, q.y, thr)) word |= 1u << b;
        }
        any = any || word;
        if (classify) mb[j] = word;
      }
      out = (!buffer || any) && q1 > q0 ? 1u : 0u;
    }
    info[k] = (uint8_t)out;
  }
}

// One warp per sequence.  fcol[k] = final colour (0..3) or kTrackNone, rank[k] = position in its cloud.  A frame's
// final colours are read by the next frame of the same warp after __syncwarp (fcol is not __restrict__: the loads
// must not go through the read-only path).  ans is scratch of K bytes: the service's answers of a frame, packed.
__global__ void __launch_bounds__(256) track_route_kernel(
    u32 n_seqs, const u32* __restrict__ seq_off, const u32* __restrict__ k_off, const u32* __restrict__ mbase,
    const uint8_t* __restrict__ info, const u32* __restrict__ bits, u32 classify, const uint8_t* __restrict__ colors,
    const u32* __restrict__ flags, uint8_t* fcol, u32* __restrict__ rank, uint8_t* ans, u32* __restrict__ cnt) {
  const u32 lane = threadIdx.x & 31;
  const u32 s = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (s >= n_seqs) return;
  const u32 lt = (1u << lane) - 1u;
  const u32 f0 = seq_off[s], f1 = seq_off[s + 1];
  for (u32 f = f0; f < f1; ++f) {
    const u32 kb = k_off[f], ke = k_off[f + 1];
    const u32 qb = f > f0 ? k_off[f - 1] : 0u;
    const u32 w = f > f0 ? (kb - qb + 31) / 32 : 0u;
    u32 n0 = 0, n1 = 0, n2 = 0, n3 = 0;  // cones per cloud so far
    u32 nneed = 0, nans = 0;
    bool bad = false;
    // pass 1: gate, carry-over (:291-306), the need list (:308-312) and the answers the service would return
    for (u32 base = kb; base < ke; base += 32) {
      const u32 k = base + lane;
      const bool valid = k < ke;
      const u32 inf = valid ? info[k] : 0u;
      u32 col = kTrackNone;
      bool need = false;
      if (inf & 1u) {
        if (!classify) {
          col = 0;
        } else {
          u32 carried = inf >> 1;
          if (f > f0) {
            const u32* mb = bits + mbase[f] + (size_t)(k - kb) * w;
            for (u32 j = 0; j < w && carried != 1; ++j) {
              for (u32 word = mb[j]; word; word &= word - 1) {
                const u32 c = fcol[qb + 32 * j + __ffs(word) - 1];
                if (c >= 1 && c <= 3 && (carried == 0 || c < carried)) carried = c;
              }
            }
          }
          if (carried) col = carried;
          else need = true;
        }
      }
      u32 r = 0;
#define CP_TRACK_RANK(c, n)                            \
  {                                                    \
    const u32 bal = __ballot_sync(kFull, col == (c));  \
    if (col == (c)) r = n + __popc(bal & lt);          \
    n += __popc(bal);                                  \
  }
      CP_TRACK_RANK(0u, n0) CP_TRACK_RANK(1u, n1) CP_TRACK_RANK(2u, n2) CP_TRACK_RANK(3u, n3)
      if (classify) {
        const u32 fl = need ? flags[k] : 0u;
        const u32 nb = __ballot_sync(kFull, need);
        const bool answered = need && !(fl & kConeEmpty);  // an empty crop is skipped (color_classifier_server.py:83-84)
        const u32 ab = __ballot_sync(kFull, answered);
        bad = bad || __any_sync(kFull, need && (fl & (kConeBadIndex | kConeBadIntensity)));
        if (need) {
          col = kTrackNeed;
          r = nneed + __popc(nb & lt);
        }
        if (answered) {
          const u32 c = colors[k];
          ans[kb + nans + __popc(ab & lt)] = (uint8_t)(c < 4 ? c : 0u);
        }
        nneed += __popc(nb);
        nans += __popc(ab);
      }
      if (valid) {
        fcol[k] = (uint8_t)col;
        rank[k] = r;
      }
    }
    __syncwarp();
    // pass 2 (:326-333, :352-361): a bad crop fails the call and every needed cone stays unknown; otherwise the
    // answers fill the need list from the front.  Needed cones follow the carried ones of their cloud.
    if (nneed) {
      for (u32 base = kb; base < ke; base += 32) {
        const u32 k = base + lane;
        const bool needed = k < ke && fcol[k] == kTrackNeed;
        u32 col = kTrackNone, r = 0;
        if (needed) {
          const u32 i = rank[k];
          col = !bad && i < nans ? ans[kb + i] : 0u;
        }
        CP_TRACK_RANK(0u, n0) CP_TRACK_RANK(1u, n1) CP_TRACK_RANK(2u, n2) CP_TRACK_RANK(3u, n3)
        if (needed) {
          fcol[k] = (uint8_t)col;
          rank[k] = r;
        }
      }
    }
#undef CP_TRACK_RANK
    if (lane == 0) {
      cnt[4 * f + 0] = n0;
      cnt[4 * f + 1] = n1;
      cnt[4 * f + 2] = n2;
      cnt[4 * f + 3] = n3;
    }
    __syncwarp();
  }
}

// One CTA: out[0..n] = exclusive scan of in[0..n).
__global__ void __launch_bounds__(kTrackScanThreads) track_scan_kernel(u32 n, const u32* __restrict__ in,
                                                                       u32* __restrict__ out) {
  __shared__ u32 wsum[kTrackScanThreads / 32];
  const u32 tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  u32 carry = 0;
  for (u32 base = 0; base < n; base += kTrackScanThreads) {
    const u32 i = base + tid;
    const u32 c = i < n ? in[i] : 0u;
    u32 s = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const u32 a = __shfl_up_sync(kFull, s, d);
      if ((int)lane >= d) s += a;
    }
    if (lane == 31) wsum[warp] = s;
    __syncthreads();
    u32 before = 0, total = 0;
    for (u32 v = 0; v < kTrackScanThreads / 32; ++v) {
      if (v < warp) before += wsum[v];
      total += wsum[v];
    }
    if (i < n) out[i] = carry + before + s - c;
    carry += total;
    __syncthreads();
  }
  if (tid == 0) out[n] = carry;
}

// Grid-stride over the K records (published cones to out[coff[4 f + color] + rank]) and over the new state entries:
// slot s holds new_off[s + 1] - new_off[s] cones, taken from frame new_src[s] of this call (the last frame of
// sequence s) or, for a slot this call leaves alone, from the old state.
__global__ void __launch_bounds__(256) track_emit_kernel(
    u32 K, const float2* __restrict__ e, const u32* __restrict__ kframe, const u32* __restrict__ k_off,
    const uint8_t* __restrict__ fcol, const u32* __restrict__ rank, const u32* __restrict__ coff,
    TrackCone* __restrict__ out, u32 n_slots, u32 n_state, const u32* __restrict__ new_off,
    const u32* __restrict__ new_src, const u32* __restrict__ old_off, const TrackCone* __restrict__ old_st,
    TrackCone* __restrict__ new_st) {
  const u32 stride = gridDim.x * blockDim.x;
  for (u32 k = blockIdx.x * blockDim.x + threadIdx.x; k < K; k += stride) {
    const u32 c = fcol[k];
    if (c < 4) {
      const float2 p = e[k];
      out[coff[4 * kframe[k] + c] + rank[k]] = TrackCone{p.x, p.y, k, c};
    }
  }
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n_state; i += stride) {
    const u32 s = frame_of(new_off, n_slots, i);
    const u32 j = i - new_off[s], src = new_src[s];
    if (src != kTrackNoIndex) {
      const u32 k = k_off[src] + j;
      const float2 p = e[k];
      new_st[i] = TrackCone{p.x, p.y, k, fcol[k]};
    } else {
      new_st[i] = old_st[old_off[s] + j];
    }
  }
}

}  // namespace cp
