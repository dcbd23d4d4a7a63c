// ellc_sequence.cu -- the pose chain of ellc_track_sequence_steps (include/ellc_gn.h): world poses and initial poses between the
// tracking waves, one thread per step, with the pose algebra of ellc_lie.cuh (the host's ellc_concat_* are the same functions, so
// the chain equals the host's bit for bit); and the per-keyframe steps of ellc_track_sequence_lc (weights, ring pushes).
#include <algorithm>

#include "ellc_internal.h"
#include "ellc_lie.cuh"

namespace ellc {

// Positions [b, e) of the sorted order are the wave just tracked: world pose = log(exp(pose) exp(world of its keyframe))
// (src/ImageFunc.cpp:305-306).  The keyframe's step lies in an earlier wave, whose world poses an earlier launch stored.
__global__ void __launch_bounds__(64) seq_world_kernel(const ellc_seq_step* __restrict__ steps, const int* __restrict__ order,
                                                       const ellc_result* __restrict__ results, float* __restrict__ world, int b, int e) {
    const int k = b + (int)(blockIdx.x * blockDim.x + threadIdx.x);
    if (k >= e) return;
    const int i = order[k];
    const ellc_seq_step& s = steps[i];
    float w[6];
    concat_relative_f(results[i].pose, s.kf_step < 0 ? s.kf_world : world + 6 * (int64_t)s.kf_step, w);
    for (int j = 0; j < 6; ++j) world[6 * (int64_t)i + j] = w[j];
}

// Positions [b, e) are the next wave: its pair records, init = log(exp(world[prev]) exp(world[kf])^-1) (src/ImageFunc.cpp:97-108).
// Both dependencies lie in earlier waves, whose world poses are stored.
__global__ void __launch_bounds__(64) seq_init_kernel(const ellc_seq_step* __restrict__ steps, const int* __restrict__ order,
                                                      const float* __restrict__ world, ellc_pair* __restrict__ pairs, int b, int e) {
    const int k = b + (int)(blockIdx.x * blockDim.x + threadIdx.x);
    if (k >= e) return;
    const int i = order[k];
    const ellc_seq_step& s = steps[i];
    ellc_pair pr;
    pr.kf_slot = s.kf_slot; pr.frame_slot = s.frame_slot; pr.flags = s.flags;
    concat_origin_f(s.prev_step < 0 ? s.prev_world : world + 6 * (int64_t)s.prev_step,
                    s.kf_step < 0 ? s.kf_world : world + 6 * (int64_t)s.kf_step, pr.init_pose);
    pairs[i] = pr;
}

// 64 threads per CTA: one step is a serial chain of fp32 / double pose algebra, so the steps of a wave are spread over many SMs
int launch_seq_world(cudaStream_t st, const ellc_seq_step* d_steps, const int* d_order, const ellc_result* d_results, float* d_world,
                     int b, int e) {
    if (e <= b) return 0;
    seq_world_kernel<<<(e - b + 63) / 64, 64, 0, st>>>(d_steps, d_order, d_results, d_world, b, e);
    return 1;
}
int launch_seq_init(cudaStream_t st, const ellc_seq_step* d_steps, const int* d_order, const float* d_world, ellc_pair* d_pairs,
                    int b, int e) {
    if (e <= b) return 0;
    seq_init_kernel<<<(e - b + 63) / 64, 64, 0, st>>>(d_steps, d_order, d_world, d_pairs, b, e);
    return 1;
}

// ---- loop-closure mode of a sequence call (ellc_track_sequence_lc) ------------------------------------------------------------------
// Frame list of every listed keyframe: the frame slots of the ELLC_PAIR_SAVE_WEIGHTS steps tracked against it, in step order (for the
// frames of one sequence, their tracking order).  One warp per keyframe walks the step table 32 steps at a time and appends the
// matches in index order (ballot + prefix count), at list_off[k]; count[k] = their number.
__global__ void __launch_bounds__(128) seq_kf_lists_kernel(const ellc_seq_step* __restrict__ steps, int n, const ellc_lc_keyframe* __restrict__ kfs,
                                                           int n_kf, const int* __restrict__ list_off, int* __restrict__ lists, int* __restrict__ count) {
    const int k = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (k >= n_kf) return;
    const int slot = kfs[k].kf_slot;
    int* __restrict__ out = lists + list_off[k];
    int m = 0;
    for (int j0 = 0; j0 < n; j0 += 32) {
        const int j = j0 + lane;
        const bool hit = j < n && steps[j].kf_slot == slot && (steps[j].flags & ELLC_PAIR_SAVE_WEIGHTS) != 0;
        const unsigned bal = __ballot_sync(0xffffffffu, hit);
        if (hit) out[m + __popc(bal & ((1u << lane) - 1u))] = steps[j].frame_slot;
        m += __popc(bal);
    }
    if (lane == 0) count[k] = m;
}

// ellc_accumulate_weights (accumulate_weights_kernel: one __fadd_rn per frame, in list order, zeros where the keyframe's mask is 0)
// followed, for a retired keyframe, by ellc_finalise_weights (finalise_weights_kernel: one __fmul_rn by the reciprocal of the count,
// rounded to float) on the same pixel: both are elementwise and the fp32 value between them is the one the composition stores, so
// the fusion is bit-identical.  Count of a level = the slot's count before the call (prior) + the frames of this call.
__global__ void __launch_bounds__(256) seq_kf_weights_kernel(float* __restrict__ kf_weight, const uint8_t* __restrict__ kf_mask,
                                                             const float* __restrict__ frw_pool, const ellc_lc_keyframe* __restrict__ kfs,
                                                             const int* __restrict__ list_off, const int* __restrict__ lists,
                                                             const int* __restrict__ count, const int* __restrict__ prior, Geometry geo) {
    const int64_t win = geo.win_off[kLevels];
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= win) return;
    const int k = blockIdx.y;
    const int slot = kfs[k].kf_slot, nf = count[k];
    const int* __restrict__ fl = lists + list_off[k];
    float* __restrict__ kf_w = kf_weight + (int64_t)slot * win;
    float w = kf_w[i];
    const bool sel = kf_mask[(int64_t)slot * win + i] != 0;
    for (int f = 0; f < nf; ++f) w = __fadd_rn(w, sel ? frw_pool[(int64_t)fl[f] * win + i] : 0.0f);
    if (kfs[k].retire_before >= 0) {
        int level = 0;
#pragma unroll
        for (int l = 1; l < kLevels; ++l) level += (i >= geo.win_off[l]);
        const int c = prior[kLevels * k + level] + nf;
        if (c > 0) w = __fmul_rn(w, (float)(1.0 / (double)c));
    }
    kf_w[i] = w;
}

__device__ __forceinline__ void seq_kf_world(const ellc_lc_keyframe& kf, const float* __restrict__ world, float w[6]) {
    const float* src = kf.world_step < 0 ? kf.world : world + 6 * (int64_t)kf.world_step;
    for (int j = 0; j < 6; ++j) w[j] = src[j];
}

// pushToArray (src/GlobalOptimize.cpp:151) of every retired keyframe: its ring entry and its query, with the world pose from the
// chain; and the rings after all pushes (position p of ring r: the last push to it in push order, else ring_in's entry).
__global__ void __launch_bounds__(64) seq_ring_push_kernel(const ellc_lc_keyframe* __restrict__ kfs, int n_kf, const float* __restrict__ world,
                                                           const ellc_lc_ring_entry* __restrict__ ring_in, int n_rings, int ring_len,
                                                           ellc_lc_ring_entry* __restrict__ push, ellc_lc_query* __restrict__ queries,
                                                           ellc_lc_ring_entry* __restrict__ ring_out) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n_kf) {
        const ellc_lc_keyframe kf = kfs[t];
        ellc_lc_ring_entry e;
        e.frame_id = kf.frame_id; e.is_valid = 1; e.frame_slot = kf.frame_slot; e.kf_slot = kf.kf_slot;
        seq_kf_world(kf, world, e.pose_world);
        push[t] = e;
        ellc_lc_query q;
        q.current_array_id = kf.current_array_id; q.match_window_beg = kf.match_window_beg; q.match_window_end = kf.match_window_end;
        q.frame_id = kf.frame_id; q.frame_slot = kf.frame_slot; q.stray = kf.stray;
        for (int j = 0; j < 6; ++j) q.pose_world[j] = e.pose_world[j];
        queries[t] = q;
    }
    if (t < n_rings * ring_len) {
        const int r = t / ring_len, pos = t - r * ring_len;
        ellc_lc_ring_entry e = ring_in[t];
        for (int j = 0; j < n_kf; ++j) {
            const ellc_lc_keyframe& kf = kfs[j];
            if (kf.retire_before < 0 || kf.ring != r || kf.ring_pos != pos) continue;
            e.frame_id = kf.frame_id; e.is_valid = 1; e.frame_slot = kf.frame_slot; e.kf_slot = kf.kf_slot;
            seq_kf_world(kf, world, e.pose_world);
        }
        ring_out[t] = e;
    }
}

int launch_seq_kf_lists(cudaStream_t st, const ellc_seq_step* d_steps, int n, const ellc_lc_keyframe* d_kfs, int n_kf, const int* d_list_off,
                        int* d_lists, int* d_count) {
    if (n_kf <= 0) return 0;
    seq_kf_lists_kernel<<<(n_kf + 3) / 4, 128, 0, st>>>(d_steps, n, d_kfs, n_kf, d_list_off, d_lists, d_count);
    return 1;
}
int launch_seq_kf_weights(cudaStream_t st, float* kf_weight, const uint8_t* kf_mask, const float* frw_pool, const ellc_lc_keyframe* d_kfs, int n_kf,
                          const int* d_list_off, const int* d_lists, const int* d_count, const int* d_prior, const Geometry& geo) {
    if (n_kf <= 0) return 0;
    seq_kf_weights_kernel<<<dim3((unsigned)((geo.win_off[kLevels] + 255) / 256), n_kf), 256, 0, st>>>(kf_weight, kf_mask, frw_pool, d_kfs, d_list_off,
                                                                                                      d_lists, d_count, d_prior, geo);
    return 1;
}
int launch_seq_ring_push(cudaStream_t st, const ellc_lc_keyframe* d_kfs, int n_kf, const float* d_world, const ellc_lc_ring_entry* d_ring_in,
                         int n_rings, int ring_len, ellc_lc_ring_entry* d_push, ellc_lc_query* d_queries, ellc_lc_ring_entry* d_ring_out) {
    const int m = std::max(n_kf, n_rings * ring_len);
    if (m <= 0) return 0;
    seq_ring_push_kernel<<<(m + 63) / 64, 64, 0, st>>>(d_kfs, n_kf, d_world, d_ring_in, n_rings, ring_len, d_push, d_queries, d_ring_out);
    return 1;
}

}  // namespace ellc
