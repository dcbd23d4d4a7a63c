// ellc_sequence.cu -- the pose chain of ellc_track_sequence_steps (include/ellc_gn.h): world poses and initial poses between the
// tracking waves, one thread per step, with the pose algebra of ellc_lie.cuh (the host's ellc_concat_* are the same functions, so
// the chain equals the host's bit for bit).
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

}  // namespace ellc
