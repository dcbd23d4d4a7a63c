// ellc_internal.h -- launch wrappers shared between the translation units of libellc_gn.so (not part of the ABI).
#pragma once

#include "ellc_common.cuh"

namespace ellc {

// ellc_preprocess.cu -- each returns the number of kernels it launched
int launch_pyramid(cudaStream_t st, uint8_t* img_pool, int64_t img_slot_stride, const int* d_slots, int n, const Geometry& geo);
int launch_pack_tex(cudaStream_t st, const uint8_t* img_pool, int64_t img_slot_stride, uint32_t* tex_pool,
                    int64_t tex_slot_stride, const int* d_slots, int n, const Geometry& geo);
int launch_select(cudaStream_t st, const float* depth_pool, const float* var_pool, int64_t win_slot_stride,
                  const uint8_t* img_pool, int64_t img_slot_stride, uint8_t* mask_pool, int* rowcount_pool,
                  int* rowoff_pool, int* count_pool, SelGeo* geo_pool, SelPix* pix_pool, float* ikf_pool, const LevelK* K,
                  const int* d_slots, int n, const Geometry& geo);

// loop-closure gating: normalised 256-bin histograms of the level-0 images of n frame slots (hist_pool: [slot][256]) and the
// per-candidate statistics (ellc_track.cu, next to the pose algebra)
int launch_frame_histograms(cudaStream_t st, const uint8_t* img_pool, int64_t img_slot_stride, const int* d_slots, int n, int n_pixels,
                            float* hist_pool);
// the ring walk of findMatch on the device: compacted, query-major list of passing (loop frame, test frame) pairs as ellc_pair records
int launch_lc_generate(cudaStream_t st, const float* hist_pool, const ellc_lc_ring_entry* d_ring, int ring_len, const ellc_lc_query* d_queries,
                       int n_queries, int min_match_difference, float match_threshold, float max_rel_view_angle, int pair_flags,
                       ellc_pair* d_seg_pairs, ellc_lc_stats* d_seg_stats, int* d_seg_count, ellc_pair* d_pairs, ellc_lc_stats* d_stats,
                       int* d_query_of_pair, int* d_total);
// ellc_track_sequence_lc: the same walk and packing, every listed keyframe k a query on its ring as of its own push (queries = n_kf)
int launch_lc_generate_seq(cudaStream_t st, const float* hist_pool, const ellc_lc_ring_entry* d_ring_in, int ring_len, const ellc_lc_keyframe* d_kfs,
                           int n_kf, const ellc_lc_ring_entry* d_push, const ellc_lc_query* d_queries, int min_match_difference,
                           float match_threshold, float max_rel_view_angle, int pair_flags, ellc_pair* d_seg_pairs, ellc_lc_stats* d_seg_stats,
                           int* d_seg_count, ellc_pair* d_pairs, ellc_lc_stats* d_stats, int* d_query_of_pair, int* d_total);
int launch_lc_gate(cudaStream_t st, const float* hist_pool, const ellc_lc_candidate* d_cand, int n, float match_threshold,
                   float max_rel_view_angle, ellc_lc_stats* d_out);
// keyframe depth / variance pyramids from hypotheses (src/DepthPropagation.cpp:1254-1306, :1637-1719); depth_slot / var_slot are
// the keyframe slot's bases in the win layout; *d_n_valid (pre-zeroed) receives the number of valid hypotheses
int launch_depth_pyramid(cudaStream_t st, const uint8_t* d_valid, const float* d_idepth, const float* d_var_s, float* depth_slot,
                         float* var_slot, uint8_t* d_valid_out, int* d_n_valid, const Geometry& geo);
// keyframe weight pyramid (src/PixelWisePyramid.cpp:546-548, src/Frame.cpp:678-695) and loop-closure records (:561-680, :938)
int launch_accumulate_weights(cudaStream_t st, float* kf_weight_slot, const uint8_t* mask_slot, const float* frw_pool,
                              int64_t win, const int* d_frame_slots, int n);
int launch_finalise_weights(cudaStream_t st, float* kf_weight_slot, const int counts[kLevels], const Geometry& geo);
int launch_lc_prepare(cudaStream_t st, const SelGeo* geo_pool, const SelPix* pix_pool, int64_t rec_slot_stride, const int* count_pool,
                      const uint8_t* img_pool, int64_t img_slot_stride, const float* weight_pool, LcRec* lc_pool, float4* lcf_pool,
                      uint32_t* lcp_pool, float* lc_H, const LevelK* K, const int* d_slots, int n, const Geometry& geo,
                      bool reference = false);   // reference: the hessian as ELLC_ARITH_REFERENCE sums it
// dst (device, 4-byte aligned, capacity rounded up to 4 bytes) <- pinned host memory read by the SMs (no copy engine)
int launch_fill_f32(cudaStream_t st, float* dst, float value, int64_t n);
int launch_pull_host(cudaStream_t st, void* dst, const void* src_host_devptr, size_t bytes);

// ellc_track.cu
// Launches the GN tracking kernel for p.n_pairs pairs with `cluster` CTAs per pair.  Returns kernels launched (1) or a
// negative value on launch-configuration failure (cudaGetLastError carries the reason).
int launch_track(cudaStream_t st, const TrackParams& p, int cluster, int arithmetic);   // arithmetic: ELLC_ARITH_*
// loop-closure (inverse-compositional constant-weight) variant: one CTA per pair, pairs = p.order[0 .. p.n_pairs)
int launch_track_lc(cudaStream_t st, const TrackParams& p, int arithmetic);
// result exchange: thread d adds n_records to *d_counters[d] (system scope)
int launch_xchg_signal(cudaStream_t st, unsigned long long* const* d_counters, int n_dst, unsigned long long n_records);
int launch_xchg_store(cudaStream_t st, unsigned long long* d_counter, unsigned long long value);
// div2_rn_shared (the pixel loop's shared-reciprocal exact division) against __fdiv_rn on n pseudo-random operand triples
int launch_div_selftest(cudaStream_t st, long long n, unsigned long long seed, unsigned long long* d_counts /*[2]*/);
int launch_unzero_selftest(cudaStream_t st, long long n, unsigned long long seed, unsigned long long* d_counts /*[1]*/);
int launch_invert6(cudaStream_t st, const float* d_in /*H36*/, float* d_out /*Hinv36 ok1*/);
// one-warp kernel running K5's LU, deltapose / weightedPose and pose update of the given flavour (ellc_solve_update)
int launch_solve_update(cudaStream_t st, const float* d_in /*H36 b6 pose6 weight6*/, float* d_out /*pose6 delta6 wp1 ok1 rt12 small1*/, int arithmetic);

// ellc_sequence.cu -- pose chain of ellc_track_sequence_steps.  Steps are visited through order[] (sorted position -> step index);
// [b, e) is one wave: seq_world stores the world poses of a tracked wave, seq_init writes the pair records of the next one.
int launch_seq_world(cudaStream_t st, const ellc_seq_step* d_steps, const int* d_order, const ellc_result* d_results, float* d_world,
                     int b, int e);
int launch_seq_init(cudaStream_t st, const ellc_seq_step* d_steps, const int* d_order, const float* d_world, ellc_pair* d_pairs,
                    int b, int e);
// ellc_track_sequence_lc (include/ellc_gn.h): per listed keyframe the frame list of its ELLC_PAIR_SAVE_WEIGHTS steps in step order
// (at d_list_off[k], count d_count[k]), accumulation + finalisation of its weight pyramid (finalised when retired; d_prior: its
// counts before the call, [k][level]), and the ring pushes: entries / queries of the retired keyframes, the rings after the call
int launch_seq_kf_lists(cudaStream_t st, const ellc_seq_step* d_steps, int n, const ellc_lc_keyframe* d_kfs, int n_kf, const int* d_list_off,
                        int* d_lists, int* d_count);
int launch_seq_kf_weights(cudaStream_t st, float* kf_weight, const uint8_t* kf_mask, const float* frw_pool, const ellc_lc_keyframe* d_kfs, int n_kf,
                          const int* d_list_off, const int* d_lists, const int* d_count, const int* d_prior, const Geometry& geo);
int launch_seq_ring_push(cudaStream_t st, const ellc_lc_keyframe* d_kfs, int n_kf, const float* d_world, const ellc_lc_ring_entry* d_ring_in,
                         int n_rings, int ring_len, ellc_lc_ring_entry* d_push, ellc_lc_query* d_queries, ellc_lc_ring_entry* d_ring_out);

// ellc_ingest.cu -- camera frame -> level-0 image (gray, undistortion, resize in one pass)
struct IngestJob { const uint8_t* src; uint8_t* dst; };                 // camera image (device), level-0 image of the slot
struct IngestGeo { int cam_w, cam_h, channels, pitch, out_w, out_h, undistort, pad; };
struct UndistortParams { double ir[9]; double fx, fy, u0, v0, k1, k2, p1, p2, k3; };
// resize taps per output column / row: (source index 0, source index 1, Q11 coefficient 0, coefficient 1)
int build_resize_taps(int cam_w, int cam_h, int out_w, int out_h, int4* cols, int4* rows);
bool invert3(const double a[9], double b[9]);
// map: (2 * out_h) x (2 * out_w) CV_16SC2 entries at the tap positions, (x | y << 16, frac)
int launch_undistort_map(cudaStream_t st, const IngestGeo& g, const UndistortParams& p, const int4* d_cols, const int4* d_rows, uint2* d_map);
int launch_ingest(cudaStream_t st, const IngestJob* d_jobs, int n, const IngestGeo& g, const int4* d_cols, const int4* d_rows, const uint2* d_map);

}  // namespace ellc
