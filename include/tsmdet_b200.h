/*
 * tsmdet_b200.h -- C ABI of libtsmdet_b200.so: the B200 (sm_100a) implementation of the
 * PointNet++ set-abstraction ops and rotated IoU / NMS of blindopen/TSM-Det-Pointcloud-.
 *
 * This is the drop-in boundary.  Every entry point takes raw DEVICE pointers, plain
 * ints/floats and a CUDA stream (cudaStream_t passed as void*; NULL = legacy default
 * stream, which is what the reference launches on).  No torch / ATen types.  All
 * functions return 0 on success, a cudaError_t value on a CUDA failure, or one of the
 * TSMDET_ERR_* codes; tsmdet_error_string() explains any of them.  Nothing here calls
 * exit(): the reference's fprintf+exit(-1) error paths (e.g. sampling_gpu.cu:255-259,
 * ball_query.cpp:20-32) become return codes that the Python shims raise as exceptions.
 *
 * Ownership (same as the reference, SURVEY.md 8b): the CALLER allocates every output.
 * Layouts are the reference's: contiguous row-major float32 / int32 tensors.
 *
 * "ref:" comments name the reference interface each function replaces; paths are
 * relative to /root/reference/pcdet/ops/.
 */
#ifndef TSMDET_B200_H_
#define TSMDET_B200_H_

#ifdef __cplusplus
extern "C" {
#endif

#define TSMDET_OK 0
#define TSMDET_ERR_INVALID 1000001  /* bad argument / unsupported size */
#define TSMDET_ERR_WATCHDOG 1000002 /* an in-kernel wait timed out */

const char* tsmdet_version(void);
const char* tsmdet_error_string(int code);
/* Reads and clears the per-device watchdog word (0 = clean). */
int tsmdet_read_status(void);

/* ---------------------------------------------------------------- sampling ----------
 * xyz (B,N,3) f32, temp (B,N) f32 scratch [in: initial min-distance, normally 1e10;
 * out: final min-distance; may be NULL], idxs (B,M) i32 out.
 * ref: pointnet2/pointnet2_batch/src/pointnet2_api.cpp:22,26  farthest_/furthest_point_sampling_wrapper
 *      (sampling.cpp:43-52, 58-67; kernels sampling_gpu.cu:100-260, 588-748) */
int tsmdet_farthest_point_sampling(int b, int n, int m, const float* xyz, float* temp, int* idxs, void* stream);

/* The same sampler with bookkeeping for CHAINED set-abstraction layers (layer l+1 samples the centres layer l
 * picked, pointnet2_backbone-style stacks).  tie_iter (B) i32 and vals (B,M) f32 record, per cloud, the first
 * iteration whose maximum was shared by points with different coordinates and every iteration's winning
 * min-distance.  Passing them as parent_tie / parent_vals (B,parent_m) to the NEXT level's call lets that call
 * return its (provably identical) result without iterating; it falls back to the full algorithm per cloud
 * whenever the record cannot prove it.  idxs are always bit-identical to tsmdet_farthest_point_sampling. */
int tsmdet_fps_chain(int b, int n, int m, const float* xyz, float* temp, int* idxs, int* tie_iter, float* vals,
                     const int* parent_tie, const float* parent_vals, int parent_m, void* stream);

/* weights (B,N) f32.  ref: pointnet2_api.cpp:28 furthest_point_sampling_weights_wrapper
 *      (sampling.cpp:112-122; sampling_gpu.cu:901-1067) */
int tsmdet_furthest_point_sampling_weights(int b, int n, int m, const float* xyz, const float* weights, float* temp,
                                           int* idxs, void* stream);

/* matrix (B,N,N) f32 pairwise distances; temp (B,N) REQUIRED.
 * ref: pointnet2_api.cpp:23,27 furthest_point_sampling_with_dist_wrapper /
 *      furthest_point_sampling_matrix_wrapper (sampling_gpu.cu:262-422, 750-899) */
int tsmdet_furthest_point_sampling_matrix(int b, int n, int m, const float* matrix, float* temp, int* idxs,
                                          void* stream);

/* ref: pointnet2_api.cpp:25 furthest_point_sampling_with_weighted_dist_wrapper (sampling_gpu.cu:424-586) */
int tsmdet_furthest_point_sampling_with_weighted_dist(int b, int n, int m, const float* matrix, const float* weights,
                                                      float* temp, int* idxs, void* stream);

/* Process-wide choice between the two d-FPS kernels (identical results): 0 = auto (by batch size), 1 = one
 * thread-block cluster per cloud (lowest pick latency while clouds <= SMs/8), 2 = one CTA per cloud with exact
 * spatial pruning (one SM per cloud; N <= 16384).  No reference counterpart (the reference has one kernel). */
int tsmdet_fps_configure(int algo);

/* Introspection: the cluster size / block size / points per thread the sampler would use. */
int tsmdet_fps_plan(int b, int n, int* csize, int* threads, int* pts_per_thread, int* smem_xyz);

/* points (B,C,N), idx (B,npoints) -> out (B,C,npoints).
 * ref: pointnet2_api.cpp:20-21 gather_points(_grad)_wrapper (sampling_gpu.cu:15-90) */
int tsmdet_gather_points(int b, int c, int n, int npoints, const float* points, const int* idx, float* out,
                         void* stream);
int tsmdet_gather_points_grad(int b, int c, int n, int npoints, const float* grad_out, const int* idx,
                              float* grad_points, void* stream);
/* xyz (B,N,3), idx (B,M) -> out (B,M,3): the transpose->gather->transpose chain of
 * pointnet2_modules.py:1143,1212-1215 in one pass. */
int tsmdet_gather_xyz(int b, int n, int m, const float* xyz, const int* idx, float* out, void* stream);

/* Input staging (SURVEY.md 8 f4): the collated batch `points (b*n, 4+c)` = [batch_idx, x, y, z, features...], frame
 * after frame with n points each, -> xyz (b,n,3) and features (b,c,n) [NULL when c == 0] in ONE pass; rows whose
 * batch index is not their frame are counted into *bad (device i32, not cleared here; may be NULL).
 * ref: pcdet/models/__init__.py:23-34 load_data_to_gpu; backbones_3d/pointnet2_backbone.py:796-800 break_up_pc,
 *      :814-823 (count check, view, permute.contiguous); pointnet2_batch/pointnet2_modules.py:1143 */
int tsmdet_stage_points(int b, int n, int c, const float* points, float* xyz, float* features, int* bad,
                        void* stream);

/* ---------------------------------------------------------------- ball query --------
 * new_xyz (B,M,3), xyz (B,N,3) -> idx_cnt (B,M) i32, idx (B,M,nsample) i32.
 * ref: pointnet2_api.cpp:11,13 ball_query_wrapper / ball_query_dilated_wrapper
 *      (ball_query.cpp:47-71; ball_query_gpu.cu:75-199) */
int tsmdet_ball_query(int b, int n, int m, float radius, int nsample, const float* new_xyz, const float* xyz,
                      int* idx_cnt, int* idx, void* stream);
int tsmdet_ball_query_dilated(int b, int n, int m, float radius_in, float radius_out, int nsample,
                              const float* new_xyz, const float* xyz, int* idx_cnt, int* idx, void* stream);

/* ---------------------------------------------------------------- grouping ----------
 * points (B,C,N), idx (B,npoints,nsample) -> out (B,C,npoints,nsample).
 * ref: pointnet2_api.cpp:14-15 group_points(_grad)_wrapper (group_points_gpu.cu:14-92) */
int tsmdet_group_points(int b, int c, int n, int npoints, int nsample, const float* points, const int* idx, float* out,
                        void* stream);
int tsmdet_group_points_grad(int b, int c, int n, int npoints, int nsample, const float* grad_out, const int* idx,
                             float* grad_points, void* stream);
/* QueryAndGroup(.Dilated).forward after the query (pointnet2_utils.py:516-530, 554-568) in one
 * pass: xyz (B,N,3), new_xyz (B,M,3), features (B,C,N)|NULL, idx (B,M,S)
 *   -> new_features (B, 3*use_xyz + C, M, S) [may be NULL], grouped_xyz (B,3,M,S) [may be NULL] */
int tsmdet_group_concat(int b, int c, int n, int m, int nsample, int use_xyz, const float* xyz, const float* new_xyz,
                        const float* features, const int* idx, float* new_features, float* grouped_xyz, void* stream);

/* ---------------------------------------------------------------- interpolation -----
 * ref: pointnet2_api.cpp:30-32 three_nn_wrapper / three_interpolate(_grad)_wrapper
 *      (interpolate.cpp; interpolate_gpu.cu:16-168).  dist2 is SQUARED distance, as in the
 *      reference (the Python caller takes the sqrt, pointnet2_utils.py:282). */
int tsmdet_three_nn(int b, int n, int m, const float* unknown, const float* known, float* dist2, int* idx,
                    void* stream);
int tsmdet_three_interpolate(int b, int c, int m, int n, const float* points, const int* idx, const float* weight,
                             float* out, void* stream);
int tsmdet_three_interpolate_grad(int b, int c, int n, int m, const float* grad_out, const int* idx,
                                  const float* weight, float* grad_points, void* stream);

/* ---------------------------------------------------------------- fused SA layer ----
 * Set-abstraction scale of _VoxelPointnetSAModuleFS(Distillation)Base.forward's layer-0
 * branch (pointnet2/pointnet2_batch/pointnet2_modules.py:1259-1268, 1297-1300):
 * group (xyz offsets + features) -> mask empty balls -> up to 3 x [1x1 conv (BN folded) + ReLU]
 * -> max over nsample, without materialising the (B,C,npoint,nsample) tensors.
 *   xyz (B,N,3), new_xyz (B,M,3), features (B,C,N)|NULL, idx (B,M,S) i32, idx_cnt (B,M) i32
 *   w[l]  (cout_l, cin_l) f32 row-major folded weights, bias[l] (cout_l) f32 folded bias
 *   out (B, out_stride_c... ) : written at out[b, out_c0 + co, p] with channel stride M and batch
 *   stride out_ctot*M, so several scales can write into one concatenated tensor.
 * precision: 0 = fp32 FMA (1e-5 parity mode), 1 = bf16 tensor cores (tcgen05 kind::f16), 2 = tf32 tensor cores
 * (tcgen05 kind::tf32: operands rounded to 10 mantissa bits, ~1e-3 relative), fp32 accumulate.  TSMDET_ERR_INVALID
 * in tf32 mode: the MLP's weights do not fit shared memory as 4-byte operands (e.g. [131,128,128,256]). */
int tsmdet_sa_mlp_maxpool(int b, int n, int m, int nsample, int c_feat, int use_xyz, const float* xyz,
                          const float* new_xyz, const float* features, const int* idx, const int* idx_cnt,
                          int num_layers, const int* channels, const float* const* weights,
                          const float* const* biases, float* out, int out_ctot, int out_c0, int precision,
                          void* stream);

/* Point-wise shared MLP over dense tensors, no pooling: out[b, out_c0 + co, i] = MLP(cat(src0[b,:,i], src1[b,:,i]))
 * with [1x1 conv (BN folded) + bias + ReLU] x num_layers.  src0 (B,c0,n), src1 (B,c1,n) | NULL (c1 = 0),
 * channels[0] == c0 + c1, out (B,out_ctot,n).  precision as above.
 * ref: pointnet2_modules.py:171,175-176 (PointnetFPModule: cat + mlp), :1320-1321 (aggregation_mlp) */
int tsmdet_pointwise_mlp(int b, int n, int c0, int c1, const float* src0, const float* src1, int num_layers,
                         const int* channels, const float* const* weights, const float* const* biases, float* out,
                         int out_ctot, int out_c0, int precision, void* stream);

/* Weights that do not change between calls (eval): build the tensor path's weight image (bf16 UMMA core matrices +
 * fp32 biases) ONCE and hand it to the *_packed entry points -- the packing kernel costs as much as a small layer.
 * dense = 0: fused SA scale (c1 ignored), 1: point-wise MLP (nsample / use_xyz ignored).  packed == NULL: only
 * *packed_bytes is set.  TSMDET_ERR_INVALID: the second-generation tensor kernel does not take this shape (nsample
 * not a power of two in 8..128, widths > 256): use the unpacked entry points. */
int tsmdet_mlp_pack(int dense, int nsample, int c_feat, int c1, int use_xyz, int num_layers, const int* channels,
                    const float* const* weights, const float* const* biases, void* packed, long long* packed_bytes,
                    void* stream);
/* features_t (optional): the features as (B,N,round_up(c_feat,8)) bf16 rows (then features may be NULL and no
 * transpose runs); out_t (optional second output): (B,M,round_up(cout,8)) bf16 rows = the next stacked layer's
 * features_t; out may be NULL when out_t is given. */
int tsmdet_sa_mlp_maxpool_packed(int b, int n, int m, int nsample, int c_feat, int use_xyz, const float* xyz,
                                 const float* new_xyz, const float* features, const void* features_t, const int* idx,
                                 const int* idx_cnt, int num_layers, const int* channels, const void* packed, float* out,
                                 void* out_t, int out_ctot, int out_c0, void* stream);
int tsmdet_pointwise_mlp_packed(int b, int n, int c0, int c1, const float* src0, const float* src1, int num_layers,
                                const int* channels, const void* packed, float* out, int out_ctot, int out_c0,
                                void* stream);
/* The same three with the tensor precision spelled out (1 = bf16, 2 = tf32; the un-suffixed forms are precision 1).
 * In tf32 mode the weight image holds tf32 operands and features_t / out_t are fp32 rows of round_up(c, 4) channels. */
int tsmdet_mlp_pack_p(int precision, int dense, int nsample, int c_feat, int c1, int use_xyz, int num_layers,
                      const int* channels, const float* const* weights, const float* const* biases, void* packed,
                      long long* packed_bytes, void* stream);
int tsmdet_sa_mlp_maxpool_packed_p(int precision, int b, int n, int m, int nsample, int c_feat, int use_xyz,
                                   const float* xyz, const float* new_xyz, const float* features, const void* features_t,
                                   const int* idx, const int* idx_cnt, int num_layers, const int* channels,
                                   const void* packed, float* out, void* out_t, int out_ctot, int out_c0, void* stream);
int tsmdet_pointwise_mlp_packed_p(int precision, int b, int n, int c0, int c1, const float* src0, const float* src1,
                                  int num_layers, const int* channels, const void* packed, float* out, int out_ctot,
                                  int out_c0, void* stream);

/* ---------------------------------------------------------------- centroid voxelisation (SURVEY.md 8 f2) ------
 * The tail of the layer-0 branch (pointnet2/pointnet2_batch/pointnet2_modules.py:1323-1355) in one call:
 * voxel indices ((xyz - range_min) / voxel_size truncated, pcdet/utils/voxel_aggregation_utils.py:48-83), the sorted
 * unique voxels with inverse indices and counts (voxel_idxs.unique(dim=0, ...), :145) and the per-voxel means of
 * [b, x, y, z, features] (:152-159), points added in ascending index order (deterministic; bit-equal to the reference
 * functions on the CPU).  new_xyz (B,M,3) f32, features (B,C,M) f32 | NULL; M <= 16384.
 * Outputs (capacity B*M rows; the first *num_unique rows of the last three are valid):
 *   voxel_idxs (B*M,4) i64 [b,z,y,x], unique_idxs (B*M) i64, centroids (.,4+C) f32, centroid_voxel_idxs (.,4) i64,
 *   labels_count (.) i64, num_unique (1) i32 device; err (1) i32 device, bit 0 = a voxel coordinate outside
 *   [-32768, 32767] (may be NULL). */
int tsmdet_voxel_centroids(int b, int m, int c, const float* new_xyz, const float* features, float vx, float vy, float vz,
                           float x0, float y0, float z0, long long* voxel_idxs, float* centroids,
                           long long* centroid_voxel_idxs, long long* labels_count, long long* unique_idxs,
                           int* num_unique, int* err, void* stream);
/* get_centroid_per_voxel (voxel_aggregation_utils.py:132-161) with the reference's own argument layout:
 * points (B*M,4+F) f32 rows [b,x,y,z,f...], voxel_idxs (B*M,4) i64 [b,z,y,x], rows grouped frame after frame with M
 * rows each (err bit 1 otherwise), num_points_in_voxel (B*M) i64 | NULL (weighted means, :147-150). */
int tsmdet_centroid_per_voxel(int b, int m, int f, const float* points, const long long* voxel_idxs,
                              const long long* num_points_in_voxel, float* centroids, long long* centroid_voxel_idxs,
                              long long* labels_count, long long* unique_idxs, int* num_unique, int* err, void* stream);
/* generate_voxel2pinds (pcdet/utils/common_utils.py:248-265): out (B,Z,Y,X) i32 = row number of the voxel in
 * indices ((n,4) i32 [b,z,y,x]), -1 elsewhere.  prev_indices != NULL: out still holds the table of prev_indices and
 * only those n_prev entries are reset (O(voxels)); NULL: the whole table is filled with -1 first. */
int tsmdet_voxel2pinds(int n, const int* indices, int n_prev, const int* prev_indices, int nb, int nz, int ny, int nx,
                       int* out, int* err, void* stream);

/* ---------------------------------------------------------------- pointnet2_stack ops (SURVEY.md 8 f3) ---------
 * ref: pointnet2/pointnet2_stack/src/pointnet2_api.cpp:13-14 voxel_query_wrapper / voxel_query_dilated_wrapper
 *      (voxel_query.cpp:27-75; voxel_query_gpu.cu:10-98, 125-215).  new_xyz (M,3), xyz (N,3), new_coords (M,4) i32
 *      [b,z,y,x], point_indices (B,R1,R2,R3) i32 dense voxel -> point table; idx (M,nsample) i32 ZEROED by the caller,
 *      cnt_unique (M) i32, idx_cnt (M) i32.  Random replacement beyond nsample hits uses cuRAND XORWOW seeded with the
 *      centre's row number, exactly as the reference: results are bit-identical to its kernels. */
int tsmdet_voxel_query(int m, int r1, int r2, int r3, int nsample, float radius, int z_range, int y_range, int x_range,
                       const float* new_xyz, const float* xyz, const int* new_coords, const int* point_indices, int* idx,
                       int* cnt_unique, void* stream);
int tsmdet_voxel_query_dilated(int m, int r1, int r2, int r3, int nsample, float former_radius, float radius, int z_range,
                               int y_range, int x_range, int z_stride, int y_stride, int x_stride, const float* new_xyz,
                               const float* xyz, const int* new_coords, const int* point_indices, int* idx, int* cnt_unique,
                               int* idx_cnt, void* stream);
/* ref: pointnet2_api.cpp:19-20 group_points(_grad)_wrapper (group_points_gpu.cu:14-95): features (N,C) stacked,
 *      idx (M,nsample) frame-local rows, *_batch_cnt (B) i32 on the device -> out (M,C,nsample). */
int tsmdet_stack_group_points(int b, int m, int c, int nsample, const float* features, const int* features_batch_cnt,
                              const int* idx, const int* idx_batch_cnt, float* out, void* stream);
int tsmdet_stack_group_points_grad(int b, int m, int c, int n, int nsample, const float* grad_out, const int* idx,
                                   const int* idx_batch_cnt, const int* features_batch_cnt, float* grad_features,
                                   void* stream);
/* ref: pointnet2_api.cpp:17 stack_farthest_point_sampling_wrapper (sampling_gpu.cu:188-345): xyz (N,3) stacked, temp (N)
 *      pre-filled (1e10; receives the final min-distances), counts (B) i32 on the device, idxs (sum M) GLOBAL rows.
 *      n_total = N.  The reference's block size is 1024 for every cloud, and so is the tie rule here. */
int tsmdet_stack_farthest_point_sampling(int n_total, int batch_size, const float* xyz, float* temp,
                                         const int* xyz_batch_cnt, int* idxs, const int* num_sampled_points, void* stream);
/* ref: pointnet2_api.cpp:15 ball_query_wrapper (ball_query.cpp:25-45; ball_query_gpu.cu:15-62): new_xyz (M,3) and
 *      xyz (N,3) stacked, new_xyz_batch_cnt / xyz_batch_cnt (B) i32 on the device, n_total = N.  idx (M,nsample) i32
 *      ZEROED by the caller receives the first min(hits, nsample) frame-local indices with d2 < radius * radius in
 *      ascending order, the remaining slots repeating the first hit; a centre without hits gets only idx[p,0] = -1.
 *      idx_cnt (M) i32, optional (NULL), receives min(hits, nsample).  global_rows = 1: frame start + index instead,
 *      and all-zero rows for centres without hits (the fused stacked SA scale's input).  No host synchronisation;
 *      TSMDET_BQ_ALGO=brute skips the per-frame grids. */
int tsmdet_stack_ball_query(int b, int m, int n_total, float radius, int nsample, const float* new_xyz,
                            const int* new_xyz_batch_cnt, const float* xyz, const int* xyz_batch_cnt, int* idx,
                            int* idx_cnt, int global_rows, void* stream);
/* Stacked features (N,C) f32 -> the fused SA kernels' feature rows (N,Cp), zero padded: precision 1 = bf16
 * (Cp = round_up(C,8), round to nearest even), 2 = tf32 as f32 bit patterns (Cp = round_up(C,4), round half away) --
 * the rounding the kernels apply to (B,C,N) planes themselves.  Pass the result as features_t of
 * tsmdet_sa_mlp_maxpool_packed_p with B = 1. */
int tsmdet_stack_feature_rows(int precision, int n, int c, const float* features, void* rows, void* stream);
/* Stacked 3-NN, ref pointnet2_stack three_nn_wrapper (interpolate.cpp, interpolate_gpu.cu): unknown (N,3), known (M,3),
 *      unknown_batch_cnt / known_batch_cnt (B) int32 on the device -> dist2 (N,3) f32 squared distances, idx (N,3) int32
 *      GLOBAL known rows.  Row p belongs to the first frame k with p < N0+..+Nk (the search stops at B-1); ties keep the
 *      smaller index; slots a frame with < 3 known points cannot fill are (+inf, the frame's known start).  One uniform
 *      grid per frame (TSMDET_NN_ALGO=brute: none); no host synchronisation. */
int tsmdet_stack_three_nn(int b, int n, int m, const float* unknown, const int* unknown_batch_cnt, const float* known,
                          const int* known_batch_cnt, float* dist2, int* idx, void* stream);
/* ref three_interpolate_wrapper (stack): features (M,C), idx / weight (N,3) -> out (N,C) (planes = 0) or (C,N)
 *      (planes != 0), out = fmaf(w2,f2, fmaf(w0,f0, w1*f1)) per element; an index outside [0,M) reads 0. */
int tsmdet_stack_three_interpolate(int n, int c, int m, const float* features, const int* idx, const float* weight,
                                   float* out, int planes, void* stream);
/* ref three_interpolate_grad_wrapper (stack): grad_out (N,C) -> grad_features (M,C) += g*w (atomic, zeroed by the
 *      caller); indices outside [0,M) are skipped. */
int tsmdet_stack_three_interpolate_grad(int n, int c, int m, const float* grad_out, const int* idx, const float* weight,
                                        float* grad_features, void* stream);
/* Vector pool (csrc/stack_vector_pool.cu; upstream OpenPCDet pointnet2_stack vector_pool_gpu.cu, restated there with
 * what was recalled rather than read).  support_xyz (N,3) and new_xyz (M,3) stacked, xyz_batch_cnt / new_xyz_batch_cnt
 * (B) i32 on the device, n_total = N; centre p belongs to the first frame k with p < M0+..+Mk.  A hit of centre p is a
 * support point of its frame with local = support - centre (fp32 per axis) inside the ball (neighbor_type 1:
 * fmaf(lz,lz, fmaf(lx,lx, ly*ly)) <= D*D) or the cube (otherwise: |l_a| <= D on every axis), D = max_neighbour_distance;
 * hits are taken in ascending index.  One uniform grid per frame (TSMDET_BQ_ALGO=brute: none).
 *
 * query_stacked_local_neighbor_idxs_wrapper_stack: the first L = min(hits, 1000, nsample if > 0) hits of every centre as
 *      GLOBAL rows; start_len (M,2) = (atomicAdd(cumsum, L), L); the list goes to stack_neighbor_idxs[offset..] except
 *      entries at or beyond avg_length_of_neighbor_idxs * M.  *cumsum (device) is not zeroed here: it ends as its old
 *      value plus the exact total of all L. */
int tsmdet_stack_local_neighbor_idxs(int b, int m, int n_total, const float* support_xyz, const int* xyz_batch_cnt,
                                     const float* new_xyz, const int* new_xyz_batch_cnt, int* stack_neighbor_idxs,
                                     int* start_len, int* cumsum, int avg_length_of_neighbor_idxs,
                                     float max_neighbour_distance, int nsample, int neighbor_type, void* stream);
/* query_three_nn_by_stacked_local_idxs_wrapper_stack: for every (p, g), the three nearest (strict-< cascade in list
 *      order, sqdist3) of centre p's list stack_neighbor_idxs[start_len[p,0] ..+ start_len[p,1]] (list_len entries exist;
 *      the rest of a list is ignored) from new_xyz_grid_centers (M,G,3) -> new_xyz_grid_idxs (M,G,3) i32 GLOBAL rows and
 *      new_xyz_grid_dist2 (M,G,3) f32; a slot the list cannot fill is (+inf, -1). */
int tsmdet_stack_three_nn_local(int m, int num_total_grids, int n_total, long long list_len, const float* support_xyz,
                                const float* new_xyz_grid_centers, const int* stack_neighbor_idxs, const int* start_len,
                                int* new_xyz_grid_idxs, float* new_xyz_grid_dist2, void* stream);
/* The two calls above in one, without the list: the same idx / dist2 as the list query (distance D, nsample,
 *      neighbor_type) followed by the list 3-NN, bit for bit; no host synchronisation. */
int tsmdet_stack_vector_three_nn(int b, int m, int n_total, int num_total_grids, const float* support_xyz,
                                 const int* xyz_batch_cnt, const float* new_xyz, const int* new_xyz_batch_cnt,
                                 const float* new_xyz_grid_centers, float max_neighbour_distance, int nsample,
                                 int neighbor_type, int* new_xyz_grid_idxs, float* new_xyz_grid_dist2, void* stream);
/* vector_pool_wrapper: G = num_grid_x*num_grid_y*num_grid_z sub-voxels per centre, cpg = c_out / G; a hit falls in
 *      g = ix*ny*nz + iy*nz + iz (i_a = floorf((l_a + D) / (D*2 / num_grid_a)), fp32), clamped as one index to [0, G-1].
 *      pooling_type 0 (average), per hit in index order: point_cnt_of_grid[p,g] += 1, new_features[p, g*cpg + i % cpg]
 *      += support_features[k,i] (i ascending), new_local_xyz[p, 3g+a] += l_a if use_xyz, one triple (k, p, g) in
 *      grouped_idxs; the hit counts toward nsample.  1 (random choice): only the first hit of each sub-voxel, assigned,
 *      count 1; it stops when (nsample > 0 && taken >= nsample) || taken >= G.  The outputs are added to (and, random
 *      choice, tested on) what the caller put there.  *num_cum_sum (device, zeroed here) = the exact number of triples;
 *      those at or beyond num_max_sum_points are not written.  planes != NULL: no rows, counts or triples; instead
 *      planes (1, G*(3+cpg), M) f32 = channel g*(3+cpg)+c of centre p: (c < 3 ? the local xyz sum c : the feature
 *      sum c-3) / max((float)count, 1e-6f), the module's normalised eval input (use_xyz implied). */
int tsmdet_stack_vector_pool(int b, int m, int n_total, int c_in, int c_out, const float* support_xyz,
                             const int* xyz_batch_cnt, const float* support_features, const float* new_xyz,
                             const int* new_xyz_batch_cnt, float* new_features, float* new_local_xyz,
                             int* point_cnt_of_grid, int* grouped_idxs, int num_grid_x, int num_grid_y, int num_grid_z,
                             float max_neighbour_distance, int use_xyz, long long num_max_sum_points, int nsample,
                             int neighbor_type, int pooling_type, int* num_cum_sum, float* planes, void* stream);
/* vector_pool_grad_wrapper: grad_support_features (N,c_in) (zeroed by the caller) += grad_new_features[p, g*cpg + i%cpg] *
 *      (1 / max(point_cnt_of_grid[p,g], 1)) for every triple (k, p, g) of grouped_idxs (num_triples,3) (atomic). */
int tsmdet_stack_vector_pool_grad(int m, int n, int c_out, int c_in, int num_total_grids, long long num_triples,
                                  const float* grad_new_features, const int* point_cnt_of_grid, const int* grouped_idxs,
                                  float* grad_support_features, void* stream);
/* The local_interpolation eval input: planes (1, G*(C+9), M) f32, channel g*(C+9)+c of centre p for sub-voxel row
 *      r = p*G+g: 0 if idx[r,0] == -1; else c < C: fmaf(w2,f2, fmaf(w0,f0, w1*f1)) (an index outside [0,N) reads 0),
 *      c = C+3s+a: new_xyz_grid_centers[r,a] - support_xyz[idx[r,s], a], a -1 slot reading row N-1. */
int tsmdet_stack_vector_interp_planes(int m, int num_total_grids, int n, int c, const float* support_features,
                                      const float* support_xyz, const float* new_xyz_grid_centers, const int* idx,
                                      const float* weight, float* planes, void* stream);

/* ---------------------------------------------------------------- roiaware_pool3d ----
 * Boxes / RoIs [cx, cy, cz, dx, dy, dz, heading] f32, (cx, cy, cz) the centre; the inside test is restated in
 * csrc/roiaware_pool3d.cu (margin 1e-5 on the GPU, 1e-2 on the CPU; a NaN coordinate is never inside).
 * ref: roiaware_pool3d/src/roiaware_pool3d.cpp (pybind names forward, backward, points_in_boxes_gpu,
 *      points_in_boxes_cpu).  Sizes must be >= 0; every voxel grid dimension in [1, 256]; max_pts_each_voxel >= 1.
 * points_in_boxes_gpu: boxes (B,T,7), pts (B,N,3), box_idx_of_points (B,N) i32 [in: the pre-fill, normally -1;
 *      out: the first box holding the point, the pre-fill where none does]. */
int tsmdet_points_in_boxes(int b, int t, int n, const float* boxes, const float* pts, int* box_idx_of_points,
                           void* stream);
/* points_in_boxes_cpu, HOST memory: boxes (M,7), pts (N,3) -> pts_indices (M,N) i32, 0 / 1 for every pair. */
int tsmdet_points_in_boxes_cpu(int m, int n, const float* boxes, const float* pts, int* pts_indices);
/* RoIAwarePool3d forward: rois (R,7), pts (P,3), pts_feature (P,C) -> pts_idx_of_voxels (R,X,Y,Z,L) i32 (slot 0 the
 *      counter, at most L-1 points in ascending index; every counter written), argmax (R,X,Y,Z,C) i32 (max pool:
 *      written everywhere, -1 for an empty voxel) and pooled_features (R,X,Y,Z,C) f32 (written for non-empty voxels
 *      only: the caller zero-fills).  pool_method 0 max, 1 avg.  No allocation. */
int tsmdet_roiaware_pool3d(int r, int p, int c, int out_x, int out_y, int out_z, int max_pts_each_voxel,
                           const float* rois, const float* pts, const float* pts_feature, int* argmax,
                           int* pts_idx_of_voxels, float* pooled_features, int pool_method, void* stream);
/* RoIAwarePool3d backward: grad_in (P,C) (zeroed by the caller) += grad_out (R,X,Y,Z,C) at argmax (max) or
 *      grad_out * (1 / max(count, 1)) at every listed point (avg); atomic. */
int tsmdet_roiaware_pool3d_grad(int r, int p, int c, int out_x, int out_y, int out_z, int max_pts_each_voxel,
                                const int* pts_idx_of_voxels, const int* argmax, const float* grad_out, float* grad_in,
                                int pool_method, void* stream);

/* ---------------------------------------------------------------- IoU / NMS ---------
 * boxes (N,7) f32 [x,y,z,dx,dy,dz,heading] on the device.
 * ref: iou3d_nms/src/iou3d_nms_api.cpp:12-13 boxes_overlap_bev_gpu / boxes_iou_bev_gpu
 *      (iou3d_nms.cpp:49-88; iou3d_nms_kernel.cu:236-265, 378-398) */
int tsmdet_boxes_overlap_bev(int num_a, const float* boxes_a, int num_b, const float* boxes_b, float* ans_overlap,
                             void* stream);
int tsmdet_boxes_iou_bev(int num_a, const float* boxes_a, int num_b, const float* boxes_b, float* ans_iou,
                         void* stream);

/* HOST memory in and out (the reference keeps this variant on the CPU for its data pipeline).
 * ref: iou3d_nms_api.cpp:16 boxes_iou_bev_cpu (iou3d_cpu.cpp:232-252) */
int tsmdet_boxes_iou_bev_cpu(int num_a, const float* boxes_a, int num_b, const float* boxes_b, float* ans_iou);

/* ref: iou3d_nms_api.cpp:14-15 nms_gpu / nms_normal_gpu (iou3d_nms.cpp:90-186).
 * boxes (n,7) device, score order; keep_host (n) int64 on the HOST (as in the reference);
 * *num_out = number kept.  Synchronises the stream, like the reference. */
int tsmdet_nms_gpu(int n, const float* boxes, float thresh, long long* keep_host, int* num_out, void* stream);
int tsmdet_nms_normal_gpu(int n, const float* boxes, float thresh, long long* keep_host, int* num_out, void* stream);

/* Device-resident, batched over frames (no host round trip):
 * boxes (frames, nmax, box_stride>=7) score-sorted per frame, counts (frames) i32 | NULL,
 * keep (frames, nmax) int64 device out, num_keep (frames) i32 device out. */
int tsmdet_nms_batch(int frames, int nmax, const float* boxes, int box_stride, const int* counts, float thresh,
                     long long* keep, int* num_keep, void* stream);
int tsmdet_nms_normal_batch(int frames, int nmax, const float* boxes, int box_stride, const int* counts, float thresh,
                            long long* keep, int* num_keep, void* stream);

/* Detection gather without a rendezvous, with credit-based flow control (csrc/peer_put.cu).  Every rank owns a ring
 * of `slots` receive buffers, each `world` rows of `slot_stride / world` floats, plus a flag array and an ack array
 * (world int64 words each), all mapped into every peer through CUDA IPC.  Step `step` (1, 2, ...) of this rank:
 *   - stores step-1 into peer_acks[r] for r < world ("this rank has consumed every earlier step": the call is
 *     stream-ordered after the caller's reads of the previous step),
 *   - waits until my_acks[r] >= step - slots for every r (the slot about to be overwritten has been released),
 *   - stores `numel` floats from `src` into rows[r] + ((step-1) % slots) * slot_stride for r < world,
 *   - publishes `step` into flags[r].
 * rows[r] = row `rank` of slot 0 of rank r's ring; flags[r] / peer_acks[r] = word `rank` of rank r's flag / ack array;
 * my_acks = this rank's own ack array; sync2 = two zero-initialised device ints owned by the caller.  src and rows
 * 16-byte aligned.  timeout_ns <= 0: 120 s.  A wait that times out records TSMDET_ERR_WATCHDOG in the status word
 * (tsmdet_read_status) and skips the stores; it never traps.
 * ref: replaces pcdet/utils/common_utils.py:224-245 merge_results_dist (pickle files + barriers). */
int tsmdet_peer_put(const float* src, long long numel, int world, void* const* rows, void* const* flags,
                    void* const* peer_acks, const long long* my_acks, int* sync2, long long step, int slots,
                    long long slot_stride, long long timeout_ns, void* stream);
/* Enables access from the current device to memory on `peer_device` (needed before kernels store into IPC-mapped
 * peer buffers); already-enabled is not an error. */
int tsmdet_enable_peer_access(int peer_device);
/* Consumer side, stream-ordered: returns once this rank's flag words (world of them) have all reached `want`, i.e.
 * every rank's records of step `want` are complete in slot (want-1) % slots.  Times out like tsmdet_peer_put. */
int tsmdet_peer_wait(const long long* flags, int world, long long want, int slots, long long timeout_ns, void* stream);

/* ---------------------------------------------------------------- runtime -----------
 * TSMDET_* tuning knobs are read from the environment once, at first use; this re-reads them. */
int tsmdet_reload_options(void);
/* Stream-ordered scratch pool: bytes in live buffers / in retired (outgrown or evicted) ones; trim frees the
 * retired ones (the caller guarantees no CUDA graph captured before the call is replayed after it). */
int tsmdet_scratch_stats(long long* live_bytes, long long* retired_bytes);
int tsmdet_scratch_trim(void);

#ifdef __cplusplus
}
#endif
#endif /* TSMDET_B200_H_ */
