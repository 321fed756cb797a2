/*
 * pn2_api.h — C ABI of libpn2_b200.so: the PointNet++ set-abstraction / feature-propagation
 * geometry ops as hand-written sm_100a CUDA kernels.
 *
 * This is the drop-in boundary for charlesq34/pointnet2's tf_ops/{sampling,grouping,
 * 3d_interpolation}.  Every entry point replaces one of the free "Launcher"/"_cpu" functions the
 * reference's TensorFlow OpKernels call (cited per function, paths relative to the reference
 * root) and keeps that function's scalar/pointer argument order, with a trailing CUDA stream.
 *
 * Conventions (all entry points):
 *   - plain C, no torch/TF types: sizes are `int`, tensors are raw pointers, `stream` is a
 *     cudaStream_t passed as void* (NULL = legacy default stream, as the reference uses).
 *   - device entry points (pn2_*): every pointer is a DEVICE pointer to a dense row-major
 *     float32 / int32 tensor, except the feature pointers of the pn2_*_h entries (`const void*` /
 *     `void*`), which hold 16-bit features of the type their leading `dtype` names.  The library
 *     allocates nothing, frees nothing and never synchronises; launches are asynchronous on `stream`.
 *     Stateless and re-entrant.
 *   - gradients accumulate with float atomics into a buffer the CALLER has zero-filled, exactly
 *     like the reference (tf_sampling.cpp:174, tf_grouping.cpp:204, tf_interpolate.cpp:258).
 *   - return value: 0 on success, otherwise a cudaError_t (argument errors return
 *     cudaErrorInvalidValue = 1).  pn2_error_string() translates.
 *   - limits: every tensor must have fewer than 2^31 elements per batch entry; n, m < 2^31
 *     (totals are indexed with 64 bits: gather / concat / interpolate are tested beyond 2^32 elements);
 *     ops that put the batch on gridDim.y (ball query, three_nn, the row kernels) take b <= 65535.
 *   - the pn2_set_* tuning hooks store one atomic word each: they may be called from any thread at any
 *     time; a launch sees either the old or the new setting, never a mixture.
 */
#ifndef PN2_API_H_
#define PN2_API_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PN2_API_VERSION 2

/* feature element types of the pn2_*_h entry points (coordinates and weights are always float32) */
#define PN2_DTYPE_BF16 1
#define PN2_DTYPE_F16 2

/* ---- sampling (replaces tf_ops/sampling/tf_sampling_g.cu launchers) ---------------------- */

/* farthestpointsamplingLauncher(b,n,m,inp,temp,out), tf_sampling_g.cu:203-205.
 * inp (b,n,3) f32; out (b,m) i32.  out[:,0] = 0; selection order and tie-break identical to the
 * reference kernel (:105-170): argmax of the running min squared distance under
 * (value desc, k mod 512 asc, k asc).  `temp` is the reference's (32,n) float scratch
 * (tf_sampling_g.cu:202).  Clouds of up to 425984 points (16 CTAs x 512 threads x 52 points) keep the
 * running minimum in registers and never touch it (temp may be NULL); larger clouds take the reference's
 * global-scratch layout and need pn2_fps_scratch_bytes(b, n) bytes there (cudaErrorInvalidValue if temp
 * is NULL then). */
int pn2_fps(int b, int n, int m, const float* inp, float* temp, int* out, void* stream);

/* Bytes of `temp` pn2_fps / pn2_fps_gather need for (b, n): 0 up to n = 425984, else
 * min(b,32)*n*sizeof(float). */
size_t pn2_fps_scratch_bytes(int b, int n);

/* Same as pn2_fps, also emitting new_xyz (b,m,3) = inp gathered at out (FPS + gather_point in one
 * launch; the pair sample_and_group always issues, utils/pointnet_util.py:40). new_xyz may be NULL. */
int pn2_fps_gather(int b, int n, int m, const float* inp, float* temp, int* out, float* new_xyz, void* stream);

/* probsampleLauncher(b,n,m,inp_p,inp_r,temp,out), tf_sampling_g.cu:198-201 (ProbSample op,
 * tf_sampling.cpp:66-92).  inp_p (b,n) f32 unnormalised probabilities; inp_r (b,m) f32 uniform
 * draws in [0,1]; temp (b,n) f32 caller-provided scratch that receives the cumulative sums (the
 * reference's allocate_temp, tf_sampling.cpp:86); out (b,m) i32 = index of the first cumulative sum
 * >= inp_r * sum.  The float32 cumulative sum keeps the reference's association, so indices are
 * bit-exact.  One CTA per row: b <= 2^31-1. */
int pn2_prob_sample(int b, int n, int m, const float* inp_p, const float* inp_r, float* temp, int* out, void* stream);

/* gatherpointLauncher(b,n,m,inp,idx,out), tf_sampling_g.cu:206-208. out (b,m,3). */
int pn2_gather_point(int b, int n, int m, const float* inp, const int* idx, float* out, void* stream);

/* scatteraddpointLauncher(b,n,m,out_g,idx,inp_g), tf_sampling_g.cu:209-211.
 * inp_g (b,n,3) must be zero-filled by the caller. */
int pn2_gather_point_grad(int b, int n, int m, const float* out_g, const int* idx, float* inp_g, void* stream);

/* ---- grouping (replaces tf_ops/grouping/tf_grouping_g.cu launchers) ----------------------- */

/* queryBallPointLauncher(b,n,m,radius,nsample,xyz1,xyz2,idx,pts_cnt), tf_grouping_g.cu:125-128.
 * xyz1 (b,n,3) data, xyz2 (b,m,3) queries; idx (b,m,nsample) i32, pts_cnt (b,m) i32.
 * First nsample hits in ascending index order, row padded with the first hit.  Rows with no hit
 * (undefined in the reference) are written as zeros with pts_cnt = 0. */
int pn2_query_ball_point(int b, int n, int m, float radius, int nsample, const float* xyz1,
                         const float* xyz2, int* idx, int* pts_cnt, void* stream);

/* Same operation and bit-identical results through a uniform grid (cell edge >= 1.01 radius: each query
 * only tests its 3x3x3 cell neighbourhood).  Clouds of 2048 <= n <= 9700 points are served by the
 * shared-memory grid kernel of pn2_ball_group (one launch, no workspace used).  Larger clouds use a
 * caller-provided device workspace of at least pn2_query_ball_point_workspace_bytes(b, n) bytes:
 * clouds whose balls are sparse are binned into a grid in that workspace;
 * the other clouds (dense or badly skewed ones, and any call with workspace == NULL or n < 2048)
 * take the brute-force path above, as does the whole batch when fewer than a quarter of its clouds
 * qualify and any cloud with a NaN coordinate (the reference counts a NaN point as a hit in every
 * ball, which only the scan reproduces).  workspace_bytes == 0 from the size query means "not applicable". */
size_t pn2_query_ball_point_workspace_bytes(int b, int n);
int pn2_query_ball_point_ws(int b, int n, int m, float radius, int nsample, const float* xyz1,
                            const float* xyz2, int* idx, int* pts_cnt, void* workspace,
                            size_t workspace_bytes, void* stream);

/* pn2_query_ball_point_ws in two halves: the grid build needs only the data points (xyz1), so it can
 * run on a second stream while farthest point sampling is still producing the queries; the second
 * half needs the queries.  Both return cudaErrorInvalidValue where pn2_query_ball_point_ws would
 * have fallen back to brute force (no workspace / n < 2048 / radius <= 1e-20). */
int pn2_ball_grid_build(int b, int n, float radius, int nsample, const float* xyz1, void* workspace,
                        size_t workspace_bytes, void* stream);
int pn2_query_ball_point_prebuilt(int b, int n, int m, float radius, int nsample, const float* xyz1,
                                  const float* xyz2, int* idx, int* pts_cnt, const void* workspace,
                                  size_t workspace_bytes, void* stream);

/* groupPointLauncher(b,n,c,m,nsample,points,idx,out), tf_grouping_g.cu:133-136.
 * points (b,n,c); idx (b,m,nsample); out (b,m,nsample,c). */
int pn2_group_point(int b, int n, int c, int m, int nsample, const float* points, const int* idx,
                    float* out, void* stream);

/* groupPointGradLauncher(b,n,c,m,nsample,grad_out,idx,grad_points), tf_grouping_g.cu:137-141.
 * grad_points (b,n,c) must be zero-filled by the caller. */
int pn2_group_point_grad(int b, int n, int c, int m, int nsample, const float* grad_out,
                         const int* idx, float* grad_points, void* stream);

/* selectionSortLauncher(b,n,m,k,dist,outi,out), tf_grouping_g.cu:129-132 (select_top_k).
 * dist (b,m,n); outi (b,m,n) i32, out (b,m,n) f32: the first k columns hold the k smallest values
 * of each row, ascending, and their indices, as k rounds of selection sort with swaps produce;
 * columns >= k hold the permuted remainder exactly as the reference leaves it. */
int pn2_selection_sort(int b, int n, int m, int k, const float* dist, int* outi, float* out, void* stream);

/* knn_point(k, xyz1, xyz2), tf_grouping.py:48-73, without the (b,m,n) distance matrix the reference's
 * graph materialises: xyz1 (b,n,3) data, xyz2 (b,m,3) queries -> val (b,m,k) f32 squared distances
 * ascending, idx (b,m,k) i32.  Bit-identical to the first k columns of selectionSortLauncher
 * (tf_grouping_g.cu:83-123, :129-132) applied to dist[b,j,i] = ((dx*dx + dy*dy) + dz*dz), every product
 * and sum rounded on its own — including the order the selection sort's SWAPS give to equal distances.
 * 1 <= k <= min(n, 128); otherwise cudaErrorInvalidValue (use pn2_selection_sort on a matrix). */
int pn2_knn_point(int b, int n, int m, int k, const float* xyz1, const float* xyz2, float* val, int* idx,
                  void* stream);

/* ---- 3d_interpolation (replaces the CPU functions of tf_interpolate.cpp; now on the GPU) -- */

/* threenn_cpu(b,n,m,xyz1,xyz2,dist,idx), tf_interpolate.cpp:60-103.
 * xyz1 (b,n,3) unknown, xyz2 (b,m,3) known; dist (b,n,3) f32 SQUARED distances ascending,
 * idx (b,n,3) i32; ties -> lower index; m < 3 -> (+inf, 0) fill.  Bit-exact with the reference's
 * x86 arithmetic (no contraction). */
int pn2_three_nn(int b, int n, int m, const float* xyz1, const float* xyz2, float* dist, int* idx, void* stream);

/* threeinterpolate_cpu(b,m,c,n,points,idx,weight,out), tf_interpolate.cpp:107-127.
 * points (b,m,c); idx, weight (b,n,3); out (b,n,c). */
int pn2_three_interpolate(int b, int m, int c, int n, const float* points, const int* idx,
                          const float* weight, float* out, void* stream);

/* threeinterpolate_grad_cpu(b,n,c,m,grad_out,idx,weight,grad_points), tf_interpolate.cpp:131-153.
 * grad_points (b,m,c) must be zero-filled by the caller. */
int pn2_three_interpolate_grad(int b, int n, int c, int m, const float* grad_out, const int* idx,
                               const float* weight, float* grad_points, void* stream);

/* The same gradient WITHOUT atomics: an inverse index (which unknown points reference each known point) is
 * built in `workspace` (pn2_three_interpolate_grad_det_workspace_bytes(b,n,m) bytes), then one warp per
 * known point adds its contributions in ascending (j, t) order — the order threeinterpolate_grad_cpu adds
 * them, every product and sum rounded on its own — so the result is run-to-run deterministic AND, for known
 * points referenced by at most 256 (j, t) pairs (every point of a non-degenerate layer), bit-identical to the
 * reference's CPU function; longer lists are summed in 8 consecutive pieces combined in order (deterministic,
 * equal to the sequential sum up to rounding).  grad_points (b,m,c) is overwritten: no zero-fill needed. */
size_t pn2_three_interpolate_grad_det_workspace_bytes(int b, int n, int m);
int pn2_three_interpolate_grad_det(int b, int n, int c, int m, const float* grad_out, const int* idx,
                                   const float* weight, float* grad_points, void* workspace,
                                   size_t workspace_bytes, void* stream);

/* ---- fused callers' glue (utils/pointnet_util.py) ------------------------------------------ */

/* sample_and_group's grouping tail, utils/pointnet_util.py:45-54 (SSG) and :179-186 (MSG), in
 * one pass: out[b,j,k,:] = concat of (xyz[idx]-new_xyz[j]) and points[idx] in the order chosen.
 *   xyz (b,n,3), new_xyz (b,m,3), points (b,n,c) or NULL (c = 0), idx (b,m,nsample)
 *   out (b,m,nsample,3+c);  grouped_xyz (b,m,nsample,3) or NULL (the 4th return of
 *   sample_and_group);  xyz_first != 0: [xyz, feats] (SSG, :50), else [feats, xyz] (MSG, :184). */
int pn2_group_concat(int b, int n, int c, int m, int nsample, const float* xyz, const float* new_xyz,
                     const float* points, const int* idx, int xyz_first, float* out,
                     float* grouped_xyz, void* stream);

/* pointnet_fp_module's front end, utils/pointnet_util.py:211-216, in one pass over the unknown
 * points: three_nn -> dist=max(dist,1e-10); w=(1/dist)/sum(1/dist) -> three_interpolate.
 *   xyz1 (b,n,3), xyz2 (b,m,3), points2 (b,m,c) -> out (b,n,c).
 *   dist/idx/weight (b,n,3) outputs are optional (NULL to skip). */
int pn2_three_nn_interpolate(int b, int n, int m, int c, const float* xyz1, const float* xyz2,
                             const float* points2, float* out, float* dist, int* idx, float* weight,
                             void* stream);

/* The whole front end of pointnet_fp_module, utils/pointnet_util.py:211-219, in one pass: the above plus the
 * concat with the dense level's own features: out (b,n,c2+c1) = [interpolated points2 (c2) | points1 (c1)].
 * points1 (b,n,c1) may be NULL with c1 = 0.  Values equal three_nn -> weights -> three_interpolate -> concat. */
int pn2_fp_interpolate_concat(int b, int n, int m, int c2, int c1, const float* xyz1, const float* xyz2,
                              const float* points1, const float* points2, float* out, void* stream);

/* ---- 16-bit features: bfloat16 / float16 twins of the feature ops ---------------------------- */

/* Each pn2_*_h entry mirrors the float32 entry named without the suffix, argument for argument, behind a
 * leading `dtype` (PN2_DTYPE_BF16 or PN2_DTYPE_F16; anything else is cudaErrorInvalidValue).  Feature
 * tensors (points, points1, points2, out, grad_out) hold that type; xyz, new_xyz, xyz1, xyz2, weight,
 * dist and grouped_xyz stay float32.  Values: every output equals the float32 op applied to the features
 * widened exactly to float32, rounded once to nearest-even into `dtype` (gathers and concats copy bits).
 * Gradients read a 16-bit grad_out and write FLOAT32 grad_points: the atomic entries accumulate into a
 * buffer the caller has zero-filled, the _det entry overwrites (same workspace size as its float32 twin,
 * and bit-identical to it applied to grad_out widened to float32). */
int pn2_group_point_h(int dtype, int b, int n, int c, int m, int nsample, const void* points, const int* idx,
                      void* out, void* stream);
int pn2_group_point_grad_h(int dtype, int b, int n, int c, int m, int nsample, const void* grad_out,
                           const int* idx, float* grad_points, void* stream);
int pn2_group_concat_h(int dtype, int b, int n, int c, int m, int nsample, const float* xyz, const float* new_xyz,
                       const void* points, const int* idx, int xyz_first, void* out, float* grouped_xyz,
                       void* stream);
int pn2_three_interpolate_h(int dtype, int b, int m, int c, int n, const void* points, const int* idx,
                            const float* weight, void* out, void* stream);
int pn2_three_interpolate_grad_h(int dtype, int b, int n, int c, int m, const void* grad_out, const int* idx,
                                 const float* weight, float* grad_points, void* stream);
int pn2_three_interpolate_grad_det_h(int dtype, int b, int n, int c, int m, const void* grad_out, const int* idx,
                                     const float* weight, float* grad_points, void* workspace,
                                     size_t workspace_bytes, void* stream);
int pn2_three_nn_interpolate_h(int dtype, int b, int n, int m, int c, const float* xyz1, const float* xyz2,
                               const void* points2, void* out, float* dist, int* idx, float* weight,
                               void* stream);
int pn2_fp_interpolate_concat_h(int dtype, int b, int n, int m, int c2, int c1, const float* xyz1,
                                const float* xyz2, const void* points1, const void* points2, void* out,
                                void* stream);

/* ---- the sampling+grouping half of a set-abstraction layer, device-resident ------------------ */

/* query_ball_point + group_point(xyz) in ONE launch (tf_grouping_g.cu:3-57 back to back, as
 * sample_and_group issues them, utils/pointnet_util.py:44-46): idx (b,m,nsample), pts_cnt (b,m) exactly as
 * pn2_query_ball_point writes them, and grouped_xyz (b,m,nsample,3) = xyz1 gathered at idx (NULL to
 * skip), minus the query when center != 0 (the tile+sub of :46, one rounding per coordinate).
 * Each cloud is binned into a uniform grid held in shared memory (or kept in index order when its
 * balls are dense), so it applies when pn2_ball_group_fits(n) != 0 (n <= 9700); otherwise
 * cudaErrorInvalidValue — use pn2_query_ball_point_ws + pn2_group_point. */
int pn2_ball_group_fits(int n);
int pn2_ball_group(int b, int n, int m, float radius, int nsample, const float* xyz1, const float* xyz2,
                   int* idx, int* pts_cnt, float* grouped_xyz, int center, void* stream);

/* farthest_point_sample + gather_point + query_ball_point + group_point(xyz)
 * (utils/pointnet_util.py:40-46) on DEVICE buffers, results bit-identical to the four separate
 * calls: fps_idx (b,m) i32 (the sampling indices; required, it is also the channel between the two
 * kernels), new_xyz (b,m,3), idx (b,m,nsample), pts_cnt (b,m), grouped_xyz (b,m,nsample,3) or NULL,
 * centred on new_xyz when center != 0.
 * When sampling runs one CTA per cloud (n <= 8192) and the cloud fits the shared-memory grid, the
 * ball query + grouping run as a programmatically dependent grid on the SMs the sampling chain
 * leaves idle and consume centroids while they are being produced; the layer then costs the sampling
 * time plus about a microsecond.  Otherwise the four kernels run back to back, using `workspace`
 * (pn2_sa_layer_device_workspace_bytes bytes, may be NULL when that is 0) for the sampling scratch
 * and the ball-query grid.  Independent batches may be issued on different streams: one layer
 * occupies 2*b SMs. */
size_t pn2_sa_layer_device_workspace_bytes(int b, int n, int m, int nsample);
/* The multi-scale form (pointnet_sa_module_msg, utils/pointnet_util.py:156-196: ONE farthest_point_sample +
 * gather_point, then query_ball_point + group_point(xyz) per scale): radii / nsamples / idx / pts_cnt /
 * grouped_xyz are HOST arrays of nscales (<= 16) entries (grouped_xyz, or any entry of it, may be NULL).
 * On the overlapped path every scale's grouping grid runs while the sampling chain is still going. */
int pn2_sa_layer_msg_device(int b, int n, int m, int nscales, const float* radii, const int* nsamples,
                            const float* xyz, int* fps_idx, float* new_xyz, int* const* idx,
                            int* const* pts_cnt, float* const* grouped_xyz, int center, void* workspace,
                            size_t workspace_bytes, void* stream);
/* tuning: grouping CTAs per cloud and scale on the overlapped path (0 = automatic: one) */
void pn2_set_sa_consumer_ctas(int ctas_per_cloud);
int pn2_sa_layer_device(int b, int n, int m, float radius, int nsample, const float* xyz, int* fps_idx,
                        float* new_xyz, int* idx, int* pts_cnt, float* grouped_xyz, int center,
                        void* workspace, size_t workspace_bytes, void* stream);

/* ---- host-buffer entry point (the reference feeds numpy through feed_dict) ----------------- */

/* One SSG set-abstraction sampling+grouping layer (farthest_point_sample + gather_point +
 * query_ball_point + group_point(xyz), utils/pointnet_util.py:40-45) on HOST buffers:
 * copies h_xyz (b,n,3) to the device, runs the four ops, copies new_xyz (b,m,3), idx (b,m,nsample),
 * pts_cnt (b,m) and grouped_xyz (b,m,nsample,3; NOT centred) back — through pn2_sa_layer_device.
 * Any of the four output pointers may be NULL: that result is neither copied back nor, for
 * grouped_xyz, computed (a caller that regroups on the host saves 3/4 of the device-to-host bytes).
 * Host buffers should be pinned for the copies to be asynchronous.  `workspace` is a device buffer of at least
 * pn2_sa_layer_workspace_bytes(b,n,m,nsample) bytes supplied by the caller.  Asynchronous on
 * `stream`: synchronise the stream before reading the outputs. */
size_t pn2_sa_layer_workspace_bytes(int b, int n, int m, int nsample);
int pn2_sa_layer_host(int b, int n, int m, float radius, int nsample, const float* h_xyz,
                      float* h_new_xyz, int* h_idx, int* h_pts_cnt, float* h_grouped_xyz,
                      void* workspace, size_t workspace_bytes, void* stream);

/* ---- introspection ------------------------------------------------------------------------- */
int pn2_api_version(void);
const char* pn2_error_string(int code);
/* number of kernel launches (not memcpys) this library has issued in this process */
unsigned long long pn2_launch_count(void);
/* the exact d2-domain threshold the ball query uses for `radius`
 * (largest float t with max(sqrtf(t),1e-20f) < radius; negative if no t qualifies) */
float pn2_ball_threshold(float radius);
/* tuning override for experiments: threads, points/thread, cluster size of the FPS kernel
 * (cluster 0 = global-scratch fallback); threads = 0 restores the built-in plan.
 * The per-step update exists in two bit-identical forms — the plain scalar chain and the packed FP32x2 /
 * value-only chain that is the built-in choice wherever it is instantiated (environment: PN2_FPS_PACKED=0/1 for
 * one CTA per cloud, PN2_FPS_PACKED_CLUSTER=0/1 for clusters).  An override can name the chain: cluster = -1 /
 * -2 = one CTA per cloud with the plain / packed chain; for cluster plans the two low bits of `threads`
 * (threads is a multiple of 128): +1 = packed, +2 = plain. */
void pn2_set_fps_config(int threads, int points_per_thread, int cluster);
/* the kernel variant pn2_fps would launch for (b, n): threads per CTA, points per thread and
 * cluster size (1 = one CTA per cloud, >= 2 = thread-block cluster per cloud, 0 = global-scratch
 * fallback) */
int pn2_fps_plan(int b, int n, int* threads, int* points_per_thread, int* cluster);
/* how many thread-block clusters of the FPS cluster kernel (threads, points/thread, cluster size) the
 * current device can hold at once (cudaOccupancyMaxActiveClusters); 0 = no such kernel / cannot launch.
 * The planner uses it to keep every cloud's cluster co-resident. */
int pn2_fps_cluster_capacity(int threads, int points_per_thread, int cluster);
/* tuning override: lanes cooperating on one ball query (1,2,4,..,32); 0 restores the heuristic */
void pn2_set_bq_group(int lanes_per_query);
/* tuning override for pn2_query_ball_point_ws: 0 = automatic, 1 = brute force only, 2 = the workspace
 * (global-memory) grid path even where the shared-memory grid kernel would apply */
void pn2_set_bq_mode(int mode);

#ifdef __cplusplus
}
#endif
#endif /* PN2_API_H_ */
