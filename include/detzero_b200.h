/*
 * detzero_b200.h -- C ABI of libdetzero_b200.so (sm_100a).
 *
 * The reference (PJLab-ADG/DetZero) has no C ABI: its native ops are pybind11 modules taking at::Tensor
 * (utils/detzero_utils/ops/iou3d_nms/src/iou3d_nms_api.cpp:10-17) and its sparse-conv / voxelizer arithmetic
 * lives in the third-party spconv wheel.  Each entry point below names the reference interface it replaces.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless marked "host"; the caller owns all buffers incl. workspace
 *   - functions only enqueue work on `stream` (a cudaStream_t): no malloc, no sync, no host loop
 *   - element counts that are only known on the device are passed as `const int* d_n` (device scalar) together
 *     with a host-side capacity `cap`; kernels are persistent / grid-stride over `cap` and read `*d_n`
 *   - return 0 on success, <0 on error (never exit(); contrast iou3d_nms.cpp:14-26); dz_last_error_string()
 *   - feature tensors are row-major (rows, channels); dense maps are NHWC
 *
 * Grid index ("coordinate index"): for a lattice (B, D, H, W) a bitmap of occupied cells + an exclusive
 * popcount prefix per 32-bit word (+ optional permutation rank->row).  cell = b*cells_pad + (z*H+y)*W+x with
 * cells_pad = round_up(D*H*W, 32).  Rank order == ascending (b,z,y,x).
 */
#ifndef DETZERO_B200_H
#define DETZERO_B200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef void* dz_stream_t;           /* cudaStream_t */

enum { DZ_OK = 0, DZ_ERR_ARG = -1, DZ_ERR_CUDA = -2, DZ_ERR_WORKSPACE = -3, DZ_ERR_UNSUPPORTED = -4 };
enum { DZ_F32 = 0, DZ_TF32 = 1, DZ_BF16 = 2, DZ_TF32X3 = 3, DZ_BF16X2 = 4 };   /* arithmetic mode of GEMM-shaped kernels:
   F32 = fp32 FMA; TF32 = one tcgen05 TF32 pass; TF32X3 = hi/lo split, 3 TF32 passes, fp32-level accuracy (sparse conv);
   BF16 / BF16X2 = bf16 operand planes (1 plane: bf16 storage; 2 planes: x = p0 + p1, 16 significand bits in 4 bytes,
   fp32-level accuracy at the cost of one TF32 pass), sparse conv only: dz_spconv_fwd_planes */

int         dz_version(void);
int         dz_sm_arch(void);                      /* 100 : built for sm_100a */
const char* dz_last_error_string(void);            /* host string, thread-local */

/* ---- grid index ---------------------------------------------------------------------------------------- */
size_t dz_grid_index_words(int B, int D, int H, int W);          /* number of u32 words in bitmap == prefix */
size_t dz_scan_ws_bytes(size_t n_words);
/* prefix[w] = base + popcount(bitmap[0..w)), *d_total = base + popcount(all); base = d_base ? *d_base : 0 */
int dz_grid_index_scan(const uint32_t* bitmap, uint32_t* prefix, size_t n_words, const int* d_base,
                       int* d_total, void* ws, size_t ws_bytes, dz_stream_t stream);
/* arbitrary site list -> index (+perm: rank -> row).  Replaces the hash table spconv builds inside
 * SparseConvTensor/indice_dict (backbone3d.py:190-195).  bitmap must be zero on entry. */
int dz_grid_index_from_coords(const int32_t* coords, const int* d_n, int cap, int B, int D, int H, int W,
                              uint32_t* bitmap, uint32_t* prefix, int32_t* perm, int* d_total,
                              void* ws, size_t ws_bytes, dz_stream_t stream);

/* ---- voxelization -------------------------------------------------------------------------------------- */
/* Hard voxelization of ONE cloud, order-exact with spconv.utils.Point2VoxelCPU3d.point_to_voxel as driven by
 * detection/detzero_det/datasets/processor/data_processor.py:61-91 (first-appearance voxel ids, first max_pts
 * points kept in input order, voxel cap in appearance order), fused with MeanVFE.forward (vfe.py:66-83).
 *   points (n, point_stride) f32; the c feature columns [xyz_off, xyz_off+c) start with x,y,z and are copied
 *   verbatim (xyz_off = 1 for a collated (N,1+C) [b,x,y,z,..] tensor, 0 for a raw (N,C) cloud)
 *   voxels (cap, max_pts, c) ; coords (cap,4) [batch_idx,z,y,x] ; num_per_voxel (cap) ; mean (cap,c) or NULL
 *   d_counters[0] = rows already used in voxels/coords (in/out), d_counters[1] = ranks already used in the
 *   index (in/out), d_counters[2] = rows wanted (in/out; > [0] iff `cap` was too small): calling once per frame with batch_idx = 0..B-1 on one stream builds a collated batch
 *   (dataset.py:260-303) without a host sync.
 *   index_* : level-0 grid index over lattice (B, iD, iH, iW) (iD = sparse_shape z = grid z + 1,
 *   backbone3d.py:133); bitmap must be zero before the first frame of a batch. */
size_t dz_voxelize_hard_ws_bytes(int n_points, int max_pts, int max_voxels, int iD, int iH, int iW);
int dz_voxelize_hard(const float* points, int n, int point_stride, int xyz_off, int c,
                     const float* range_xyz6_host, const float* vsize_xyz3_host, const int* grid_zyx3_host,
                     int max_pts, int max_voxels, int batch_idx,
                     float* voxels, int32_t* coords, int32_t* num_per_voxel, float* mean, int cap,
                     int* d_counters,
                     int B, int iD, int iH, int iW, uint32_t* index_bitmap, uint32_t* index_prefix,
                     int32_t* index_perm,
                     void* ws, size_t ws_bytes, dz_stream_t stream);
/* The same for the B frames of a batch in ONE call (frames = batch indices 0..B-1, d_counters zero or carried on entry):
 * the frames run on internal streams forked from / joined to `stream` and only wait for each other's running totals, so
 * their latency-bound kernels overlap.  points_host / n_host are HOST arrays of device pointers / point counts.
 * Identical results to B calls of dz_voxelize_hard in frame order. */
size_t dz_voxelize_hard_batch_ws_bytes(int n_max, int B, int max_pts, int max_voxels, int iD, int iH, int iW);
int dz_voxelize_hard_batch(const float* const* points_host, const int* n_host, int B, int point_stride, int xyz_off, int c,
                           const float* range6_host, const float* vsize3_host, const int* grid_zyx3_host, int max_pts,
                           int max_voxels, float* voxels, int32_t* coords, int32_t* num_per_voxel, float* mean, int cap,
                           int* d_counters, int iD, int iH, int iW, uint32_t* index_bitmap, uint32_t* index_prefix,
                           int32_t* index_perm, void* ws, size_t ws_bytes, dz_stream_t stream);

/* MeanVFE.forward (vfe.py:66-83) on an already voxelized batch: out (M,C) = voxels.sum(1) / max(num,1) */
int dz_mean_vfe(const float* voxels, const int32_t* num_per_voxel, int M, int P, int C, float* out,
                dz_stream_t stream);

/* Dynamic mean voxelization of a collated batch: DynamicMeanVFE.forward (vfe.py:110-147): floor((p-lo)/vs),
 * in-range mask, key b*XYZ + x*YZ + y*Z + z, unique (sorted), scatter_mean of all c columns.
 *   points (n, 1+c) [b,x,y,z,...] ; out feats (cap,c), coords (cap,4) [b,z,y,x] ordered by ascending key ;
 *   *d_m = number of voxels.  bitmap_xyz: B*round_up(X*Y*Z,32)/32 words, zero on entry. */
size_t dz_voxelize_dynamic_ws_bytes(int n_points, int cap, int B, int X, int Y, int Z);
int dz_voxelize_dynamic_mean(const float* points, int n, int c, int B,
                             const float* range_xyz6_host, const float* vsize_xyz3_host,
                             const int* grid_xyz3_host, float* feats, int32_t* coords, int cap, int* d_m,
                             void* ws, size_t ws_bytes, dz_stream_t stream);

/* ---- rulebook ------------------------------------------------------------------------------------------ */
/* Neighbour-table form of the spconv rulebook.  Two layouts, each optional (NULL = not wanted, at least one given):
 *   nbr  k-major  (K, cap):  nbr[k*cap + o] = input row feeding output row o through kernel offset
 *                            k = (kz*KH+ky)*KW+kx, or -1            (exact-fp32 kernel; what the parity tests read)
 *   tab  row-major (cap, 32): tab[o*32 + k] = the same entry for k < K, -1 up to 26, [27] = bit mask of the live
 *                            offsets, [28..31] = 0: one 128-byte line per output row   (tensor-core kernels)
 * The pair set {(k, nbr, o)} equals spconv's indice pairs (SubMConv3d: backbone3d.py:68,93-100,136 ;
 * SparseConv3d: :70-71,169-170,183-184).
 * sched_ws (optional, needs tab; dz_rulebook_schedule_ws_bytes(cap) bytes): the kernel also leaves what
 * dz_rulebook_schedule needs (mask digests, scanned histogram) there. */
int dz_rulebook_subm(const int32_t* coords, const int* d_n, int cap, int B, int D, int H, int W,
                     const int* ksize3_host, const uint32_t* bitmap, const uint32_t* prefix,
                     const int32_t* perm, int32_t* nbr, int32_t* tab, void* sched_ws, int sched_frame_major,
                     dz_stream_t stream);
/* Strided conv: generates the output site set (sorted ascending (b,z,y,x)), its grid index and the table(s).
 * out_bitmap must be zero on entry. */
int dz_rulebook_conv(const int32_t* in_coords, const int* d_n_in, int in_cap, int B,
                     const int* in_dhw3_host, const int* ksize3_host, const int* stride3_host,
                     const int* pad3_host, const uint32_t* in_bitmap, const uint32_t* in_prefix,
                     const int32_t* in_perm, int32_t* out_coords, int* d_n_out, int out_cap,
                     uint32_t* out_bitmap, uint32_t* out_prefix, int32_t* nbr, int32_t* tab,
                     void* ws, size_t ws_bytes, void* sched_ws, int sched_frame_major, dz_stream_t stream);
/* Tile schedule for the tensor-core conv (no reference counterpart; spconv's implicit-GEMM "mask sort" plays the same
 * role).  order (cap + ceil(cap/128) ints): order[p] = output row at tile position p -- rows with alike neighbour
 * masks become adjacent, so a 128-row tile skips the kernel offsets none of its rows uses -- and order[cap + j] = the
 * tile the j-th CTA takes (most live offsets first).  Hand it to dz_spconv_fwd as row_order; results are bit-identical
 * to the unscheduled call.  sched_ws must be the one the rulebook call filled for this tab.
 * sched_frame_major (same value in the rulebook call and here; B = frames in the batch): sort by (frame, mask) and order the
 * tiles frame by frame (heaviest first inside a frame), so that the rows the CTAs gather at any moment belong to ONE frame's
 * feature map and stay L2-resident at batch sizes whose level no longer fits L2. */
size_t dz_rulebook_schedule_ws_bytes(int cap);
int dz_rulebook_schedule(const int32_t* tab, int cap, const int* d_n, int32_t* order, void* sched_ws,
                         size_t ws_bytes, int B, int sched_frame_major, int K, int32_t* tab_tiles, dz_stream_t stream);
/* tab_tiles (optional; ceil(cap/128) * (K+1) * 128 ints): the scheduled table again, TILE-major: tile j = (K+1) planes of 128
 * ints, plane k < K = neighbour row of tile position p through offset k, plane K = the output row order[j*128+p] (-1 beyond the
 * count).  With it `order` must have cap + 2*ceil(cap/128) ints: order[cap + tiles + j] = OR of tile j's row masks.  The
 * persistent bf16-plane conv (dz_spconv_fwd_planes) fetches a tile's block with ONE bulk copy. */

/* Direct path to tab_tiles without a row-major table (the schedule + tile-major table of the bf16-plane conv; same pair set as
 * spconv's generate_subm_conv_inds / generate_conv_inds_stage{1,2}).  Two calls per rulebook:
 *   1. dz_rulebook_subm_masks / dz_rulebook_conv_masks: the mask pass.  Leaves in sched_ws exactly what dz_rulebook_subm /
 *      dz_rulebook_conv leave there (neighbour masks, digests, scanned histogram) and writes no table.  The strided variant
 *      also produces the output sites, their count and their grid index, as dz_rulebook_conv does.  perm_walk (needs perm):
 *      visit the rows in lattice (rank) order.
 *   2. dz_rulebook_schedule_direct: the schedule and the tile-major table from the masks and the INPUT grid index.  coords,
 *      cap, d_n are the OUTPUT sites (the rulebook's rows); in_dhw3 / ksize3 / stride3 / pad3 the conv geometry; subm = 1 for a
 *      submanifold conv (stride and pad are then ignored: 1 and (k-1)/2).  order: cap + 2*ceil(cap/128) ints and tab_tiles:
 *      ceil(cap/128) * (K+1) * 128 ints, both as dz_rulebook_schedule with K given.  Plane k of every row equals the entry
 *      the row-major table would hold. */
int dz_rulebook_subm_masks(const int32_t* coords, const int* d_n, int cap, int B, int D, int H, int W,
                           const int* ksize3_host, const uint32_t* bitmap, const uint32_t* prefix, const int32_t* perm,
                           void* sched_ws, int sched_frame_major, int perm_walk, dz_stream_t stream);
int dz_rulebook_conv_masks(const int32_t* in_coords, const int* d_n_in, int in_cap, int B,
                           const int* in_dhw3_host, const int* ksize3_host, const int* stride3_host,
                           const int* pad3_host, const uint32_t* in_bitmap, const uint32_t* in_prefix,
                           const int32_t* in_perm, int32_t* out_coords, int* d_n_out, int out_cap,
                           uint32_t* out_bitmap, uint32_t* out_prefix, void* ws, size_t ws_bytes,
                           void* sched_ws, int sched_frame_major, dz_stream_t stream);
int dz_rulebook_schedule_direct(const int32_t* coords, int cap, const int* d_n, int B, const int* in_dhw3_host,
                                const int* ksize3_host, const int* stride3_host, const int* pad3_host, int subm,
                                const uint32_t* in_bitmap, const uint32_t* in_prefix, const int32_t* in_perm,
                                int32_t* order, void* sched_ws, size_t ws_bytes, int sched_frame_major,
                                int32_t* tab_tiles, dz_stream_t stream);

/* ---- sparse convolution -------------------------------------------------------------------------------- */
/* out[o,:] = act( (sum_k in[nbr[k][o],:] @ W[k]) * scale + shift (+ residual[o,:]) )
 * Replaces SubMConv3d/SparseConv3d forward + BatchNorm1d(eval) + bias + residual add + ReLU
 * (backbone3d.py:64-83,105-121).  weight packed (K, cin, cout) f32 (host side repacks spconv's
 * (cout,KD,KH,KW,cin) layout, SURVEY A.3; DZ_TF32 expects (cout, K*cin_pad)).  in_rows = allocated rows of `in`
 * (bounds the TMA gather).  mode: DZ_F32 exact-fp32 FMA (nbr = k-major table), DZ_TF32 / DZ_TF32X3 tcgen05 tensor
 * cores (nbr = ROW-major table `tab`, nbr_cap = its rows).
 * row_order: NULL, or the tile schedule of dz_rulebook_schedule (tensor-core modes only). */
int dz_spconv_fwd(const float* in, int cin, int in_rows, const int32_t* nbr, int K, int nbr_cap,
                  const int32_t* row_order, const int* d_n_out,
                  int out_cap, const float* weight, const float* scale, const float* shift,
                  const float* residual, int relu, float* out, int cout, int mode, dz_stream_t stream);

/* Backward of dz_spconv_fwd on the same k-major table (exact fp32; SURVEY.md 8f row 1; the reference trains through spconv's
 * autograd, detection/tools/train_utils.py:59-68).  dz_rulebook_transpose: nbrT (K, cap_in), nbrT[k][j] = o for every pair
 * (k, j = nbr[k][o], o), -1 elsewhere.  dgrad = dz_spconv_fwd(d_out, nbrT, weight^T (K, cout, cin)); the transposed table with its own
 * weights is SparseInverseConv3d (backbone3d.py:72-73).  dz_spconv_wgrad: dW (K, cin, cout) = sum_o in[nbr[k][o]]^T (x) d_out[o]. */
int dz_rulebook_transpose(const int32_t* nbr, int K, int cap_out, const int* d_n_out, int32_t* nbrT, int cap_in,
                          dz_stream_t stream);
int dz_spconv_wgrad(const float* in, int cin, const int32_t* nbr, int K, int nbr_cap, const int* d_n_out, int out_cap,
                    const float* dout, int cout, float* dW, dz_stream_t stream);

/* The same layer on bf16 operand PLANES (modes DZ_BF16: planes = 1, DZ_BF16X2: planes = 2), csrc/spconv_bf16.cu: a persistent
 * warp-specialised tcgen05 kernel.  Feature tensors `in`, `residual`, `out` are (rows, planes * C) bf16, a row = [p0 | p1] with
 * x ~ p0 (+ p1), p0 = RN_bf16(x), p1 = RN_bf16(x - p0); cin <= 8 is stored padded to 8 channels per plane.  weight: (planes * cout,
 * K * cin_pad) bf16, rows [w0 ; w1] split the same way.  tab = ROW-major table, row_order = NULL or the tile schedule,
 * tab_tiles = NULL or the tile-major table dz_rulebook_schedule wrote next to row_order (fast path).  With tab_tiles and
 * row_order, tab may be NULL (direct rulebook path); tab_rows is then the rulebook's capacity.
 * No reference counterpart for the storage format (spconv keeps fp32 rows); dz_to_planes / dz_from_planes convert at the
 * boundary: out[r, p, 0..c_pad) <- x[r, 0..c) (zero padded), x[r, c] <- p0 + p1. */
int dz_spconv_fwd_planes(const void* in, int cin, int in_rows, const int32_t* tab, int K, int tab_rows,
                         const int32_t* row_order, const int* d_n_out, int out_cap, const void* weight,
                         const float* scale, const float* shift, const void* residual, int relu, void* out, int cout,
                         int planes, const int32_t* tab_tiles, dz_stream_t stream);
int dz_to_planes(const float* x, const int* d_n, int cap, int c, int c_pad, int planes, void* out, dz_stream_t stream);
int dz_from_planes(const void* x, const int* d_n, int cap, int c, int planes, float* out, dz_stream_t stream);

/* ---- BEV ------------------------------------------------------------------------------------------------ */
/* SparseConvTensor.dense() + reshape(N, C*D, H, W) (height_compression.py:20-25) into NHWC:
 * out[b,y,x,c*D+z] = feats[i,c].  out must be zero on entry. */
int dz_sparse_to_bev(const float* feats, const int32_t* coords, const int* d_n, int cap, int c,
                     int B, int D, int H, int W, float* out, dz_stream_t stream);
/* the same from a bf16 planes tensor (rows, planes * c) */
int dz_sparse_to_bev_planes(const void* feats, const int32_t* coords, const int* d_n, int cap, int c, int planes,
                            int B, int D, int H, int W, float* out, dz_stream_t stream);
/* NHWC conv2d (cross-correlation) with fused per-channel affine (folded BatchNorm2d / bias) and ReLU; output
 * written at channel offset into a tensor with out_cstride channels (fused torch.cat, backbone2d.py:107-108).
 * weight packed (KH, KW, cin, cout).  Replaces nn.Conv2d(+ZeroPad2d)+BatchNorm2d+ReLU stacks at
 * backbone2d.py:34-48 and center_head.py:25-31,81-88. */
int dz_conv2d_fwd(const float* in, int B, int H, int W, int cin, int in_cstride, const float* weight, int KH, int KW,
                  int stride, int pad, const float* scale, const float* shift, int relu,
                  float* out, int Ho, int Wo, int cout, int out_coff, int out_cstride, int mode,
                  dz_stream_t stream);
/* ConvTranspose2d with kernel == stride (backbone2d.py:52-60): out[b,y*s+dy,x*s+dx,co] = sum_ci in*W[dy,dx,ci,co]
 * weight packed (s, s, cin, cout). */
int dz_deconv2d_fwd(const float* in, int B, int H, int W, int cin, const float* weight, int s,
                    const float* scale, const float* shift, int relu, float* out, int cout, int out_coff,
                    int out_cstride, int mode, dz_stream_t stream);

/* ---- CenterHead decode + NMS --------------------------------------------------------------------------- */
/* centernet_utils.decode_bbox_from_heatmap / _topk (centernet_utils.py:138-230) on the fused head map
 * (B,H,W,ch) NHWC with channel layout given by ch_* offsets.  Produces, per frame, up to K candidates in
 * descending score order that pass POST_CENTER_LIMIT_RANGE and SCORE_THRESH:
 *   cand_boxes (B,K,7), cand_scores (B,K), cand_labels (B,K) int32 (0-based class), d_cand_n (B). */
size_t dz_centerhead_decode_ws_bytes(int B, int H, int W, int num_class, int K);
int dz_centerhead_decode(const float* head, int B, int H, int W, int ch, int ch_center, int ch_z, int ch_dim,
                         int ch_rot, int ch_iou, int ch_hm, int num_class, int K,
                         const float* range_xyz6_host, const float* vsize_xyz3_host, int fmap_stride,
                         const float* post_limit6_host, float score_thresh, int use_iou,
                         float* cand_boxes, float* cand_scores, int32_t* cand_labels, int* d_cand_n,
                         void* ws, size_t ws_bytes, dz_stream_t stream);
/* Rotated-BEV NMS fully on device: replaces model_nms_utils.class_agnostic_nms -> nms_gpu
 * (model_nms_utils.py:6-25, iou3d_nms_utils.py:154-170, iou3d_nms.cpp:114-160, iou3d_nms_kernel.cu:386-430).
 * Input per frame: n<=cap boxes in descending score order.  Output: out (B, post_max, 9) rows
 * [x,y,z,dx,dy,dz,heading,score,label+label_offset], zero padded, d_out_n (B). */
size_t dz_nms_bev_ws_bytes(int B, int cap);
int dz_nms_bev(const float* boxes, const float* scores, const int32_t* labels, const int* d_n, int B, int cap,
               float thresh, int post_max, int label_offset, float* out, int* d_out_n,
               void* ws, size_t ws_bytes, dz_stream_t stream);
/* pairwise rotated BEV IoU (iou3d_nms_kernel.cu:370-384 boxes_iou_bev_kernel) */
int dz_boxes_iou_bev(const float* boxes_a, int na, const float* boxes_b, int nb, float* out, dz_stream_t stream);

/* ---- on-disk frame -> collated device points (SURVEY.md 8f row 4) ---------------------------------------- */
/* raw: a frame file as waymo_utils.py:284-302 writes it, (n, 6) f32 [x,y,z,intensity,elongation,NLZ_flag], already on the device
 * (pinned-host -> device copy of the file bytes).  Does DatasetTemplate.merge_sweeps (dataset.py:167-196) + the collate batch
 * column (:275-283) on the device: keep NLZ_flag == -1 in file order, tanh(intensity), xyz <- [x y z 1] @ T[:3,:].T in double
 * (transform12_host: row-major 3x4 of inv(current_pose) @ sweep_pose, NULL = identity), append time_offset (with_time),
 * prepend batch_idx.  Rows (1 + 5 + with_time floats) are appended at d_count[0]; d_count[1] = rows wanted (> cap: overflow). */
size_t dz_prepare_points_ws_bytes(int n);
int dz_prepare_points(const float* raw, int n, const double* transform12_host, float time_offset, int with_time, int batch_idx,
                      float* out, int cap, int* d_count, void* ws, size_t ws_bytes, dz_stream_t stream);

/* ---- tracker association matrices + object crop (SURVEY.md 8f rows 2, 3) ---------------------------------- */
/* out (na, nb) = kind(boxes_a[i], boxes_b[j]); boxes are rows of >= 7 floats [x,y,z,dx,dy,dz,heading,...] with row strides
 * lda / ldb floats, so the matrices can be computed straight from the all-gathered (F, 500, 9) detection tensor.
 * kind 0: rotated-BEV IoU (IoUBEV_dis_mat -> boxes_iou_bev_gpu), 1: BEV overlap area (bev_overlap_gpu, the tracker's overlap
 * filter), 2: 3-D IoU (IoU3D_dis_mat -> boxes_iou3d_gpu, iou3d_nms_utils.py:74-107), 3: axis-aligned 2-D IoU on (x,y,dx,dy)
 * (IoU2D_dis_mat).  Replaces tracking/detzero_track/models/tracking_modules/data_association/distance.py:44-141. */
int dz_boxes_pairwise(const float* boxes_a, int na, int lda, const float* boxes_b, int nb, int ldb, int kind, float* out,
                      dz_stream_t stream);
/* Object crop: which points (rows of pt_stride >= 3 floats, x,y,z first) lie inside which box -- points_in_boxes_gpu_v2
 * (roiaware_pool3d_kernel.cu:23-36,352-372; daemon/prepare_object_data.py:264-311) -- as the ORDERED index list the daemon builds
 * on the host: idx (n_boxes, cap) = indices of box t's points in input order (-1 padded, first cap kept), num (n_boxes) = true
 * counts.  dz_points_in_boxes_mask writes the reference's own (n_boxes, n_pts) int32 mask. */
size_t dz_crop_points_ws_bytes(int n_pts, int n_boxes);
int dz_crop_points_in_boxes(const float* points, int n_pts, int pt_stride, const float* boxes, int n_boxes, int ldb,
                            int32_t* idx, int cap, int* num, void* ws, size_t ws_bytes, dz_stream_t stream);
int dz_points_in_boxes_mask(const float* points, int n_pts, int pt_stride, const float* boxes, int n_boxes, int ldb,
                            int32_t* mask, dz_stream_t stream);

/* ---- refiner (GRM / PRM / CRM) ------------------------------------------------------------------------- */
/* y = act((x @ W^T) * scale + shift): x (M,K) row-major, W (N,K) row-major (nn.Linear / 1x1 Conv layout).
 * Replaces F.linear and the Conv1d/Conv2d(k=1)+BN+ReLU MLP stacks (utils/detzero_utils/model_utils.py:81-134). */
int dz_linear_fwd(const float* x, int M, int K, const float* w, int N, const float* scale, const float* shift,
                  int relu, float* y, int ldy, int mode, dz_stream_t stream);
/* The same with a per-row-GROUP shift: y[m] = act((x[m] W^T) * scale + shift + gshift[m / gsize]), gshift (M/gsize, N).  Serves the
 * PointNet "concatenate the max-pooled global feature back onto every point, then Linear" step (position_transformer.py:118-123,
 * geometry_transformer.py:131-136, confidence_pointnet.py:88-100) without materialising the concatenation: W = [W_g | W_p],
 * gshift = (g W_g^T) * scale computed once per group, x = the per-point half. */
int dz_linear_fwd_grouped(const float* x, int M, int K, const float* w, int N, const float* scale, const float* shift,
                          const float* gshift, int gsize, int relu, float* y, int ldy, int mode, dz_stream_t stream);
/* Linear (+folded BN +ReLU) fused with the max over groups of `group` consecutive rows (group % 128 == 0, K % 32 == 0, N % 4 == 0,
 * tensor-core mode): y (M/group, N).  The last layer of a PointNet encoder + torch.max over the points in one kernel. */
int dz_linear_max_fwd(const float* x, int M, int K, const float* w, int N, const float* scale, const float* shift, int relu,
                      int group, float* y, int mode, dz_stream_t stream);
/* max over `group` consecutive rows: x (G*group, C) -> y (G, C)  (torch.max over points,
 * position_transformer.py:109,118) */
int dz_group_max(const float* x, int G, int group, int C, float* y, dz_stream_t stream);
/* softmax(q k^T + key_padding) v per (batch, head); q already scaled.  q (B,Pq,H*dh), k/v (B,Pk,H*dh) with
 * row strides ldq/ldk/ldv ; key_padding_mask (B,Pk) u8 (non-zero = masked, as masked_fill(-inf)) or NULL.
 * Replaces multi_head_attention.py:266-286 without materialising the (B*H,Pq,Pk) score tensor. */
int dz_attention_fwd(const float* q, int ldq, const float* k, int ldk, const float* v, int ldv,
                     const unsigned char* key_padding_mask, int B, int Pq, int Pk, int H, int dh, float* out,
                     int ldo, int mode, dz_stream_t stream);
/* y = LayerNorm(x + r) * gamma + beta over the last dim C (decoder.py:73-75,85-90) ; r may be NULL */
int dz_layernorm_residual(const float* x, const float* r, const float* gamma, const float* beta, float eps,
                          int M, int C, float* y, dz_stream_t stream);

/* out = a + b, n % 4 == 0 (with_pos_embed, decoder.py:45-46) */
int dz_add(const float* a, const float* b, size_t n, float* out, dz_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif
