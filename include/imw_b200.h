/* imw_b200 -- C ABI of the B200-native image-pair matching hot path.
 *
 * Drop-in boundary for the reference's plugin layer (imcui/hloc/utils/base_model.py:9-55): every
 * entry point below replaces the forward pass of one BaseModel plugin.  The reference is pure
 * Python + PyTorch, so the reference-side binding is a ctypes stub inside the plugin's
 * `_forward` (see INTEGRATION.md); signatures carry only raw device pointers, sizes and a
 * cudaStream_t -- no torch types.
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless stated; fp32 / int32; no allocation, no host
 *     synchronisation and no implicit stream inside any call (ui/api callers own memory + stream);
 *   - `*_workspace_bytes` returns the scratch size the matching call needs;
 *   - return value: 0 = ok, <0 = error (imw_last_error() holds the message); the Python shim turns
 *     errors into the exceptions the reference raises (ValueError / AssertionError);
 *   - empty inputs are not errors (counts may be 0), as in the reference (SURVEY.md 8(b)).
 */
#ifndef IMW_B200_H
#define IMW_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* imw_stream_t; /* == cudaStream_t */

const char* imw_last_error(void);
int imw_version(void);
/* number of kernels this library has launched so far in this process (bench.py: gpu_launches) */
unsigned long long imw_launch_count(void);
/* Launch-site profiler (measurement aid, bench.py): between imw_prof_begin(stream) and imw_prof_end() every kernel launch
 * of the library records a CUDA event behind itself on the launching stream; imw_prof_end synchronises them and writes
 * "launcher signature:line<TAB>launches<TAB>total_ms" lines (one per launch site) into buf.  Returns the number of
 * launches seen (<0 = error).  Off by default: no events, no synchronisation. */
int imw_prof_begin(imw_stream_t stream);
long long imw_prof_end(char* buf, size_t buf_bytes);

/* ------------------------------------------------------------------------------------------------
 * Image pre-processing of the extraction drivers.
 * Replaces: hloc/extract_features.py:120-162 (preprocess + the RGB2GRAY of extract) and hloc/match_dense.py:588-640:
 * cv2.cvtColor(RGB2GRAY) on uint8, astype(float32), cv2.resize(INTER_AREA) for resize_max and force_resize
 * (INTER_LINEAR when up-sampling, :30-31), / 255, torchvision antialias resize down to a multiple of dfactor.
 * Bit-identical to the libraries the reference calls for gray / INTER_AREA / /255 / antialias (oracle/preprocess.py);
 * the INTER_LINEAR up-sampling branch follows OpenCV's own arithmetic (pip builds route it through IPP: ~4e-6 relative).
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
  int grayscale;    /* conf["grayscale"]: RGB frames are converted to gray first */
  int resize_max;   /* conf["resize_max"]; <= 0: none.  Only ever down-scales (extract_features.py:124-129) */
  int force_resize; /* conf["force_resize"]: resize to (width, height) */
  int width, height;
  int dfactor;      /* output size is floored to a multiple of dfactor (antialias resize when it changes) */
} imw_pre_conf;

/* output geometry of one frame size (host-only arithmetic, no GPU work): channels / height / width of the tensor
 * imw_preprocess writes, and the per-image workspace */
int imw_preprocess_plan(const imw_pre_conf* conf, int height, int width, int channels, int* out_channels, int* out_height,
                        int* out_width, size_t* workspace_bytes);
size_t imw_preprocess_workspace_bytes(const imw_pre_conf* conf, int batch, int height, int width, int channels);
/* images [B][H][W][channels] uint8 on the DEVICE (channels 1 = gray, 3 = RGB interleaved, as decoded), same size for the
 * batch -> out [B][out_channels][out_height][out_width] fp32 in [0,1]. */
int imw_preprocess(const imw_pre_conf* conf, int batch, int height, int width, int channels, const unsigned char* images,
                   float* out, void* workspace, size_t workspace_bytes, imw_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Match post-processing.
 * Replaces: hloc/match_features.py:236-257 (valid = matches0 > -1, gather of the matched keypoints, rescale to the
 * original image with (k + 0.5) * s - 0.5) for a batch of pairs, on the device, in ascending keypoint order.
 * keypoints [2P][cap][2], matches [2P][cap] (matches0 in even slots), matching_scores [2P][cap] (nullable),
 * counts [2P], scales [2P][2] = original_size / size per image as fp32 (nullable: 1).
 * Outputs: mkpts0/1 [P][cap][2] (resized-image coordinates), mkpts0/1_orig [P][cap][2] (nullable pair), mconf [P][cap]
 * (nullable), mcount [P].
 * ---------------------------------------------------------------------------------------------- */
int imw_gather_matches(int n_pairs, int cap, const float* keypoints, const int* matches, const float* matching_scores,
                       const int* counts, const float* scales, float* mkpts0, float* mkpts1, float* mkpts0_orig,
                       float* mkpts1_orig, float* mconf, int* mcount, imw_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Dense-match aggregation (per-pair array work of hloc/match_dense.py:37-121).
 * imw_quantize_keypoints: `to_cpts` (:37-40): cells [n][cap][2] = rint((k + 0.5) / cell_size) and coords [n][cap][2] = the
 *   fp32 tuple np.round(cell * cell_size - 0.5, 2) the reference uses as dictionary key (cell_size 0: the raw keypoint).
 * imw_nearest_point: `assign_keypoints(update=False)` (:52-59): id of the nearest of `points` [M][2] per query, -1 beyond
 *   max_error.
 * imw_unique_matches: `kpids_to_matches0` (:99-121) for a batch of pairs: ids0/ids1/scores [P][cap] (ids -1 = unassigned,
 *   < id_cap), counts [P] -> matches0 [P][id_cap] (-1 = none), scores0 [P][id_cap] fp16, n_kps0 [P] (= max kept id0 + 1,
 *   the length the reference's arrays have).  n-to-1 conflicts keep the best-scoring match per id on BOTH sides.
 * ---------------------------------------------------------------------------------------------- */
int imw_quantize_keypoints(int n_sets, int cap, const float* keypoints, const int* counts, float cell_size, int* cells,
                           float* coords, imw_stream_t stream);
int imw_nearest_point(int n_query, const float* query, int n_points, const float* points, float max_error, int* ids,
                      imw_stream_t stream);
size_t imw_unique_matches_workspace_bytes(int n_pairs, int id_cap);
int imw_unique_matches(int n_pairs, int cap, int id_cap, const int* ids0, const int* ids1, const float* scores, const int* counts,
                       int* matches0, void* scores0_f16, int* n_kps0, void* workspace, size_t workspace_bytes, imw_stream_t stream);

/* keypoints [n_sets][cap][2], counts [n_sets] (nullable: all cap rows), scales [n_sets][2] -> out = (k + 0.5) * s - 0.5
 * (hloc/match_features.py:251-254, hloc/match_dense.py:655-659) */
int imw_rescale_keypoints(int n_sets, int cap, const float* keypoints, const int* counts, const float* scales, float* out,
                          imw_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * SuperPoint extractor.
 * Replaces: hloc/extractors/superpoint.py:56-57 (SuperPoint._forward) ->
 *           third_party/SuperGluePretrainedNetwork/models/superpoint.py:145-206.
 * Weights: conv kernels re-laid out by the host to [ky*3+kx][Cin][Cout] (1x1: [Cout][Cin]).
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
  const float* w[12]; /* conv1a,1b,2a,2b,3a,3b,4a,4b,Pa,Pb,Da,Db */
  const float* b[12];
  /* optional: 3x3 kernels of conv1b..conv4b, convPa, convDa as two fp16 planes [2][9][Cout][Cin]
     (w = hi + lo * 2^-11, lo stored pre-scaled by 2^11: csrc/split_planes.cuh) for the tcgen05 split-precision path; NULL entries -> CUDA-core path only.
     wp[9] / wp[11] (optional): the 1x1 heads as planes [2][1][Cout_p][256], convPb's 65 outputs zero-padded to
     Cout_p = 128 -- then b[9] must hold 128 values (65 + zeros) */
  const void* wp[12];
} imw_sp_weights;

typedef struct {
  int nms_radius;           /* conf["nms_radius"]        (re-read every call, superpoint.py:145-150) */
  float keypoint_threshold; /* conf["keypoint_threshold"] */
  int max_keypoints;        /* conf["max_keypoints"]; -1 = no cap; 0 or < -1 -> error (superpoint.py:139-141) */
  int remove_borders;       /* conf["remove_borders"] */
  int use_tensor_cores;     /* 1: encoder convs on tcgen05 (two fp16 planes per operand, three products = fp32-equivalent), 0: fp32 CUDA cores */
  int fix_sampling;         /* conf["fix_sampling"] (hloc/extractors/superpoint.py:16-30,46-47): descriptors sampled at
                               (k + 0.5) / (8 [w, h]) with align_corners=False instead of superpoint.py:80-92 */
} imw_sp_conf;

size_t imw_superpoint_workspace_bytes(int batch, int height, int width);

/* image [B][1][H][W] in [0,1] (H,W multiples of 8).
 * keypoints [B][cap][2] (x,y) pixel coords, scores [B][cap], descriptors [B][cap][256] (token-major;
 * the plugin exposes the [256,N] view the reference returns), counts [2][B] = {written[B], total[B]}:
 * total > written means `cap` was too small for max_keypoints = -1 (call again with a larger cap).
 * Optional debug outputs (may be NULL): dense_scores [B][H][W] (before NMS). */
int imw_superpoint_forward(const imw_sp_weights* weights, const imw_sp_conf* conf, int batch, int height, int width,
                           const float* image, int cap, float* keypoints, float* scores, float* descriptors,
                           int* counts, float* dense_scores, void* workspace, size_t workspace_bytes,
                           imw_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * LightGlue matcher.
 * Replaces: hloc/matchers/lightglue.py:54-75 (LightGlue._forward) ->
 *           third_party/LightGlue/lightglue/lightglue.py:488-634, for a batch of independent pairs
 *           (each pair keeps the reference's B=1 semantics: own early exit, own pruning).
 * ---------------------------------------------------------------------------------------------- */
#define IMW_LG_MAX_LAYERS 16

typedef struct {
  /* self block: qkv_w [768][256] rows permuted to [q|k|v][head][dim]; cross block: [to_qk; to_v] [512][256] */
  const float *qkv_w, *qkv_b, *out_w, *out_b;
  const float *ffn0_w, *ffn0_b, *ln_g, *ln_b, *ffn3_w, *ffn3_b;
} imw_lg_block;

typedef struct {
  imw_lg_block self_blk, cross_blk;
} imw_lg_layer;

typedef struct {
  int n_layers;
  int input_dim;              /* 256 (Identity input_proj) or 128 (ALIKED / DISK: Linear input_proj, lightglue.py:392-395) */
  const float* posenc_wr;     /* [32][2] */
  const float *token_w, *token_b; /* [L-1][256], [L-1]   token_confidence */
  const float *final_w, *final_b; /* [L][256][256], [L][256] log_assignment.final_proj */
  const float *match_w, *match_b; /* [L][256], [L]       log_assignment.matchability */
  imw_lg_layer layers[IMW_LG_MAX_LAYERS];
  const float *input_proj_w, *input_proj_b; /* [256][input_dim], [256]; used when input_dim != 256 */
  /* 1: every linear weight matrix W [N][K] above (qkv_w, out_w, ffn0_w, ffn3_w, input_proj_w) is followed in memory by its
     TF32 lo plane W - trunc_tf32(W) [N][K]: the 3xTF32 tcgen05 GEMM then splits activations only.
     2 (ops.lg_pack_weights): followed by its split-fp16 planes [2][N][K] __half (hi = fp16(w), lo = fp16((w - hi) 2^11); the same
     N*K*4 bytes): the linears run on the split-fp16 tcgen05 GEMM (kind::f16, three products per fp32-equivalent product) */
  int has_lo_planes;
  int posenc_dim;   /* 2 (0 is read as 2): posenc_wr [32][2]; 4: add_scale_ori features (sift / doghardnet, lightglue.py:366-377,
                       500-506): posenc_wr [32][4] over (x, y, scale, orientation) */
} imw_lg_weights;

typedef struct {
  float depth_confidence; /* <= 0 disables early stopping (conf -1) */
  float width_confidence; /* <= 0 disables point pruning */
  float filter_threshold; /* hloc: = match_threshold (hloc/matchers/lightglue.py:50) */
  int pruning_min_kpts;   /* lightglue.py:339-344: 1536 = CUDA+flash, 1024 = CUDA, -1 = CPU semantics */
  int use_tensor_cores;   /* linear layers: 1 = tcgen05 3xTF32 split precision (fp32-equivalent, default),
                             2 = tcgen05 single TF32 (fast mode), 0 = fp32 CUDA cores; 1/2 need cap % 128 == 0 */
} imw_lg_conf;

size_t imw_lightglue_workspace_bytes(int n_pairs, int cap);

/* Slot s = 2*pair + side.  keypoints [2P][cap][2], descriptors [2P][cap][256], counts [2P].
 * Outputs: matches [2P][cap] (matches0 in even slots, matches1 in odd; -1 = unmatched),
 * matching_scores [2P][cap], stop [P], prune [2P][cap]. */
int imw_lightglue_forward(const imw_lg_weights* weights, const imw_lg_conf* conf, int n_pairs, int cap,
                          const float* keypoints, const float* descriptors, const int* counts, int* matches,
                          float* matching_scores, int* stop, int* prune, void* workspace, size_t workspace_bytes,
                          imw_stream_t stream);
/* the same with the per-keypoint scales / orientations [2P][cap] of the add_scale_ori features (NULL otherwise) */
int imw_lightglue_forward_so(const imw_lg_weights* weights, const imw_lg_conf* conf, int n_pairs, int cap,
                             const float* keypoints, const float* scales, const float* oris, const float* descriptors,
                             const int* counts, int* matches, float* matching_scores, int* stop, int* prune, void* workspace,
                             size_t workspace_bytes, imw_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * SuperGlue matcher.
 * Replaces: hloc/matchers/superglue.py:42-43 (SuperGlue._forward) ->
 *           third_party/SuperGluePretrainedNetwork/models/superglue.py:228-283, batch of independent pairs.
 * Weights are prepared by the host: BatchNorm (eval) folded into the preceding 1x1 conv, attention projection
 * rows / merge columns permuted from the reference's channel order d*4+h to h*64+d, first keypoint-encoder
 * layer zero-padded from 3 to 16 inputs.
 * ---------------------------------------------------------------------------------------------- */
#define IMW_SG_MAX_LAYERS 32

typedef struct {
  const float *qkv_w, *qkv_b;     /* [768][256]: proj[0..2] stacked */
  const float *merge_w, *merge_b; /* [256][256] */
  const float *mlp0_w, *mlp0_b;   /* [512][512] (BN folded), ReLU */
  const float *mlp1_w, *mlp1_b;   /* [256][512] */
  int is_cross;                   /* GNN_layers[i] == "cross" */
  int pad_;
} imw_sg_layer;

typedef struct {
  int n_layers;
  float bin_score;
  const float* kenc_w[5]; /* [32][16], [64][32], [128][64], [256][128], [256][256] (BN folded) */
  const float* kenc_b[5];
  const float *final_w, *final_b; /* [256][256] */
  imw_sg_layer layers[IMW_SG_MAX_LAYERS];
} imw_sg_weights;

typedef struct {
  int sinkhorn_iterations; /* conf["sinkhorn_iterations"] */
  float match_threshold;   /* conf["match_threshold"] */
  int use_tensor_cores;    /* as imw_lg_conf */
} imw_sg_conf;

size_t imw_superglue_workspace_bytes(int n_pairs, int cap);

/* keypoints [2P][cap][2], scores [2P][cap], descriptors [2P][cap][256] token-major, counts [2P],
 * image_wh [2P][2] = (width, height) of the image each keypoint set came from (superglue.py:65-72).
 * Outputs: matches [2P][cap] (-1 = none), matching_scores [2P][cap]. */
int imw_superglue_forward(const imw_sg_weights* weights, const imw_sg_conf* conf, int n_pairs, int cap, const float* keypoints,
                          const float* scores, const float* descriptors, const int* counts, const int* image_wh, int* matches,
                          float* matching_scores, void* workspace, size_t workspace_bytes, imw_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Mutual nearest neighbour.   Replaces hloc/matchers/nearest_neighbor.py:38-66.
 * Dual-softmax.               Replaces hloc/matchers/dual_softmax.py:50-71.
 * descriptors [2P][cap][dim] token-major (dim % 4 == 0, dim <= 256), counts [2P].
 * matches0 [P][cap] (int32, -1 = none), scores0 [P][cap].
 * ---------------------------------------------------------------------------------------------- */
size_t imw_matcher_workspace_bytes(int n_pairs, int cap);

int imw_nearest_neighbor(int n_pairs, int cap, int dim, const float* descriptors, const int* counts,
                         float ratio_threshold /* <=0: none */, float distance_threshold /* <=0: none */,
                         int do_mutual_check, int use_tensor_cores /* 1: 3xTF32 tcgen05 similarity tiles when cap % 128 == 0 and
                         dim % 32 == 0 (fp32-equivalent); 0: fp32 CUDA cores */, int* matches0, float* scores0, void* workspace,
                         size_t workspace_bytes, imw_stream_t stream);

int imw_dual_softmax(int n_pairs, int cap, int dim, const float* descriptors, const int* counts, float match_threshold,
                     float inv_temperature, int use_tensor_cores, int* matches0, float* scores0, void* workspace,
                     size_t workspace_bytes, imw_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * ALIKED (aliked-n16) extractor.
 * Replaces: hloc/extractors/aliked.py:12-32 -> third_party/LightGlue/lightglue/aliked.py:757-775 (ALIKED.forward:
 * extract_dense_map :709-740, DKD :94-261, SDDH :479-609, deformable convolutions :291-349).
 * Weights prepared by the host (ops.aliked_pack_weights): fp32, BatchNorm folded, conv kernels as [tap][Cin][Cout]
 * (block1.conv1 Cin padded 3 -> 4; the 18-channel offset convolutions padded to 24 outputs), 1x1 kernels as [Cin][Cout].
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
  const float *b1c1_w, *b1c1_b, *b1c2_w, *b1c2_b;                                       /* block1: 3(4) -> 16 -> 16 */
  const float *b2c1_w, *b2c1_b, *b2c2_w, *b2c2_b, *b2ds_w, *b2ds_b;                     /* block2: 16 -> 32, shortcut 1x1 (+bias) */
  const float *b3o1_w, *b3o1_b, *b3c1_w, *b3c1_b, *b3o2_w, *b3o2_b, *b3c2_w, *b3c2_b, *b3ds_w, *b3ds_b; /* block3 (DCN): 32 -> 64 */
  const float *b4o1_w, *b4o1_b, *b4c1_w, *b4c1_b, *b4o2_w, *b4o2_b, *b4c2_w, *b4c2_b, *b4ds_w, *b4ds_b; /* block4 (DCN): 64 -> 128 */
  const float *conv1_w, *conv2_w, *conv3_w, *conv4_w;                                   /* aggregation heads [Cin][32] */
  const float *s0_w, *s2_w, *s4_w, *s6_w;                                               /* score head: [128][8], [9][8][4], [9][4][4], [9][4][1] */
  const float *sd_off0_w, *sd_off0_b, *sd_off2_w, *sd_off2_b, *sd_sf_w, *sd_agg;        /* SDDH: [9][128][32], [32], [32][32], [32], [128][128], [16][128][128] */
} imw_aliked_weights;

typedef struct {
  float detection_threshold;   /* 0.2; <= 0: top-k mode (max_num_keypoints > 0) or mean threshold */
  int max_num_keypoints;       /* -1: up to 20000 (n_limit_max) */
  int nms_radius;              /* 2 */
} imw_aliked_conf;

size_t imw_aliked_workspace_bytes(int n_images, int height, int width, int cap);

/* images [B][channels][H][W] fp32 in [0,1] (channels 1 = gray, repeated to RGB; 3 = RGB), same size for the batch.
 * keypoints [B][cap][2] (x, y sub-pixel, pixel units), scores [B][cap], descriptors [B][cap][128] (L2-normalised),
 * counts [2B]: [0,B) keypoints written, [B,2B) keypoints the reference returns (> cap = overflow).
 * dbg_score_map [B][H][W] / dbg_feature_map [B][H][W][128]: optional copies of the dense maps (NULL to skip). */
int imw_aliked_forward(const imw_aliked_weights* weights, const imw_aliked_conf* conf, int n_images, int channels, int height,
                       int width, const float* images, int cap, float* keypoints, float* scores, float* descriptors, int* counts,
                       float* dbg_score_map, float* dbg_feature_map, void* workspace, size_t workspace_bytes, imw_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * SIFT extractor.
 * Replaces: hloc/extractors/sift.py (opencv backend) -> cv2.SIFT_create(...).detectAndCompute on uint8(trunc(x * 255))
 * with firstOctave -1, then the LightGlue wrapper glue (lightglue/sift.py): filter_dog_point (nms_radius 0), top-k on the
 * response, RootSIFT.  No weights.
 * ---------------------------------------------------------------------------------------------- */
#define IMW_SIFT_MAX_TAPS 64

typedef struct {
  int n_octave_layers;      /* cv2 nOctaveLayers (the wrapper passes its num_octaves = 4 here) */
  float contrast_threshold; /* cv2 contrastThreshold (wrapper: detection_threshold) */
  float edge_threshold;     /* cv2 edgeThreshold */
  double sigma;             /* 1.6 (a double, as cv::SIFT keeps it: the pyramid sigmas are computed from it in double) */
  int max_keypoints;        /* cv2 nfeatures and the wrapper's top-k; <= 0: all */
  int nms_radius;           /* -1: no pixel filter (None), 0: filter_dog_point's one-keypoint-per-pixel rule */
  int rootsift;             /* 1: RootSIFT descriptors (unit L2 norm), 0: cv2's integer-valued descriptors */
} imw_sift_conf;

/* host-only: octave count of a height x width input and the Gaussian kernels of the pyramid (ksizes [L+3], taps
 * [L+3][IMW_SIFT_MAX_TAPS]; index 0 is the blur of the doubled base image).  Any output may be NULL. */
int imw_sift_plan(const imw_sift_conf* conf, int height, int width, int* n_octaves, int* ksizes, float* taps);
size_t imw_sift_workspace_bytes(const imw_sift_conf* conf, int batch, int height, int width);
/* images [B][H][W] fp32 gray in [0,1] (H, W <= 4096).  Outputs in descending response order: keypoints [B][cap][2] (x, y),
 * scores [B][cap] (response), scales [B][cap] (size), oris [B][cap] (radians), descriptors [B][cap][128];
 * counts [2B]: [0,B) written, [B,2B) keypoints the reference returns (> cap: call again with a larger cap; -1: more
 * extrema than the internal per-image capacity).  dbg_pyramid (nullable): the Gaussian layers, per image octave after octave,
 * (L+3) layers of (2H >> o) x (2W >> o) each. */
int imw_sift_forward(const imw_sift_conf* conf, int batch, int height, int width, const float* images, int cap, float* keypoints,
                     float* scores, float* scales, float* oris, float* descriptors, int* counts, float* dbg_pyramid,
                     void* workspace, size_t workspace_bytes, imw_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * LoFTR dense matcher.
 * Replaces: hloc/matchers/loftr.py:41-71 -> kornia.feature.LoFTR == third_party/SE2LoFTR/src/loftr/loftr.py:29-75
 * (ResNet-FPN backbone, coarse linear-attention transformer, dual-softmax coarse matching, fine refinement).
 * Weights prepared by the host: BatchNorm folded, conv kernels as two fp16 planes [2][k*k][Cout][Cin] with the
 * 196-channel tensors zero-padded to 256, encoder q/k/v stacked to [3*d][d].
 * ---------------------------------------------------------------------------------------------- */
typedef struct { const void* w; const float* b; int cin, cout, ksize, stride; } imw_loftr_conv;
typedef struct {
  const float *conv1_w, *conv1_b;        /* 7x7 stem: [49][128] fp32 (BN folded), [128] */
  imw_loftr_conv l1[4], l2[4], l2_down, l3[4], l3_down; /* BasicBlocks: conv1, conv2 of block 0 then block 1 */
  imw_loftr_conv l3_out, l2_out, l2_out2[2], l1_out, l1_out2[2];
} imw_loftr_backbone;
typedef struct {
  const float *qkv_w, *merge_w, *mlp0_w, *mlp2_w, *norm1_g, *norm1_b, *norm2_g, *norm2_b;
  int is_cross, pad_;
} imw_loftr_layer;
typedef struct {
  imw_loftr_backbone backbone;
  const float* pos_enc;                  /* [hc*wc][256] for the current image size (position_encoding.py:6-42) */
  int n_coarse, n_fine;
  imw_loftr_layer coarse[8], fine[2];
  const float *down_proj_w, *down_proj_b, *merge_feat_w, *merge_feat_b; /* [128][256],[128],[128][256],[128] */
  /* 1 (ops.loftr_pack_weights): every encoder weight matrix W [N][K] (qkv_w, merge_w, mlp0_w, mlp2_w) is followed in memory by its
     split-fp16 planes [2][N][K] __half: the coarse linears then run on the split-fp16 tcgen05 GEMM (see imw_lg_weights) */
  int has_f16_planes;
} imw_loftr_weights;
typedef struct {
  float match_threshold; /* match_coarse.thr */
  float temperature;     /* match_coarse.dsmax_temperature (0.1) */
  int border_rm;         /* match_coarse.border_rm (2) */
  int use_tensor_cores;  /* encoder linears: 1 = 3xTF32, 2 = TF32, 0 = fp32 CUDA cores (convs are always tcgen05 split-fp16) */
} imw_loftr_conf;

size_t imw_loftr_workspace_bytes(int n_pairs, int height, int width, int max_matches);
size_t imw_loftr_workspace_bytes_hw(int n_pairs, int height0, int width0, int height1, int width1, int max_matches);

/* images [2P][H][W] fp32 (H, W multiples of 8): slot 2p indexes the rows of the confidence matrix ("image0" of the LoFTR
 * module), slot 2p+1 its columns; the sub-pixel refinement moves the slot-2p+1 keypoint.
 * keypoints0/1 [P][max_matches][2], confidence [P][max_matches], counts [P] (matches in ascending row-cell order).
 * dbg_* may be NULL: coarse features after the transformer [2P][cap][256] (cap = L rounded up to 128) / after the
 * backbone [2P][L][256]. */
int imw_loftr_forward(const imw_loftr_weights* weights, const imw_loftr_conf* conf, int n_pairs, int height, int width,
                      const float* images, int max_matches, float* keypoints0, float* keypoints1, float* confidence, int* counts,
                      float* dbg_feat_c, float* dbg_backbone_c, void* workspace, size_t workspace_bytes, imw_stream_t stream);

/* The same for pairs whose two images differ in size (the LoFTR module then runs its backbone per image,
 * third_party/SE2LoFTR/src/loftr/loftr.py:48-56; hloc's minima_loftr / loftr_aachen-style confs do not force a common size).
 * images0 [P] frames of height0 x width0 (rows of the confidence matrix), images1 [P] frames of height1 x width1; stride0 /
 * stride1 = floats between consecutive frames of a side.  weights->pos_enc is the position encoding of side 0
 * ([height0/8 * width0/8][256]), pos_enc1 that of side 1 (NULL: same as side 0).  dbg_* are laid out for max(L0, L1). */
int imw_loftr_forward_hw(const imw_loftr_weights* weights, const imw_loftr_conf* conf, int n_pairs, int height0, int width0,
                         int height1, int width1, const float* images0, long long stride0, const float* images1, long long stride1,
                         const float* pos_enc1, int max_matches, float* keypoints0, float* keypoints1, float* confidence, int* counts,
                         float* dbg_feat_c, float* dbg_backbone_c, void* workspace, size_t workspace_bytes, imw_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * MAGSAC++ geometric verification.
 * Replaces: imcui/ui/utils.py:352-372 (cv2.findHomography / cv2.findFundamentalMat, method=cv2.USAC_MAGSAC) for a
 * batch of correspondence sets.  pts0/pts1 [n_sets][cap][2] pixel coordinates, counts [n_sets].
 * model_type 0 = homography, 1 = fundamental matrix.  Outputs: models [n_sets][9] (fp64, row-major, last element 1;
 * all zeros = no model), masks [n_sets][cap] (1 = inlier: residual <= threshold), n_inliers / n_iters [n_sets].
 * ---------------------------------------------------------------------------------------------- */
int imw_magsac(int n_sets, int cap, const float* pts0, const float* pts1, const int* counts, int model_type, float threshold,
               float confidence, int max_iters, unsigned seed, double* models, unsigned char* masks, int* n_inliers,
               int* n_iters, imw_stream_t stream);

/* Unit-test hooks: out[M][N] = A[M][K] W[N][K]^T + bias on the tcgen05 path (split = 1: single TF32,
 * split = 3: 3xTF32 fp32-equivalent, split = 4: the same with W [2N][K] = weights + host-computed lo plane, split = 5: the
 * split-fp16 GEMM the linears run on, W [2N][K] = weights + their two fp16 planes, split = 6: the same with A handed over as
 * split-fp16 planes [2][M][K] too, as a producer kernel writes them) and on the CUDA-core fp32 path. */
int imw_debug_gemm_tf32(const float* A, const float* W, const float* bias, float* out, int M, int N, int K, int split,
                        imw_stream_t stream);
int imw_debug_gemm_fp32(const float* A, const float* W, const float* bias, float* out, int M, int N, int K,
                        imw_stream_t stream);

/* One 3x3 conv layer of the SuperPoint stack (NHWC fp32 in/out, weights [9][Cin][Cout], optional ReLU and fused
 * 2x2 max-pool): bench.py times the dominant kernel alone through this hook. */
/* Attention on q/k/v [slots][4 heads][cap][64] -> ctx [slots][cap][256]; use_tc: tcgen05 3xTF32 kernel vs fp32 CUDA cores */
int imw_debug_attention(const float* q, const float* k, const float* v, const int* counts, int slots, int cap, float scale,
                        int cross, int use_tc, float* ctx, void* scratch, size_t scratch_bytes, imw_stream_t stream);
int imw_debug_conv3x3_tc(const float* in, const float* w_tap_cin_cout, const float* bias, float* out, int batch, int height,
                         int width, int cin, int cout, int relu, int pool, void* scratch, size_t scratch_bytes,
                         imw_stream_t stream);
/* the tcgen05 conv alone on pre-split operands: in [2][B][H][W][Cin] fp16, w [2][9][Cout][Cin] fp16, out planes */
int imw_debug_conv3x3_tc_planes(const void* in_planes, const void* w_planes, const float* bias, void* out_planes, int batch,
                                int height, int width, int cin, int cout, int relu, int pool, imw_stream_t stream);
/* SuperPoint conv1a (1 -> 64) evaluated inside the conv1b (64 -> 64) tcgen05 kernel: image [B][H][W] fp32, w1a [9][64],
 * w1b_planes [2][9][64][64] fp16 -> conv1b output planes [2][B][H/2][W/2][64] (pool = 1) */
/* tuning hook: images per pass of the SuperPoint conv stack (default 8); returns the value in effect */
int imw_debug_set_sp_sub(int n);
/* 1 (default): 3x3 stride-1 tcgen05 convs with W % 8 == 0 use the halo-copy kernel, 0: the per-tap generic kernel; < 0: query */
int imw_debug_set_conv_halo(int on);
/* 1 (default) = 3x3 stride-1 convs with W % 8 == 0 (and the fused first layer) on CTA pairs, tcgen05 cta_group::2; 0 = their
 * single-CTA predecessors; 2 = probe (B halves of the two CTAs swapped: wrong results); 1 + 256 / 512 / 1024 = timing ablations of
 * the 64-channel pair kernel (no conv1a arithmetic / no epilogue arithmetic / no MMAs: garbage results); < 0 = query */
int imw_debug_set_conv_pair(int mode);
/* timing ablations of the split-fp16 GEMM: bit 1 = no operand split, bit 2 = no epilogue (garbage results); 0 = off; < 0 = query */
int imw_debug_set_gemm_ablate(int mode);
int imw_debug_conv1ab_fused(const float* image, const float* w1a, const float* b1a, const void* w1b_planes, const float* b1b,
                            void* out_planes, int batch, int height, int width, int pool, imw_stream_t stream);
int imw_debug_conv3x3(const float* in, const float* w, const float* bias, float* out, int batch, int height, int width,
                      int cin, int cout, int relu, int pool, imw_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* IMW_B200_H */
