/*
 * linetr_b200 - C ABI of the B200-native LineTR line-descriptor + NN-matcher hot path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch types, no exceptions.
 * Every entry point replaces a piece of the reference's Python call surface (paths are
 * relative to the reference checkout, yosungho/LineTR):
 *
 *   ltr_create / ltr_destroy   <- LineTransformer.__init__ + load_state_dict
 *                                 (models/line_transformer.py:203-223): takes the raw
 *                                 checkpoint tensors by their state-dict names, folds the
 *                                 eval-mode BatchNorms, repacks heads, uploads to the GPU.
 *   ltr_encode                 <- LineTransformer.forward (models/line_transformer.py:225-249)
 *                                 = normalize_keylines (:22-38) + KeylineEncoder.forward
 *                                 (:107-130, models/line_attention.py:42-94) +
 *                                 SelfAttentionalLayer.forward (:176-183) + final_proj +
 *                                 F.normalize (:245-246).
 *   ltr_match                  <- get_dist_matrix (models/line_process.py:198-201) +
 *                                 LineTransformer.subline2keyline (models/line_transformer.py:277-282)
 *                                 + nn_matcher_distmat (models/nn_matcher.py:3-31); with
 *                                 descriptors as input it is nn_matcher (models/nn_matcher.py:33-43).
 *   ltr_match_distmat          <- nn_matcher_distmat on a caller-supplied distance matrix.
 *
 * Conventions: return 0 on success, a negative LTR_E_* code on failure (message via
 * ltr_last_error(), thread-local).  All device pointers are caller-owned and must live on
 * the device the model was created on.  Calls are asynchronous with respect to the host
 * and ordered on the given CUDA stream (pass the cudaStream_t as void*; NULL = default
 * stream).  There is no CPU fallback: every function fails if no CUDA device is usable.
 */
#ifndef LINETR_B200_H_
#define LINETR_B200_H_

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LTR_ABI_VERSION 3

#define LTR_OK 0
#define LTR_E_INVALID (-1)   /* bad argument / missing checkpoint tensor / shape mismatch */
#define LTR_E_CUDA (-2)      /* CUDA runtime error (no device, launch failure, OOM) */
#define LTR_E_WORKSPACE (-3) /* caller workspace too small */
#define LTR_E_UNSUPPORTED (-4)

typedef struct LtrModel LtrModel;

/* One checkpoint tensor, fp32, host memory, in the reference state-dict layout
 * (SURVEY.md 8a "State-dict contract"); `name` is the state-dict key. */
typedef struct {
  const char* name;
  const float* data;
  int64_t numel;
} LtrTensor;

typedef struct {
  int32_t d_model;        /* 256  (config 'descriptor_dim') */
  int32_t n_heads;        /* 4    (config 'n_heads') */
  int32_t d_inner;        /* 1024 (config 'd_inner') */
  int32_t n_desc_layers;  /* config 'n_line_descriptive_layers'; only the LAST layer is live
                             in the reference (line_transformer.py:123-125 never chains) */
  int32_t n_sig_layers;   /* 7 (line_transformer.py:213) */
} LtrConfig;

/* Tokenised lines of a batch of images, rows of all images concatenated.
 * Image i owns lines [cu_lines[i], cu_lines[i+1]).  For a uniform batch [B, L, ...] pass
 * cu_lines_host = cu_lines_dev = NULL and lines_per_image = L.
 * The token mask ('mask_sublines') is deliberately absent: in the reference it masks
 * query rows of which only the always-valid CLS row is consumed (models/line_attention.py:
 * 15-16,62-63; models/line_transformer.py:128), so it cannot change the output. */
typedef struct {
  const float* sublines;  /* [n_lines, 2, 2] end points, pixels */
  const float* resp;      /* [n_lines, 1] */
  const float* angle;     /* [n_lines, 2] */
  const float* pnt;       /* [n_lines, n_tokens, 2] token positions, pixels */
  const float* desc;      /* [n_lines, n_tokens, d_model] sampled descriptors */
  const float* score;     /* [n_lines, n_tokens, 1] */
  const int32_t* cu_lines_host; /* [n_images + 1] or NULL (uniform) */
  const int32_t* cu_lines_dev;  /* device copy of the same, or NULL (uniform) */
  int32_t n_images;
  int32_t n_lines;         /* total lines over all images */
  int32_t n_tokens;        /* T (config 'max_tokens'), 1..128 */
  int32_t lines_per_image; /* used when cu_lines_* are NULL */
  float image_width;       /* LineTransformer.image_shape (ctor-time, :206,238) */
  float image_height;
} LtrEncodeInput;

/* Bytes of device scratch ltr_encode needs for this problem size. */
int64_t ltr_encode_workspace_bytes(const LtrModel* m, int32_t n_images, int32_t n_lines,
                                   int32_t n_tokens);

int ltr_create(const LtrTensor* tensors, int32_t n_tensors, const LtrConfig* cfg,
               int32_t device, LtrModel** out);
void ltr_destroy(LtrModel* m);

/* Outputs of ltr_encode (device, caller-owned; any of them may be NULL).
 * desc_cf:    unit-norm descriptors channel-first, image i at offset d_model*cu_lines[i],
 *             element (c, l) at c*L_i + l - for a uniform batch exactly the reference's
 *             line_desc [B, d_model, L].
 * desc_rows:  the same descriptors row-major [n_lines, d_model] (matcher layout).
 * desc_tiles: the same descriptors as the split-bf16 "tile image" the tensor-core matcher
 *             contracts (ltr_desc_tiles_bytes(n_lines) bytes, opaque): hand it to ltr_match
 *             (LtrMatchInput.tiles0/1) and the matcher skips its own fp32 -> tile conversion.
 *             Needs desc_rows != NULL and desc_cf == NULL (it is written by the same fused
 *             projection + L2-normalisation launch as desc_rows). */
typedef struct {
  float* desc_cf;
  float* desc_rows;
  void* desc_tiles;
} LtrEncodeOutput;

int64_t ltr_desc_tiles_bytes(int32_t n_lines);

int ltr_encode(LtrModel* m, const LtrEncodeInput* in, const LtrEncodeOutput* out,
               void* workspace, int64_t workspace_bytes, void* stream);

#define LTR_LAYOUT_ROWS 0          /* [n, d] */
#define LTR_LAYOUT_CHANNEL_FIRST 1 /* [d, n] per image */

/* A batch of independent image pairs.  Side s of pair p owns sublines
 * [cu_s[p], cu_s[p+1]) (uniform: p*n_s .. (p+1)*n_s when cu_s == NULL).
 * Keyline merging (LineTransformer.subline2keyline): the adjacency of
 * models/line_process.py:163-167 is block-constant with weight 1/n_sub over contiguous
 * sublines, so it is passed as CSR offsets: keyline g (global numbering over the whole
 * batch) owns sublines [sub_off_s[g], sub_off_s[g+1]) in global subline numbering and pair
 * p owns keylines [cuk_s[p], cuk_s[p+1]).  With sub_off0 == sub_off1 == NULL every subline
 * is its own keyline (A = I) and no merging pass runs. */
typedef struct {
  const float* desc0;
  const float* desc1;
  int32_t layout;          /* LTR_LAYOUT_* of desc0/desc1 */
  int32_t d;               /* descriptor dim, multiple of 16 */
  int32_t n_pairs;
  int32_t n0, n1;          /* sublines per image when cu0/cu1 are NULL */
  const int32_t* cu0;      /* device [n_pairs+1] or NULL */
  const int32_t* cu1;
  const int32_t* sub_off0; /* device [total keylines side 0 + 1] or NULL */
  const int32_t* sub_off1;
  const int32_t* cuk0;     /* device [n_pairs+1] keyline offsets, required iff sub_off0 != NULL */
  const int32_t* cuk1;
  int32_t max_n0, max_n1;  /* max sublines per image on each side (grid sizing; var-len only) */
  int32_t max_k0, max_k1;  /* max keylines per image on each side (keyline merging only) */
  int64_t dist_pair_stride; /* elements between consecutive pairs' matrices in `dist_key`;
                               0 = max_k0*max_k1 (or max_n0*max_n1 without merging) */
  float nn_thresh;         /* strict '<' (models/nn_matcher.py:18) */
  int32_t mutual;
  int32_t total_n0, total_n1; /* total sublines per side (required with cu0/cu1; 0 = n_pairs*n0/n1) */
  int32_t dist_mode;       /* 0: 2 - 2<a,b> (unit descriptors; models/nn_matcher.py:37-38,
                              models/line_process.py:199-200); 1: |a|^2 + |b|^2 - 2<a,b>
                              (evaluations/matcher.py:66-70); mode 1 needs d == 256, no merging */
  /* Optional: descriptor tile images written by ltr_encode (LtrEncodeOutput.desc_tiles) for the SAME
   * descriptors as desc0/desc1.  Usable when d == 256, the batch is uniform (cu0 == cu1 == NULL),
   * n0 % 128 == 0, n1 % 128 == 0 and tiles_row0_s % 128 == 0; tiles_lines_s = the n_lines the image
   * was produced for, tiles_row0_s = row of this side's first line inside it (both sides may live in
   * one image: one ltr_encode over 2P images).  NULL = the matcher converts desc0/desc1 itself. */
  const void* tiles0;
  const void* tiles1;
  int32_t tiles_lines0, tiles_lines1;
  int32_t tiles_row0_0, tiles_row0_1;
} LtrMatchInput;

/* Multi-GPU: the path's ONE collective - every rank learns the per-pair match counts of all ranks - fused
 * into the matcher's last kernel.  The caller owns a SYMMETRIC int32 buffer (same size on every rank, peer
 * mapped over NVLink, e.g. torch.distributed._symmetric_memory) laid out as
 *     counts[LTR_GATHER_SLOTS][world][n_pairs]  followed by  flags[LTR_GATHER_SLOTS][world].
 * The thread block of the matcher's exact kernel that completes the last pair's counts (block 0 when no
 * decision needed the exact path) stores this rank's n_pairs counts into row `rank` of slot `slot`
 * of EVERY rank's buffer - one multimem.st per element through the NVSwitch multicast address when `mc_base`
 * is given, else plain stores through the `world` peer pointers - and then publishes flags[slot][rank] =
 * epoch the same way.  No NCCL kernel, no extra launch on the producing side; ltr_gather_wait (one tiny
 * block) waits for the `world` flags of a slot and copies the gathered counts out.  A rank may run at most
 * LTR_GATHER_SLOTS - 2 steps ahead of its own ltr_gather_wait calls. */
#define LTR_GATHER_SLOTS 8
typedef struct {
  void* mc_base;               /* multicast address of the symmetric buffer or NULL */
  void* const* peer_bases;     /* device array [world]: address of the buffer on every rank (used if !mc_base) */
  int32_t rank, world;
  int32_t slot;                /* 0 .. LTR_GATHER_SLOTS-1 */
  int32_t epoch;               /* > 0, increasing per use of a slot */
} LtrPeerGather;

/* Waits (on the stream) until flags[slot][0..world) of the LOCAL symmetric buffer have all reached `epoch`, then
 * copies counts[slot] (world * n_pairs int32) to `out`. */
int ltr_gather_wait(const void* local_base, int32_t world, int32_t n_pairs, int32_t slot, int32_t epoch,
                    int32_t* out, int32_t device, void* stream);

/* Outputs (device).  Keyline k of side 0 lives at index cuk0[p]+k (cu0[p]+k without
 * merging, p*n0+k for a uniform batch); likewise side 1.
 * matches0[k] = index (local to the pair) of the matched keyline in side 1, or -1;
 * scores0[k]  = distance to the nearest neighbour;
 * nn1[k1]     = nearest side-0 keyline of every side-1 keyline (only written if mutual);
 * counts[p]   = number of matches of pair p;
 * dist_key    = keyline distance matrices, pair p at p*dist_pair_stride, row-major
 *               [K0_p, K1_p] (Matching's 'matching_scores_l');
 * dist_sub    = scratch for subline distances [n_pairs, max_n0*max_n1], merging only.
 * workspace   = device scratch of ltr_match_workspace_bytes(in) bytes (tile images, per-line
 *               argmin slots).
 * dist_key may be NULL when there is no key-line merging and d == 256: the distance matrix is
 * then never materialised (row argmin lives in the epilogue of the tensor-core contraction).
 * matches0 == NULL (with scores0, nn1, counts) computes dist_key only (get_dist_matrix). */
typedef struct {
  int32_t* matches0;
  float* scores0;
  int32_t* nn1;
  int32_t* counts;
  float* dist_key;
  float* dist_sub;
  void* workspace;
  int64_t workspace_bytes;
  const LtrPeerGather* gather;   /* optional (d == 256, no merging): publish `counts` to all ranks, see above */
} LtrMatchOutput;

int64_t ltr_match_workspace_bytes(const LtrMatchInput* in);

int ltr_match(const LtrMatchInput* in, const LtrMatchOutput* out, int32_t device, void* stream);

/* nn_matcher_distmat on caller-supplied distance matrices (device, row-major [n0, n1],
 * pair p at p*dist_pair_stride, 0 = n0*n1); negative entries are clipped to 0 as the
 * reference does (models/nn_matcher.py:12). */
int ltr_match_distmat(const float* dist, int32_t n_pairs, int32_t n0, int32_t n1,
                      int64_t dist_pair_stride, float nn_thresh, int32_t mutual,
                      int32_t* matches0, float* scores0, int32_t* nn1, int32_t* counts,
                      int32_t device, void* stream);

/* LineTransformer.subline2keyline alone: dist_key[p] = A0_p @ dist_sub[p] @ A1_p^T with the
 * adjacencies given as CSR offsets (see LtrMatchInput).  dist_sub: pair p at p*stride_sub,
 * row-major [S0_p, S1_p]; dist_key: pair p at p*stride_key, row-major [K0_p, K1_p]. */
int ltr_merge_sublines(const float* dist_sub, int64_t stride_sub, int32_t n_pairs,
                       const int32_t* cuk0, const int32_t* cuk1, const int32_t* sub_off0,
                       const int32_t* sub_off1, int32_t max_k0, int32_t max_k1, float* dist_key,
                       int64_t stride_key, int32_t device, void* stream);

/* GPU line tokenizer - the step that feeds ltr_encode (reference line_tokenizer +
 * sample_descriptors, models/line_process.py:86-196).  The host supplies per key line (device
 * arrays): start point, end point before and after the in-place clip to (W-0.6, H-0.6) [K,2]
 * float64, detector length [K] float64, angle code [K,2] float32, n_tok = ceil(length /
 * token_distance) [K], first subline index sub0 [K+1] and the key line of every subline [S].
 * Outputs (device, fp32) in the tokenizer's layout: sublines [S,2,2], pnt [S,T,2], mask
 * [S,T+1,1], resp [S,1], angle [S,2], desc [S,T,256] (bilinear grid_sample of dense_desc
 * [256,desc_h,desc_w] + L2 normalisation), score [S,T,1] (dense_score [score_h,score_w] at the
 * rounded token position). */
typedef struct {
  const double* sp;
  const double* ep;
  const double* ep_clipped;
  const double* length;
  const float* angle;
  const int32_t* n_tok;
  const int32_t* sub0;
  const int32_t* sub2line;
  int32_t n_keylines, n_sublines, n_tokens;
  double token_distance;
  const float* dense_desc;
  int32_t desc_channels, desc_h, desc_w;
  const float* dense_score;
  int32_t score_h, score_w;
  int32_t align_corners;   /* the reference keys this on the torch version (line_process.py:93) */
} LtrTokenizeInput;

int ltr_tokenize(const LtrTokenizeInput* in, float* sublines, float* pnt, float* mask, float* resp,
                 float* angle, float* desc, float* score, int32_t device, void* stream);

/* Generic row-major linear layer Y = act(X W^T + b) (+ R) on the library's GEMM engine;
 * exported so the engine can be unit-tested in isolation.  act: 0 none, 1 relu, 2 gelu(erf). */
int ltr_linear(const float* x, int32_t ldx, const float* w, const float* bias, const float* res,
               int32_t ldr, float* y, int32_t ldy, int32_t m, int32_t n, int32_t k, int32_t act,
               int32_t device, void* stream);

/* The same on the tensor-core engine (gemm_img.cuh: persistent, TMA-fed split-bf16 tile images,
 * tcgen05): x is converted to a
 * split-bf16 tile image, the GEMM writes fp32 rows into `y` (may be NULL) and - when
 * `y_from_image` is given - also the split-bf16 image of the result, which is converted back
 * to fp32 rows [m, n] there so that both outputs can be checked.  n % 64 == 0, k % 64 == 0;
 * bn_hint: 0 (auto), 64, 128 or 256.  Synchronous; unit-test hook only. */
int ltr_linear_img(const float* x, int32_t ldx, const float* w_host, const float* bias,
                   const float* res, int32_t ldr, float* y, int32_t ldy, float* y_from_image,
                   int32_t m, int32_t n, int32_t k, int32_t act, int32_t bn_hint, int32_t device,
                   void* stream);

/* ltr_linear_img with the row-normalising epilogue the encoder uses (n = 256 fixed): norm = 1:
 * y = LayerNorm(x W^T + b (+ res); eps) * gamma + beta (+ add)   - MultiHeadAttention / FeedForward
 * tails, models/line_attention.py:51-53,73-75, plus the `klines_pos +` of models/line_transformer.py:128;
 * norm = 2: y = (x W^T + b) / max(||.||_2, 1e-12)               - final_proj + F.normalize,
 * models/line_transformer.py:245-246.  Synchronous; unit-test hook only. */
int ltr_linear_img_norm(const float* x, int32_t ldx, const float* w_host, const float* bias,
                        const float* res, int32_t ldr, int32_t norm, float eps, const float* gamma,
                        const float* beta, const float* add, int32_t ldadd, float* y, int32_t ldy,
                        float* y_from_image, int32_t m, int32_t k, int32_t device, void* stream);

/* Instrumentation.  Kernel launches issued by this library since the last reset. */
int64_t ltr_launch_count(void);
void ltr_reset_launch_count(void);
/* Per-kernel-class device timing with CUDA events on the launching stream.
 * ltr_profile_begin() arms it; ltr_profile_end() synchronises, fills `names` (pointers to
 * static strings), `ms` (summed elapsed per class) and `launches`, returns the class count. */
void ltr_profile_begin(void);
int ltr_profile_end(const char** names, float* ms, int32_t* launches, int32_t max_classes);

const char* ltr_last_error(void);
int ltr_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* LINETR_B200_H_ */
