/*
 * psalm_b200 — C ABI of the B200-native PSALM inference hot path.
 *
 * Plain pointers and sizes only (no torch / ATen types).  Every entry point
 *   - takes DEVICE pointers unless the parameter name ends in `_host`,
 *   - enqueues work on `stream` (a cudaStream_t passed as void*) and never synchronises,
 *   - returns 0 on success or a negative PSALM_E_* code; psalm_last_error() holds the message.
 *     (The reference only printf()s launch failures — ms_deform_im2col_cuda.cuh:953-957 — and its
 *      Python caller swallows every exception — ops/modules/ms_deform_attn.py:117; we never do.)
 *
 * Reference interfaces each entry point replaces are cited per function as
 * (path relative to /root/reference/psalm/model/…:line).
 */
#ifndef PSALM_B200_H_
#define PSALM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PSALM_ABI_VERSION 1

/* element types */
enum { PSALM_F32 = 0, PSALM_F16 = 1, PSALM_BF16 = 2, PSALM_U8 = 3 };

/* error codes */
enum {
  PSALM_OK = 0,
  PSALM_E_ARG = -1,      /* bad argument (shape, dtype, alignment, null pointer) */
  PSALM_E_UNSUPPORTED = -2,
  PSALM_E_CUDA = -3      /* CUDA runtime / launch error */
};

int psalm_abi_version(void);
const char* psalm_last_error(void);
/* compute capability the library was compiled for (100 => sm_100a) */
int psalm_compiled_arch(void);

/* ------------------------------------------------------------------------------------------
 * Multi-scale deformable attention, forward (sampling + aggregation).
 *
 * Replaces: ms_deform_attn_forward (mask_decoder/Mask2Former_Simplify/modeling/pixel_decoder/
 *   ops/src/ms_deform_attn.h:25-44 -> ops/src/cuda/ms_deform_attn_cuda.cu:25-85 ->
 *   ms_deformable_im2col_gpu_kernel, ops/src/cuda/ms_deform_im2col_cuda.cuh:243-304).
 *
 *   out[b,q,m,:] = sum_{l,p} w[b,q,m,l,p] * bilinear(value_l[b,:,m,:], loc[b,q,m,l,p,:])
 *   zero padding outside the map, pixel-centre convention (x_im = loc_x * W_l - 0.5).
 *
 *   value   [B,S,M,D]      (value_layout 0, the reference layout)   dtype value_dtype
 *           [B,M,S,D]      (value_layout 1, head-major, used by the fused pipeline)
 *   shapes  [L,2] int64 (H_l, W_l), starts [L] int64 — DEVICE pointers as in the reference
 *           (spatial_shapes.data<int64_t>()), or HOST pointers when shapes_on_host != 0.
 *   loc     [B,Lq,M,L,P,2], w [B,Lq,M,L,P]                          dtype loc_dtype
 *           (the reference requires loc_dtype == value_dtype; PSALM_F32 is always accepted)
 *   out     [B,Lq,M*D]                                              dtype value_dtype
 *   All tensors contiguous; out is fully overwritten (no pre-zeroing needed).
 * ------------------------------------------------------------------------------------------ */
int psalm_msda_forward(const void* value, const int64_t* shapes, const int64_t* starts,
                       const void* loc, const void* w, void* out,
                       int B, int S, int M, int D, int L, int Lq, int P,
                       int value_dtype, int loc_dtype, int value_layout, int shapes_on_host,
                       void* stream);

/* Fused sampling for the encoder layer: takes the raw outputs of the sampling_offsets /
 * attention_weights Linear layers and does softmax(L*P) + reference-point generation
 * (get_reference_points, pixel_decoder/msdeformattn.py:76-87, valid_ratios == 1) +
 * location arithmetic (ops/modules/ms_deform_attn.py:104-110) + sampling in one kernel, so
 * `sampling_locations` and `attention_weights` never exist in HBM.
 *
 *   value  [B,M,S,D] head-major, dtype value_dtype
 *   ow     [B,Lq,M*L*P*3]: per query, first M*L*P*2 offsets (m,l,p,xy order), then M*L*P logits
 *          dtype ow_dtype (F32 / F16 / BF16).  Lq must equal S (encoder self-attention).
 *   out    [B,Lq,M*D] dtype value_dtype
 *   shapes_host/starts_host: HOST int64 arrays.
 * Three kernels sit behind the call (psalm_set_msda_impl: 0 = auto (= 1), 1, 2, 3):
 *   1  one lane group per (query, head), corners gathered from global memory / L1 (measured fastest);
 *   2  paired columns (the two x-adjacent bilinear corners are one contiguous access);
 *   3  (16-bit storage, M=8, D=32, L=3, P=4, levels ordered coarse to fine) value tiles of a 16x16 cell of the finest
 *      level (+ halo) staged in shared memory by TMA (cp.async.bulk.tensor.4d, zero fill = the op's zero padding), the
 *      gather + weighted sum as ldmatrix gathers + mma.sync (csrc/msda_smem.cu); samples beyond the halo
 *      (psalm_set_msda_halo, default 5 pixels) read global memory - results do not depend on the halo.  Correct,
 *      selectable, measured slower than 1 (DESIGN.md section 5). */
int psalm_set_msda_impl(int impl);
int psalm_set_msda_halo(int halo);
int psalm_msda_encoder_fused(const void* value, const void* ow, void* out,
                             const int64_t* shapes_host, const int64_t* starts_host,
                             int B, int S, int M, int D, int L, int P,
                             int value_dtype, int ow_dtype, void* stream);

/* ------------------------------------------------------------------------------------------
 * Swin windowed multi-head self-attention (W-MSA / SW-MSA), fused.
 * Replaces: WindowAttention.forward + the roll / pad / window_partition / window_reverse copies of
 *   SwinTransformerBlock.forward (multimodal_encoder/swin_trans.py:117-149, 207-245) and the shift
 *   mask of BasicLayer.forward (swin_trans.py:370-387).
 *   qkv      [B, H*W, 3*C]  output of the qkv Linear on norm1(x), UNPADDED and UNSHIFTED token order
 *   qkv_bias [3*C]          value of a zero-padded token after the Linear (swin_trans.py:207-214)
 *   rel_bias [nh, (2*ws-1)^2] fp32: the checkpoint's relative_position_bias_table TRANSPOSED (head-major).
 *            Entry (dy + ws - 1) * (2 ws - 1) + (dx + ws - 1) is the bias between a query at window
 *            position (yi, xi) and a key at (yi - dy, xi - dx) — the value relative_position_index
 *            (swin_trans.py:93-103) selects for that pair; the dense [ws^2, ws^2] gather (:137-141, 83 KB per
 *            head) never exists.  Same meaning for every dtype / kernel path.
 *   out      [B, H*W, C]    attention output before `proj`, original token order (padding cropped)
 * ------------------------------------------------------------------------------------------ */
int psalm_window_attention(const void* qkv, const void* qkv_bias, const float* rel_bias, void* out,
                           int B, int H, int W, int C, int nh, int ws, int shift, int dtype, void* stream);

/* Attention implementation selector: 0 = auto (tensor-core kernels for fp16/bf16 storage, fp32 SIMT
 * kernels for fp32 storage; split-K cross-attention with <= 4 splits reduces its partials inside a thread-block
 * cluster over distributed shared memory, larger split counts go through the workspace + a combine kernel),
 * 1 = force the fp32-math SIMT kernels for every storage type (parity runs), 2 / 3 = tensor-core kernels with
 * the split-K reduction always through the workspace / always inside a cluster (<= 16 splits). */
int psalm_set_attention_impl(int impl);

/* Causal prefill attention of the LLM (third-party PhiAttention eager path; call site
 * language_model/llava_phi.py:1354-1363).  qkv [B,T,3,nh,hd] with rotary already applied
 * (psalm_rotary_inplace); key_valid [B,T] uint8 (attention_mask) or NULL; out [B,T,nh*hd].
 * fp32 softmax as in the reference.  16-bit storage, head_dim 64, 256 <= T <= 2048: tcgen05 + TMEM kernel
 * (128-query tiles, S and O accumulators in tensor memory); otherwise the mma.sync flash kernel; fp32
 * storage: SIMT kernel.  psalm_set_causal_impl: 0 = auto, 1 = mma.sync, 2 = tcgen05 (error if unsupported). */
int psalm_set_causal_impl(int impl);
int psalm_causal_attention(const void* qkv, const uint8_t* key_valid, void* out, int B, int T, int nh,
                           int hd, int dtype, void* stream);

/* Partial rotary embedding in place on q and k of qkv [B,T,3,nh,hd]; cos/sin [T, rd/2] fp32
 * (PhiRotaryEmbedding + apply_rotary_pos_emb on the first rd dims). */
int psalm_rotary_inplace(void* qkv, const float* cos_t, const float* sin_t, int B, int T, int nh, int hd,
                         int rd, int dtype, void* stream);

/* Masked cross-attention / query self-attention of the Mask2Former decoder.
 * Replaces nn.MultiheadAttention's core in CrossAttentionLayer / SelfAttentionLayer
 *   (transformer_decoder/mask2former_transformer_decoder.py:93-105, 35-45) after the in-projections.
 *   q [B,Lq,nh*hd], k,v [B,Lk,nh*hd], out [B,Lq,nh*hd]
 *   mask_bits [B,Lq,ceil(Lk/32)] uint32, bit = 1 -> key blocked (identical for all heads), or NULL
 *   row_open  [B,Lq] uint8, 1 -> every key of the row is blocked -> the row attends everywhere
 *             (mask2former_transformer_decoder.py:647), or NULL
 *   splits > 1 -> split-K over the keys; workspace of psalm_cross_attention_workspace_bytes(). */
size_t psalm_cross_attention_workspace_bytes(int B, int nh, int hd, int Lq, int splits);
int psalm_cross_attention(const void* q, const void* k, const void* v, const uint32_t* mask_bits,
                          const uint8_t* row_open, void* out, float* workspace, int B, int Lq, int Lk,
                          int nh, int hd, int splits, int dtype, void* stream);

/* Prediction head pieces (mask2former_transformer_decoder.py:695-762).
 *   psalm_mask_logits: out[b,q,p] = sum_c mask_embed[b,q,c] * feats[b,p,c]
 *       (= einsum("bqc,bchw->bqhw") at :750 with the feature map stored token-major [B,HW,C])
 *   psalm_bilinear_tokens: F.interpolate(bilinear, align_corners=False) on token-major maps
 *       [B,Hi,Wi,C] -> [B,Ho,Wo,C]; accumulate != 0 adds into `out` (FPN top-down add, msdeformattn.py:306)
 *   psalm_attn_mask_bits: bits = (logit < 0)  (== sigmoid < 0.5, :757-759), row_open = all blocked */
/* Intermediate prediction heads in one kernel (16-bit storage, C == 256, Q <= 112): bits = (mask_embed .
 * feats^T < 0) packed 32 keys / word + row_open; the logits are never written. */
int psalm_mask_bits_fused(const void* mask_embed, const void* feats, uint32_t* bits, uint8_t* row_open, int B,
                          int Q, int P, int C, int dtype, void* stream);
/* Implementation selector of psalm_mask_logits for 16-bit storage: 0 = auto (tcgen05 + TMEM kernel for
 * P >= 8192, warp-level mma.sync below), 1 = mma.sync, 2 = tcgen05. */
int psalm_set_mask_proj_impl(int impl);
int psalm_mask_logits(const void* mask_embed, const void* feats, void* out, int B, int Q, int P, int C,
                      int dtype, int out_dtype, void* stream);
int psalm_bilinear_tokens(const void* in, void* out, int B, int Hi, int Wi, int Ho, int Wo, int C, int dtype,
                          int out_dtype, int accumulate, void* stream);
int psalm_attn_mask_bits(const void* logits, uint32_t* bits, uint8_t* row_open, int rows, int P, int dtype,
                         void* stream);

/* Fused residual add + LayerNorm:  s = x (+ r1) (+ r2);  y = LN(s) * weight + bias;  sum_out (nullable)
 * receives s.  Replaces the `x = shortcut + ...; norm(x)` pairs of swin_trans.py:207,247-251, the
 * parallel-residual sum of PhiDecoderLayer followed by the next input_layernorm, and the post-norm
 * layers of msdeformattn.py:59-65 / mask2former_transformer_decoder.py:42-43,102-103,160-161.
 * x, r1, r2, y, sum_out: [rows, C]; C in {128,256,512,1024,2048}; fp32 statistics (two-pass). */
int psalm_add_layernorm(const void* x, const void* r1, const void* r2, const void* weight, const void* bias,
                        void* sum_out, void* y, long long rows, int C, float eps, int dtype, void* stream);

/* GroupNorm (+ optional ReLU) of a token-major map x [B,N,C] (statistics over N x C/groups per group),
 * msdeformattn.py:199-203,244-252.  Deterministic (no atomics).
 * pre_bias [C] or NULL: per-channel bias of the conv / Linear that produced x, added before the statistics
 * (GroupNorm(x + pre_bias)): the producer runs without its separate broadcast bias-add pass.
 * stats_workspace: at least 8 * B * groups * (1 + ceil(N / 256)) bytes. */
int psalm_groupnorm_tokens(const void* x, const void* pre_bias, const void* weight, const void* bias, void* y,
                           double* stats_workspace, int B, int N, int C, int groups, float eps, int relu,
                           int dtype, void* stream);

/* Fused post-processing of eval_seg (llava_phi.py:1399-1406 up-sampling + the task heads :325-447) for the
 * common case where the up-sampled map needs no further crop / resize.  Reads the low-resolution mask
 * logits [Q,H4,W4] and produces, without materialising [Q,H,W] tensors:
 *   sem_seg    [ncls,H,W] fp32 = softmax(cls)[:, :-1]^T . sigmoid(up(logits))   (probsT_f16: [144,112] fp16,
 *              class-major, zero padded; NULL together with sem_seg to skip)
 *   ids / in_mask [H,W]: arg-max_q (wq[q] * sigmoid + negq[q]) and (sigmoid >= 0.5 at the winner)
 *              (panoptic_inference, llava_phi.py:341-361; NULL x4 to skip)
 *   inst_masks [K,H,W] fp32 = (up(logits)[slot_query[k]] > 0); slots with query -1 are not written
 *   partials   [rows, Q, 5] per-CTA sums: count(x>0), sum(sigmoid*[x>0]), count(x>=0), area, inter
 *              (rows from psalm_postproc_partials for the same arguments); the caller reduces over the first axis.
 * Two kernels sit behind the call: a tensor-core formulation (16-bit logits, x1..x8 power-of-two up-sampling:
 * up-sampling and the semantic einsum are both mma GEMMs, persistent CTAs) and a generic one (any dtype /
 * resize factor).  psalm_set_postproc_impl: 0 = auto, 1 = generic, 2 = tensor-core (error if unsupported). */
int psalm_set_postproc_impl(int impl);
int psalm_postproc_partials(int Q, int H4, int W4, int H, int W, int ncls, int K, int dtype, int* rows);
int psalm_postproc_fused(const void* logits, const void* probsT_f16, const float* wq, const float* negq,
                         const int* slot_query, float* sem_seg, float* inst_masks, int* ids,
                         unsigned char* in_mask, float* partials, int Q, int H4, int W4, int H, int W, int ncls,
                         int K, int dtype, void* stream);

/* Same outputs for the reference's eval flow with a padded / resized image (detectron2 sem_seg_postprocess inside
 * eval_seg, llava_phi.py:1418-1430): the low-resolution logits are up-sampled to the padded input size (Hp, Wp), cropped
 * to the un-padded box (oh, ow) and resized to the output size (H, W) - composed inside the kernel (4 x 4 separable taps
 * per pixel), the [Q,Hp,Wp] tensor never exists.  psalm_postproc_crop_supported: 1 when the geometry fits the kernel's
 * shared-memory source window (otherwise callers use the step-by-step path).  partials rows:
 * psalm_postproc_crop_partials(H, W). */
int psalm_postproc_crop_supported(int Q, int H4, int W4, int Hp, int Wp, int oh, int ow, int H, int W, int ncls);
int psalm_postproc_crop_partials(int H, int W, int* rows);
int psalm_postproc_fused_crop(const void* logits, const void* probsT_f16, const float* wq, const float* negq,
                              const int* slot_query, float* sem_seg, float* inst_masks, int* ids, unsigned char* in_mask,
                              float* partials, int Q, int H4, int W4, int Hp, int Wp, int oh, int ow, int H, int W,
                              int ncls, int K, int dtype, void* stream);

/* ------------------------------------------------------------------------------------------
 * Masked cross-attention of the Mask2Former decoder, all 8 heads of a key range per CTA, K/V through TMA
 * (csrc/xattn_tma.cu).  Same mathematics as psalm_cross_attention; replaces CrossAttentionLayer.forward_post's
 * nn.MultiheadAttention call (transformer_decoder/mask2former_transformer_decoder.py:93-105) for 16-bit storage.
 *   q        [B,Lq,256]  projected queries (8 heads x 32), Lq <= 112
 *   k, v     [B,Lk,256]  projected keys / values as ROW-STRIDED views: row n of image b starts at
 *            base + (b*Lk + n) * kv_row_stride elements (kv_row_stride = 256 for separate contiguous tensors, 768
 *            when the K (or V) projections of the three decoder layers sharing a feature level are one GEMM)
 *   mask_bits [B,Lq,ceil(Lk/32)] bit j of word w = key 32w+j BLOCKED (shared by the heads), or NULL
 *   row_open  [B,Lq] != 0: ignore the mask for that row (fully blocked rows attend everywhere, :647), or NULL
 *   workspace: psalm_masked_cross_attention_workspace_bytes(B, Lq, Lk) bytes (split-K partials), may be NULL if 0
 * ------------------------------------------------------------------------------------------ */
/* implementation selector: 0 = auto (tcgen05 + TMEM kernel, csrc/xattn_tc5.cu), 1 = warp-level mma.sync kernel
 * (csrc/xattn_tma.cu), 2 = tcgen05.  Both are fed by TMA. */
int psalm_set_cross_impl(int impl);
size_t psalm_masked_cross_attention_workspace_bytes(int B, int Lq, int Lk);
int psalm_masked_cross_attention(const void* q, const void* k, const void* v, long long kv_row_stride,
                                 const uint32_t* mask_bits, const uint8_t* row_open, void* out, float* workspace,
                                 size_t workspace_bytes, int B, int Lq, int Lk, int nh, int hd, int dtype, void* stream);

/* ------------------------------------------------------------------------------------------
 * Autoregressive decode of the LLM (chat path: psalm/serve/cli.py:89-96 -> PSALM.generate; single-token branch
 * language_model/llava_phi.py:773-778): paged KV cache + single-token causal attention (csrc/decode.cu).
 * Replaces HF's DynamicCache growth by torch.cat (a full cache copy per layer per token) and the eager
 * [B,32,1,T] score / softmax / matmul chain of PhiAttention.
 *   cache pages  [num_pages, nh, page_size, hd] (K and V separately), block_table [B,max_pages] int32
 *   psalm_kv_cache_write: rows t = 0..T-1 of qkv [B,T,3,nh,hd] (rotary applied) go to positions start_pos[b] + t
 *   psalm_paged_decode_attention: q [B,nh,hd] with batch stride q_batch_stride elements (e.g. 3*nh*hd inside a qkv
 *     buffer) against the first seq_lens[b] cached keys -> out [B, nh*hd]
 * ------------------------------------------------------------------------------------------ */
int psalm_kv_cache_write(const void* qkv, void* kcache, void* vcache, const int* block_table, const int* start_pos, int B,
                         int T, int nh, int hd, int page_size, int max_pages, int dtype, void* stream);
int psalm_paged_decode_attention(const void* q, long long q_batch_stride, const void* kcache, const void* vcache,
                                 const int* block_table, const int* seq_lens, void* out, int B, int nh, int hd, int page_size,
                                 int max_pages, int dtype, void* stream);

/* ------------------------------------------------------------------------------------------
 * Input pipeline on the device (SURVEY.md section 8 f2): pixel normalisation + zero padding to the patch grid +
 * unfold into the operand of the patch-embedding GEMM, one pass.
 * Replaces: `(image - pixel_mean) / pixel_std` on the host (datasets_mapper/coco_panoptic_mapper.py:161; the
 *   image can then be uploaded as uint8), PatchEmbed's F.pad and the unfold inside its stride-4 convolution
 *   (multimodal_encoder/swin_trans.py:427-441).
 *   images  [B,Cin,H,W] in_dtype (PSALM_U8 / F32 / F16 / BF16)
 *   mean, stdv [Cin] fp32 or both NULL (input already normalised)
 *   patches [B, ceil(H/4)*ceil(W/4), Cin*16] out_dtype; element (c,i,j) of patch (py,px) is the normalised
 *           pixel (c, 4py+i, 4px+j), 0 beyond the image border (zero padding AFTER normalisation, as F.pad does).
 * ------------------------------------------------------------------------------------------ */
int psalm_patchify(const void* images, void* patches, const float* mean, const float* stdv, int B, int Cin,
                   int H, int W, int patch, int in_dtype, int out_dtype, void* stream);

/* ------------------------------------------------------------------------------------------
 * Linear layer with a fused epilogue (tcgen05 + TMEM accumulators, operands through TMA; csrc/gemm_tc5.cu):
 *   out = epilogue(a · wᵀ + bias), 16-bit storage (PSALM_BF16 / PSALM_F16), fp32 accumulation.
 * Replaces the library GEMM + the separate elementwise pass of
 *   epilogue 1: Swin `Mlp.fc1` followed by the exact-erf `nn.GELU` (multimodal_encoder/swin_trans.py:37-44);
 *   epilogue 2: MSDeformAttn `value_proj` (ops/modules/ms_deform_attn.py:95-99) stored HEAD-MAJOR
 *               [M / rows_per_image, N / 32, rows_per_image, 32] - the layout psalm_msda_encoder_fused reads - instead of
 *               [M, N] followed by a transposing copy;
 *   epilogue 0: bias only (plain nn.Linear).
 *   a [M, K] with row stride a_row_stride elements (K contiguous), w [N, K] contiguous (nn.Linear weight), bias [N] or NULL.
 * Shapes: N % 256 == 0, K % 64 == 0 (psalm_linear_fused_supported returns 1 when the kernel applies).
 * ------------------------------------------------------------------------------------------ */
int psalm_linear_fused_supported(long long M, int N, int K, int epilogue, long long rows_per_image, int dtype);
int psalm_linear_fused(const void* a, long long a_row_stride, const void* w, const void* bias, void* out, long long M, int N,
                       int K, int epilogue, long long rows_per_image, int dtype, void* stream);

/* PatchMerging's 2x2 gather + LayerNorm over the 4C concatenated channels (multimodal_encoder/swin_trans.py:269-296:
 * F.pad to even H / W, x0..x3 strided slices, torch.cat, self.norm) in one pass: x [B,H,W,C] token-major ->
 * y [B, ceil(H/2)*ceil(W/2), 4C] normalised, ready for the `reduction` Linear.  C in {128, 256, 512}. */
int psalm_patch_merge_layernorm(const void* x, const void* weight, const void* bias, void* y, int B, int H, int W, int C,
                                float eps, int dtype, void* stream);

/* Region prompts (SURVEY.md section 8 f3): features of R regions = mean over P points of the bilinear samples
 * (F.grid_sample, align_corners=True, zero padding) of the projector's token map.
 * Replaces `region_pooling.forward` (visual_prompt_module/context_cluster.py:333-400, point_sample :43-68).
 *   tokens [B, h*w, C] token-major (dtype), points [R, P, 2] fp32 = (y, x) in [0, 1] (mask pixel / mask size, as
 *   context_cluster.py:349-352 builds them), region_image [R] int32 = image of every region, out [R, C] (dtype). */
int psalm_region_pool(const void* tokens, const float* points, const int* region_image, void* out, int B, int h, int w,
                      int C, int R, int P, int dtype, void* stream);

/* ------------------------------------------------------------------------------------------
 * COCO run-length encoding of binary masks (csrc/rle.cu), byte for byte what pycocotools' maskApi.c rleEncode +
 * rleToString produce.  Replaces `pycocotools.mask.encode` as called on the dense masks of eval_seg's results, after
 * a copy of the dense masks to the host: detectron2's instances_to_coco_json behind COCOEvaluator.process
 * (psalm/eval/instance_segmentation.py:128,150; instance_evaluation.py:13,17) and the region script
 * (psalm/eval/region_segmentation.py:282-283).
 *   masks   [K,H,W] contiguous, row-major, dtype PSALM_F32 / F16 / BF16 / U8 (uint8 or bool).  A pixel is foreground
 *           when its value is non-zero; masks are expected to hold 0 / 1 (other values, NaN included, are outside the
 *           contract).  K >= 1, H, W >= 1, H * W < 2^31.
 *   counts  uint32 run lengths of every mask in COLUMN-MAJOR pixel order, alternating 0-runs and 1-runs and starting
 *           with a 0-run (of length 0 when pixel (0, 0) is set); mask k's runs are counts[run_offsets[k] ..
 *           run_offsets[k+1]).
 *   strings the compressed counts strings of rleToString, mask k's at strings[str_offsets[k] .. str_offsets[k+1])
 *           (no terminating NUL).
 * Three calls on one stream, each sizing the output of the next, so that every buffer has its exact size:
 *   psalm_mask_rle_sizes   -> run_offsets [K+1] int64 (read run_offsets[K] to size `counts`)
 *   psalm_mask_rle_runs    -> counts, str_offsets [K+1] int64 (read str_offsets[K] to size `strings`)
 *   psalm_mask_rle_write   -> strings
 * `workspace` (psalm_mask_rle_workspace_bytes(K, H, W) bytes: the masks as column-major bits + 8 bytes per column) is
 * written by _sizes and read by _runs.
 * ------------------------------------------------------------------------------------------ */
size_t psalm_mask_rle_workspace_bytes(int K, int H, int W);
int psalm_mask_rle_sizes(const void* masks, void* workspace, size_t workspace_bytes, int64_t* run_offsets, int K, int H,
                         int W, int dtype, void* stream);
int psalm_mask_rle_runs(const void* workspace, size_t workspace_bytes, const int64_t* run_offsets, uint32_t* counts,
                        int64_t* str_offsets, int K, int H, int W, void* stream);
int psalm_mask_rle_write(const uint32_t* counts, const int64_t* run_offsets, const int64_t* str_offsets, char* strings,
                         int K, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PSALM_B200_H_ */
