/* arp_b200.h — C ABI of the B200-native reward-labeling hot path.
 *
 * The reference (csmile-1006/ARP) has no FFI for this path: it is plain Python calling PyTorch
 * (arp_dt/label_reward.py). This header is the boundary a maintainer would bind from that Python
 * with ctypes (see INTEGRATION.md): plain pointers and sizes, no torch types, int status codes,
 * nothing thrown across the ABI. Each entry point names the reference code it replaces.
 *
 * Conventions
 *   - one ArpHandle per GPU, used from one host thread at a time;
 *   - device pointers are caller-owned; work is stream-ordered on the `stream` argument
 *     (a cudaStream_t passed as void*; NULL = the legacy default stream);
 *   - return 0 (ARP_OK) or a negative ArpStatus; arp_last_error() gives the message;
 *   - there is NO CPU fallback: without an sm_100 device arp_create fails with ARP_ERR_NO_DEVICE.
 *
 * Instruction sets ("text groups"): arp_set_text_groups sets G sets of instruction embeddings at once, and every
 * labeling call then scores all of them from ONE decode + encoder pass. Outputs become group-major: reward / rtg
 * [G, T], stacked arrays [G, T, F]; group g's rows are bit-identical to a call after arp_set_text(group g's rows).
 * arp_set_text is the G = 1 case, and with G = 1 every output has the shape it always had.
 *
 * Stored embeddings: labeling splits into an image side (decode, ViT, the head's projection / adapter) and an
 * instruction side (cosine, group reduction, return-to-go scan). arp_embed_host / arp_embed_file run the image side once
 * and return one fp32 vector per frame; arp_label_embeddings runs the instruction side on such vectors, with no frames
 * and no image-side weights, and gives arp_label's outputs bit for bit. A new instruction, inst_type, reduce mode or
 * text-head variant of the same checkpoint then costs a read of the vectors and one memory-bound head launch.
 *
 * CLIP tower records (adapter heads): the adapter heads' stored embedding depends on the adapter checkpoint, but
 * fine-tuning freezes CLIP, so what the adapter reads from the CLIP tower is the same for every checkpoint made from the
 * same CLIP. arp_embed_tower_host / arp_embed_tower_file run the frozen tower once and return one fp32 record of
 * arp_tower_dim() = 12*768 + 512 = 9728 floats per frame: the 12 class-token taps (block l at columns [l*768, (l+1)*768),
 * each the value the image_intermediate_linear GEMM multiplies), then the un-normalised CLIP feature. arp_label_tower
 * runs only the adapter (three GEMMs, the gate, the head) and the scan on such records, with no frames and no visual.*
 * weights, and gives arp_label's outputs bit for bit — also for an adapter checkpoint other than the one the records were
 * written with. A new fine-tuned adapter then costs 0.468 GFLOP per frame instead of the ViT's 35.1.
 *
 * Compressed rows: the recorder writes `ob` as gzip-chunked HDF5 with one row (F stacked frames) per chunk, and HDF5's
 * deflate filter stores every chunk as one plain zlib stream. arp_label_zfile / arp_embed_zfile / arp_embed_tower_zfile
 * take the file offset and size of every row's chunk (h5py: DatasetID.get_chunk_info), pread() the compressed bytes and
 * inflate them on the device (one warp per row, Adler-32 checked) before the unchanged encoder pass. No HDF5 parsing
 * happens here: the caller's chunk index says where the streams are.
 *
 * Compressed chunks of any shape: a gzip dataset that was re-chunked (h5py's own chunk guess, several rows per chunk,
 * frames split along F, H, W or the channels) is one zlib stream per chunk, each inflating to the full chunk volume,
 * edge chunks included. arp_label_zchunks / arp_embed_zchunks / arp_embed_tower_zchunks take the dataset's
 * ArpChunkLayout and its chunk table (logical origin, file offset, size), read and inflate only the chunks that hold a
 * scored frame, and gather the scored frames into dense [n, H, W, 3] frames on the device (gather_frames_kernel)
 * before the unchanged encoder pass. The arp_*_zfile calls are the (1, F, H, W, 3) case of the same code.
 */
#ifndef ARP_B200_H_
#define ARP_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ARP_B200_ABI_VERSION 11  /* 3: + arp_encode_taps_chw, 4: + arp_operand_dtype, 5: + ARP_PREC_F32RESID, arp_ln_gemm, arp_resid_gemm_stats, arp_label_file, arp_wants_weight, 6: + arp_set_text_groups, arp_text_groups, 7: + arp_embedding_dim, arp_embed_host, arp_embed_file, arp_label_embeddings, 8: + arp_tower_dim, arp_embed_tower_host, arp_embed_tower_file, arp_label_tower, 9: + ArpInflateStatus, arp_inflate_rows, arp_label_zfile, arp_embed_zfile, arp_embed_tower_zfile, 10: + ArpChunkLayout, arp_label_zchunks, arp_embed_zchunks, arp_embed_tower_zchunks, arp_gather_frames, 11: + arp_cls_attention */

#define ARP_MAX_TEXT 16          /* texts of one instruction set (arp_set_text's n_text, one group's size) */
#define ARP_MAX_TEXT_GROUPS 16   /* instruction sets of one arp_set_text_groups call */
#define ARP_MAX_TEXT_TOTAL 64    /* texts of all groups together */

#if defined(__GNUC__)
#define ARP_API __attribute__((visibility("default")))
#else
#define ARP_API
#endif

typedef enum ArpStatus {
  ARP_OK = 0,
  ARP_ERR_INVALID = -1,     /* bad argument / unsupported geometry */
  ARP_ERR_CUDA = -2,        /* a CUDA runtime / driver call failed */
  ARP_ERR_STATE = -3,       /* weights or text embeddings not set yet */
  ARP_ERR_NO_DEVICE = -4,   /* no CUDA device, or not compute capability 10.x */
  ARP_ERR_UNKNOWN_KEY = -5  /* arp_set_weight: name is not part of the model */
} ArpStatus;

/* Per-row result of the device zlib inflate (arp_inflate_rows' status_dev; named by arp_last_error after a failed
 * arp_*_zfile call). The first violation stops the row. */
typedef enum ArpInflateStatus {
  ARP_INFLATE_OK = 0,
  ARP_INFLATE_TRUNCATED = 1,          /* a read past the row's compressed bytes */
  ARP_INFLATE_BAD_HEADER = 2,         /* zlib header: CM != 8, CINFO > 7, FCHECK wrong, or FDICT set */
  ARP_INFLATE_BAD_BLOCK = 3,          /* block type 3, or a stored block whose LEN / NLEN disagree */
  ARP_INFLATE_BAD_CODE = 4,           /* over-subscribed or invalid Huffman code, bad code-length repeat, symbol 286-287 / 30-31 */
  ARP_INFLATE_DISTANCE_TOO_FAR = 5,   /* a back-reference before the start of the row */
  ARP_INFLATE_TOO_LONG = 6,           /* more than row_bytes of output */
  ARP_INFLATE_TOO_SHORT = 7,          /* the stream ended before row_bytes of output */
  ARP_INFLATE_BAD_ADLER = 8           /* the Adler-32 trailer does not match the inflated row */
} ArpInflateStatus;

/* label_reward.py:109-121 vs clip_multiscale_adapter.py:121-133 */
typedef enum ArpPreprocess { ARP_PRE_PIL_BICUBIC = 0, ARP_PRE_BILINEAR = 1 } ArpPreprocess;
/* label_reward.py:128 "clip" | :166 "clip_ft" | :217-222 3-D feature branch | :148,180 goal-conditioned */
typedef enum ArpHead {
  ARP_HEAD_CLIP = 0,
  ARP_HEAD_ADAPTER = 1,
  ARP_HEAD_ADAPTER_ENSEMBLE = 2,
  ARP_HEAD_CLIP_GOAL = 3,
  ARP_HEAD_ADAPTER_GOAL = 4
} ArpHead;
/* label_reward.py:142-145: row 0 of logits_per_text is what the reference takes (SURVEY.md Q1);
 * MEAN is the envs/vl_reward.py:19-22 behaviour. */
typedef enum ArpReduce { ARP_REDUCE_FIRST = 0, ARP_REDUCE_MEAN = 1 } ArpReduce;

typedef enum ArpDType { ARP_F32 = 0, ARP_BF16 = 1, ARP_F16 = 2 } ArpDType;
/* Arithmetic of the model path.
 * ARP_PREC_BF16 (0; the name is historical — read "16-bit tensor-core path"): the product path. tcgen05 tensor cores,
 *   16-bit operands in the build's operand format (arp_operand_dtype(): fp16 by default, the format the reference's own
 *   CUDA route runs CLIP in, clip.load label_reward.py:126), fp32 accumulation, 16-bit residual stream updated by TMA
 *   reduce-add, LayerNorm folded algebraically into the QKV / c_fc GEMM epilogues from fp32 row moments.
 * ARP_PREC_F32RESID (2): same tensor-core GEMMs and attention with an fp32 residual stream and standalone fp32 LayerNorm
 *   kernels (round 1's pipeline): ~2x closer to fp32, ~10 % slower.
 * ARP_PREC_F32 (1): verification path — every weight, activation and contraction in fp32 on the FMA pipe, what
 *   clip.load(...).float() computes on the reference's CPU route (label_reward.py:126-141); used to check the restated
 *   algorithm at the 1e-5 bar, ~50x slower. */
typedef enum ArpPrecision { ARP_PREC_BF16 = 0, ARP_PREC_F32 = 1, ARP_PREC_F32RESID = 2 } ArpPrecision;

typedef struct ArpHandle ArpHandle;

typedef struct ArpConfig {
  int32_t struct_size; /* sizeof(ArpConfig), for forward compatibility */
  int32_t device;      /* CUDA device ordinal */
  int32_t patch;       /* 16 = ViT-B/16 (label_reward.py:126), 32 = ViT-B/32 */
  int32_t width;       /* 768 */
  int32_t layers;      /* 12 */
  int32_t heads;       /* 12 (width / 64) */
  int32_t embed_dim;   /* 512 */
  int32_t in_h, in_w;  /* dataset frame size (64 or 256 for procgen) */
  int32_t use_crop;    /* label_reward.py:90-106: centre crop to (H//2, W//2) before the resize */
  int32_t preprocess;  /* ArpPreprocess */
  int32_t head;        /* ArpHead */
  int32_t reduce;      /* ArpReduce */
  int32_t max_batch;   /* frames per internal chunk (workspace is sized for this) */
  int32_t precision;   /* ArpPrecision */
} ArpConfig;

/* ------------------------------------------------------------------------------------------------
 * lifetime
 * ---------------------------------------------------------------------------------------------- */
/* replaces clip.load("ViT-B/16", device) + transform construction (label_reward.py:89-130, :165-178) */
ARP_API int arp_create(const ArpConfig* cfg, ArpHandle** out);
ARP_API void arp_destroy(ArpHandle* h);
ARP_API const char* arp_last_error(const ArpHandle* h); /* h may be NULL: last error of arp_create */
ARP_API int arp_abi_version(void);
/* ArpDType of the 16-bit operand format this build runs its contractions in: ARP_F16 (default build; the reference's
 * own CUDA path keeps CLIP in fp16, clip.load) or ARP_BF16 (-DARP_OP_FP16=0). The "bf16" buffers of the test hooks
 * below (arp_gemm_bf16, arp_ln_gemm, arp_layernorm_bf16, arp_attention) are in THIS format. */
ARP_API int arp_operand_dtype(void);

/* ------------------------------------------------------------------------------------------------
 * weights: one call per state_dict entry, names exactly as in openai/CLIP's state_dict
 * ("visual.conv1.weight", "visual.transformer.resblocks.3.attn.in_proj_weight", "visual.proj", ...)
 * and, for the adapter heads, finetune_module/clip_multiscale_adapter.py's
 * ("image_intermediate_linear.weight", "image_adapter.layers.0.weight", "image_adapter.layers.3.bias",
 *  "image_residual_weight"). `data` is a DEVICE pointer to a contiguous tensor of `dtype`; the library
 * keeps its own packed copy (bf16 for GEMM operands, fp32 for norms / biases / tables).
 * Text-tower keys are accepted and ignored (ARP_OK); unknown keys give ARP_ERR_UNKNOWN_KEY.
 * replaces model.load_state_dict(torch.load(model_ckpt_dir), strict=False) (label_reward.py:175-176)
 * ---------------------------------------------------------------------------------------------- */
ARP_API int arp_set_weight(ArpHandle* h, const char* name, const void* data, int32_t dtype, const int64_t* shape,
                   int32_t ndim, void* stream);
/* 1 if `name` is a tensor this handle stores (so a caller can skip uploading the text tower etc.), else 0 */
ARP_API int arp_wants_weight(const ArpHandle* h, const char* name);
/* number of weights still missing for the configured head (0 = ready) */
ARP_API int arp_missing_weights(const ArpHandle* h, char* names_out, int64_t names_cap);

/* Cached instruction embedding(s): fp32 [n_text, dim] DEVICE rows, already L2-normalised
 * (per 512-wide scale for ARP_HEAD_ADAPTER_ENSEMBLE); dim = 512 (clip) or 6656 (adapter heads); 1 <= n_text <= ARP_MAX_TEXT.
 * logit_scale_exp = model.logit_scale.exp() (label_reward.py:141, :213-216).
 * Sets ONE group (arp_text_groups() == 1): the outputs of the calls below are [T] / [T, F].
 * replaces clip.tokenize + encode_text, which the reference re-runs every episode (:135-138). */
ARP_API int arp_set_text(ArpHandle* h, const float* text_emb_dev, int32_t n_text, int32_t dim, float logit_scale_exp,
                 void* stream);
/* G instruction sets scored in one pass (the reference relabels the same demonstrations once per inst_type).
 *   text_emb_dev        fp32 [n_text_total, dim] DEVICE rows of all groups, concatenated, normalised as for arp_set_text
 *   group_offsets_host  int32 [n_groups + 1] HOST: group g = rows [off[g], off[g+1]); off[0] = 0, off[G] = n_text_total
 * Each group is reduced on its own (ArpConfig.reduce: its first row or its mean). Limits: 1..ARP_MAX_TEXT_GROUPS groups of
 * 1..ARP_MAX_TEXT texts, at most ARP_MAX_TEXT_TOTAL in all; ARP_ERR_INVALID otherwise, and for goal-conditioned heads
 * (they take no text). After it, with G = n_groups:
 *   arp_label / arp_label_host / arp_label_file   reward, rtg [G, T]; reward_stacked, rtg_stacked [G, T, F]
 *   arp_compute_reward                            reward [G, T]; logits [T, n_text_total]
 *   arp_online_reward                             ARP_ERR_INVALID for G > 1
 * Group g's values are bit-identical to the same call after arp_set_text(group g's rows). arp_set_text resets to G = 1. */
ARP_API int arp_set_text_groups(ArpHandle* h, const float* text_emb_dev, int32_t n_text_total, int32_t dim,
                        const int32_t* group_offsets_host, int32_t n_groups, float logit_scale_exp, void* stream);
/* the current number of text groups G: 1 after arp_set_text (and before any text is set) */
ARP_API int arp_text_groups(const ArpHandle* h);

/* ------------------------------------------------------------------------------------------------
 * the hot path
 * ---------------------------------------------------------------------------------------------- */
/* Score T dataset rows and build the per-episode return-to-go tokens. Replaces the whole episode loop
 * label_reward.py:265-271 (compute_reward + discount_cumsum + stack_outputs x2).
 *   ob_dev            uint8, row t's image to score starts at ob_dev + t*row_stride_bytes
 *                     (for the reference layout ob[T,F,H,W,3] pass &ob[0,F-1] and stride F*H*W*3: label_reward.py:268)
 *   ep_offsets_dev    int64 [n_eps+1] DEVICE: episode e = rows [off[e], min(off[e+1], T))   (:82-83, :267)
 *   num_frames        F of the stacked outputs (:81)
 *   reward_dev        fp32 [T] per-frame reward (may be NULL)
 *   rtg_dev           fp32 [T] per-frame return-to-go (may be NULL)
 *   reward_stacked_dev, rtg_stacked_dev   fp32 [T,F] = the two datasets the reference writes (:270-271)
 * With G text groups (arp_set_text_groups) the four outputs are [G, T] and [G, T, F], group-major.
 */
ARP_API int arp_label(ArpHandle* h, const uint8_t* ob_dev, int64_t T, int64_t row_stride_bytes,
              const int64_t* ep_offsets_dev, int32_t n_eps, int32_t num_frames, float* reward_dev, float* rtg_dev,
              float* reward_stacked_dev, float* rtg_stacked_dev, void* stream);

/* Same contract with HOST buffers (G groups: [G, T] / [G, T, F] as for arp_label): frames are streamed to the device in
 * chunks on a copy stream, overlapped with compute, and the four outputs are copied back. Pinned (cudaHostAlloc / cudaHostRegister) frames are copied directly;
 * pageable ones — e.g. a pointer into the memory-mapped dataset itself — are gathered by a few internal worker threads
 * through a ring of pinned slots, so page-cache reads, PCIe and the GPU overlap and ONE call can cover a whole shard.
 * This is the call a drop-in label_reward() makes per image key; it synchronises before returning. */
ARP_API int arp_label_host(ArpHandle* h, const uint8_t* ob_host, int64_t T, int64_t row_stride_bytes,
                   const int64_t* ep_offsets_host, int32_t n_eps, int32_t num_frames, float* reward_host,
                   float* rtg_host, float* reward_stacked_host, float* rtg_stacked_host);

/* Same call with the frames read straight from a FILE: row t's scored image is the frame_bytes (= in_h*in_w*3) at
 * file_offset + t*row_stride_bytes of the open descriptor `fd` — an .npy memory-map's backing file, or a contiguous
 * (unchunked, uncompressed) HDF5 dataset at its data offset. The gather threads pread() into the pinned ring, which
 * avoids the page-table work of touching tens of GB through a mapping (faults on the way in, a long munmap on the way out).
 * Outputs as for arp_label_host ([G, T] / [G, T, F] with G text groups).
 * replaces g[img_key][traj, -1] (label_reward.py:268) for containers whose rows sit contiguously in a file. */
ARP_API int arp_label_file(ArpHandle* h, int32_t fd, int64_t file_offset, int64_t T, int64_t row_stride_bytes,
                   const int64_t* ep_offsets_host, int32_t n_eps, int32_t num_frames, float* reward_host,
                   float* rtg_host, float* reward_stacked_host, float* rtg_stacked_host);

/* Per-frame embedding width: 512 for the clip heads (ARP_HEAD_CLIP, ARP_HEAD_CLIP_GOAL), 13*512 for the adapter heads. */
ARP_API int arp_embedding_dim(const ArpHandle* h);   /* 512 (clip heads) or 13*512 (adapter heads) */
/* The image side of arp_label_host, stopped before the instruction: the per-frame embedding [T, dim] fp32 is written to
 * emb_host (clip heads: encode_image un-normalised, label_reward.py:156; adapter heads: the gated feature
 * a = sigmoid(w) * feat + (1 - sigmoid(w)) * mlp(feat) before F.normalize, clip_multiscale_adapter.py:145-151). Same
 * frame arguments, staging and encoder pass as arp_label_host / arp_label_file; the result is assembled on the device and
 * copied to the host once at the end (T * dim * 4 bytes of device memory, freed before the call returns). Synchronises.
 * replaces the image half of compute_reward (label_reward.py:132-146, :200-230) when its output is to be kept. */
/* per-frame embedding [T, dim] fp32 (clip: encode_image un-normalised; adapter: gated feature before F.normalize) */
ARP_API int arp_embed_host(ArpHandle* h, const uint8_t* ob_host, int64_t T, int64_t row_stride_bytes, float* emb_host);
ARP_API int arp_embed_file(ArpHandle* h, int32_t fd, int64_t file_offset, int64_t T, int64_t row_stride_bytes,
                           float* emb_host);
/* arp_label's outputs ([G,T] / [G,T,F] with text groups) from stored embeddings; needs no image-side weights */
/* emb_dev [T, arp_embedding_dim] fp32 DEVICE rows from arp_embed_* of a handle with the same checkpoint; the other
 * arguments and the four outputs are those of arp_label. Bit-identical to arp_label on the frames the rows came from. An
 * embedding serves every head of its family: a clip row labels on ARP_HEAD_CLIP and ARP_HEAD_CLIP_GOAL, an adapter row on
 * ARP_HEAD_ADAPTER, ARP_HEAD_ADAPTER_ENSEMBLE and ARP_HEAD_ADAPTER_GOAL. Works on a handle whose image-side weights were
 * never set. ARP_ERR_STATE only when a text head has no text. Text heads make exactly two launches (head, scan).
 * replaces compute_reward's cosine + discount_cumsum + stack_outputs (label_reward.py:141-146, :213-254) */
ARP_API int arp_label_embeddings(ArpHandle* h, const float* emb_dev, int64_t T, const int64_t* ep_offsets_dev,
                                 int32_t n_eps, int32_t num_frames, float* reward_dev, float* rtg_dev,
                                 float* reward_stacked_dev, float* rtg_stacked_dev, void* stream);

/* CLIP tower record width: 9728 (12 class-token taps of 768 + the 512-wide CLIP feature) for the adapter heads, 0 for the
 * clip heads. The layout is the same for every precision and operand format. */
ARP_API int arp_tower_dim(const ArpHandle* h);
/* The frozen-CLIP side of arp_label_host / arp_label_file on an adapter head, stopped after the CLIP feature: one record
 * [T, arp_tower_dim] fp32 per frame is written to rec_host. Columns [0, 9216): the class-token taps the adapter's
 * image_intermediate_linear reads (the 16-bit paths: the operand-format taps widened to fp32, which is exact; block 11's
 * is the 16-bit rounding of the pruned last block's fp32 class row; ARP_PREC_F32: the fp32 taps). Columns [9216, 9728):
 * encode_image before normalisation (clip_multiscale_adapter.py:136,145). Same frame arguments, staging and encoder pass
 * as arp_embed_host; the result is assembled on the device and copied to the host once at the end (T * 38 912 bytes of
 * device memory, freed before the call returns). Synchronises. ARP_ERR_INVALID on clip heads. */
ARP_API int arp_embed_tower_host(ArpHandle* h, const uint8_t* ob_host, int64_t T, int64_t row_stride_bytes,
                                 float* rec_host);
ARP_API int arp_embed_tower_file(ArpHandle* h, int32_t fd, int64_t file_offset, int64_t T, int64_t row_stride_bytes,
                                 float* rec_host);

/* Compressed rows. Row t of the call is one zlib stream (RFC 1950) of chunk_bytes_host[t] bytes at byte
 * chunk_offset_host[t] of the open descriptor `fd`, and inflates to exactly row_bytes = F * in_h * in_w * 3 bytes, F in
 * [1, 64] (the row's F stacked frames; the LAST one is scored). The gather threads pread() each row's compressed bytes
 * into the pinned ring (slots sized from the call's largest chunk), each max_batch chunk crosses PCIe compressed, and
 * inflate_rows_kernel writes the whole rows into a device scratch of max_batch * row_bytes bytes that the encoder reads
 * with row stride row_bytes. Outputs as for arp_label_file / arp_embed_file / arp_embed_tower_file, bit for bit what
 * those give on the same rows stored uncompressed. ARP_ERR_INVALID for fd < 0, T < 0, null tables, a negative offset or
 * size, a bad row_bytes, and for a row that does not inflate: arp_last_error then names the first such row (its index
 * in the call) and its ArpInflateStatus, no output is written, and the handle stays usable. Synchronises.
 * replaces g[img_key][traj, -1] (label_reward.py:268) for gzip datasets chunked (1, F, H, W, 3). */
ARP_API int arp_label_zfile(ArpHandle* h, int32_t fd, const int64_t* chunk_offset_host, const int64_t* chunk_bytes_host,
                            int64_t T, int64_t row_bytes, const int64_t* ep_offsets_host, int32_t n_eps,
                            int32_t num_frames, float* reward_host, float* rtg_host, float* reward_stacked_host,
                            float* rtg_stacked_host);
ARP_API int arp_embed_zfile(ArpHandle* h, int32_t fd, const int64_t* chunk_offset_host, const int64_t* chunk_bytes_host,
                            int64_t T, int64_t row_bytes, float* emb_host);
ARP_API int arp_embed_tower_zfile(ArpHandle* h, int32_t fd, const int64_t* chunk_offset_host,
                                  const int64_t* chunk_bytes_host, int64_t T, int64_t row_bytes, float* rec_host);
/* The inflate kernel alone, on DEVICE buffers: row r's zlib stream is src_dev[src_off_dev[r], + src_bytes_dev[r]) (the
 * caller keeps those ranges inside src_dev), it is inflated to out_dev[r * row_bytes, (r + 1) * row_bytes) and
 * status_dev[r] (int32) receives its ArpInflateStatus. Rows that fail leave the rest of their output unwritten.
 * Stream-ordered, does not synchronise; ARP_ERR_INVALID only for bad arguments (row_bytes as for arp_label_zfile). */
ARP_API int arp_inflate_rows(ArpHandle* h, const uint8_t* src_dev, const int64_t* src_off_dev,
                             const int64_t* src_bytes_dev, int64_t n, int64_t row_bytes, uint8_t* out_dev,
                             int32_t* status_dev, void* stream);

/* Compressed chunks of any shape. A uint8 dataset [T, F, H, W, 3] (ndim 5) or [T, H, W, 3] (ndim 4, read as F = 1) with
 * H, W = in_h, in_w is stored as chunks of shape `chunk` (every extent >= 1; HDF5 compresses an edge chunk at the full
 * chunk size, including the part past the dataset's extent, so every chunk inflates to exactly
 * prod(chunk) bytes). */
typedef struct ArpChunkLayout {
  int32_t struct_size;   /* sizeof(ArpChunkLayout) */
  int32_t ndim;          /* 4 or 5 */
  int64_t shape[5];      /* dataset shape (first ndim entries) */
  int64_t chunk[5];      /* chunk shape (first ndim entries) */
} ArpChunkLayout;

/* Maximum device scratch for the inflated chunks of one max_batch batch (and so for one chunk). */
#define ARP_ZCHUNK_SCRATCH_BYTES (4LL << 30)
/* Maximum compressed size of one needed chunk: one pinned staging slot, so the pinned ring (8 slots) stays within
 * 512 MiB. */
#define ARP_ZCHUNK_MAX_COMPRESSED_BYTES (64LL << 20)

/* Scores dataset rows [row_lo, row_lo + T), frame F-1 of each (the call's row t is dataset row row_lo + t). Chunk i of
 * the table has logical origin origins_host[i * ndim .. + ndim) (h5py: StoreInfo.chunk_offset) and is one zlib stream of
 * bytes_host[i] bytes at offsets_host[i] of `fd`. Only the chunks holding a scored frame are read: the row-chunks that
 * cover the call's rows, at the F-chunk of frame F-1, all H, W and channel chunks. The table may hold more (the whole
 * dataset's, or only a shard's part); the others are never read. Per max_batch batch the gather threads pread() the
 * batch's needed chunks into the pinned ring, they cross PCIe compressed, inflate_rows_kernel inflates each to its chunk
 * volume (one warp per chunk), and gather_frames_kernel copies each row's scored frame into a dense [n, H, W, 3] buffer
 * for the encoder. When every chunk is (1, cF, H, W, 3) the scored frames already sit at a fixed stride and the gather
 * is skipped. A row-chunk that straddles a batch boundary (or row_lo) is read and inflated once per batch it serves.
 * ep_offsets_host are relative to row_lo (0 .. T) and the outputs are those of arp_label_zfile, bit for bit what
 * arp_label_file gives on the same rows uncompressed. ARP_ERR_INVALID, with nothing written and the handle usable, for
 * a bad layout (ndim, H, W, 3 channels, a chunk extent < 1), rows outside the dataset, null tables, a negative offset or
 * size, an origin that is not a multiple of the chunk shape or lies outside the dataset, a duplicated origin, a needed
 * chunk missing from the table, one batch's inflated chunks needing more than ARP_ZCHUNK_SCRATCH_BYTES, more than 2^26
 * needed chunks, a needed chunk of more than ARP_ZCHUNK_MAX_COMPRESSED_BYTES compressed, and a needed
 * chunk that does not inflate to its chunk volume: arp_last_error names the chunk's logical origin (and
 * ArpInflateStatus). Synchronises. */
ARP_API int arp_label_zchunks(ArpHandle* h, int32_t fd, const ArpChunkLayout* layout, const int64_t* origins_host,
                              const int64_t* offsets_host, const int64_t* bytes_host, int64_t n_chunks, int64_t row_lo,
                              int64_t T, const int64_t* ep_offsets_host, int32_t n_eps, int32_t num_frames,
                              float* reward_host, float* rtg_host, float* reward_stacked_host, float* rtg_stacked_host);
ARP_API int arp_embed_zchunks(ArpHandle* h, int32_t fd, const ArpChunkLayout* layout, const int64_t* origins_host,
                              const int64_t* offsets_host, const int64_t* bytes_host, int64_t n_chunks, int64_t row_lo,
                              int64_t T, float* emb_host);
ARP_API int arp_embed_tower_zchunks(ArpHandle* h, int32_t fd, const ArpChunkLayout* layout,
                                    const int64_t* origins_host, const int64_t* offsets_host, const int64_t* bytes_host,
                                    int64_t n_chunks, int64_t row_lo, int64_t T, float* rec_host);
/* The gather kernel alone, on DEVICE buffers: chunks_dev holds, for the row-chunks row0 / chunk[0] ..
 * (row0 + n - 1) / chunk[0], every (H, W, channel) chunk at the F-chunk of frame F-1, in the order (row-chunk, H-chunk,
 * W-chunk, channel-chunk), each inflated to prod(chunk) bytes. out_dev[n, H, W, 3] receives frame F-1 of dataset rows
 * [row0, row0 + n). Stream-ordered, does not synchronise; ARP_ERR_INVALID for bad arguments or layout. */
ARP_API int arp_gather_frames(ArpHandle* h, const ArpChunkLayout* layout, int64_t row0, int64_t n,
                              const uint8_t* chunks_dev, uint8_t* out_dev, void* stream);
/* arp_label's outputs ([G,T] / [G,T,F] with text groups, the goal-conditioned adapter head included) from tower records:
 * rec_dev [T, arp_tower_dim] fp32 DEVICE rows (16-byte aligned) from arp_embed_tower_* of a handle with the same CLIP
 * weights, arch, frame size, crop and precision; the other arguments and the four outputs are those of arp_label. Needs
 * only the image-adapter tensors (image_intermediate_linear.weight, image_adapter.layers.{0,3}.*, image_residual_weight):
 * works on a handle whose visual.* weights were never set, and with any adapter checkpoint of that CLIP. Bit-identical to
 * arp_label on the frames the records came from, with this handle's adapter. Per max_batch chunk: one unpack launch and
 * the adapter's launches; one scan for the call. ARP_ERR_INVALID on clip heads, a null or unaligned buffer, T < 0, bad
 * offsets, num_frames outside [1, 64]; ARP_ERR_STATE when an adapter tensor is missing or a text head has no text.
 * replaces compute_reward's model(images, text) for a new adapter checkpoint (label_reward.py:200-230) */
ARP_API int arp_label_tower(ArpHandle* h, const float* rec_dev, int64_t T, const int64_t* ep_offsets_dev,
                            int32_t n_eps, int32_t num_frames, float* reward_dev, float* rtg_dev,
                            float* reward_stacked_dev, float* rtg_stacked_dev, void* stream);

/* Latency mode — the online reward of a rollout (arp_dt/envs/vl_reward.py:11-23 get_torch_clip_reward, :44-59
 * get_torch_clip_adapter_reward, and the two encode_image calls of the goal-conditioned variants :26-41, :62-77;
 * called once per environment step from envs/rollout_procgen.py:133-150). Scores n (1..max_batch) HOST frames
 * uint8 [n,H,W,3] and returns, each optional: reward [n] (row 0 or the mean over texts, per ArpConfig.reduce),
 * logits [n, n_text], features [n, feat_dim] (CLIP: un-normalised encode_image; adapter heads: normalised).
 * The kernel sequence is captured into a CUDA graph on first use per n; the call synchronises. Goal heads give
 * features only (the caller takes -||f_obs - f_goal||). One text group only: ARP_ERR_INVALID after arp_set_text_groups
 * with G > 1. */
ARP_API int arp_online_reward(ArpHandle* h, const uint8_t* ob_host, int32_t n, float* reward_host, float* logits_host,
                      float* feat_host);

/* Consumer side — ProcgenDataset.preprocess_rtgs (arp_dt/data_procgen.py:132-174), which turns the labeler's
 * per-frame rewards into the return-to-go tokens and the conditioning statistic of DT training:
 *   reward_dev [T] fp32 (column -1 of the "<key>_<vl_type>_pos_reward" dataset, :142-146)
 *   stats_host[0..1] = min, max of the rewards over all T rows (:147-148)
 *   use_normalize: shifted_dev [T] = reward - min (:150-151), and the scan runs on it
 *   rtg_dev [T], rtg_stacked_dev [T, num_frames]: per-episode discount_cumsum(gamma=1) + window stack (:155-168)
 *   stats_host[2..3] = min, max over the stacked return-to-go values (:171, CoinRun's return_to_go before //100*100)
 * Synchronises. The 0.9-quantile branch (:173) takes its two order statistics from arp_quantile_f32. */
ARP_API int arp_preprocess_rtgs(ArpHandle* h, const float* reward_dev, int64_t T, const int64_t* ep_offsets_dev,
                        int32_t n_eps, int32_t num_frames, int32_t use_normalize, float* shifted_dev, float* rtg_dev,
                        float* rtg_stacked_dev, float* stats_host, void* stream);
/* Exact order statistics of n device floats: lo_hi_host[0] = k_lo-th smallest, [1] = k_hi-th smallest (0-based),
 * by MSB-first radix select. np.quantile(x, q) (data_procgen.py:173) interpolates between the two. Synchronises. */
ARP_API int arp_quantile_f32(ArpHandle* h, const float* x_dev, int64_t n, int64_t k_lo, int64_t k_hi, float* lo_hi_host,
                     void* stream);

/* compute_reward only (label_reward.py:132-146 / :200-230): per-frame rewards [T], optional [T,n_text] logits;
 * with G text groups reward is [G, T] and logits [T, n_text_total]. */
ARP_API int arp_compute_reward(ArpHandle* h, const uint8_t* ob_dev, int64_t T, int64_t row_stride_bytes, float* reward_dev,
                       float* logits_dev, void* stream);

/* model.encode_image (un-normalised, [T, embed_dim]) resp. the adapter's encode_image ([T, 13*512], normalised).
 * Goal-conditioned heads and parity tests use it (label_reward.py:156, :187). */
ARP_API int arp_encode_image(ArpHandle* h, const uint8_t* ob_dev, int64_t T, int64_t row_stride_bytes, float* feat_dev,
                     void* stream);

/* The frozen-CLIP side of adapter fine-tuning (finetune_module/clip_multiscale_adapter.py:135-143 inside forward
 * :179-252; CLIP's parameters are frozen, finetune.py:147-148): images the caller has already resized / augmented /
 * normalised (`preprocess(x, train=True)`, :121-133), fp32 [T,3,224,224] DEVICE ->
 *   taps_dev fp32 [T, layers*width]  class-token row of every resblock's output (what the forward hooks capture,
 *                                    finetune_module/utils.py:6-18), block l at columns [l*width, (l+1)*width)
 *   feat_dev fp32 [T, embed_dim]     clip_model.encode_image(image)
 * Either output may be NULL. Clip heads only (the trainable adapter stays with the caller's autograd). */
ARP_API int arp_encode_taps_chw(ArpHandle* h, const float* chw_dev, int64_t T, float* taps_dev, float* feat_dev,
                        void* stream);

/* ------------------------------------------------------------------------------------------------
 * seams of the reference (unit-test hooks; same kernels the hot path runs)
 * ---------------------------------------------------------------------------------------------- */
/* transform(img) for every row (label_reward.py:92-121) or model.preprocess (clip_multiscale_adapter.py:121-133):
 * fp32 [T,3,224,224] */
ARP_API int arp_decode_only(ArpHandle* h, const uint8_t* ob_dev, int64_t T, int64_t row_stride_bytes, float* chw_dev,
                    void* stream);
/* discount_cumsum + stack_outputs (label_reward.py:232-254). Needs no weights. h may come from any config. */
ARP_API int arp_scan_only(ArpHandle* h, const float* reward_dev, int64_t T, const int64_t* ep_offsets_dev, int32_t n_eps,
                  int32_t num_frames, float gamma, float* rtg_dev, float* reward_stacked_dev,
                  float* rtg_stacked_dev, void* stream);
/* C[M,N] = act(A[M,K] W[N,K]^T + bias) (+ resid): the tcgen05 GEMM behind every linear layer.
 * A, W in the operand format (arp_operand_dtype) on the device; out in that format (out_dtype = it) or fp32; act 0 none,
 * 1 QuickGELU, 2 ReLU; bias fp32 or NULL; resid NULL or a buffer of out's dtype (may alias out_dev: the residual
 * stream is then updated in place by TMA reduce-add, fp32 or 16-bit); N % 256 == 0, K % 64 == 0. */
ARP_API int arp_gemm_bf16(ArpHandle* h, const void* a_dev, const void* w_dev, void* out_dev, int32_t out_dtype, int64_t M,
                  int32_t N, int32_t K, const float* bias_dev, const void* resid_dev, int32_t act, void* stream);
/* The default path's residual update: x[M,N] (operand format, in place) = fl16(x + A[M,K] W[N,K]^T + bias) done in the
 * GEMM epilogue's registers, which also writes stats[M][2] = (rstd, -mean*rstd) of every updated row (eps 1e-5, moments
 * of the ROUNDED values over all N columns; the epilogue emits one partial (mean, M2) per 128 columns and the consuming
 * GEMM merges them — here a small kernel does) — the LayerNorm statistics the next GEMM folds in (out_proj -> ln_2,
 * c_proj -> next ln_1). N % 256 == 0, K % 64 == 0; fp32 stats on the device. Test seam. */
ARP_API int arp_resid_gemm_stats(ArpHandle* h, const void* a_dev, const void* w_dev, const float* bias_dev, void* x_dev,
                         float* stats_dev, int64_t M, int32_t N, int32_t K, void* stream);
/* out[M,N] = act(LayerNorm(x; gamma, beta) W^T + bias) with the LayerNorm FOLDED into the GEMM as on the default path
 * (ln_1 -> in_proj, ln_2 -> c_fc; openai/CLIP ResidualAttentionBlock): x [M,768] in the operand format is multiplied raw
 * by gamma-folded weights and the epilogue applies the row's (rstd, -mean*rstd). w fp32 [N,768], gamma / beta [768],
 * bias [N] fp32 DEVICE; out in the operand format; act 0 none, 1 QuickGELU. Allocates its temporaries per call: test seam. */
ARP_API int arp_ln_gemm(ArpHandle* h, const void* x_dev, const float* gamma_dev, const float* beta_dev, const float* w_f32_dev,
                const float* bias_dev, void* out_dev, int64_t M, int32_t N, int32_t act, void* stream);
/* y = LayerNorm(x) over 768-wide rows, fp32 in, bf16 out */
ARP_API int arp_layernorm_bf16(ArpHandle* h, const float* x_dev, const float* gamma_dev, const float* beta_dev, void* y_dev,
                       int64_t M, void* stream);
/* softmax(QK^T/8)V for qkv bf16 [B*tokens, 3*width] -> bf16 [B*tokens, width]; tokens = 197 or 50 */
ARP_API int arp_attention(ArpHandle* h, const void* qkv_dev, void* out_dev, int32_t B, int32_t tokens, void* stream);
/* the pruned last block's class-token attention: softmax(q K^T/8) V of ONE query row per (frame, head), q [B, width]
 * (head h at columns 64h), K and V of the frame's tokens in qkv [B*tokens, 3*width] as arp_attention takes it (the Q
 * third is not read) -> out [B, width]; operand format throughout, tokens = 197 or 50. Test seam. */
ARP_API int arp_cls_attention(ArpHandle* h, const void* q_dev, const void* qkv_dev, void* out_dev, int32_t B,
                              int32_t tokens, void* stream);

/* counters: kernels launched by this handle since creation (bench.py's gpu_launches) */
ARP_API int64_t arp_launch_count(const ArpHandle* h);

/* Optional per-kernel-class timing. Between begin and end every launch is bracketed by CUDA events on the
 * stream it is launched on; end synchronises the device and fills stats[class] for
 * class 0 GEMM, 1 attention, 2 LayerNorm, 3 decode, 4 head, 5 scan, 6 other. `flops` / `bytes` are the
 * ALGORITHMIC work of those launches (2MNK; operand + result bytes), not hardware counters. */
typedef struct ArpProfileStats {
  int64_t launches;
  double total_ms;
  double flops;
  double bytes;
} ArpProfileStats;
#define ARP_PROFILE_CLASSES 7
ARP_API int arp_profile_begin(ArpHandle* h);
ARP_API int arp_profile_end(ArpHandle* h, ArpProfileStats* stats, int32_t n_classes);

#ifdef __cplusplus
}
#endif
#endif /* ARP_B200_H_ */
