/* ance_b200.h — C ABI of libance_b200.so: the B200-native replacement for the native arithmetic on
 * microsoft/ANCE's ANN-refresh path (drivers/run_ann_data_gen.py + model/models.py).
 *
 * The reference has no FFI of its own: the native work on this path is done by un-vendored
 * libraries called directly from Python.  Each entry point below names the reference call site it
 * replaces.  Plain C, opaque handles, int status (0 = ok), ance_last_error() for the message, no
 * exceptions and no torch types across the boundary.  All *_dev pointers are CUDA device pointers
 * on the device that was current when the handle was created; `stream` is a cudaStream_t passed as
 * void*.  Handles are not thread-safe; distinct handles may be used concurrently.
 *
 * There is NO CPU fallback: every compute entry point fails with ANCE_ERR_CUDA when no sm_100
 * device is present.
 */
#ifndef ANCE_B200_H_
#define ANCE_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum {
  ANCE_OK = 0,
  ANCE_ERR_INVALID = 1,     /* bad argument */
  ANCE_ERR_CUDA = 2,        /* CUDA runtime / driver error, or no sm_100 device */
  ANCE_ERR_NOMEM = 3,
  ANCE_ERR_UNSUPPORTED = 4  /* shape outside what the kernels were built for */
};

/* 16-bit operand format of the tensor-core passes (tcgen05 kind::f16 runs both at the same rate). */
enum { ANCE_FMT_FP16 = 0, ANCE_FMT_BF16 = 1 };

const char* ance_version(void);
const char* ance_last_error(void);
/* number of kernels this library has launched in the calling process (bench.py's gpu_launches) */
int64_t ance_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * Flat inner-product index  — replaces faiss.IndexFlatIP(dim) / .add / .search
 *   reference: drivers/run_ann_data_gen.py:269-276,303 ; drivers/run_ann_data_gen_dpr.py:238-252
 * Semantics (faiss IndexFlatIP): for each query the k rows with the largest fp32 inner product,
 * sorted by score descending; labels are row numbers in insertion order (+ row_offset), int64;
 * when fewer than k rows exist the tail is label -1 / score -FLT_MAX.  Ties are broken by the
 * smaller row number (faiss leaves tie order unspecified; ours is deterministic).
 * Scores are the exact fp32-input dot product accumulated in fp64 and rounded once to fp32.
 * k is at most 2048 (faiss's GPU flat index has the same limit): ance_index_search and ance_index_search_exact fail with
 * ANCE_ERR_INVALID and an error message naming the limit for k > 2048.  k <= 512 runs the register-resident coarse
 * epilogue; 512 < k <= 2048 keeps larger candidate reservoirs in global memory (up to 1.2 GB of scratch on a 148-SM
 * device, allocated the first time such a k is searched) and gives the same exact, certified results.
 * ance_index_search fails with ANCE_ERR_UNSUPPORTED when an index row or a query is non-finite after rounding to the
 * 16-bit operand format (inf / NaN input, or |x| > 65504 with ANCE_FMT_FP16) instead of returning unverifiable results.
 * ------------------------------------------------------------------------------------------------ */
typedef struct ance_index* ance_index_t;

typedef struct {
  int64_t nq;             /* queries in the last search */
  int64_t n_tier2;        /* queries the first coarse pass could not certify -> second pass from their own thresholds */
  int64_t n_uncertified;  /* queries no coarse pass could certify -> exact brute-force fallback */
  int64_t n_candidates;   /* candidates rescored in fp32/fp64 */
  int32_t kprime;         /* candidates kept per (query, split) by the coarse pass */
  int32_t n_splits;       /* row-range splits of the corpus per query tile */
  float max_eps;          /* largest per-query coarse-score error bound used by the certificate */
} ance_search_stats;

int ance_index_create(int dim, int64_t capacity_rows, int operand_fmt, ance_index_t* out);
/* Same, over CALLER-OWNED fp32 row storage rows_dev [capacity_rows, dim] (16-byte aligned, must outlive the index; never
 * freed by it).  A producer that writes rows i .. i+n straight into rows_dev + i*dim and then calls
 * ance_index_add(idx, rows_dev + i*dim, n) adds them WITHOUT a copy: this is how the refresher keeps one fp32 copy of the
 * corpus instead of the reference's three (per-batch arrays -> concatenation -> faiss storage,
 * drivers/run_ann_data_gen.py:160-193,271). */
int ance_index_create_over(int dim, int64_t capacity_rows, int operand_fmt, float* rows_dev, ance_index_t* out);
int ance_index_destroy(ance_index_t idx);
int ance_index_reset(ance_index_t idx);                       /* ntotal = 0, storage kept */
int64_t ance_index_ntotal(ance_index_t idx);
/* IndexFlatIP.add: append n rows (fp32, row-major [n, dim], device memory). */
int ance_index_add(ance_index_t idx, const float* rows_dev, int64_t n, void* stream);
/* Build the 16-bit operands of the coarse pass from ALL rows added so far: the rows are centred on their column mean
 * (<q, p> = <q, p - mu> + <q, mu>: the ranking does not change, the certificate's error bound shrinks to the centred rows'
 * norms) and rounded to operand_fmt.  ance_index_search does this itself when rows were added since the last time
 * (8.84M rows: ~10 ms); call it explicitly to keep that cost out of the first search. */
int ance_index_prepare(ance_index_t idx, void* stream);
/* IndexFlatIP.search: Q [nq, dim] fp32 -> D [nq, k] fp32, I [nq, k] int64 (all device memory). */
int ance_index_search(ance_index_t idx, const float* q_dev, int64_t nq, int k, float* D_dev, int64_t* I_dev,
                      int64_t row_offset, void* stream);
/* Same contract, computed entirely by the exact fp32->fp64 brute-force kernel (validation path). */
int ance_index_search_exact(ance_index_t idx, const float* q_dev, int64_t nq, int k, float* D_dev,
                            int64_t* I_dev, int64_t row_offset, void* stream);
/* Statistics of the last search (ance_index_search has already synchronised its stream). */
int ance_index_last_stats(ance_index_t idx, ance_search_stats* out);
/* Tunables: "kprime" (0 = auto: about 1.44 k for fp16 operands, 2 k for bf16; a multiple of 32 up to 4128 = 2 * 2048 + 32;
 * a k' below k sends the search to the exact path), "n_splits" (0 = auto), "cta_group" (1|2),
 * "max_ctas" (0 = all SMs), "tier2" (0|1), "exact_fallback" (0|1: measurement only — results of uncertified queries are
 * then NOT guaranteed), "pace_window" (tiles a sweeping CTA pair may run ahead of the slowest one; 0 = no soft
 * barrier), "operand_fmt" (ANCE_FMT_*: the rows already added are re-rounded from the fp32 copy at the next prepare / search),
 * "center" (0|1, default 1: centre the rows before rounding). */
int ance_index_set_param(ance_index_t idx, const char* name, double value);

/* Host k-way merge of per-shard results — replaces utils/util.py:87-146 barrier_array_merge +
 * the rank-0-only search (the reference's own precedent: utils/eval_mrr.py:175-183).
 * D[s], I[s]: [nq, k] sorted descending per shard (labels already global).  Output [nq, k]. */
int ance_merge_topk_host(const float* const* D, const int64_t* const* I, int n_shards, int64_t nq, int k,
                         float* D_out, int64_t* I_out, int n_threads);

/* ann_training_data_N writer (host only) — replaces the per-query formatting loop of drivers/run_ann_data_gen.py:318-329.
 * Line i = "qid \t pos \t n1,n2,...\n" of query order[i]; neg [n, neg_stride] holds counts[q] valid ids per row. */
int ance_write_training_data_host(const char* path, const int64_t* qids, const int64_t* pos, const int64_t* neg,
                                  const int64_t* counts, const int64_t* order, int64_t n, int neg_stride,
                                  int64_t* lines_written);

/* ------------------------------------------------------------------------------------------------
 * Dual-encoder forward — replaces the HF RobertaModel/BertModel forward + embeddingHead + norm
 *   reference: model/models.py:149-157 (RobertaDot_NLL_LN.query_emb/body_emb),
 *              model/models.py:165-199 (MultiChunk body_emb, caller reshapes [B,2048]->[4B,512]),
 *              model/models.py:223-259 (BiEncoder / HFBertEncoder, CLS of last layer, no head)
 * ------------------------------------------------------------------------------------------------ */
typedef struct ance_encoder* ance_encoder_t;

enum { ANCE_ARCH_ROBERTA = 0, ANCE_ARCH_BERT = 1 };

typedef struct {
  int arch;        /* ANCE_ARCH_ROBERTA: position ids = cumsum(ids != pad) * (ids != pad) + pad_id
                      ANCE_ARCH_BERT   : position ids = 0..L-1 */
  int n_layer, hidden, heads, ffn, vocab, max_pos, type_vocab, pad_id;
  float ln_eps;
  int has_head;    /* 1: out = LayerNorm(Linear(CLS)) (models.py:152-153); 0: out = CLS (models.py:237-239) */
  int operand_fmt; /* ANCE_FMT_FP16 (recommended) or ANCE_FMT_BF16: 16-bit storage format of weights and activations.
                      Both run the tensor cores at the same rate with fp32 accumulation; fp16 keeps 11 significant bits
                      instead of 8, i.e. 8x closer to the reference's fp32 forward.  A checkpoint whose activations
                      leave the fp16 range (|x| > 65504) produces non-finite embeddings, which ance_encoder_check
                      reports as ANCE_ERR_UNSUPPORTED: use ANCE_FMT_BF16 for such a model. */
} ance_encoder_config;

/* All weight pointers are HOST fp32 arrays in the checkpoint's own layout (Linear weight = [out, in]);
 * the library converts and uploads them once (Linear weights -> operand_fmt; embedding tables, biases and LayerNorm
 * parameters stay fp32). */
typedef struct {
  const float *q_w, *q_b, *k_w, *k_b, *v_w, *v_b;   /* attention.self.{query,key,value} */
  const float *ao_w, *ao_b, *ln1_g, *ln1_b;         /* attention.output.{dense,LayerNorm} */
  const float *ff1_w, *ff1_b;                       /* intermediate.dense */
  const float *ff2_w, *ff2_b, *ln2_g, *ln2_b;       /* output.{dense,LayerNorm} */
} ance_layer_weights;

typedef struct {
  const float *word_emb, *pos_emb, *type_emb, *emb_ln_g, *emb_ln_b;
  const ance_layer_weights* layers;                 /* [n_layer] */
  const float *head_w, *head_b, *head_ln_g, *head_ln_b; /* embeddingHead, norm (has_head only) */
} ance_encoder_weights;

int ance_encoder_create(const ance_encoder_config* cfg, const ance_encoder_weights* w, int max_tokens,
                        ance_encoder_t* out);
int ance_encoder_destroy(ance_encoder_t enc);
/* ids_dev [B, L] int32.  Attention mask: lens_dev [B] int32 (mask = 1^len 0^(L-len), the
 * data/msmarco_data.py:275-303 form) or mask_dev [B, L] uint8 (data/DPR_data.py:283 form); exactly one
 * non-null.  Masked keys get the additive -10000 of HF 2.3.0, so an all-pad sequence yields the
 * finite "uniform attention" vector the reference yields.  out_dev [B, hidden] fp32. */
int ance_encoder_forward(ance_encoder_t enc, const int32_t* ids_dev, const int32_t* lens_dev,
                         const uint8_t* mask_dev, int B, int L, float* out_dev, void* stream);
/* Variable-length form of the same forward for L <= 128 (the MS MARCO passage / query caches): sequence b has lens[b]
 * real tokens followed by padding (data/msmarco_data.py:275-303), and only the real tokens are computed.  Whole sequences
 * are packed into 128-row attention tiles (a tile holds sequences of ANY lengths, none straddles a tile, every sequence
 * attends to its own tokens only), the linear layers and LayerNorms run on the packed token matrix, the CLS rows are
 * gathered for the last layer and the head.  lens_dev and lens_host hold the same B lengths, each in [1, L] (the tile
 * packing is planned on the host); B is unlimited (the call splits by the handle's max_tokens).  With the default
 * "varlen_align" = 1 the embeddings equal those of ance_encoder_forward up to fp32 summation order inside the softmax / P*V
 * of a tile (a sequence's terms are grouped by its offset in the tile; tests: |diff| <= 1e-2, both within the gate of the
 * fp32 reference); with "varlen_align" = 16 every sequence starts at a multiple of the tensor core's K step and the result
 * is bit-identical to ance_encoder_forward and independent of the batch composition, at ~12 % fewer real tokens per tile. */
int ance_encoder_forward_varlen(ance_encoder_t enc, const int32_t* ids_dev, const int32_t* lens_dev,
                                const int32_t* lens_host, int B, int L, float* out_dev, void* stream);
/* Tunables: "prune_last_layer" (default 1): in the last layer only token 0 of every sequence is read
 * downstream, so out-projection / FFN / LayerNorm run on those rows only (result-identical; bench.py reports
 * the executed FLOPs beside the algorithmic ones).  "ln_rows_per_warp" (1, 2, 4, or 3 = two rows held packed; default 2, process-wide): rows a warp
 * of the LayerNorm kernel normalises side by side (bit-identical results; 2 is the fastest on B200).  "varlen_align" (1 | 16):
 * see ance_encoder_forward_varlen. */
int ance_encoder_set_param(ance_encoder_t enc, const char* name, double value);
/* Input / output validation, deferred so that forward stays asynchronous: synchronises `stream` and returns
 * ANCE_ERR_INVALID if any forward since the last check saw a token id outside [0, vocab_size) or a position
 * beyond max_position_embeddings (such lookups are clamped on the device; the reference's nn.Embedding raises
 * an index error, model/models.py:150-155 -> transformers modeling_roberta.py embeddings), ANCE_ERR_UNSUPPORTED if
 * any forward produced a non-finite embedding (fp16 range exceeded, or NaN weights).  The drivers call it once per
 * encode pass. */
int ance_encoder_check(ance_encoder_t enc, void* stream);
/* Debug / parity: copy the hidden states after layer `layer` (0 = embeddings) of the last forward
 * into out_dev [B*L, hidden] fp32 (with prune_last_layer the last layer holds its B CLS rows first). */
int ance_encoder_debug_hidden(ance_encoder_t enc, int layer, float* out_dev, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Device-time profile by kernel class (bench.py's roofline numbers): CUDA events recorded around every
 * launch on the launch stream.  Classes: 0 encoder GEMM, 1 attention, 2 LayerNorm/embedding/gather,
 * 3 operand quantisation, 4 coarse search GEMM, 5 exact rescore, 6 exact brute force, 7-10 encoder
 * GEMMs by role (QKV, attention out-proj, FFN up, FFN down; class 0 then holds the head GEMM only).
 * ance_profile_read synchronises the device, returns milliseconds and launch counts per class
 * (arrays of length n <= 12) and optionally resets the accumulators.
 * ------------------------------------------------------------------------------------------------ */
int ance_profile_enable(int on);
int ance_profile_read(double* ms_by_class, int64_t* launches_by_class, int n, int reset);

/* ------------------------------------------------------------------------------------------------
 * Bring-up / test hooks (not part of the drop-in surface)
 * ------------------------------------------------------------------------------------------------ */
/* D[M,N] = act(A[M,K] * B[N,K]^T + bias) + R ; A,B 16-bit device arrays in `fmt`; outputs optional.
 * variant: 0 = BN 256 CG 1, 1 = BN 128 CG 1, 2 = BN 256 CG 2, 3 = BN 128 CG 2, 4 = BN 64 CG 1 */
/* Host-only: the tile plan ance_encoder_forward_varlen makes for the first chunk of lens_host[0..B) on a handle created with
 * `max_tokens`: row0_out[i] = packed row of sequence i's first token (i < *n_placed), lo/hi_out [*n_tiles * 128] = own-sequence
 * key range of every packed row (may be null). */
int ance_dbg_pack_varlen(const int32_t* lens_host, int B, int max_tokens, int align, int32_t* row0_out, uint8_t* lo_out,
                         uint8_t* hi_out, int* n_placed, int* n_tiles);
int ance_dbg_gemm(const void* A_dev, const void* B_dev, int M, int N, int K, int fmt, int variant,
                  const float* bias_dev, const void* residual_bf16_dev, int act, void* C_bf16_dev,
                  float* C_f32_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ANCE_B200_H_ */
