/* sealdec.h — C ABI of the B200-native constrained beam-search decode for SEAL.
 *
 * Replaces, behind the reference's own Python surface (seal_b200/beam_search.py mirrors
 * /root/reference/seal/beam_search.py), the per-step work of
 *   - IndexBasedLogitsProcessor.__call__            seal/beam_search.py:62-140
 *   - constrained_beam_search's step                seal/beam_search.py:219-345
 *   - BeamSearchScorerWithMemory.process/finalize   seal/beam_search.py:614-735
 *   - the BART-large forward the reference gets from transformers 4.13 (call sites
 *     seal/beam_search.py:231-238,481-483; model = BartForConditionalGeneration)
 * Plain pointers and sizes only.  Status codes and sealfm_last_error() as in sealfm.h.
 * Everything runs on the GPU; there is no CPU path.
 */
#ifndef SEALDEC_H
#define SEALDEC_H
#include <stdint.h>
#include "sealfm.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ---- stateless logits-processor hook (HF LogitsProcessor protocol) ------------------------------ */

typedef struct {
    int32_t num_beams;
    int32_t pad_token_id;              /* IndexBasedLogitsProcessor defaults: 0          (:43) */
    int32_t eos_token_id;              /*                                     2          (:44) */
    int32_t stop_at_count;             /* 0 = off                                        (:46) */
    int32_t always_allow_eos;          /*                                                (:47) */
    int32_t forced_bos_token_id;       /* -1 = None                                      (:48) */
    int32_t n_force_decoding_from;     /* length of force_decoding_from, 0 = None        (:45) */
    const int64_t* force_decoding_from;/* host pointer                                         */
    int32_t shift;                     /* seal/index.py:16 SHIFT = 10                           */
} sealdec_processor_cfg_t;

/* scores_out[r][v] = scores_in[r][v] + (allowed(r,v) ? 0 : -inf)  — seal/beam_search.py:62-140.
 * input_ids_d: int64 [R][t] (device), scores: float32 [R][ld] (device; in == out allowed).
 * occurring_mask_d: uint32 [ceil(V/32)] bitmask of index.occurring_distinct (first-step rule :73-77).
 * No host synchronisation. */
int sealdec_apply_index_mask_d(const sealfm_t* fm, sealfm_stream_t stream,
                               const sealdec_processor_cfg_t* cfg,
                               const int64_t* input_ids_d, int64_t R, int64_t t,
                               const uint32_t* occurring_mask_d,
                               const float* scores_in_d, float* scores_out_d, int64_t V, int64_t ld);

/* ---- BART weights ----------------------------------------------------------------------------- */

typedef struct sealbart sealbart_t;

typedef struct {
    int32_t vocab_size;        /* 50265 after resize (seal/retrieval.py:570)   */
    int32_t d_model;           /* 1024                                         */
    int32_t encoder_layers;    /* 12                                           */
    int32_t decoder_layers;    /* 12                                           */
    int32_t heads;             /* 16 (head_dim must be 64)                     */
    int32_t ffn_dim;           /* 4096                                         */
    int32_t max_positions;     /* 1024 (+2 learned offset)                     */
    int32_t scale_embedding;   /* 0 for bart-large                             */
    int32_t gemm_mode;         /* 5 = 3xFP16 on CTA pairs (cta_group::2, 256x256 tiles; mode 3's kernel with split-K for small problems; default), 3 = 3xFP16, one CTA per 128x256 tile, 2 = 3xTF32 (fp32 range).  All tcgen05 + TMA + TMEM. */
} sealbart_config_t;

int  sealbart_create(const sealbart_config_t* cfg, int device, sealbart_t** out);
void sealbart_free(sealbart_t* m);
/* Copies one tensor of an HF BartForConditionalGeneration state_dict (float32, host pointer,
 * row-major, `numel` elements) by its state_dict key, e.g.
 * "model.decoder.layers.3.encoder_attn.q_proj.weight".  Unknown keys return SEALFM_EINVAL. */
int  sealbart_set_tensor(sealbart_t* m, const char* key, const float* host, uint64_t numel);
/* After all tensors are set: checks completeness, ties lm_head to model.shared if it was not
 * given, derives fused/pre-split copies. */
int  sealbart_finalize(sealbart_t* m);
uint64_t sealbart_device_bytes(const sealbart_t* m);

/* ---- fused generate --------------------------------------------------------------------------- */

typedef struct {
    int32_t num_beams;
    int32_t min_length;
    int32_t max_length;
    float   length_penalty;
    int32_t eos_token_id;            /* scorer / processor eos (fm_index_generate kwarg, :403)        */
    int32_t pad_token_id;            /* model.config.pad_token_id (1)                                */
    int32_t decoder_start_token_id;  /* model.config.decoder_start_token_id (2)                      */
    int32_t model_eos_token_id;      /* model.config.eos_token_id: MinLength processor (SURVEY §H3)  */
    int32_t forced_eos_token_id;     /* model.config.forced_eos_token_id, -1 = None (§H3)            */
    int32_t forced_bos_token_id;     /* -1 = None                                                    */
    int32_t stop_at_count;
    int32_t always_allow_eos;
    int32_t disable_fm_index;
    int32_t remove_invalid_values;   /* InfNanRemoveLogitsProcessor (:445)                           */
    int32_t n_force_decoding_from;
    const int64_t* force_decoding_from;   /* host pointer */
    int32_t shift;                   /* 10 */
} sealdec_params_t;

/* Number of hypothesis records per query that sealdec_generate writes:
 * (max_length-1) * 2*num_beams + num_beams   (process :662-668 every step + finalize :717-725). */
int64_t sealdec_hyps_per_query(const sealdec_params_t* p);

/* fm_index_generate(model, index, input_ids, attention_mask, ..., keep_history=True)
 * seal/beam_search.py:391-557.  HOST buffers in and out (copies are part of the call):
 *   input_ids, attention_mask  int64 [Q][S]
 *   out_scores   float32 [Q][H]      sum_logprobs of each recorded hypothesis (:667); caller applies
 *                                    score/len**lp * len**lp (:754,:555) — identity for lp = 0
 *   out_len      int32   [Q][H]      tokens in the hypothesis (incl. decoder_start)
 *   out_tokens   int32   [Q][H][max_length]
 *   out_valid    uint8   [Q][H]      1 iff the pick's CONSTRAINED score was finite (SURVEY §H4);
 *                                    finalize records carry 2
 *   out_lo/out_hi uint64 [Q][H]      SA range [lo,hi) of the hypothesis' tokens[1:] (0,0 if invalid
 *                                    or FM index disabled); may be NULL
 * H = sealdec_hyps_per_query(p).  Returns SEALFM_EINVAL("beam") if some query had fewer than
 * num_beams non-EOS candidates (the reference raises ValueError, :687-690).  If an activation leaves the fp16
 * range of the default GEMM mode the pass is repeated with the 3xTF32 kernels (sealbart_get_stat "overflow_fallbacks"). */
int sealdec_generate(sealbart_t* model, const sealfm_t* fm, const uint32_t* occurring_mask_host,
                     const sealdec_params_t* p, const int64_t* input_ids, const int64_t* attention_mask,
                     int64_t Q, int64_t S, float* out_scores, int32_t* out_len, int32_t* out_tokens,
                     uint8_t* out_valid, uint64_t* out_lo, uint64_t* out_hi);

/* Same, inputs and outputs already resident on the model's device; asynchronous on `stream` except for
 * workspace (re)allocation and -- without a source-token count, see sealdec_generate_dx -- one 16-byte read-back
 * of the real source-token count.  *_d pointers are device pointers.
 * error_flag_d: int32[4] on the device, zeroed by the call and raised by its kernels:
 *   [0] some query had fewer than num_beams non-EOS candidates   (the reference raises ValueError, :687-690)
 *   [1] an activation left the fp16 range of the 3xFP16 GEMM modes (|x| > 65504; operands were saturated): the
 *       results are NOT to be used -- re-run after sealbart_set_option(model, "gemm_mode", 2) (3xTF32, fp32 range).
 *       sealdec_generate (host buffers) does that by itself.
 *   [2] src_tokens_hint did not match the attention mask
 *   [3] reserved */
int sealdec_generate_d(sealbart_t* model, const sealfm_t* fm, const uint32_t* occurring_mask_d,
                       const sealdec_params_t* p, const int64_t* input_ids_d,
                       const int64_t* attention_mask_d, int64_t Q, int64_t S, sealfm_stream_t stream,
                       float* out_scores_d, int32_t* out_len_d, int32_t* out_tokens_d,
                       uint8_t* out_valid_d, uint64_t* out_lo_d, uint64_t* out_hi_d,
                       int32_t* error_flag_d);
/* sealdec_generate_d plus what the caller knows about the sources:
 *   src_tokens_hint >= 1  the number of non-zero attention_mask entries, masks right-padded (the only kind SEAL
 *                         builds): the encoder runs on the real tokens only and the call never touches the host;
 *                         a wrong count raises error_flag_d[2];
 *                   -1    unknown (sealdec_generate_d): one 16-byte device->host read to learn it;
 *                   -2    compute the padded positions too (no host access either).
 * On a non-default stream, batches of at most 4096 rows (queries x beams) are replayed from a CUDA graph of the
 * whole call from the third call with the same shapes, parameters and buffer addresses on (a generate of 20
 * queries is ~1 900 short kernels: launch-bound); sealbart_set_option(model, "cuda_graph", 0 / 1 / -1) forces it
 * off / on / back to automatic. */
int sealdec_generate_dx(sealbart_t* model, const sealfm_t* fm, const uint32_t* occurring_mask_d,
                        const sealdec_params_t* p, const int64_t* input_ids_d,
                        const int64_t* attention_mask_d, int64_t Q, int64_t S, sealfm_stream_t stream,
                        float* out_scores_d, int32_t* out_len_d, int32_t* out_tokens_d,
                        uint8_t* out_valid_d, uint64_t* out_lo_d, uint64_t* out_hi_d,
                        int32_t* error_flag_d, int64_t src_tokens_hint);
/* Options: "cuda_graph" (-1 auto, 0 off, 1 on), "gemm_mode" (switch between the 3xFP16 modes 3/5 and 2 = 3xTF32;
 * the TF32 operand copies are made on first use).  Stats: "last_used_graph", "overflow_fallbacks", "gemm_mode",
 * "cached_graphs" (-1 for an unknown name). */
int     sealbart_set_option(sealbart_t* model, const char* name, int64_t value);
int64_t sealbart_get_stat(const sealbart_t* model, const char* name);

/* ---- teacher-forced scoring: SURVEY.md section 8(f) rank 1 ------------------------------------------
 * The decoder pass behind rescore_keys (seal/keys.py:64-141) and compute_unigram_scores (:145-176).
 * dec_ids: int64 [N][T] decoder inputs (row r = decoder_start + key tokens, right-padded), row r is
 * scored against encoder input row_query[r] (sorted ascending).  HOST pointers.
 *   out_logprob [N][T-1]: log_softmax(logits_p / temperature)[dec_ids[r][p+1]] for p = 0..T-2
 *                         (full-vocabulary normalisation; the caller masks padding and sums, :131-135)
 *   out_full    [N][V]  : if non-NULL, the whole log-prob vector of position out_full_pos (:167-172) */
int sealdec_teacher_forced(sealbart_t* model, const int64_t* input_ids, const int64_t* attention_mask,
                           int64_t Q, int64_t S, const int64_t* dec_ids, const int32_t* row_query,
                           int64_t N, int64_t T, float temperature, float* out_logprob,
                           int64_t out_full_pos, float* out_full);

/* Test / profiling hooks: one decoder step's logits for explicit decoder inputs (teacher forcing).
 * decoder_input_ids int64 [R][t] host, R = Q*num_beams rows laid out query-major like the
 * reference's expanded batch (:517-521); writes float32 [R][V] host logits of the last position. */
int sealdec_debug_step_logits(sealbart_t* model, const int64_t* input_ids, const int64_t* attention_mask,
                              int64_t Q, int64_t S, int32_t num_beams, const int64_t* decoder_input_ids,
                              int64_t t, float* out_logits);
/* Stand-alone GEMM C[M,N] = A[M,K] W[N,K]^T + bias (+GELU) through the model's GEMM kernels
 * (mode 2 = 3xTF32, 3 = 3xFP16, 5 = 3xFP16 on CTA pairs), host pointers; if iters > 0 also reports the average
 * device time per call (CUDA events, includes the activation split). */
int sealdec_debug_gemm(int mode, int64_t M, int32_t N, int32_t K, const float* A, const float* W,
                       const float* bias, float* C, int32_t gelu, int32_t iters, double* avg_us);
/* The same GEMM with the output written as the fp16 split (h1, h2) that the next 3xFP16 GEMM consumes (modes 3 and 5):
 * halves_sum float32 [M][N] host receives h1 + h2; *overflow (may be NULL) = 1 if an output left the fp16 range
 * (|x| > 65504, saturated), else 0. */
int sealdec_debug_gemm_split(int mode, int64_t M, int32_t N, int32_t K, const float* A, const float* W,
                             const float* bias, int32_t gelu, float* halves_sum, int32_t* overflow);
/* in-kernel timeline of CTA 0 of the mode-3/4 GEMM kernel (development aid): out20 (may be NULL) receives
 * the stamps of the last traced launch -- SM cycles at 0 entry, 1 prologue done, 2 first operands landed,
 * 3 last MMA issued, 4 last chunk complete, 5 tile stored, 6 exit; 7/8 globaltimer ns at entry / exit --
 * 9..16 the epilogue's four store passes (staged / stored) -- then tracing is switched on (enable != 0) or off. */
int sealdec_debug_gemm_trace(int enable, int64_t out20[20]);
/* kernel launches issued by the last sealdec_generate* call on this model (own kernels only) */
int64_t sealdec_last_launch_count(const sealbart_t* model);
/* GEMM profiling: enable != 0 makes every following GEMM launch of this model be bracketed by CUDA
 * events on its stream.  When total_us/launches/flops are non-NULL the call first drains the device
 * and returns the summed device time, launch count and 2MNK flops recorded since the previous call,
 * then clears the record. */
int sealdec_profile_gemm(sealbart_t* model, int enable, double* total_us, int64_t* launches, double* flops);
/* microseconds spent (CUDA events) in the last generate, split by phase:
 * 0 encoder, 1 decoder layers, 2 lm_head, 3 select+expand (FM index), 4 total */
int sealdec_last_phase_us(const sealbart_t* model, double out5[5]);

#ifdef __cplusplus
}
#endif
#endif /* SEALDEC_H */
