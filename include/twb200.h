/*
 * twb200.h — C ABI of the B200-native Whisper transcription hot path.
 *
 * This is the drop-in boundary (SURVEY.md §8b).  The reference (crmorton/Turbo-Whisper-Workspace)
 * has no native code: its hot path is `AudioProcessingPipeline.transcribe`
 * (ref: vocalis/core/audio_pipeline.py:323-369) calling a Hugging Face ASR pipeline object
 * (ref: vocalis/core/audio_pipeline.py:195-200,351-358).  All arithmetic behind that call lives in
 * `transformers` ($TF = transformers 5.5.0 as installed; the reference pins 4.54.1).  Each entry
 * point below names the $TF function whose arithmetic it replaces.  The Python host side
 * (`turbo-whisper-workspace_b200/pipeline.py`) keeps the HF pipeline call signature and binds these
 * symbols with ctypes; INTEGRATION.md shows the reference-side stub.
 *
 * Conventions
 *  - plain pointers and sizes only; no torch types.  `void* stream` is a `cudaStream_t`.
 *  - device pointers are borrowed for the duration of the call (stream-ordered); the caller
 *    (PyTorch, as the device allocator) owns every buffer.  The library allocates nothing on the
 *    device.
 *  - bf16 tensors are passed as `void*` (16-bit storage), row-major unless stated.
 *  - every function returns 0 on success; on failure a non-zero status and `tw_last_error()`
 *    (thread-local, NUL-terminated) describes it.  Nothing is launched on argument errors.
 *  - there is no CPU fallback: without an sm_100 device the launch functions fail.
 */
#ifndef TWB200_H_
#define TWB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TW_ABI_VERSION 1

const char* tw_last_error(void);
int tw_abi_version(void);

/* ------------------------------------------------------------------------------------------------
 * K1  log-mel front end.
 * Replaces WhisperFeatureExtractor._torch_extract_fbank_features
 * ($TF/models/whisper/feature_extraction_whisper.py:135-164) for clips already cut to <= 30 s:
 * zero-pad to 480000 samples, reflect-padded 400-point STFT at hop 160 (periodic Hann), power,
 * 128 (or, through the *_n entry points, 80) slaney mel filters, log10(max(.,1e-10)), max(x, clipmax-8), (x+4)/4.
 * ---------------------------------------------------------------------------------------------- */
size_t tw_logmel_tables_bytes(void);
size_t tw_logmel_scratch_bytes(int32_t batch);
/* mel_filters: host fp32 [201,128] exactly as WhisperFeatureExtractor.mel_filters (cast to fp32). */
int tw_logmel_init(void* tables_dev, const float* mel_filters_host_201x128);
/* pcm: device fp32 [batch, pcm_stride] (pcm_stride >= 480000); n_valid: device int32 [batch] number
 * of real samples per clip (NULL = 480000), samples beyond it are treated as zeros.
 * out_f32: device fp32 [batch,128,3000] or NULL.  out_bf16_t: device bf16 time-major
 * [batch, rows, 128] or NULL, frame t is written to row (out_t_row_off + t); out_t_bstride in
 * elements. */
int tw_logmel(const void* tables_dev, const float* pcm, int64_t pcm_stride, const int32_t* n_valid,
              int32_t batch, void* scratch, float* out_f32, void* out_bf16_t,
              int64_t out_t_bstride, int32_t out_t_row_off, void* stream);
/* Whole-clip features for un-chunked long-form input (WhisperFeatureExtractor with truncation=False over the full
 * waveform, $TF/models/whisper/feature_extraction_whisper.py:135-164; the ASR pipeline's path for > 30 s without
 * chunk_length_s, $TF/pipelines/automatic_speech_recognition.py:446-454).  pcm_long: device fp32, covered by n_windows
 * overlapping 30 s windows that start hop_samples apart (window b = pcm_long[b*hop_samples .. +480000), readable and
 * zero beyond the clip; the caller appends the 200 reflected samples of the clip's end).  Window b writes its frames
 * [frame_lo[b], frame_hi[b]) to rows out_t_row_off + out_row0[b].. of out_bf16_t (time-major [rows,128]); the max - 8
 * clamp uses the maximum over all written frames (max_scratch: one device uint32).  The arrays are device int32. */
int tw_logmel_long(const void* tables_dev, const float* pcm_long, int64_t hop_samples, int32_t n_windows,
                   const int32_t* frame_lo, const int32_t* frame_hi, const int32_t* out_row0, uint32_t* max_scratch,
                   void* out_bf16_t, int64_t total_frames, int32_t out_t_row_off, void* stream);
/* The same three functions for a given mel-bin count: n_mels is 128 (the large-v3 family; what the functions above
 * use) or 80 (large-v2 and older checkpoints, WhisperFeatureExtractor(feature_size=80)); any other count is an error.
 * mel_filters_host is fp32 [201, n_mels]; every [.., 128] / [.., 128, ..] shape above has n_mels in place of 128, so an
 * 80-bin frame is one 160-byte row of the time-major output.  The tables are laid out per count: launch with the count
 * they were initialised for.  tw_logmel_tables_bytes() covers either layout. */
int tw_logmel_init_n(void* tables_dev, const float* mel_filters_host, int32_t n_mels);
int tw_logmel_n(const void* tables_dev, const float* pcm, int64_t pcm_stride, const int32_t* n_valid,
                int32_t batch, void* scratch, float* out_f32, void* out_bf16_t,
                int64_t out_t_bstride, int32_t out_t_row_off, int32_t n_mels, void* stream);
int tw_logmel_long_n(const void* tables_dev, const float* pcm_long, int64_t hop_samples, int32_t n_windows,
                     const int32_t* frame_lo, const int32_t* frame_hi, const int32_t* out_row0, uint32_t* max_scratch,
                     void* out_bf16_t, int64_t total_frames, int32_t out_t_row_off, int32_t n_mels, void* stream);
/* Whole-clip features of SEVERAL clips in one launch (plus one floor launch): the clips' buffers (each laid out as for
 * tw_logmel_long) are concatenated in pcm; window b reads pcm + win_offset[b] (samples), belongs to clip win_clip[b] and
 * writes its frames [frame_lo[b], frame_hi[b]) to rows out_row0[b].. of out_bf16_t (time-major [total_frames, n_mels]).
 * Clip c owns rows [clip_row0[c], clip_row0[c + 1]) and gets its own max - 8 clamp (max_scratch: n_clips device
 * uint32).  win_offset, clip_row0 (n_clips + 1 entries): device int64; the other arrays device int32.  A clip computed
 * alone or together with others gives the same bits. */
int tw_logmel_long_multi(const void* tables_dev, const float* pcm, const int64_t* win_offset, const int32_t* win_clip,
                         int32_t n_windows, const int32_t* frame_lo, const int32_t* frame_hi, const int32_t* out_row0,
                         int32_t n_clips, const int64_t* clip_row0, uint32_t* max_scratch, void* out_bf16_t,
                         int64_t total_frames, int32_t n_mels, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K4  LayerNorm over the last dimension, fp32 in -> bf16 out (eps as nn.LayerNorm, 1e-5).
 * Replaces the nn.LayerNorm calls of WhisperEncoderLayer / WhisperDecoderLayer
 * ($TF/models/whisper/modeling_whisper.py:380-414, 449-506) and the final layer_norm (:640, :789).
 * ---------------------------------------------------------------------------------------------- */
int tw_layernorm(const float* x, const float* gamma, const float* beta, void* out_bf16,
                 int64_t rows, int32_t cols, float eps, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K5  TMA-fed tcgen05/TMEM bf16 GEMM with fused epilogue:
 *       out[b, r, n] = act( sum_k A[b, a_row_off[b] + r, k] * W[n, k] + bias[n] ) + resid[b, r, n]
 * A is a (possibly overlapping-row) strided view: element (b, r, k) lives at
 *   a + b*a_batch_stride + r*a_row_stride + k   (strides in elements, multiples of 8).
 * That view expresses nn.Linear (batches = 1) and both Conv1d layers of the encoder stem as
 * implicit GEMMs over time-major activations (im2col is a stride trick, never materialised).
 * Replaces nn.Linear / nn.Conv1d + GELU + residual adds in WhisperEncoder.forward and
 * WhisperAttention ($TF/models/whisper/modeling_whisper.py:284-357, 380-414, 593-647).
 * ---------------------------------------------------------------------------------------------- */
typedef struct tw_gemm_args {
    const void* a;          /* bf16 */
    int64_t a_row_stride;   /* elements */
    int64_t a_batch_stride; /* elements */
    int32_t a_rows;         /* addressable rows per batch in the view (TMA bound; OOB reads 0) */
    const int32_t* a_row_off; /* device int32 [batches] or NULL */
    const void* w;          /* bf16 [N, K] row-major (nn.Linear weight layout) */
    int32_t batches;
    int32_t rows;           /* output rows per batch (M) */
    int32_t n;              /* N, multiple of 8 */
    int32_t k;              /* K, multiple of 8 */
    const float* bias;      /* fp32 [N] or NULL */
    int32_t act;            /* 0 none, 1 exact-erf GELU */
    const float* resid;     /* fp32 or NULL; element (b, r, n) at resid + (b*resid_batch_rows + r)*resid_ld + n */
    int64_t resid_ld;
    int64_t resid_batch_rows;
    void* out;              /* element (b, r, n) at out + (b*out_batch_rows + out_row_off + r)*out_ld + n */
    int32_t out_f32;        /* 0: bf16, 1: fp32 */
    int64_t out_ld;
    int64_t out_batch_rows;
    int32_t out_row_off;
    int32_t out_mode;       /* 0: row-major as above; 1: head-major out[n/64][b][r][n%64] (K/V for decode attention) */
} tw_gemm_args;
int tw_gemm_bf16(const tw_gemm_args* args, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K6  encoder self-attention (non-causal, no mask, head_dim 64), flash-style on tcgen05/TMEM.
 * qkv: bf16 [batch*seq, 3*heads*64] = the fused q|k|v projection (q already scaled by 1/8, which
 * the engine folds into Wq/bq).  out: bf16 [batch*seq, out_ld] with head h at columns 64h..64h+63.
 * Replaces the attention_interface call of WhisperAttention.forward for the encoder
 * ($TF/models/whisper/modeling_whisper.py:335-352; sdpa/eager softmax(QK^T)V with scaling=1.0).
 * ---------------------------------------------------------------------------------------------- */
int tw_attention_enc(const void* qkv_bf16, void* out_bf16, int32_t batch, int32_t seq, int32_t heads,
                     int64_t out_ld, void* stream);
/* profiling hook: device int64[192] that CTA (0,0,0) fills with clock64() stamps of its MMA thread ([0,64)) and of
 * query row 0's softmax thread ([64,128)); NULL disables (default). */
int tw_attention_enc_set_trace(void* dev_buf_int64_x192);

/* Gather a seek-shifted 30 s window of time-major features (WhisperGenerationMixin._get_input_segment,
 * $TF/models/whisper/generation_whisper.py:1831-1850): dst[b, row_off + t, :] =
 * src[src_row[b], row_off + seek[b] + t, :] for t < frames - seek[b], zeros after.  bf16 [*, rows, cols]. */
int tw_shift_frames(const void* src_bf16, void* dst_bf16, const int32_t* src_row, const int32_t* seek,
                    int32_t batch, int32_t frames, int32_t cols, int64_t batch_stride, int32_t row_off,
                    void* stream);
/* The same gather for the long-form seek loop, every row from the whole-clip features of its own clip:
 * dst[b, dst_row_off + t, :] = src_rows[b][seek[b] + t, :] for t < min(window, frames[b] - seek[b]), zeros up to window.
 * src_rows: device array of batch pointers, each to 16-byte aligned time-major bf16 features [frames[b], cols];
 * frames, seek: device int32 [batch]; dst: bf16, row b at dst_bf16 + b * dst_batch_stride (elements).  One launch. */
int tw_gather_frames(const void* const* src_rows, const int32_t* frames, const int32_t* seek, int32_t batch,
                     int32_t window, int32_t cols, void* dst_bf16, int64_t dst_batch_stride, int32_t dst_row_off,
                     void* stream);

/* ------------------------------------------------------------------------------------------------
 * K7 / K8  batched greedy decode step (<= 32 rows per call).  All per-row state lives on the
 * device so a step is a fixed launch sequence (CUDA-graph capturable):
 *   row_state: tw_row_state [batch] (below; passed as void*)
 *   self-attention KV cache is paged: pool layer base bf16 [2][n_pages][64][D],
 *   block_table int32 [batch][pages_per_row].
 * Replaces WhisperDecoder.forward / WhisperDecoderLayer with cache
 * ($TF/models/whisper/modeling_whisper.py:691-796, 449-506), DynamicLayer.update
 * ($TF/cache_utils.py:102-119), the logits processors and GenerationMixin._sample's
 * fp32-logits -> processors -> argmax -> pad-if-finished step ($TF/generation/utils.py:2762-2797).
 * ---------------------------------------------------------------------------------------------- */
/* Decoding state of one decode row (8 x int32, 32 bytes).  text_lo / ts_lo / ts_hi / begin encode what
 * WhisperTimeStampLogitsProcessor and the two Suppress* processors allow for the NEXT token
 * ($TF/generation/logits_process.py:1812-2043). */
typedef struct tw_row_state {
    int32_t pos;        /* index in tokens[] of the token fed this step */
    int32_t finished;   /* row has emitted eos */
    int32_t last_ts;    /* last timestamp token generated so far, or -1 */
    int32_t text_lo;    /* non-timestamp ids < text_lo are forbidden next step */
    int32_t ts_lo;      /* timestamp ids < ts_lo forbidden */
    int32_t ts_hi;      /* timestamp ids > ts_hi forbidden (ts_hi < ts_lo: none allowed) */
    int32_t begin;      /* 1 if the next token is the first generated one (begin-suppress applies) */
    int32_t mode;       /* bit 0: language detection at this step (only language ids allowed, cleared afterwards);
                         * bit 1: row generates without timestamps (suppress lists only, plain arg-max) */
} tw_row_state;

typedef struct tw_skinny_args {
    const void* w;      /* bf16, n rounded up to 16 rows x k, FRAGMENT-MAJOR: [n/16][k/32][2][8][4][8] with element
                         * W[16*slab + 8*half + g][32*kstep + 8*tg + e] (zero rows beyond n) — each warp load of the
                         * mma.m16n8k16 A fragments is then 512 contiguous bytes; engine.pack_skinny_weight builds it */
    const void* x;      /* bf16 [batch, ldx] */
    int32_t ldx;
    const float* bias;  /* fp32 [n] or NULL */
    int32_t batch;      /* 1..32 */
    int32_t n;
    int32_t k;          /* multiple of 256 */
    /* residual epilogue only (tw_dec_linear epilogue 2): when ln_out_bf16 is given, the last CTA to finish
     * writes LayerNorm(updated fp32 rows; gamma, beta, eps 1e-5) as bf16 [batch, n] (n <= 1280) — the operand of
     * the next projection — so the decoder needs no separate LayerNorm launches.  ln_counter: zero-initialised
     * device uint32, re-armed by the kernel. */
    const float* ln_gamma;
    const float* ln_beta;
    void* ln_out_bf16;
    uint32_t* ln_counter;
    /* LayerNorm FOLDED into the next projection:  W LN(x) + b = rstd (W' x - mean c) + d  with W' = W diag(gamma),
     * c = row sums of the bf16 W', d = W beta + b.
     * Producer (residual epilogue): with ln_part_out given, every CTA also stores bf16(updated x) into x_bf16_out
     * [batch, n] and (mean, M2) of its 16 values per row into the scratch ln_part_out[n / 16][32] (float2); the last CTA
     * to finish (ln_counter) reduces them in a fixed order to ln_stats_out[32] = (mean, rstd) per row — a tail of a few
     * hundred loads instead of a LayerNorm over batch x n values.
     * Consumer (tw_dec_linear epilogues 0 / 3, tw_dec_qkv): with ln_stats_in given, `w` holds W', `bias` holds d, `x` is
     * the producer's x_bf16_out, ln_c = c [n]; rstd / mean are applied in the epilogue. */
    void* ln_part_out;
    void* x_bf16_out;
    void* ln_stats_out;
    const void* ln_stats_in;
    const float* ln_c;
} tw_skinny_args;

typedef struct tw_grammar {
    int32_t eos, pad, no_timestamps, ts_begin, vocab, lang_first, lang_last, max_initial_ts, begin_index;
} tw_grammar;

/* Decode kernels are launched with programmatic dependent launch (each prefetches its weights before waiting for
 * its predecessor); tw_set_pdl(0) falls back to plain stream ordering (debugging). */
int tw_set_pdl(int32_t enabled);
/* x[b,:] = tok_emb[tokens[b, pos_b], :] + pos_emb[pos_b, :]   (fp32 residual stream [batch, d_model]);
 * optionally also ln_out[b,:] = LayerNorm(x[b,:]; ln_gamma, ln_beta) as bf16 (first layer's self_attn_layer_norm). */
int tw_dec_embed(const int32_t* tokens, int32_t tokens_ld, const void* row_state, const void* tok_emb_bf16,
                 const float* pos_emb, float* x, int32_t batch, int32_t d_model, const float* ln_gamma,
                 const float* ln_beta, void* ln_out_bf16, void* stream);
/* out = x W^T + bias with epilogue 0: bf16 [batch, ldo]; 3: GELU -> bf16 [batch, ldo];
 * 2: fp32 residual update in place, out[b, n] += result (out is fp32 [batch, n]). */
int tw_dec_linear(const tw_skinny_args* args, int32_t epilogue, void* out, int32_t ldo, void* stream);
/* fused q|k|v projection (n = 3*D): q -> q_out bf16 [batch, D]; k, v -> paged cache at position pos_b. */
int tw_dec_qkv(const tw_skinny_args* args, void* q_out_bf16, void* kv_pool_layer, const int32_t* block_table,
               int32_t pages_per_row, int32_t n_pages, const void* row_state, void* stream);
int tw_dec_self_attn(const void* q_bf16, void* out_bf16, const void* kv_pool_layer, const int32_t* block_table,
                     int32_t pages_per_row, int32_t n_pages, const void* row_state, int32_t batch, int32_t heads,
                     void* stream);
/* cross-attention of one query per (row, head) over src_len encoder positions; K row j of decode row b, head h at
 * k + enc_row[b]*kv_batch_stride + h*kv_head_stride + j*kv_row_stride (elements; V likewise).  The engine stores
 * K/V head-major ([head][row][pos][64], tw_gemm_bf16 out_mode 1) so every CTA streams one contiguous block.
 * `splits` CTAs per (row, head) with a last-CTA combine (part: fp32 [batch][heads][splits][66], counters:
 * zero-initialised uint32 [batch][heads]).
 * tw_set_cross_attn_stream(1) (or TWB200_CROSS_ATTN=stream in the environment) selects the persistent TMA-fed kernel
 * of csrc/cross_attn.cu for dense head-major K/V (kv_row_stride 64, kv_batch_stride src_len*64, src_len >= 128):
 * `splits` is then the capacity of `part`, the kernel picks the split count that balances the SMs.  Same results to
 * fp32 rounding; faster at >= 72 rows, slower at <= 24 (DESIGN.md K7), so it is off by default. */
int tw_set_cross_attn_stream(int32_t enabled);
/* host only: the key-split plan the streaming kernel would use for `rows` decode rows on a device with `sms` SMs
 * (splits per (row, head), 128-key chunks per split, CTAs launched); no device is touched. */
int tw_cross_attn_plan(int32_t rows, int32_t heads, int32_t src_len, int32_t split_cap, int32_t sms, int32_t* splits,
                       int32_t* chunks_per_split, int32_t* grid);
int tw_dec_cross_attn(const void* q_bf16, void* out_bf16, const void* k_bf16, const void* v_bf16,
                      int64_t kv_row_stride, int64_t kv_batch_stride, int64_t kv_head_stride, const int32_t* enc_row,
                      int32_t src_len, int32_t batch, int32_t heads, int32_t splits, float* part, uint32_t* counters,
                      void* stream);
/* LM head (tied embedding, no bias) + logits processors + per-CTA partial arg-max / log-sum-exp.
 * part_val fp32 [batch][parts][3], part_idx int32 [batch][parts][2], parts = tw_dec_lmhead_parts(vocab).
 * logits_out: optional raw fp32 logits [batch, vocab] (parity tests), else NULL. */
int32_t tw_dec_lmhead_parts(int32_t vocab);
/* row stride of the LayerNorm scratch buffers (ln_part_out [n / 16][rows], ln_stats [rows]) = the most decode rows a
 * tw_dec_linear / tw_dec_qkv launch accepts (128); tw_dec_lmhead accepts up to 48 per launch (the engine launches it per
 * 48-row chunk).  Beyond 32 rows the projections walk the rows in chunks of 24 with ONE pass over their weights. */
int32_t tw_dec_max_rows(void);
int tw_dec_lmhead(const tw_skinny_args* args, const tw_grammar* g, const void* row_state,
                  const uint32_t* suppress_bits, const uint32_t* begin_suppress_bits, float* part_val,
                  int32_t* part_idx, float* logits_out, void* stream);
/* combine partials, pick the token (forced[b, i] >= 0 overrides index i; finished rows emit pad),
 * write tokens[b, pos_b + 1] and advance row_state.  choices: optional int32 [batch, tokens_ld] that
 * receives the engine's own pick before the forced override (teacher-forced parity tests), or NULL. */
int tw_dec_finalize(const float* part_val, const int32_t* part_idx, int32_t n_parts, int32_t* tokens,
                    int32_t tokens_ld, const int32_t* forced, int32_t* choices, void* row_state,
                    const tw_grammar* g, int32_t batch, void* stream);

/* ---- decoder prefill (generate(prompt_ids=...)) ----------------------------------------------------------------
 * Runs positions 0 .. n_pos - 1 of `rows` decode rows through the decoder in one pass, so that the step loop continues
 * at position n_pos as if it had fed those tokens itself.  Prompt row r, position t is activation row r * n_pos + t of
 * every buffer below.  The projections are tw_gemm_bf16 launches over rows * n_pos rows (the engine's
 * WhisperEngine.prefill); these functions are the rest of WhisperDecoderLayer for those rows
 * ($TF/models/whisper/modeling_whisper.py:449-506, :736-759).
 * x[r * n_pos + t, :] = tok_emb[tokens[r, t], :] + pos_emb[t, :]   (fp32 [rows * n_pos, d_model]) */
int tw_prefill_embed(const int32_t* tokens, int32_t tokens_ld, int32_t rows, int32_t n_pos, const void* tok_emb_bf16,
                     const float* pos_emb, float* x, int32_t d_model, void* stream);
/* K and V columns of the fused q|k|v projection (bf16 [rows * n_pos, 3 * d_model]) -> the paged self-attention cache
 * at positions 0 .. n_pos - 1, in the layout tw_dec_qkv writes (pool layer base [2][n_pages][64][d_model]). */
int tw_prefill_kv_store(const void* qkv_bf16, int32_t rows, int32_t n_pos, int32_t d_model, void* kv_pool_layer,
                        const int32_t* block_table, int32_t pages_per_row, int32_t n_pages, void* stream);
/* causal self-attention of the prompt positions (head_dim 64, q pre-scaled) read from the fused q|k|v projection;
 * out: bf16 [rows * n_pos, heads * 64].  n_pos <= 448. */
int tw_prefill_self_attn(const void* qkv_bf16, void* out_bf16, int32_t rows, int32_t n_pos, int32_t heads,
                         void* stream);
/* cross-attention of the prompt queries (q: bf16 row r * n_pos + t at q + (r * n_pos + t) * q_ld) over src_len encoder
 * positions; K / V addressing as tw_dec_cross_attn (row r reads window enc_row[r], NULL = r).
 * out: bf16 [rows * n_pos, heads * 64]. */
int tw_prefill_cross_attn(const void* q_bf16, int64_t q_ld, void* out_bf16, const void* k_bf16, const void* v_bf16,
                          int64_t kv_row_stride, int64_t kv_batch_stride, int64_t kv_head_stride,
                          const int32_t* enc_row, int32_t src_len, int32_t rows, int32_t n_pos, int32_t heads,
                          void* stream);

/* ---- word-level timestamps (return_timestamps="word") --------------------------------------------------------
 * Replaces the `output_attentions` plumbing + WhisperGenerationMixin._extract_token_timestamps
 * ($TF/models/whisper/generation_whisper.py:241-381; _median_filter :43-61, _dynamic_time_warping :64-112).
 * tw_dec_align_tap runs inside the decode step of an alignment layer, right after the cross-attention query
 * projection: for the layer's alignment heads it writes softmax(q_h K_h^T) (fp32, all src_len encoder positions) of
 * every decode row to probs[row][slot0 + i][pos_row][:]  (probs: fp32 [batch][n_slots][max_len][src_len]; pos_row =
 * row_state[row].pos).  K addressing as in tw_dec_cross_attn.  heads_dev: device int32 [n_heads]. */
int tw_dec_align_tap(const void* q_bf16, int32_t q_ld, const void* k_bf16, int64_t kv_row_stride,
                     int64_t kv_batch_stride, int64_t kv_head_stride, const int32_t* enc_row, const void* row_state,
                     const int32_t* heads_dev, int32_t n_heads, int32_t slot0, int32_t n_slots, int32_t max_len,
                     int32_t src_len, int32_t batch, float* probs, void* stream);
/* matrix[row][t][f] = mean over slots of median_filter_f((probs[row][slot][t0 + t][f] - mean_t) / std_t) for
 * t < n_tok, f < n_frames_dev[row] (population std over the n_tok token positions; reflect-padded median of odd
 * width <= 15).  stats: scratch fp32 [batch][n_slots][src_len][2]; matrix: fp32 [batch][max_len][src_len]. */
int tw_align_matrix(const float* probs, const int32_t* n_frames_dev, int32_t batch, int32_t n_slots, int32_t max_len,
                    int32_t src_len, int32_t t0, int32_t n_tok, int32_t filter_width, float* stats, float* matrix,
                    void* stream);
/* host: dynamic time warping over -matrix (fp32 [n_tok][ld], n_frames columns used) with HF's float32 cost table and
 * tie rules; token_frame[t] = first encoder frame of token t's run on the warping path (timestamp = frame * 0.02 s). */
int tw_dtw_token_frames(const float* matrix, int64_t ld, int32_t n_tok, int32_t n_frames, int32_t* token_frame);
/* the same for `batch` independent windows (matrix b at matrices + b*batch_stride, n_frames[b] columns used, 0 allowed:
 * every token then gets frame -1 as in HF) on up to n_threads host threads; token_frames: int32 [batch][n_tok]. */
int tw_dtw_token_frames_batch(const float* matrices, int64_t batch_stride, int64_t ld, int32_t batch, int32_t n_tok,
                              const int32_t* n_frames, int32_t* token_frames, int32_t n_threads);

/* ---- audio ingest: format conversion + channel down-mix + polyphase windowed-sinc resampling ---------------
 * Replaces torchaudio.functional.resample (sinc_interp_hann, lowpass_filter_width 6, rolloff 0.99) in the pipeline's
 * preprocess ($TF/pipelines/automatic_speech_recognition.py:394-407) and the sample conversion / `-ac 1` down-mix
 * of the file reader ($TF/pipelines/audio_utils.py:9-45).  `in`: device, [n_in, channels] interleaved float32 or
 * int16 (scaled by 1/32768); rates already divided by their gcd; filt: device fp32 [new_rate, 2*width + orig_rate]
 * (the torchaudio filter bank), span: device int32 [new_rate, 2] = first non-zero tap and tap count per phase;
 * out: device fp32 [n_out], n_out <= ceil(new_rate * n_in / orig_rate). */
int tw_resample(const void* in, int32_t in_is_int16, int32_t channels, int64_t n_in, float* out, int64_t n_out,
                const float* filt, const int32_t* span, int32_t orig_rate, int32_t new_rate, int32_t width,
                void* stream);

/* ---- host: native FLAC reader (the reference's example input is FLAC; HF spawns ffmpeg per file) --------------
 * Replaces the container decode of ffmpeg_read ($TF/pipelines/audio_utils.py:9-45) for FLAC streams (RFC 9639:
 * CONSTANT / VERBATIM / FIXED / LPC subframes, Rice residuals, stereo decorrelation; frame CRC-8 / CRC-16 verified).
 * The decoded interleaved PCM goes to tw_resample for conversion, down-mix and resampling on the GPU. */
typedef struct tw_flac_info {
    int32_t sample_rate, channels, bits_per_sample, max_block;
    int64_t total_samples;      /* per channel; 0 = unknown (count with tw_flac_decode(out = NULL)) */
    uint8_t md5[16];            /* of the decoded little-endian interleaved samples; all zero = not recorded */
} tw_flac_info;
int tw_flac_info_read(const uint8_t* data, int64_t n, tw_flac_info* out);
/* out: int32 [out_cap_samples][channels] interleaved, or NULL to count only; n_decoded = samples per channel. */
int tw_flac_decode(const uint8_t* data, int64_t n, int32_t* out, int64_t out_cap_samples, int64_t* n_decoded);

/* ---- host: per-window token streams -> timestamped chunks ------------------------------------------------
 * Replaces tokenizer._decode_asr / _find_longest_common_sequence for return_timestamps in {False, True}
 * ($TF/models/whisper/tokenization_whisper.py:901-1150, 1153-1270; called from the pipeline's postprocess,
 * $TF/pipelines/automatic_speech_recognition.py:562-656).  Token ids in, token ids + times out; no device work. */
typedef struct tw_asr_window {
    const int32_t* tokens;      /* generated ids of one window (prompt, specials, timestamps and text) */
    int32_t n_tokens;
    int32_t has_stride;         /* 0: the window carries no stride triple */
    double chunk_len, stride_left, stride_right;   /* seconds, as the pipeline's postprocess passes them */
} tw_asr_window;

typedef struct tw_asr_config {
    int32_t timestamp_begin;          /* id of <|0.00|> */
    int32_t prompt_token_id;          /* <|startofprev|> */
    int32_t decoder_start_token_id;   /* <|startoftranscript|> */
    int32_t return_timestamps;        /* 0 / 1 (word timestamps are not handled here) */
    int32_t segment_size;             /* encoder positions per window (1500) */
    int32_t n_special;
    const int32_t* special_ids;       /* sorted ascending: tokenizer.all_special_ids */
    const int32_t* special_lang;      /* per special id: language index >= 0, or -1 for any other special token */
    double time_precision;            /* seconds per timestamp step (0.02) */
} tw_asr_config;

/* Chunk c owns out_tokens[chunk_offsets[c] .. chunk_offsets[c+1]); chunk_t0 / chunk_t1 are NaN where Python has
 * None; chunk_lang is a language index or -1.  flags bit 0: the last chunk has no closing timestamp.
 * Capacities: out_tokens_cap >= total input tokens, max_chunks (+1 offsets) >= total input tokens + 1. */
int tw_decode_asr(const tw_asr_window* windows, int32_t n_windows, const tw_asr_config* cfg, int32_t* out_tokens,
                  int64_t out_tokens_cap, int64_t* chunk_offsets, double* chunk_t0, double* chunk_t1,
                  int32_t* chunk_lang, int32_t max_chunks, int32_t* n_chunks_out, int32_t* flags_out);

/* ---- beam search on the device (generate_kwargs={"num_beams": k}) -----------------------------------------
 * Replaces GenerationMixin._beam_search ($TF/generation/utils.py:3076-3400, helpers :2876-3075) and the Whisper
 * logits processors applied to log-probabilities ($TF/generation/logits_process.py:1812-2043) for
 * n_windows x num_beams decode rows (row = window * num_beams + beam), early_stopping = False, do_sample = False.
 * One call = one search step appended to a decode step whose LM head tapped the raw logits: per-row log-softmax +
 * processors + best 2K continuations, per-window running / finished bookkeeping, the next token / position of every
 * decode row, and the paged self-attention cache re-gathered by beam of origin as a block-table permutation (full
 * pages by pointer, the partial current page copied into the row's own slot of the other page bank).  All state is
 * device resident, so the step is CUDA-graph capturable; the host only polls ctrl[1] (search over). */
typedef struct tw_beam_config {
    int32_t num_beams;        /* K <= 8 */
    int32_t vocab;
    int32_t max_length;       /* generation_config.max_length (<= tokens_ld) */
    int32_t prompt_len;       /* decoder prompt tokens per row */
    int32_t eos, pad, no_timestamps;
    int32_t max_initial_ts;   /* max_initial_timestamp_index, -1: none */
    int32_t timestamps;       /* 0: generate(return_timestamps=False): suppress lists only */
    int32_t track_indices;    /* 1: keep HF's beam_indices next to the tokens (word timestamps) */
    float length_penalty;
} tw_beam_config;
/* W = tw_beam_record_width(cfg): a hypothesis record is [max_length tokens | max_length beam indices (if tracked)].
 * Initial state (set by the caller): hist[0][w][k][:prompt_len] = prompt, pad elsewhere; run_score[w][0] = 0, others
 * -1e9; fin_score = -1e9; fin_flag = fin_len = 0; gram = {0, 1, -1, 0}; improvable = 1; ctrl = 0. */
typedef struct tw_beam_state {
    int32_t* hist;        /* [2][n][K][W] running hypotheses, double-buffered by ctrl[0] */
    int32_t* fin;         /* [2][n][K][W] finished hypotheses (slot 0 = best) */
    float* run_score;     /* [n][K] */
    float* fin_score;     /* [n][K] score / generated_length ** length_penalty */
    int32_t* fin_flag;    /* [n][K] */
    int32_t* fin_len;     /* [n][K] generated length */
    int32_t* gram;        /* [n][K][4] timestamp-grammar state of the running rows */
    int32_t* improvable;  /* [n] */
    int32_t* hits_all;    /* [n] */
    int32_t* ctrl;        /* [8]: [0] record parity, [1] search over, [2] scratch, [3] KV page bank, [4] steps taken */
} tw_beam_state;
int32_t tw_beam_record_width(const tw_beam_config* cfg);
/* logits: fp32 [R][vocab] of this step (tw_dec_lmhead's tap); row_state as in the decode kernels (pos = position just
 * fed; the step sets pos + 1); tokens[r][pos + 1] receives the token row r feeds next.  block_table [R][pages_per_row]
 * must start as bank-0 identity (row r, page q -> r * pages_per_row + q); the pool holds n_pages >= 2 * bank_pages
 * pages per (layer, k|v).  cand_val / cand_tok: scratch [R][2K]; copy_src / copy_dst: scratch int32 [R]; copy_len:
 * scratch int32 [1]; origin_out: int32 [R], the previous row every new row continues. */
int tw_beam_step(const tw_beam_config* cfg, const tw_beam_state* state, const float* logits, void* row_state,
                 const uint32_t* suppress_bits, const uint32_t* begin_suppress_bits, float* cand_val,
                 int32_t* cand_tok, int32_t* tokens, int32_t tokens_ld, int32_t* block_table, int32_t pages_per_row,
                 int32_t bank_pages, void* kv_pool, int32_t n_pages, int32_t layers, int32_t d_model,
                 int32_t* copy_src, int32_t* copy_dst, int32_t* copy_len, int32_t* origin_out, int32_t n_windows,
                 void* stream);
/* host: the same step on HOST buffers (same scalar code; no device involved) for the CPU test suite.  cur = index the new
 * token is written to; next_tokens / origin_out: int32 [R]. */
int tw_beam_step_host(const tw_beam_config* cfg, const tw_beam_state* state, const float* logits, int32_t cur,
                      const uint32_t* suppress_bits, const uint32_t* begin_suppress_bits, int32_t* next_tokens,
                      int32_t* origin_out, int32_t n_windows);

#ifdef __cplusplus
}
#endif
#endif /* TWB200_H_ */
