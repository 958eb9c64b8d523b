// Decoder-side kernel interface (decoder.cu / search.cu).  Token loop of ctranslate2.models.Whisper.generate
// (/root/reference/main.py:687-692; SURVEY.md section 8a rows A10-A14).
#pragma once
#include "common.cuh"
#include "kernels.h"

namespace wisb {

constexpr int DEC_MAX_ROWS = 8;    // rows (utterances x beams) one decoder pass handles
constexpr int MAX_BEAM = 8;
constexpr int MAX_CAND = 2 * MAX_BEAM;
constexpr int TOPK_CHUNKS = 32;

// Everything the captured decode graphs read at run time lives in device memory so one graph serves every step.
struct DecState {
  int pos;        // position of the token being fed this step
  int gen_step;   // 0-based index of the token being generated (valid once pos >= prompt_len - 1)
  int n_done;     // utterances finished
  int all_done;   // n_done == n_utt
  int ticket;     // CTAs of search_tail_kernel that finished this step's bookkeeping (the last one advances the step)
};

enum GemvEpi : int {
  GV_STORE = 0,   // out[r, n] = v
  GV_RESID = 1,   // out[r, n] += v
  GV_GELU = 2,    // out[r, n] = gelu(v)
  GV_QKV = 3,     // n < d: q[r, n] = v ; d <= n < 2d: kcache[slot r][pos][n - d] ; else vcache
};

struct GemvArgs {
  const float* x = nullptr;   // [R, K] fp32
  const float* ln_g = nullptr;  // LayerNorm prologue when non-null
  const float* ln_b = nullptr;
  const __half* w = nullptr;  // [N, K] fp16
  const float* bias = nullptr;
  float* out = nullptr;       // fp32 [R, ldo]
  long long ldo = 0;
  int R = 0, N = 0, K = 0;
  int epi = GV_STORE;
  // GV_QKV
  __half* kcache = nullptr;   // [R_slots][t_max][d]
  __half* vcache = nullptr;
  int d_model = 0, t_max = 0;
  const DecState* st = nullptr;
};
void gemv_run(const GemvArgs& a, cudaStream_t stream);

// x[r, :] = tok_emb[token[r], :] + pos_emb[pos, :]
void dec_embed_run(const int* tokens, const __half* tok_emb, const float* pos_emb, float* x, int R, int d,
                   const DecState* st, cudaStream_t stream);

// causal self-attention over the cache, with beam indirection: position t of row r lives in slot indir[r][t]
// (two ping-pong indirection tables; *flip says which one is current)
void dec_self_attn_run(const float* q /*[R,d]*/, const __half* kcache, const __half* vcache, const int* indir0,
                       const int* indir1, const int* flip, float* ctx /*[R,d]*/, int R, int d, int H, int t_max,
                       const DecState* st, cudaStream_t stream);

// cross-attention: rows of utterance u share K/V [H][1536][64]; grid = (H, n_utt) x cluster of 8 CTAs over the keys
void dec_cross_attn_run(const float* q /*[R,d]*/, const __half* k /*[n_utt_total][H][1536][64]*/, const __half* v,
                        float* ctx, int n_utt, int beam, int d, int H, cudaStream_t stream);

struct SearchArgs {
  // inputs
  const float* logits = nullptr;  // [R, ldl]
  long long ldl = 0;
  int n_vocab = 0;
  const unsigned char* mask = nullptr;  // [V] bit0: suppressed always, bit1: suppressed at the first generated step
  int n_utt = 0, beam = 0, n_cand = 0;
  int max_new = 0, max_hyp = 0, eot = 0, t_max = 0, prompt_len = 0;
  float length_penalty = 1.f;
  // workspaces / state (device)
  float* row_lse = nullptr;       // [R]
  float* part_max = nullptr;      // [R][TOPK_CHUNKS] chunk max of the processed logits
  float* part_sum = nullptr;      // [R][TOPK_CHUNKS] chunk sum exp(logit - chunk max)
  float* cum = nullptr;           // [R] cumulative log-prob of the alive beams
  unsigned long long* part = nullptr;  // [R][TOPK_CHUNKS][MAX_CAND] packed (score, ~index)
  float* cand_score = nullptr;    // [n_utt][MAX_CAND]
  int* cand_idx = nullptr;        // [n_utt][MAX_CAND]   beam * V + token
  int* tokens = nullptr;          // [R] token fed next step
  int* seq[2] = {nullptr, nullptr};    // [R][max_new] generated tokens of the alive beams (ping-pong)
  int* indir[2] = {nullptr, nullptr};  // [R][t_max] cache indirection (ping-pong)
  int* flip = nullptr;            // which of the ping-pong buffers is current (device int)
  int* done = nullptr;            // [n_utt]
  int* n_hyp = nullptr;           // [n_utt]
  float* best_score = nullptr;    // [n_utt]
  int* best_len = nullptr;        // [n_utt]
  int* best_tokens = nullptr;     // [n_utt][max_new]
  DecState* st = nullptr;
  int* row_pos = nullptr;         // [R] position fed by every row this step (batched pass); advanced with st->pos
  int* row_slot = nullptr;        // [R] cache slot every row writes this step's K/V to (= its own row)
  const int* max_new_u = nullptr; // optional [n_utt]: per-utterance cap on generated tokens (<= max_new)
  // timestamp rules (search.cu): first timestamp token (<|notimestamps|> + 1), -1 = off; largest index of the first
  // timestamp above ts_begin
  int ts_begin = -1, max_init_ts = 0;
};
void search_step_run(const SearchArgs& a, cudaStream_t stream);
// prompt prefill: no search, just feed the next prompt token and advance the position
void prefill_advance_run(int* tokens, const int* prompt /*[n_utt][prompt_len]*/, int prompt_len, int R, int beam,
                         DecState* st, cudaStream_t stream);
void search_init_run(const SearchArgs& a, const int* prompt, cudaStream_t stream, int shared_prefix = 0);
// rows of a batched prefill pass: row i = prompt position p0 + i % chunk of utterance i / chunk, cache slot = the
// utterance's first beam
void prefill_rows_run(int* tokens, int* row_pos, int* row_slot, const int* prompt, int prompt_len, int n_utt, int p0,
                      int chunk, int beam, cudaStream_t stream);

// ------------------------------------------------------------------ batched decoder pass (decoder_batch.cu)
struct BatchLayer {
  GemmPlan qkv, o, cq, co, fc1, fc2;  // built for the row capacity of the workspaces; o / co / fc2 write split-K partials
  const float *ln1g = nullptr, *ln1b = nullptr;      // LayerNorm before the QKV GEMM (only layer 0's is applied by the embedding kernel)
  const float *ob = nullptr, *ln2g = nullptr, *ln2b = nullptr;    // out-proj bias, LayerNorm before cross-attention
  const float *cob = nullptr, *ln3g = nullptr, *ln3b = nullptr;   // cross out-proj bias, LayerNorm before the MLP
  const float *fc2b = nullptr, *next_g = nullptr, *next_b = nullptr;  // fc2 bias, the NEXT LayerNorm (layer l+1's ln1 or the final one)
  const __half* ck = nullptr;   // cross K / V of this layer for utterance 0 of the pass: [n_utt][H][1536][64]
  const __half* cv = nullptr;
  __half* kcache = nullptr;     // self-attention cache of this layer: [slots][t_cap][d]
  __half* vcache = nullptr;
};
struct BatchArgs {
  int R = 0, d = 0, H = 0, n_utt = 0, rows_per_utt = 0, t_cap = 0, t_ind = 0, prefill = 0, with_logits = 0, pdl = 0;
  const int* tokens = nullptr;    // [R]
  const int* row_pos = nullptr;   // [R]
  const int* row_slot = nullptr;  // [R]
  const __half* tok_emb = nullptr;
  const float* pos_emb = nullptr;
  float* x = nullptr;             // [rows_cap, d] fp32 residual stream
  __half* xn = nullptr;           // [rows_cap, d] LayerNorm output (GEMM A operand)
  float* q = nullptr;             // [rows_cap, d]
  __half* ctx = nullptr;          // [rows_cap, d] attention output (GEMM A operand)
  float* part = nullptr;          // split-K partial slabs [splits][rows_cap][d]
  long long part_stride = 0;
  const int* indir0 = nullptr;
  const int* indir1 = nullptr;
  const int* flip = nullptr;
  const int* done = nullptr;      // [n_utt] or null (prefill)
  const GemmPlan* vocab = nullptr;
  // tcgen05 cross-attention: one tensor map over the whole cross-K/V buffer viewed as [rows][64] fp16
  int cross_tc = 1, num_sms = 148;
  const CUtensorMap* ckv_map = nullptr;
  const __half* ckv_base = nullptr;
  // optional per-kernel-family timing hook (engine option "profile", eager launches only):
  // cat 0 GEMM, 1 cross-attention, 2 LayerNorm / embedding, 3 self-attention; begin = 1 / 0
  void (*prof)(void* ctx, int cat, int begin) = nullptr;
  void* prof_ctx = nullptr;
};
// returns the number of kernels launched
int batch_pass_run(const BatchArgs& a, const BatchLayer* layers, int n_layers, cudaStream_t stream);

// ------------------------------------------------------------------ persistent decoder pass (decoder_mega.cu)
struct MegaGemv {
  const __half* w = nullptr;     // [N, K] fp16; K > 1536: chunk-major [chunk][N][K/chunks] (mega_chunk_major); warp-MMA pass: mega_mma_image
  const float* bias = nullptr;
  const float* ln_g = nullptr;   // LayerNorm gamma (x is multiplied by it while staged), K <= 1536
  const float* ln_s2 = nullptr;  // non-null = LayerNorm folded: s2[n] = sum_k g_k W[n,k]; `bias` then holds bias + sum_k b_k W[n,k]
  const float* x = nullptr;      // [R, K] fp32 activations
  float* out = nullptr;
  long long ldo = 0;
  int N = 0, K = 0, epi = GV_STORE;
  int shape = 0;                 // warp-MMA pass: 0 qkv, 1 d x d (o / cross-q / cross-o), 2 fc1, 3 fc2, 4 vocabulary (geometry table)
  // fp16 activation exchange images [K/64][R][64] (decoder_mega.cu act16_off): input read with one bulk copy / GELU output
  const __half* x16 = nullptr;
  __half* out16 = nullptr;
  const float* next_g = nullptr;  // GV_RESID: gain of the LayerNorm that reads the new residual rows next
};
struct MegaLayer {
  MegaGemv qkv, o, cq, co, fc1, fc2;
  const __half* ck = nullptr;    // cross K of this layer for the utterances of the pass: [n_utt][H][1536][64]
  const __half* cv = nullptr;
  __half* kcache = nullptr;      // self-attention cache of this layer: [slots][t_max][d]
  __half* vcache = nullptr;
};
struct MegaArgs {
  const MegaLayer* layers = nullptr;  // device array [n_layers]
  int n_layers = 0;
  MegaGemv vocab;
  int with_logits = 0;
  int R = 0, d = 0, H = 0, n_utt = 0, beam = 0, t_max = 0;
  // prompt prefill in one pass: rows = n_utt x pf_len prompt positions (beam := pf_len for the cross-attention phase),
  // tokens -> prompt [n_utt][pf_tok_stride], K/V written to cache slot u * pf_slot_stride; 0 = normal decoding step
  int pf_len = 0, pf_tok_stride = 0, pf_slot_stride = 0;
  const int* tokens = nullptr;
  const __half* tok_emb = nullptr;
  const float* pos_emb = nullptr;
  float* x = nullptr;      // [R, d] residual stream
  float* q = nullptr;      // [R, d]
  float* ctx = nullptr;    // [R, d]
  __half* ctx16 = nullptr; // warp-MMA pass: attention output as an fp16 exchange image instead of `ctx`
  __half* q16 = nullptr;   // warp-MMA pass: cross-attention queries [head][R][64] fp16, pre-scaled by 1/8
  __half* xn16 = nullptr;  // warp-MMA pass: residual rows times the next LayerNorm's gain, fp16 exchange image
  float* xstat = nullptr;  // warp-MMA pass: [CTA][R][2] per-CTA shares of the rows' (sum, sum of squares)
  const int* indir0 = nullptr;
  const int* indir1 = nullptr;
  const int* flip = nullptr;
  const DecState* st = nullptr;
  float* cross_part = nullptr;   // [n_utt][H][S<=16][MAX_BEAM][68] (64 acc, m, l, pad)
  unsigned* cross_flags = nullptr;  // [n_utt * H][16] epoch-tagged 'partial written' flags, one 128-byte line each
  unsigned* flags = nullptr;     // grid-barrier epoch flags, one 128-byte line per CTA
  unsigned* epoch_base = nullptr;
  int barrier_mode = 0;          // 0: per-CTA epoch flags, 1: shared counter (red.release + spin)
  int tc = 0;                    // 1: GEMV phases on the warp-level tensor path (dec_pass_mma_kernel)
  int dbg = 0;                   // diagnostics (timing experiments, results are garbage): bit 1 = stream a quarter of every weight unit
  int trace_cta = 0, trace_layer = 0, trace_cap = 0;  // event trace: which CTA, which layer opens the window, events kept
  unsigned long long* trace = nullptr;  // optional: [2*k] = time phase k starts, [2*k+1] = time CTA 0 reached barrier k
};
size_t mega_flags_words();
int mega_k_chunks(int K);
void mega_chunk_major(const __half* src, __half* dst, int N, int K, cudaStream_t stream);
// W [N, K] -> the image the warp-MMA pass streams with one bulk copy per ring unit (N x K halves)
void mega_mma_image(const __half* src, __half* dst, int N, int K, int grid, cudaStream_t stream);
// s2[n] = sum_k g[k] W[n,k];  biasf[n] = bias[n] + sum_k b[k] W[n,k]   (bias may be null)
void mega_ln_fold(const __half* w, const float* g, const float* b, const float* bias, float* s2, float* biasf, int N, int K,
                  cudaStream_t stream);
void dec_pass_run(const MegaArgs& a, int num_sms, cudaStream_t stream);

// tcgen05 skinny GEMV (gemv_tc.cu), diagnostics entry: returns the average kernel time in microseconds
float gemv_tc_debug_run(const float* x, const __half* w, const float* bias, float* out, int R, int N, int K, int num_sms,
                        int iters, cudaStream_t stream);

// language detection head: softmax over lang ids of the logits of row u*beam (one step on <|startoftranscript|>)
void lang_probs_run(const float* logits, long long ldl, const int* lang_ids, int n_lang, int n_utt, int row_stride,
                    float* probs /*[n_utt][n_lang]*/, cudaStream_t stream);

}  // namespace wisb
