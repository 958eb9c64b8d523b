// Device-side token search: logits processors, log-softmax, top-k over beam x vocabulary and the CTranslate2-style
// beam / greedy bookkeeping, all without a host round trip (the host only polls DecState::all_done).
//
// Semantics restated from CTranslate2 4.1.0 as listed in SURVEY.md section 8a rows A11-A13 (the reference call is
// /root/reference/main.py:687-692 with the library defaults patience=1, length_penalty=1, suppress_blank=True,
// suppress_tokens=[-1], num_hypotheses=1):
//   * processors: `suppress_ids` -> -inf every step; {blank, eot} -> -inf at the first generated step
//   * timestamp rules when the prompt has no <|notimestamps|> (SearchArgs::ts_begin >= 0): see ts_rules below
//   * scores: log_softmax(logits) + cumulative beam score, divided by (step+1)^length_penalty
//   * candidates: top 2*beam of beam*V (ties: lowest flat index); at step 0 only beam 0 is live
//   * the first `beam` candidates that end in eot (or any at the last step) become hypotheses and are replaced by the
//     next non-eot candidates; an utterance is finished once round(beam*patience) hypotheses exist or at the last step
//   * result: best normalised score, first one on ties; eot itself is not part of the output
//   * beam_size == 1 is the same procedure with 2 candidates, i.e. greedy arg-max decoding
#include "decoder.cuh"

namespace wisb {

namespace {

__device__ __forceinline__ unsigned f2ord(float f) {
  unsigned u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(unsigned u) {
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}
// larger key == better candidate: higher score first, then lower index
__device__ __forceinline__ unsigned long long pack_key(float score, unsigned idx) {
  return (static_cast<unsigned long long>(f2ord(score)) << 32) | static_cast<unsigned long long>(~idx);
}

__device__ __forceinline__ float masked_logit(const SearchArgs& a, const float* row, int v, bool first_step) {
  const unsigned char m = a.mask[v];
  if ((m & 1) || (first_step && (m & 2))) return -INFINITY;
  return row[v];
}

// block-wide selection of the `n_cand` largest keys among each thread's private keys[0..cnt)
template <int PER>
__device__ void block_select(unsigned long long (&keys)[PER], int n_cand, unsigned long long* out,
                             unsigned long long* s_red /*[32]*/) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nwarps = blockDim.x >> 5;
  for (int c = 0; c < n_cand; ++c) {
    unsigned long long best = 0ull;
    int bi = -1;
#pragma unroll
    for (int i = 0; i < PER; ++i)
      if (keys[i] > best) {
        best = keys[i];
        bi = i;
      }
    unsigned long long wbest = best;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const unsigned long long other = __shfl_xor_sync(0xffffffffu, wbest, o);
      wbest = other > wbest ? other : wbest;
    }
    if (lane == 0) s_red[warp] = wbest;
    __syncthreads();
    unsigned long long bbest = s_red[0];
    for (int w = 1; w < nwarps; ++w) bbest = s_red[w] > bbest ? s_red[w] : bbest;
    __syncthreads();
    if (bi >= 0 && best == bbest && best != 0ull) {  // keys are unique (index is part of the key)
#pragma unroll
      for (int i = 0; i < PER; ++i)
        if (i == bi) keys[i] = 0ull;
    }
    if (tid == 0) out[c] = bbest;
  }
}

// grid (TOPK_CHUNKS, R): partial top-n_cand of one chunk of one row
constexpr int TK_THREADS = 256;
constexpr int TK_PER = 8;  // 256 * 8 = 2048 >= ceil(51865 / 32) = 1621 (timestamp mode: ceil(50364 / 31) = 1625, 1501)

// Timestamp mode (a.ts_begin >= 0): the rules of HF WhisperTimeStampLogitsProcessor (a port of openai-whisper's
// ApplyTimestampRules) for row r at generation step `gen`, derived from the row's own generated tokens
// seq[*flip][r][0, gen) -- already per beam and reordered by the bookkeeping, so no extra per-row state is carried.
// The chunk layout changes too: the text tokens [0, ts_begin) are spread over chunks 0 .. TOPK_CHUNKS-2 and the
// timestamps [ts_begin, n_vocab) form the last chunk alone, so that the merge finds the timestamps' (max, sum exp) and
// the text maximum among the partials as they are (rule 5).  Outputs: the chunk [v0, v1) and the tokens of it the rules
// let through, [lo, hi) minus `hole`.  Called by every thread of the block.
__device__ void ts_rules(const SearchArgs& a, int r, int gen, int chunk, int& v0, int& v1, int& lo, int& hi, int& hole,
                         int* s_i /*[TK_THREADS / 32]*/) {
  const int tb = a.ts_begin;
  const int* hist = a.seq[*a.flip] + static_cast<long long>(r) * a.max_new;
  int li = -1;  // position of the last timestamp in the history
  for (int t = threadIdx.x; t < gen; t += blockDim.x)
    if (hist[t] >= tb) li = t;
  li = __reduce_max_sync(0xffffffffu, li);
  if ((threadIdx.x & 31) == 0) s_i[threadIdx.x >> 5] = li;
  __syncthreads();
  for (int w = 0; w < TK_THREADS / 32; ++w) li = max(li, s_i[w]);
  const bool last_ts = gen >= 1 && hist[gen - 1] >= tb;
  const bool pen_ts = gen < 2 || hist[gen - 2] >= tb;
  int text_lo = 0, ts_lo = tb, ts_hi = a.n_vocab;
  if (last_ts) {
    if (pen_ts) ts_hi = tb;  // a pair was just completed (or the history is one timestamp): text next
    else text_lo = a.eot;    // a segment was just closed: another timestamp or <|endoftext|> next
  }
  // timestamps never decrease; right after a segment closes the next one may open at the same time
  if (li >= 0) ts_lo = max(ts_lo, hist[li] + ((last_ts && !pen_ts) ? 0 : 1));
  if (gen == 0) {  // the first generated token is a timestamp no later than ts_begin + max_init_ts
    text_lo = tb;
    ts_hi = min(a.n_vocab, tb + a.max_init_ts + 1);
  }
  if (chunk == TOPK_CHUNKS - 1) {
    v0 = tb;
    v1 = a.n_vocab;
    lo = ts_lo;
    hi = ts_hi;
  } else {
    const int per = (tb + TOPK_CHUNKS - 2) / (TOPK_CHUNKS - 1);
    v0 = chunk * per;
    v1 = min(tb, v0 + per);
    lo = text_lo;
    hi = v1;
    hole = tb - 1;  // <|notimestamps|> is never generated
  }
}

__global__ void __launch_bounds__(TK_THREADS) topk_partial_kernel(const SearchArgs a) {
  // Within one row the ranking by processed logit equals the ranking by score, so the per-chunk stage needs no
  // log-sum-exp: it emits the chunk's top-n_cand logits plus (max, sum exp) partials; the merge stage turns them into
  // the row's lse and into scores.  (This replaced a separate two-pass lse kernel: 55 us -> 0.)
  __shared__ unsigned long long s_red[32];
  __shared__ float s_f[32];
  __shared__ int s_i[TK_THREADS / 32];
  if (a.st->all_done) return;  // a step enqueued ahead of the host's poll
  const int chunk = blockIdx.x, r = blockIdx.y;
  const int gen = a.st->gen_step;
  const bool first = gen == 0;
  const float* row = a.logits + static_cast<long long>(r) * a.ldl;
  int v0, v1, lo, hi, hole = -1;
  if (a.ts_begin < 0) {
    const int per_chunk = (a.n_vocab + TOPK_CHUNKS - 1) / TOPK_CHUNKS;
    v0 = chunk * per_chunk;
    v1 = min(a.n_vocab, v0 + per_chunk);
    lo = v0;
    hi = v1;
  } else {
    ts_rules(a, r, gen, chunk, v0, v1, lo, hi, hole, s_i);
  }
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  unsigned long long keys[TK_PER];
  float lg[TK_PER];
  float mx = -INFINITY;
#pragma unroll
  for (int i = 0; i < TK_PER; ++i) {
    const int v = v0 + tid + i * TK_THREADS;
    keys[i] = 0ull;
    lg[i] = -INFINITY;
    if (v < v1) {
      lg[i] = (v < lo || v >= hi || v == hole) ? -INFINITY : masked_logit(a, row, v, first);
      if (lg[i] != -INFINITY) keys[i] = pack_key(lg[i], static_cast<unsigned>(v));
      mx = fmaxf(mx, lg[i]);
    }
  }
  mx = warp_max(mx);
  if (lane == 0) s_f[warp] = mx;
  __syncthreads();
  mx = s_f[0];
  for (int w = 1; w < TK_THREADS / 32; ++w) mx = fmaxf(mx, s_f[w]);
  __syncthreads();
  float se = 0.f;
#pragma unroll
  for (int i = 0; i < TK_PER; ++i)
    if (lg[i] != -INFINITY) se += __expf(lg[i] - mx);
  se = warp_sum(se);
  if (lane == 0) s_f[warp] = se;
  __syncthreads();
  if (tid == 0) {
    float t = 0.f;
    for (int w = 0; w < TK_THREADS / 32; ++w) t += s_f[w];
    a.part_max[r * TOPK_CHUNKS + chunk] = mx;
    a.part_sum[r * TOPK_CHUNKS + chunk] = t;
  }
  block_select<TK_PER>(keys, a.n_cand, a.part + (static_cast<long long>(r) * TOPK_CHUNKS + chunk) * MAX_CAND, s_red);
}

// grid (n_utt): merge beam * TOPK_CHUNKS * n_cand partial keys -> sorted candidate list
constexpr int TM_PER = (MAX_BEAM * TOPK_CHUNKS * MAX_CAND + TK_THREADS - 1) / TK_THREADS;  // 16

__device__ __forceinline__ void topk_merge_body(const SearchArgs& a, unsigned long long* s_red, unsigned long long* s_out, float* s_lse,
                                                int* s_ts_only) {
  const int u = blockIdx.x;
  const int gen = a.st->gen_step;
  const bool first = gen == 0;
  const float norm = (a.length_penalty != 0.f) ? powf(static_cast<float>(gen + 1), a.length_penalty) : 1.f;
  if (threadIdx.x < a.beam) {  // row log-sum-exp from the chunk partials
    const int r = u * a.beam + threadIdx.x;
    float mx = -INFINITY;
    for (int c = 0; c < TOPK_CHUNKS; ++c) mx = fmaxf(mx, a.part_max[r * TOPK_CHUNKS + c]);
    float t = 0.f;
    for (int c = 0; c < TOPK_CHUNKS; ++c) {
      const float pm = a.part_max[r * TOPK_CHUNKS + c];
      if (pm != -INFINITY) t += a.part_sum[r * TOPK_CHUNKS + c] * __expf(pm - mx);
    }
    float lse = mx + logf(t);
    int ts_only = 0;
    if (a.ts_begin >= 0) {
      // timestamp rule 5: when the timestamps' total probability beats every single text token, text is banned and the
      // row is renormalised over the timestamps (the last chunk holds exactly them; the log-softmax shift cancels)
      const int cts = TOPK_CHUNKS - 1;
      float mtext = -INFINITY;
      for (int c = 0; c < cts; ++c) mtext = fmaxf(mtext, a.part_max[r * TOPK_CHUNKS + c]);
      const float pm = a.part_max[r * TOPK_CHUNKS + cts];
      const float lse_ts = pm == -INFINITY ? -INFINITY : pm + logf(a.part_sum[r * TOPK_CHUNKS + cts]);
      if (lse_ts > mtext) {
        lse = lse_ts;
        ts_only = 1;
      }
    }
    s_lse[threadIdx.x] = lse;
    s_ts_only[threadIdx.x] = ts_only;
    a.row_lse[r] = lse;
  }
  __syncthreads();
  const int total = a.beam * TOPK_CHUNKS * a.n_cand;
  unsigned long long keys[TM_PER];
#pragma unroll
  for (int i = 0; i < TM_PER; ++i) {
    const int j = threadIdx.x + i * TK_THREADS;
    keys[i] = 0ull;
    if (j < total) {
      const int c = j % a.n_cand;
      const int rc = j / a.n_cand;       // (beam row, chunk)
      const int k = rc / TOPK_CHUNKS;    // beam index
      const unsigned long long pk = a.part[(static_cast<long long>(u * a.beam) * TOPK_CHUNKS + rc) * MAX_CAND + c];
      // at the first step every beam holds the same prefix: only beam 0 counts
      if (pk != 0ull && !(first && k > 0) && !(s_ts_only[k] && rc % TOPK_CHUNKS != TOPK_CHUNKS - 1)) {
        const float lg = ord2f(static_cast<unsigned>(pk >> 32));
        const unsigned v = ~static_cast<unsigned>(pk & 0xffffffffull);
        const float sc = ((lg - s_lse[k]) + a.cum[u * a.beam + k]) / norm;
        keys[i] = pack_key(sc, static_cast<unsigned>(k * a.n_vocab) + v);
      }
    }
  }
  block_select<TM_PER>(keys, a.n_cand, s_out, s_red);
  __syncthreads();
  if (threadIdx.x < a.n_cand) {
    const unsigned long long key = s_out[threadIdx.x];
    const bool valid = key != 0ull;
    a.cand_score[u * MAX_CAND + threadIdx.x] = valid ? ord2f(static_cast<unsigned>(key >> 32)) : -INFINITY;
    a.cand_idx[u * MAX_CAND + threadIdx.x] = valid ? static_cast<int>(~static_cast<unsigned>(key & 0xffffffffull)) : -1;
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// one warp: the CTranslate2 bookkeeping for one utterance
__device__ __forceinline__ void search_bookkeeping_body(const SearchArgs& a, int* s_pick, int& s_best_k, int& s_finished) {
  const int u = blockIdx.x, lane = threadIdx.x;
  const int beam = a.beam, V = a.n_vocab, nc = a.n_cand;
  const int gen = a.st->gen_step, pos = a.st->pos;
  const int cur = *a.flip, nxt_buf = cur ^ 1;
  const int* seq_cur = a.seq[cur];
  int* seq_nxt = a.seq[nxt_buf];
  const int* ind_cur = a.indir[cur];
  int* ind_nxt = a.indir[nxt_buf];

  if (a.done[u]) {
    // frozen utterance: carry the state over unchanged so the ping-pong buffers stay coherent
    for (int k = 0; k < beam; ++k) {
      const int r = u * beam + k;
      for (int t = lane; t < a.max_new; t += 32) seq_nxt[r * a.max_new + t] = seq_cur[r * a.max_new + t];
      for (int t = lane; t < a.t_max; t += 32) ind_nxt[r * a.t_max + t] = (t == pos) ? r : ind_cur[r * a.t_max + t];
    }
    return;
  }
  const float* cs = a.cand_score + u * MAX_CAND;
  const int* ci = a.cand_idx + u * MAX_CAND;
  const bool is_last = (gen + 1 >= (a.max_new_u != nullptr ? a.max_new_u[u] : a.max_new));
  const float norm = (a.length_penalty != 0.f) ? powf(static_cast<float>(gen + 1), a.length_penalty) : 1.f;
  if (lane == 0) {
    int n_hyp = a.n_hyp[u];
    float best = a.best_score[u];
    int best_k = -1;
    int secondary = beam;
    for (int k = 0; k < beam; ++k) {
      int pick = k;
      const int idx = ci[k];
      const int tok = idx < 0 ? a.eot : idx % V;
      if (idx >= 0 && (tok == a.eot || is_last)) {
        ++n_hyp;
        if (cs[k] > best) {  // strict: the first best hypothesis wins ties
          best = cs[k];
          best_k = k;
        }
        for (int j = secondary; j < nc; ++j) {
          if (ci[j] >= 0 && ci[j] % V != a.eot) {
            pick = j;
            secondary = j + 1;
            break;
          }
        }
      }
      s_pick[k] = pick;
    }
    a.n_hyp[u] = n_hyp;
    a.best_score[u] = best;
    s_best_k = best_k;
    const int fin = (is_last || n_hyp >= a.max_hyp) ? 1 : 0;
    s_finished = fin;
    if (fin) {
      a.done[u] = 1;
      const int nd = atomicAdd(&a.st->n_done, 1) + 1;
      if (nd == gridDim.x) a.st->all_done = 1;
    }
  }
  __syncwarp();
  if (s_best_k >= 0) {  // record the new best hypothesis (tokens of its parent beam + the last token unless eot)
    const int k = s_best_k;
    const int idx = ci[k];
    const int parent = idx / V, tok = idx % V;
    const int pr = u * beam + parent;
    for (int t = lane; t < gen; t += 32) a.best_tokens[u * a.max_new + t] = seq_cur[pr * a.max_new + t];
    if (lane == 0) {
      int len = gen;
      if (tok != a.eot) {
        a.best_tokens[u * a.max_new + gen] = tok;
        len = gen + 1;
      }
      a.best_len[u] = len;
    }
  }
  // next alive beams (also written when finished: harmless, keeps buffers defined)
  for (int k = 0; k < beam; ++k) {
    const int r = u * beam + k;
    const int idx = ci[s_pick[k]];
    const int parent = idx < 0 ? k : idx / V;
    const int tok = idx < 0 ? a.eot : idx % V;
    const int pr = u * beam + parent;
    for (int t = lane; t < gen; t += 32) seq_nxt[r * a.max_new + t] = seq_cur[pr * a.max_new + t];
    for (int t = lane; t < pos; t += 32) ind_nxt[r * a.t_max + t] = ind_cur[pr * a.t_max + t];
    if (lane == 0) {
      if (gen < a.max_new) seq_nxt[r * a.max_new + gen] = tok;
      ind_nxt[r * a.t_max + pos] = pr;  // this step's K/V were written by the parent row into its own slot
      a.tokens[r] = tok;
      a.cum[r] = (idx < 0) ? -INFINITY : cs[s_pick[k]] * norm;
    }
  }
}

// grid (n_utt) x TK_THREADS: candidate merge, then (warp 0) the bookkeeping of the utterance, then -- by the last CTA to get
// there -- the step advance (position, generation step, ping-pong flip, per-row positions).  One launch instead of three:
// the tail of a decoding step is launch-latency bound.
__global__ void __launch_bounds__(TK_THREADS) search_tail_kernel(const SearchArgs a) {
  __shared__ unsigned long long s_red[32];
  __shared__ unsigned long long s_out[MAX_CAND];
  __shared__ float s_lse[MAX_BEAM];
  __shared__ int s_ts_only[MAX_BEAM];
  __shared__ int s_pick[MAX_BEAM];
  __shared__ int s_best_k;
  __shared__ int s_finished;
  __shared__ int s_last;
  if (a.st->all_done) return;  // a step enqueued ahead of the host's poll: nothing left to do
  topk_merge_body(a, s_red, s_out, s_lse, s_ts_only);
  __syncthreads();  // the candidate list (global) is complete for this CTA's readers
  if (threadIdx.x < 32) search_bookkeeping_body(a, s_pick, s_best_k, s_finished);
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const int t = atomicAdd(&a.st->ticket, 1);
    s_last = t == static_cast<int>(gridDim.x) - 1;
  }
  __syncthreads();
  if (s_last) {  // every utterance has read this step's position / generation step / flip
    if (threadIdx.x == 0) {
      a.st->ticket = 0;
      a.st->pos += 1;
      a.st->gen_step += 1;
      *a.flip ^= 1;
    }
    if (a.row_pos != nullptr)
      for (int i = threadIdx.x; i < a.n_utt * a.beam; i += blockDim.x) a.row_pos[i] += 1;
  }
}

__global__ void prefill_rows_kernel(int* tokens, int* row_pos, int* row_slot, const int* prompt, int prompt_len, int rows,
                                    int p0, int chunk, int beam) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows) return;
  const int u = i / chunk, p = p0 + i % chunk;
  tokens[i] = prompt[u * prompt_len + p];
  row_pos[i] = p;
  row_slot[i] = u * beam;
}

__global__ void prefill_advance_kernel(int* tokens, const int* prompt, int prompt_len, int R, int beam, DecState* st) {
  const int next = st->pos + 1;
  for (int r = threadIdx.x; r < R; r += blockDim.x) tokens[r] = prompt[(r / beam) * prompt_len + next];
  __syncthreads();
  if (threadIdx.x == 0) st->pos = next;
}

// shared_prefix: the prompt prefix (all but the last prompt token) is forwarded once per utterance into the cache slot of
// its first beam by a single prefill pass; decoding then starts at the last prompt token and every beam's indirection
// points at that slot.
__global__ void search_init_kernel(const SearchArgs a, const int* prompt, int shared_prefix) {
  const int R = a.n_utt * a.beam;
  const int tid = blockIdx.x * blockDim.x + threadIdx.x, n = gridDim.x * blockDim.x;
  if (tid == 0) {
    a.st->pos = shared_prefix ? a.prompt_len - 1 : 0;
    a.st->gen_step = 0;
    a.st->n_done = 0;
    a.st->all_done = 0;
    a.st->ticket = 0;
    *a.flip = 0;
  }
  for (int i = tid; i < R; i += n) {
    a.tokens[i] = prompt[(i / a.beam) * a.prompt_len + (shared_prefix ? a.prompt_len - 1 : 0)];
    a.cum[i] = 0.f;
    if (a.row_pos != nullptr) {
      a.row_pos[i] = shared_prefix ? a.prompt_len - 1 : 0;
      a.row_slot[i] = i;
    }
  }
  for (int i = tid; i < a.n_utt; i += n) {
    a.done[i] = 0;
    a.n_hyp[i] = 0;
    a.best_score[i] = -INFINITY;
    a.best_len[i] = 0;
  }
  for (int i = tid; i < R * a.t_max; i += n) {
    const int r = i / a.t_max;
    const int slot = shared_prefix ? (r / a.beam) * a.beam : r;  // else identity: every row holds its own prefix copy
    a.indir[0][i] = slot;
    a.indir[1][i] = slot;
  }
}

__global__ void lang_probs_kernel(const float* logits, long long ldl, const int* lang_ids, int n_lang, int row_stride,
                                  float* probs) {
  __shared__ float s_v[128];
  const int u = blockIdx.x;
  const float* row = logits + static_cast<long long>(u) * row_stride * ldl;
  float mx = -INFINITY;
  for (int i = threadIdx.x; i < n_lang; i += blockDim.x) {
    s_v[i] = row[lang_ids[i]];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 0; i < n_lang; ++i) mx = fmaxf(mx, s_v[i]);
    float s = 0.f;
    for (int i = 0; i < n_lang; ++i) s += expf(s_v[i] - mx);
    for (int i = 0; i < n_lang; ++i) probs[u * n_lang + i] = expf(s_v[i] - mx) / s;
  }
}

}  // namespace

void search_step_run(const SearchArgs& a, cudaStream_t stream) {
  const int R = a.n_utt * a.beam;
  WISB_REQUIRE(a.beam >= 1 && a.beam <= MAX_BEAM && a.n_cand <= MAX_CAND, "search: beam_size must be in [1, 8]");
  WISB_REQUIRE((a.n_vocab + TOPK_CHUNKS - 1) / TOPK_CHUNKS <= TK_THREADS * TK_PER, "search: vocabulary too large");
  if (a.ts_begin >= 0) {
    WISB_REQUIRE(a.ts_begin > a.eot && a.ts_begin < a.n_vocab, "search: the vocabulary has no timestamp tokens");
    WISB_REQUIRE(a.max_init_ts >= 0 && a.max_init_ts < a.n_vocab - a.ts_begin, "search: max_initial_timestamp_index out of range");
    WISB_REQUIRE(cdiv(a.ts_begin, TOPK_CHUNKS - 1) <= TK_THREADS * TK_PER && a.n_vocab - a.ts_begin <= TK_THREADS * TK_PER,
                 "search: vocabulary too large for timestamp decoding");
  }
  topk_partial_kernel<<<dim3(TOPK_CHUNKS, R), TK_THREADS, 0, stream>>>(a);
  search_tail_kernel<<<a.n_utt, TK_THREADS, 0, stream>>>(a);
  WISB_CUDA(cudaGetLastError());
}

void prefill_rows_run(int* tokens, int* row_pos, int* row_slot, const int* prompt, int prompt_len, int n_utt, int p0,
                      int chunk, int beam, cudaStream_t stream) {
  const int rows = n_utt * chunk;
  prefill_rows_kernel<<<cdiv(rows, 256), 256, 0, stream>>>(tokens, row_pos, row_slot, prompt, prompt_len, rows, p0, chunk, beam);
  WISB_CUDA(cudaGetLastError());
}

void prefill_advance_run(int* tokens, const int* prompt, int prompt_len, int R, int beam, DecState* st, cudaStream_t stream) {
  prefill_advance_kernel<<<1, 64, 0, stream>>>(tokens, prompt, prompt_len, R, beam, st);
  WISB_CUDA(cudaGetLastError());
}

void search_init_run(const SearchArgs& a, const int* prompt, cudaStream_t stream, int shared_prefix) {
  search_init_kernel<<<8, 256, 0, stream>>>(a, prompt, shared_prefix);
  WISB_CUDA(cudaGetLastError());
}

void lang_probs_run(const float* logits, long long ldl, const int* lang_ids, int n_lang, int n_utt, int row_stride,
                    float* probs, cudaStream_t stream) {
  WISB_REQUIRE(n_lang <= 128, "detect_language: more than 128 language ids");
  lang_probs_kernel<<<n_utt, 128, 0, stream>>>(logits, ldl, lang_ids, n_lang, row_stride, probs);
  WISB_CUDA(cudaGetLastError());
}

}  // namespace wisb
