// libwisb200.so host side: handle, weight blob, workspaces, encoder / decoder orchestration and the C ABI
// declared in include/wisb200.h.  Mirrors the call surface WIS uses on ctranslate2 (main.py:341-355, 638-640, 685-692).
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/wisb200.h"
#include "decoder.cuh"
#include "kernels.h"

namespace wisb {

namespace {

thread_local std::string g_last_error;

struct TensorRef {
  const uint8_t* ptr = nullptr;
  int dtype = 0, ndim = 0;
  long long shape[4] = {1, 1, 1, 1};
  long long numel() const { return shape[0] * shape[1] * shape[2] * shape[3]; }
};

struct Dims {
  int d_model, n_heads, n_enc_layers, n_dec_layers, n_vocab, n_vocab_pad, n_text_ctx, n_mels, n_audio_ctx, sot, eot,
      transcribe, translate, no_timestamps, sot_prev, sot_lm, no_speech, blank, lang_first, n_langs;
};
static_assert(sizeof(Dims) == WISB_N_DIMS * sizeof(int), "Dims must mirror the blob header");

template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  void ensure(size_t count, bool zero = false) {
    if (count <= n) return;
    release();
    WISB_CUDA(cudaMalloc(&p, count * sizeof(T)));
    n = count;
    if (zero) WISB_CUDA(cudaMemset(p, 0, count * sizeof(T)));
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
  }
  ~DevBuf() { release(); }
};

template <typename T>
struct PinBuf {
  T* p = nullptr;
  size_t n = 0;
  void ensure(size_t count) {
    if (count <= n) return;
    if (p) cudaFreeHost(p);
    WISB_CUDA(cudaMallocHost(&p, count * sizeof(T)));
    n = count;
  }
  ~PinBuf() {
    if (p) cudaFreeHost(p);
  }
};

struct EncLayerPlans {
  GemmPlan qkv, o, fc1, fc2;
};

struct DecLayerW {
  const float *ln1g, *ln1b, *qkvb, *ob, *ln2g, *ln2b, *cqb, *cob, *ln3g, *ln3b, *fc1b, *fc2b;
  const __half *qkvw, *ow, *cqw, *cow, *fc1w, *fc2w;
};

struct GraphKey {
  int n_utt, beam, prompt_len, max_new, max_hyp, u0, b_total, batched, ts_begin, max_init_ts;
  float lp;
  bool operator<(const GraphKey& o) const {
    return memcmp(this, &o, sizeof(GraphKey)) < 0;
  }
};
struct DecGraphs {
  cudaGraphExec_t prefill = nullptr, step = nullptr;
};

}  // namespace

}  // namespace wisb

using namespace wisb;

struct wisb_handle {
  int device = 0;
  int num_sms = 148;
  std::mutex mu;
  cudaStream_t stream = nullptr;
  Dims dims{};
  // weights
  uint8_t* blob = nullptr;
  bool own_blob = false;
  size_t blob_bytes = 0;
  std::map<std::string, TensorRef> tensors;
  std::vector<DecLayerW> dec_w;
  // options
  int use_graphs = 1, attn_v_mn = 1, attn_ref = 0, decode_poll = 1, decoder_mega = 1;
  // front end
  DevBuf<float> lm_tables;
  DevBuf<unsigned> lm_max;
  DevBuf<uint8_t> pcm_dev;
  DevBuf<long long> pcm_off;
  DevBuf<int> pcm_n;
  DevBuf<float> mel;  // [B,80,3000]
  int mel_B = 0;      // utterances currently held in `mel`
  // encoder workspaces (capacity enc_cap utterances)
  int enc_cap = 0;
  DevBuf<__half> h1, xn, qkv, vt, ctx, hbuf, enc_out, ckv;
  DevBuf<float> x;
  GemmPlan plan_conv2, plan_ckv;
  CUtensorMap ckv_map;
  std::vector<EncLayerPlans> enc_plans;
  AttnPlan attn_plan;
  int plans_B = 0, plans_vmn = -1, plans_pdl = -1;
  // decoder workspaces
  DevBuf<float> dx, dq, dctx, dh, logits;
  DevBuf<__half> dctx16, dh16, dxn16, dq16;
  DevBuf<float> dxstat;  // warp-MMA pass: fp16 exchange images of the attention output and the MLP hidden rows
  DevBuf<__half> kcache, vcache;  // [L][16][448][d]
  DevBuf<uint8_t> mask_base, mask_cur;
  std::vector<int> mask_extra;
  DevBuf<float> row_lse, cum, cand_score, best_score, lang_probs, part_max, part_sum;
  DevBuf<unsigned long long> part;
  DevBuf<int> cand_idx, tokens, seq0, seq1, ind0, ind1, flip, done, n_hyp, best_len, best_tokens, prompt_dev, lang_ids;
  DevBuf<DecState> st;
  DevBuf<int> row_pos, row_slot, max_new_u;
  int search_rows = 0;  // rows the search / state buffers above are sized for
  int search_gen = 0, bd_search_gen = -1;  // reallocation count of those buffers / the one the batched-pass plans were built for
  // batched decoder pass (more than DEC_MAX_ROWS rows): workspaces for bd_rows (multiple of 128) rows, bd_tcap positions
  int batch_rows = 320, batch_pdl = 1, decoder_batch = 1, mega_barrier = 1, cross_tc = 1, debug_chunk = 1;  // options: row capacity of one shared pass; programmatic dependent launch
  int bd_rows = 0, bd_tcap = 0, bd_launches_step = 0;
  DevBuf<float> bx, bq, bpart, blogits;
  DevBuf<__half> bxn, bctx, bh, bkc, bvc;
  std::vector<BatchLayer> bd_layers;
  GemmPlan bd_vocab;
  DevBuf<MegaLayer> mega_layers;
  DevBuf<__half> mega_img;  // warp-MMA pass: decoder weights as per-CTA shared-memory images (mega_mma_image)
  int enc_pdl = 1;  // encoder: programmatic dependent launch along the whole kernel chain (227 launches per window)
  int mega_tc = 1, mega_dbg = 0;  // mega_dbg (timing experiments only): bit 0 every layer streams layer 0's weights and cross K/V (L2 resident), bit 1 a quarter of every weight unit
  DevBuf<unsigned> mega_flags;
  // optional reuse of the encoder output + cross K/V between consecutive calls on identical host features
  // (detect_language -> generate -> translate on one window, main.py:633-644, 514-547): option "encoder_cache"
  int encoder_cache = 0;
  std::vector<float> mel_cache;
  int mel_cache_B = 0;
  bool enc_valid = false;
  int ckv_sw = 0, ckv_is_sw = 0;  // cross K/V layout wanted by the decoder pass of this call / layout of what is in HBM
  DevBuf<float> cross_part;
  DevBuf<unsigned> cross_flags;
  DevBuf<float> ln_fold;       // per LN-GEMV: s2[N] and folded bias[N] (qkv, cq, fc1 of every decoder layer, vocab)
  DevBuf<__half> fc2_chunked;  // decoder fc2 weights in chunk-major layout for the persistent pass kernel
  DevBuf<unsigned long long> mega_trace;
  int mega_trace_on = 0, mega_trace_cta = 0, mega_trace_layer = 0;
  cudaEvent_t ev_flag[2] = {nullptr, nullptr};  // decode loop: `all_done` copies of the last two steps
  PinBuf<MegaLayer> mega_layers_host;
  PinBuf<int> pin_i;
  PinBuf<float> pin_f;
  PinBuf<uint8_t> pin_b;
  std::map<GraphKey, DecGraphs> graphs;
  // timing
  cudaEvent_t ev[8] = {};
  float timing[16] = {};
  int launches = 0;
  // optional per-kernel-family profile of the encoder (option "profile"): event pairs on the launching stream
  int profile = 0;
  std::vector<cudaEvent_t> prof_ev;
  std::vector<int> prof_cat;  // category of pair i: 0 gemm, 1 attention, 2 layernorm, 3 conv1
  size_t prof_used = 0;
  void prof_begin(int cat) {
    if (!profile) return;
    if (prof_used + 2 > prof_ev.size()) {
      cudaEvent_t a, b;
      WISB_CUDA(cudaEventCreate(&a));
      WISB_CUDA(cudaEventCreate(&b));
      prof_ev.push_back(a);
      prof_ev.push_back(b);
    }
    prof_cat.push_back(cat);
    WISB_CUDA(cudaEventRecord(prof_ev[prof_used], stream));
  }
  void prof_end() {
    if (!profile) return;
    WISB_CUDA(cudaEventRecord(prof_ev[prof_used + 1], stream));
    prof_used += 2;
  }
  void prof_collect() {  // call after a stream synchronize
    for (int i = 8; i < 16; ++i) timing[i] = 0.f;
    if (!profile) return;
    for (size_t i = 0; i + 1 < prof_used; i += 2) {
      float ms = 0.f;
      WISB_CUDA(cudaEventElapsedTime(&ms, prof_ev[i], prof_ev[i + 1]));
      const int cat = prof_cat[i / 2];
      timing[8 + cat] += ms;
      if (cat == 0) timing[12] += 1.f;
    }
    prof_used = 0;
    prof_cat.clear();
  }

  const TensorRef& T(const std::string& name) const {
    auto it = tensors.find(name);
    if (it == tensors.end()) throw Error(1, "weight blob is missing tensor '" + name + "'");
    return it->second;
  }
  const __half* H(const std::string& n) const { return reinterpret_cast<const __half*>(T(n).ptr); }
  const float* F(const std::string& n) const { return reinterpret_cast<const float*>(T(n).ptr); }
};

namespace {

constexpr int T_MAX = 448;

void parse_blob(wisb_handle* h, const std::vector<uint8_t>& head) {
  WISB_REQUIRE(head.size() >= 256 && memcmp(head.data(), "WISB200\0", 8) == 0, "not a WISB200 weight blob");
  uint32_t version, n_tensors;
  memcpy(&version, head.data() + 8, 4);
  memcpy(&n_tensors, head.data() + 12, 4);
  WISB_REQUIRE(version == 1, "unsupported weight blob version");
  memcpy(&h->dims, head.data() + 16, sizeof(Dims));
  WISB_REQUIRE(head.size() >= 256 + 96ull * n_tensors, "truncated weight blob table");
  for (uint32_t i = 0; i < n_tensors; ++i) {
    const uint8_t* e = head.data() + 256 + 96ull * i;
    char name[49] = {0};
    memcpy(name, e, 48);
    TensorRef t;
    uint32_t dt, nd;
    memcpy(&dt, e + 48, 4);
    memcpy(&nd, e + 52, 4);
    t.dtype = static_cast<int>(dt);
    t.ndim = static_cast<int>(nd);
    for (int k = 0; k < 4; ++k) {
      int64_t s;
      memcpy(&s, e + 56 + 8 * k, 8);
      t.shape[k] = s;
    }
    uint64_t off;
    memcpy(&off, e + 88, 8);
    WISB_REQUIRE(t.dtype >= 0 && t.dtype <= 2 && t.ndim >= 0 && t.ndim <= 4, "bad tensor dtype / rank in the weight blob");
    long long n_el = 1;
    for (int k = 0; k < 4; ++k) {
      WISB_REQUIRE(t.shape[k] >= 0 && t.shape[k] <= (1ll << 40), "bad tensor shape in the weight blob");
      n_el *= (k < t.ndim ? t.shape[k] : 1);
      WISB_REQUIRE(n_el <= (1ll << 40), "bad tensor shape in the weight blob");
    }
    const unsigned long long bytes = static_cast<unsigned long long>(n_el) * (t.dtype == 0 ? 2 : 4);
    WISB_REQUIRE(off <= h->blob_bytes && bytes <= h->blob_bytes - off, std::string("tensor '") + name + "' reaches outside the weight blob");
    t.ptr = h->blob + off;
    h->tensors[name] = t;
  }
  const Dims& d = h->dims;
  WISB_REQUIRE(d.d_model % 128 == 0 && d.d_model == 64 * d.n_heads && d.d_model <= 1536,
               "engine requires head_dim 64 and d_model a multiple of 128 (<= 1536)");
  WISB_REQUIRE(d.n_mels == N_MELS && d.n_audio_ctx == T_ENC, "engine is built for 80 mels x 1500 positions");
  WISB_REQUIRE(d.n_text_ctx <= T_MAX, "n_text_ctx > 448");
  WISB_REQUIRE(d.n_langs <= 128, "more than 128 languages");
  WISB_REQUIRE(d.n_vocab > 0 && d.n_vocab_pad >= d.n_vocab && d.n_vocab_pad % 128 == 0 && d.n_enc_layers > 0 && d.n_dec_layers > 0,
               "bad vocabulary / layer counts in the weight blob");
  // every tensor the kernels index must have exactly the shape the dimensions imply (a truncated or mismatched blob
  // must fail here, not read out of bounds on the device)
  auto expect = [&](const std::string& name, int dtype, std::initializer_list<long long> shape) {
    auto it = h->tensors.find(name);
    WISB_REQUIRE(it != h->tensors.end(), "weight blob is missing tensor '" + name + "'");
    const TensorRef& t = it->second;
    bool ok = t.dtype == dtype && t.ndim == static_cast<int>(shape.size());
    int k = 0;
    for (long long v : shape) ok = ok && t.shape[k++] == v;
    WISB_REQUIRE(ok, "tensor '" + name + "' has the wrong dtype / shape for this model");
  };
  const long long dd = d.d_model;
  expect("enc.conv1.w", 0, {dd, 3ll * d.n_mels});
  expect("enc.conv2.w", 0, {dd, 3 * dd});
  expect("enc.pos", 1, {d.n_audio_ctx, dd});
  expect("dec.tok_emb", 0, {d.n_vocab_pad, dd});
  expect("dec.pos", 1, {d.n_text_ctx, dd});
  expect("dec.crosskv.w", 0, {2ll * d.n_dec_layers * dd, dd});
  expect("dec.crosskv.b", 1, {2ll * d.n_dec_layers * dd});
  for (int side = 0; side < 2; ++side) {
    const int nl = side == 0 ? d.n_enc_layers : d.n_dec_layers;
    for (int i = 0; i < nl; ++i) {
      const std::string p = std::string(side == 0 ? "enc." : "dec.") + std::to_string(i) + ".";
      expect(p + "qkv.w", 0, {3 * dd, dd});
      expect(p + "qkv.b", 1, {3 * dd});
      expect(p + "o.w", 0, {dd, dd});
      expect(p + "o.b", 1, {dd});
      expect(p + "fc1.w", 0, {4 * dd, dd});
      expect(p + "fc1.b", 1, {4 * dd});
      expect(p + "fc2.w", 0, {dd, 4 * dd});
      expect(p + "fc2.b", 1, {dd});
      expect(p + "ln1.g", 1, {dd});
      expect(p + "ln2.g", 1, {dd});
      if (side == 1) {
        expect(p + "cq.w", 0, {dd, dd});
        expect(p + "co.w", 0, {dd, dd});
        expect(p + "ln3.g", 1, {dd});
      }
    }
  }
  for (const char* nm : {"meta.suppress_ids", "meta.suppress_ids_begin"}) {
    auto it = h->tensors.find(nm);
    WISB_REQUIRE(it != h->tensors.end() && it->second.dtype == 2 && it->second.ndim <= 1, std::string("bad '") + nm + "' in the weight blob");
  }
}

void drop_graphs(wisb_handle* h) {
  for (auto& kv : h->graphs) {
    if (kv.second.prefill) cudaGraphExecDestroy(kv.second.prefill);
    if (kv.second.step) cudaGraphExecDestroy(kv.second.step);
  }
  h->graphs.clear();
}

// search / beam state for R rows (rows = utterances x beams of one shared decoder pass)
void ensure_search(wisb_handle* h, int rows) {
  if (rows <= h->search_rows) return;
  WISB_CUDA(cudaStreamSynchronize(h->stream));
  drop_graphs(h);  // captured graphs hold the old pointers
  const size_t R = static_cast<size_t>(rows);
  h->row_lse.ensure(R); h->cum.ensure(R);
  h->part_max.ensure(R * TOPK_CHUNKS); h->part_sum.ensure(R * TOPK_CHUNKS);
  h->part.ensure(R * TOPK_CHUNKS * MAX_CAND);
  h->cand_score.ensure(R * MAX_CAND); h->cand_idx.ensure(R * MAX_CAND);
  h->tokens.ensure(R);
  h->seq0.ensure(R * T_MAX, true); h->seq1.ensure(R * T_MAX, true);
  h->ind0.ensure(R * T_MAX, true); h->ind1.ensure(R * T_MAX, true);
  h->done.ensure(R); h->n_hyp.ensure(R); h->best_score.ensure(R); h->best_len.ensure(R);
  h->best_tokens.ensure(R * T_MAX, true);
  h->prompt_dev.ensure(R * T_MAX);
  h->row_pos.ensure(R, true); h->row_slot.ensure(R, true); h->max_new_u.ensure(R, true);
  h->lang_probs.ensure(R * 128);
  h->pin_i.ensure(4 + R * (T_MAX + 2));
  h->pin_f.ensure(R * 130);
  h->search_rows = rows;
  ++h->search_gen;  // whoever baked these pointers into plans must rebuild them
}

void finish_create(wisb_handle* h) {
  const Dims& d = h->dims;
  const bool has_model = h->blob != nullptr;
  cudaDeviceProp prop;
  WISB_CUDA(cudaGetDeviceProperties(&prop, h->device));
  WISB_REQUIRE(prop.major == 10, "libwisb200 is built for sm_100a (Blackwell B200) only");
  h->num_sms = prop.multiProcessorCount;
  WISB_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  for (auto& e : h->ev) WISB_CUDA(cudaEventCreate(&e));
  h->lm_tables.ensure(logmel_table_floats());
  logmel_init_tables(h->lm_tables.p, h->stream);
  if (!has_model) {  // front-end-only handle (wisb_create_frontend)
    WISB_CUDA(cudaStreamSynchronize(h->stream));
    return;
  }
  // per-layer decoder weight pointers
  h->dec_w.resize(d.n_dec_layers);
  for (int i = 0; i < d.n_dec_layers; ++i) {
    const std::string p = "dec." + std::to_string(i) + ".";
    DecLayerW& w = h->dec_w[i];
    w.ln1g = h->F(p + "ln1.g"); w.ln1b = h->F(p + "ln1.b");
    w.qkvw = h->H(p + "qkv.w"); w.qkvb = h->F(p + "qkv.b");
    w.ow = h->H(p + "o.w"); w.ob = h->F(p + "o.b");
    w.ln2g = h->F(p + "ln2.g"); w.ln2b = h->F(p + "ln2.b");
    w.cqw = h->H(p + "cq.w"); w.cqb = h->F(p + "cq.b");
    w.cow = h->H(p + "co.w"); w.cob = h->F(p + "co.b");
    w.ln3g = h->F(p + "ln3.g"); w.ln3b = h->F(p + "ln3.b");
    w.fc1w = h->H(p + "fc1.w"); w.fc1b = h->F(p + "fc1.b");
    w.fc2w = h->H(p + "fc2.w"); w.fc2b = h->F(p + "fc2.b");
  }
  // suppression mask: bit0 = always (suppress_ids), bit1 = at the first generated step (suppress_ids_begin)
  std::vector<uint8_t> mask(d.n_vocab, 0);
  auto fetch_ids = [&](const char* name) {
    const TensorRef& t = h->T(name);
    std::vector<int> ids(static_cast<size_t>(t.numel()));
    if (!ids.empty()) WISB_CUDA(cudaMemcpy(ids.data(), t.ptr, ids.size() * 4, cudaMemcpyDeviceToHost));
    return ids;
  };
  for (int id : fetch_ids("meta.suppress_ids"))
    if (id >= 0 && id < d.n_vocab) mask[id] |= 1;
  for (int id : fetch_ids("meta.suppress_ids_begin"))
    if (id >= 0 && id < d.n_vocab) mask[id] |= 2;
  h->mask_base.ensure(d.n_vocab);
  h->mask_cur.ensure(d.n_vocab);
  WISB_CUDA(cudaMemcpy(h->mask_base.p, mask.data(), mask.size(), cudaMemcpyHostToDevice));
  WISB_CUDA(cudaMemcpy(h->mask_cur.p, mask.data(), mask.size(), cudaMemcpyHostToDevice));
  // decoder workspaces for DEC_MAX_ROWS rows (the persistent SIMT pass); the batched pass grows the search state later
  const size_t R = DEC_MAX_ROWS;
  h->dx.ensure(R * d.d_model, true);
  h->dq.ensure(R * d.d_model, true);
  h->dctx.ensure(R * d.d_model, true);
  h->dh.ensure(R * 4 * d.d_model, true);
  h->dctx16.ensure(R * d.d_model, true);
  h->dh16.ensure(R * 4 * d.d_model, true);
  h->dxn16.ensure(R * d.d_model, true);
  h->dq16.ensure(R * d.d_model, true);
  h->dxstat.ensure(static_cast<size_t>(h->num_sms) * R * 2, true);
  h->logits.ensure(R * d.n_vocab_pad, true);
  const size_t cache = static_cast<size_t>(d.n_dec_layers) * R * T_MAX * d.d_model;
  h->kcache.ensure(cache, true);
  h->vcache.ensure(cache, true);
  h->flip.ensure(1, true);
  h->st.ensure(1, true);
  ensure_search(h, DEC_MAX_ROWS);
  h->mega_layers.ensure(d.n_dec_layers);
  h->mega_layers_host.ensure(d.n_dec_layers);
  h->mega_flags.ensure(mega_flags_words(), true);
  h->cross_flags.ensure(static_cast<size_t>(DEC_MAX_ROWS) * d.n_heads * 16 * 32, true);
  {
    // LayerNorm fold vectors for the persistent pass kernel (decoder_mega.cu consume_gemv)
    const size_t per_layer = 2ull * (3 * d.d_model + d.d_model + 4 * d.d_model);
    h->ln_fold.ensure(per_layer * d.n_dec_layers + 2ull * d.n_vocab_pad);
    for (int i = 0; i < d.n_dec_layers; ++i) {
      const DecLayerW& w = h->dec_w[i];
      float* base = h->ln_fold.p + per_layer * i;
      mega_ln_fold(w.qkvw, w.ln1g, w.ln1b, w.qkvb, base, base + 3 * d.d_model, 3 * d.d_model, d.d_model, h->stream);
      base += 6 * d.d_model;
      mega_ln_fold(w.cqw, w.ln2g, w.ln2b, w.cqb, base, base + d.d_model, d.d_model, d.d_model, h->stream);
      base += 2 * d.d_model;
      mega_ln_fold(w.fc1w, w.ln3g, w.ln3b, w.fc1b, base, base + 4 * d.d_model, 4 * d.d_model, d.d_model, h->stream);
    }
    float* vb = h->ln_fold.p + per_layer * d.n_dec_layers;
    mega_ln_fold(h->H("dec.tok_emb"), h->F("dec.ln.g"), h->F("dec.ln.b"), nullptr, vb, vb + d.n_vocab_pad, d.n_vocab, d.d_model, h->stream);
  }
  if (mega_k_chunks(4 * d.d_model) > 1) {
    const size_t per = static_cast<size_t>(4) * d.d_model * d.d_model;
    h->fc2_chunked.ensure(per * d.n_dec_layers);
    for (int i = 0; i < d.n_dec_layers; ++i)
      mega_chunk_major(h->dec_w[i].fc2w, h->fc2_chunked.p + per * i, d.d_model, 4 * d.d_model, h->stream);
  }
  h->cross_part.ensure(static_cast<size_t>(DEC_MAX_ROWS) * d.n_heads * 16 * MAX_BEAM * 68, true);
  if (4 * d.d_model <= 5120 && d.d_model % 64 == 0) {
    // warp-MMA pass: a second copy of the decoder weights laid out as the shared-memory image each CTA streams
    // (decoder_mega.cu mma_image_kernel); per layer qkv | o | cq | co | fc1 | fc2, then the vocabulary projection
    const size_t dd = d.d_model;
    const size_t per_layer = 14 * dd * dd;
    const size_t vocab_rows = static_cast<size_t>(d.n_vocab);
    h->mega_img.ensure(per_layer * d.n_dec_layers + vocab_rows * dd);
    for (int i = 0; i < d.n_dec_layers; ++i) {
      const DecLayerW& w = h->dec_w[i];
      __half* p = h->mega_img.p + per_layer * i;
      mega_mma_image(w.qkvw, p, 3 * d.d_model, d.d_model, h->num_sms, h->stream);
      mega_mma_image(w.ow, p + 3 * dd * dd, d.d_model, d.d_model, h->num_sms, h->stream);
      mega_mma_image(w.cqw, p + 4 * dd * dd, d.d_model, d.d_model, d.n_heads, h->stream);  // head-major: the cross phase projects its own queries
      mega_mma_image(w.cow, p + 5 * dd * dd, d.d_model, d.d_model, h->num_sms, h->stream);
      mega_mma_image(w.fc1w, p + 6 * dd * dd, 4 * d.d_model, d.d_model, h->num_sms, h->stream);
      mega_mma_image(w.fc2w, p + 10 * dd * dd, d.d_model, 4 * d.d_model, h->num_sms, h->stream);
    }
    mega_mma_image(h->H("dec.tok_emb"), h->mega_img.p + per_layer * d.n_dec_layers, d.n_vocab, d.d_model, h->num_sms, h->stream);
  } else {
    h->mega_tc = 0;
  }
  WISB_CUDA(cudaStreamSynchronize(h->stream));
}

// feature buffer [B,80,3000] (+ the per-utterance maxima of the log-mel kernel); growing it drops what it held
void ensure_mel(wisb_handle* h, int B) {
  h->lm_max.ensure(B);
  const size_t n = static_cast<size_t>(B) * N_MELS * N_FRAMES;
  if (n <= h->mel.n) return;
  h->mel.ensure(n);
  h->mel_B = 0;
}

void ensure_encoder(wisb_handle* h, int B) {
  if (h->blob == nullptr) return;  // front-end-only handle
  const Dims& dm = h->dims;
  const int d = dm.d_model, H = dm.n_heads;
  const long long M = static_cast<long long>(B) * T_ENC_PAD;
  if (B > h->enc_cap) {
    h->plans_B = 0;
    drop_graphs(h);  // captured decoder graphs hold pointers into the buffers reallocated below
    h->h1.release();
    h->h1.ensure((static_cast<size_t>(B) * H1_ROWS + 8) * d, true);
    h->x.ensure(M * d, true);
    h->xn.ensure(M * d, true);
    h->qkv.ensure(M * 3 * d, true);
    h->vt.ensure(M * d, true);
    h->ctx.ensure(M * d, true);
    h->hbuf.ensure(M * 4 * d, true);
    h->enc_out.ensure(M * d, true);
    h->ckv.ensure(static_cast<size_t>(dm.n_dec_layers) * 2 * M * d, true);
    // the whole cross-K/V buffer as rows of one head's 64 values (for the tcgen05 cross-attention of the batched pass)
    make_tmap_f16_2d(&h->ckv_map, h->ckv.p, HEAD_DIM, static_cast<long long>(h->ckv.n / HEAD_DIM), HEAD_DIM, HEAD_DIM, 128);
    h->enc_cap = B;
  }
  if (h->plans_B == B && h->plans_vmn == h->attn_v_mn && h->plans_pdl == h->enc_pdl) return;
  const int Mi = static_cast<int>(M);
  {
    GemmEpi e;
    e.mode = EPI_CONV2;
    e.bias = h->F("enc.conv2.b");
    e.out = h->x.p;
    e.ldo = d;
    e.pos = h->F("enc.pos");
    gemm_plan(h->plan_conv2, h->h1.p, 2LL * d, h->H("enc.conv2.w"), Mi, d, 3 * d, e, h->num_sms, 0, 2 * d);
  }
  h->enc_plans.assign(dm.n_enc_layers, EncLayerPlans());
  for (int i = 0; i < dm.n_enc_layers; ++i) {
    const std::string p = "enc." + std::to_string(i) + ".";
    EncLayerPlans& pl = h->enc_plans[i];
    GemmEpi e;
    e.mode = h->attn_v_mn ? EPI_F16 : EPI_QKV_VT;
    e.bias = h->F(p + "qkv.b");
    e.out = h->qkv.p;
    e.ldo = 3 * d;
    e.aux = h->vt.p;
    e.d_model = d;
    e.n_heads = H;
    e.batch = B;
    gemm_plan(pl.qkv, h->xn.p, d, h->H(p + "qkv.w"), Mi, 3 * d, d, e, h->num_sms);
    GemmEpi eo;
    eo.mode = EPI_RESID_F32;
    eo.bias = h->F(p + "o.b");
    eo.out = h->x.p;
    eo.ldo = d;
    gemm_plan(pl.o, h->ctx.p, d, h->H(p + "o.w"), Mi, d, d, eo, h->num_sms);
    GemmEpi e1;
    e1.mode = EPI_F16_GELU;
    e1.bias = h->F(p + "fc1.b");
    e1.out = h->hbuf.p;
    e1.ldo = 4 * d;
    gemm_plan(pl.fc1, h->xn.p, d, h->H(p + "fc1.w"), Mi, 4 * d, d, e1, h->num_sms);
    GemmEpi e2;
    e2.mode = EPI_RESID_F32;
    e2.bias = h->F(p + "fc2.b");
    e2.out = h->x.p;
    e2.ldo = d;
    gemm_plan(pl.fc2, h->hbuf.p, 4LL * d, h->H(p + "fc2.w"), Mi, d, 4 * d, e2, h->num_sms);
  }
  {
    GemmEpi e;
    e.mode = EPI_CROSSKV;
    e.bias = h->F("dec.crosskv.b");
    e.out = h->ckv.p;
    e.d_model = d;
    e.n_heads = H;
    e.batch = B;
    gemm_plan(h->plan_ckv, h->enc_out.p, d, h->H("dec.crosskv.w"), Mi, dm.n_dec_layers * 2 * d, d, e, h->num_sms);
  }
  enc_attn_plan(h->attn_plan, h->qkv.p, h->vt.p, h->ctx.p, B, d, H, h->attn_v_mn != 0);
  h->attn_plan.pdl = h->enc_pdl != 0;
  h->plan_conv2.pdl = h->plan_ckv.pdl = h->enc_pdl;
  for (EncLayerPlans& pl : h->enc_plans) pl.qkv.pdl = pl.o.pdl = pl.fc1.pdl = pl.fc2.pdl = h->enc_pdl;
  h->plans_pdl = h->enc_pdl;
  h->plans_B = B;
  h->plans_vmn = h->attn_v_mn;
}

// the persistent warp-MMA pass (<= 8 rows) reads the cross K/V rows chunk-swizzled (ldmatrix without bank conflicts); every
// other decoder path reads them linear
bool want_ckv_swizzle(const wisb_handle* h, int rows) {
  return rows <= DEC_MAX_ROWS && h->decoder_batch != 2 && h->decoder_mega && h->mega_tc;
}

// mel (device, [B,80,3000]) -> enc_out fp16 [B*1536, d] (+ cross K/V when with_ckv)
void run_encoder(wisb_handle* h, int B, int n_layers, bool with_ckv, int mel_first = 0) {
  const Dims& dm = h->dims;
  const int d = dm.d_model;
  const int M = B * T_ENC_PAD;
  cudaStream_t s = h->stream;
  ensure_encoder(h, B);
  h->enc_valid = false;  // callers that want the result cached re-validate it after a full encode
  h->prof_begin(3);
  conv1_gelu_run(h->mel.p + static_cast<size_t>(mel_first) * N_MELS * N_FRAMES, h->H("enc.conv1.w"), h->F("enc.conv1.b"), h->h1.p, B, d, s);
  h->prof_end();
  h->prof_begin(0);
  gemm_run(h->plan_conv2, s);
  h->prof_end();
  const int nl = (n_layers < 0 || n_layers > dm.n_enc_layers) ? dm.n_enc_layers : n_layers;
  for (int i = 0; i < nl; ++i) {
    const std::string p = "enc." + std::to_string(i) + ".";
    EncLayerPlans& pl = h->enc_plans[i];
    h->prof_begin(2);
    layernorm_f32_to_f16_run(h->x.p, h->F(p + "ln1.g"), h->F(p + "ln1.b"), h->xn.p, M, d, s, h->enc_pdl != 0);
    h->prof_end();
    h->prof_begin(0);
    gemm_run(pl.qkv, s);
    h->prof_end();
    h->prof_begin(1);
    if (h->attn_ref)
      enc_attn_ref_run(h->qkv.p, h->ctx.p, B, d, dm.n_heads, s);
    else
      enc_attn_run(h->attn_plan, s);
    h->prof_end();
    h->prof_begin(0);
    gemm_run(pl.o, s);
    h->prof_end();
    h->prof_begin(2);
    layernorm_f32_to_f16_run(h->x.p, h->F(p + "ln2.g"), h->F(p + "ln2.b"), h->xn.p, M, d, s, h->enc_pdl != 0);
    h->prof_end();
    h->prof_begin(0);
    gemm_run(pl.fc1, s);
    h->prof_end();
    h->prof_begin(0);
    gemm_run(pl.fc2, s);
    h->prof_end();
  }
  h->prof_begin(2);
  layernorm_f32_to_f16_run(h->x.p, h->F("enc.ln_post.g"), h->F("enc.ln_post.b"), h->enc_out.p, M, d, s, h->enc_pdl != 0);
  h->prof_end();
  h->launches += 2 + 7 * nl + 1;
  if (with_ckv) {
    WISB_CUDA(cudaEventRecord(h->ev[3], s));
    h->prof_begin(0);
    h->plan_ckv.epi.kv_swizzle = h->ckv_sw;
    gemm_run(h->plan_ckv, s);
    h->ckv_is_sw = h->ckv_sw;
    h->prof_end();
    h->launches += 1;
  }
}

// Places the features of this call in h->mel.  Returns true when the encoder output and cross K/V already in HBM belong
// to exactly these features (option "encoder_cache", host features of <= 2 windows compared byte for byte), in which
// case the caller skips the encoder.  Off by default: a benchmark that feeds the same utterance every step must not
// silently skip work.
bool upload_mel(wisb_handle* h, const float* mel, int B) {
  ensure_mel(h, B);
  if (mel == nullptr) {
    WISB_REQUIRE(h->mel_B == B, "mel == NULL but wisb_logmel(keep_on_device) did not leave features for this batch size");
    h->mel_cache_B = 0;
    return false;
  }
  const size_t n = static_cast<size_t>(B) * N_MELS * N_FRAMES;
  if (h->encoder_cache && B <= 2) {
    if (h->enc_valid && h->mel_cache_B == B && memcmp(h->mel_cache.data(), mel, n * sizeof(float)) == 0) return true;
    h->mel_cache.assign(mel, mel + n);
    h->mel_cache_B = B;
  } else {
    h->mel_cache_B = 0;
  }
  h->enc_valid = false;
  WISB_CUDA(cudaMemcpyAsync(h->mel.p, mel, n * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  h->mel_B = B;
  return false;
}

// encoder + cross K/V for the features placed by upload_mel, unless they are already there
void encode_for_decode(wisb_handle* h, int B, bool reuse) {
  if (reuse) {
    WISB_CUDA(cudaEventRecord(h->ev[3], h->stream));  // keeps the stage timings well defined (both read ~0)
    return;
  }
  run_encoder(h, B, -1, true);
  h->enc_valid = h->encoder_cache != 0 && h->mel_cache_B == B;
}

struct DecodeCfg {
  int u0, n_utt, B_total, beam, prompt_len, max_new, max_hyp;
  float lp;
  int per_utt_max_new = 0;  // h->max_new_u holds a per-utterance cap (<= max_new)
  int ts_begin = -1, max_init_ts = 0;  // timestamp rules (SearchArgs): first timestamp token, -1 = off
};

SearchArgs make_search_args(wisb_handle* h, const DecodeCfg& c) {
  const Dims& dm = h->dims;
  SearchArgs a;
  a.logits = h->logits.p;
  a.ldl = dm.n_vocab_pad;
  a.n_vocab = dm.n_vocab;
  a.mask = h->mask_cur.p;
  a.n_utt = c.n_utt;
  a.beam = c.beam;
  a.n_cand = 2 * c.beam;
  a.max_new = c.max_new;
  a.max_hyp = c.max_hyp;
  a.eot = dm.eot;
  a.t_max = T_MAX;
  a.prompt_len = c.prompt_len;
  a.length_penalty = c.lp;
  a.row_lse = h->row_lse.p;
  a.part_max = h->part_max.p;
  a.part_sum = h->part_sum.p;
  a.cum = h->cum.p;
  a.part = h->part.p;
  a.cand_score = h->cand_score.p;
  a.cand_idx = h->cand_idx.p;
  a.tokens = h->tokens.p;
  a.seq[0] = h->seq0.p;
  a.seq[1] = h->seq1.p;
  a.indir[0] = h->ind0.p;
  a.indir[1] = h->ind1.p;
  a.flip = h->flip.p;
  a.done = h->done.p;
  a.n_hyp = h->n_hyp.p;
  a.best_score = h->best_score.p;
  a.best_len = h->best_len.p;
  a.best_tokens = h->best_tokens.p;
  a.st = h->st.p;
  a.row_pos = h->row_pos.p;
  a.row_slot = h->row_slot.p;
  a.max_new_u = c.per_utt_max_new ? h->max_new_u.p : nullptr;
  a.ts_begin = c.ts_begin;
  a.max_init_ts = c.max_init_ts;
  return a;
}

// descriptors of the persistent decoder pass for this batch slice (device array of per-layer pointers)
void upload_mega_layers(wisb_handle* h, const DecodeCfg& c) {
  const Dims& dm = h->dims;
  const int d = dm.d_model, H = dm.n_heads;
  const size_t layer_cache = static_cast<size_t>(DEC_MAX_ROWS) * T_MAX * d;
  const size_t head_block = static_cast<size_t>(H) * T_ENC_PAD * HEAD_DIM;
  for (int i = 0; i < dm.n_dec_layers; ++i) {
    const DecLayerW& w = h->dec_w[i];
    MegaLayer& m = h->mega_layers_host.p[i];
    m = MegaLayer();
    // (LayerNorm-fused GEMVs: `bias` is the folded bias, ln_s2 the fold vector, both precomputed at load)
    auto set = [&](MegaGemv& g, const __half* wt, const float* bias, const float* lg, const float* s2, const float* x,
                   float* out, long long ldo, int N, int K, int epi) {
      g.w = wt; g.bias = bias; g.ln_g = lg; g.ln_s2 = s2; g.x = x; g.out = out; g.ldo = ldo; g.N = N; g.K = K; g.epi = epi;
    };
    const size_t per_layer = 2ull * (3 * d + d + 4 * d);
    const float* fb = h->ln_fold.p + per_layer * i;
    set(m.qkv, w.qkvw, fb + 3 * d, w.ln1g, fb, h->dx.p, h->dq.p, d, 3 * d, d, GV_QKV);
    set(m.o, w.ow, w.ob, nullptr, nullptr, h->dctx.p, h->dx.p, d, d, d, GV_RESID);
    set(m.cq, w.cqw, fb + 7 * d, w.ln2g, fb + 6 * d, h->dx.p, h->dq.p, d, d, d, GV_STORE);
    set(m.co, w.cow, w.cob, nullptr, nullptr, h->dctx.p, h->dx.p, d, d, d, GV_RESID);
    set(m.fc1, w.fc1w, fb + 12 * d, w.ln3g, fb + 8 * d, h->dx.p, h->dh.p, 4 * d, 4 * d, d, GV_GELU);
    const __half* fc2w = (h->fc2_chunked.p && !h->mega_tc) ? h->fc2_chunked.p + static_cast<size_t>(4) * d * d * i : w.fc2w;
    set(m.fc2, fc2w, w.fc2b, nullptr, nullptr, h->dh.p, h->dx.p, d, d, 4 * d, GV_RESID);
    if (h->mega_tc) {
      m.o.x16 = h->dctx16.p;
      m.co.x16 = h->dctx16.p;
      m.fc1.out16 = h->dh16.p;
      m.fc2.x16 = h->dh16.p;
      m.qkv.x16 = m.cq.x16 = m.fc1.x16 = h->dxn16.p;
      m.cq.out16 = h->dq16.p;
      m.qkv.shape = 0;
      m.o.shape = m.cq.shape = m.co.shape = 1;
      m.fc1.shape = 2;
      m.fc2.shape = 3;
      m.o.next_g = w.ln2g;
      m.co.next_g = w.ln3g;
      m.fc2.next_g = i + 1 < dm.n_dec_layers ? h->dec_w[i + 1].ln1g : h->F("dec.ln.g");
      const size_t dd = d;
      const __half* img = h->mega_img.p + 14 * dd * dd * ((h->mega_dbg & 1) ? 0 : i);
      m.qkv.w = img;
      m.o.w = img + 3 * dd * dd;
      m.cq.w = img + 4 * dd * dd;
      m.co.w = img + 5 * dd * dd;
      m.fc1.w = img + 6 * dd * dd;
      m.fc2.w = img + 10 * dd * dd;
    }
    const int ikv = (h->mega_dbg & 1) ? 0 : i;
    m.ck = h->ckv.p + (static_cast<size_t>(ikv * 2 + 0) * c.B_total + c.u0) * head_block;
    m.cv = h->ckv.p + (static_cast<size_t>(ikv * 2 + 1) * c.B_total + c.u0) * head_block;
    m.kcache = h->kcache.p + i * layer_cache;
    m.vcache = h->vcache.p + i * layer_cache;
  }
  WISB_CUDA(cudaMemcpyAsync(h->mega_layers.p, h->mega_layers_host.p, sizeof(MegaLayer) * dm.n_dec_layers,
                            cudaMemcpyHostToDevice, h->stream));
}

int enqueue_decoder_forward_mega(wisb_handle* h, const DecodeCfg& c, bool with_logits, bool prefill_pass = false) {
  const Dims& dm = h->dims;
  MegaArgs a;
  a.layers = h->mega_layers.p;
  a.n_layers = dm.n_dec_layers;
  a.vocab.w = h->H("dec.tok_emb");
  a.vocab.ln_g = h->F("dec.ln.g");
  {
    const size_t per_layer = 2ull * 8 * dm.d_model;
    const float* vb = h->ln_fold.p + per_layer * dm.n_dec_layers;
    a.vocab.ln_s2 = vb;
    a.vocab.bias = vb + dm.n_vocab_pad;
  }
  a.vocab.x = h->dx.p;
  a.vocab.out = h->logits.p;
  a.vocab.ldo = dm.n_vocab_pad;
  a.vocab.N = dm.n_vocab;
  a.vocab.K = dm.d_model;
  a.vocab.epi = GV_STORE;
  if (h->mega_tc) {
    a.vocab.w = h->mega_img.p + static_cast<size_t>(14) * dm.d_model * dm.d_model * dm.n_dec_layers;
    a.tc = 1;
    a.dbg = h->mega_dbg;
    a.ctx16 = h->dctx16.p;
    a.xn16 = h->dxn16.p;
    a.q16 = h->dq16.p;
    a.xstat = h->dxstat.p;
    a.vocab.x16 = h->dxn16.p;
    a.vocab.shape = 4;
  }
  a.with_logits = with_logits ? 1 : 0;
  a.R = c.n_utt * c.beam;
  a.d = dm.d_model;
  a.H = dm.n_heads;
  a.n_utt = c.n_utt;
  a.beam = c.beam;
  a.t_max = T_MAX;
  a.tokens = h->tokens.p;
  if (prefill_pass) {  // the whole prompt prefix of every utterance in ONE pass (rows = utterances x prefix positions)
    a.pf_len = c.prompt_len - 1;
    a.pf_tok_stride = c.prompt_len;
    a.pf_slot_stride = c.beam;
    a.R = c.n_utt * a.pf_len;
    a.beam = a.pf_len;
    a.tokens = h->prompt_dev.p;
  }
  a.tok_emb = h->H("dec.tok_emb");
  a.pos_emb = h->F("dec.pos");
  a.x = h->dx.p;
  a.q = h->dq.p;
  a.ctx = h->dctx.p;
  a.indir0 = h->ind0.p;
  a.indir1 = h->ind1.p;
  a.flip = h->flip.p;
  a.st = h->st.p;
  a.cross_part = h->cross_part.p;
  a.cross_flags = h->cross_flags.p;
  a.flags = h->mega_flags.p;
  a.epoch_base = h->mega_flags.p + 160 * 32;
  a.barrier_mode = h->mega_barrier;
  if (h->mega_trace_on) {
    h->mega_trace.ensure(2048 + 160 * 264, true);
    a.trace = h->mega_trace.p;
    a.trace_cta = h->mega_trace_cta;
    a.trace_layer = h->mega_trace_layer;
    a.trace_cap = h->mega_tc ? 380 : 70;
  }
  dec_pass_run(a, h->num_sms, h->stream);
  return 1;
}

// one decoder forward for R rows at position st->pos; returns kernels launched
int enqueue_decoder_forward(wisb_handle* h, const DecodeCfg& c, bool with_logits) {
  if (h->decoder_mega) return enqueue_decoder_forward_mega(h, c, with_logits);
  const Dims& dm = h->dims;
  const int d = dm.d_model, H = dm.n_heads, R = c.n_utt * c.beam;
  cudaStream_t s = h->stream;
  const DecState* st = h->st.p;
  int n = 0;
  dec_embed_run(h->tokens.p, h->H("dec.tok_emb"), h->F("dec.pos"), h->dx.p, R, d, st, s);
  ++n;
  const size_t layer_cache = static_cast<size_t>(DEC_MAX_ROWS) * T_MAX * d;
  const size_t head_block = static_cast<size_t>(H) * T_ENC_PAD * HEAD_DIM;  // one utterance, one of K/V
  for (int i = 0; i < dm.n_dec_layers; ++i) {
    const DecLayerW& w = h->dec_w[i];
    GemvArgs g;
    g.R = R;
    g.st = st;
    // LN1 + QKV (+ cache append)
    g.x = h->dx.p; g.ln_g = w.ln1g; g.ln_b = w.ln1b; g.w = w.qkvw; g.bias = w.qkvb;
    g.out = h->dq.p; g.ldo = d; g.N = 3 * d; g.K = d; g.epi = GV_QKV;
    g.kcache = h->kcache.p + i * layer_cache; g.vcache = h->vcache.p + i * layer_cache; g.d_model = d; g.t_max = T_MAX;
    gemv_run(g, s);
    dec_self_attn_run(h->dq.p, h->kcache.p + i * layer_cache, h->vcache.p + i * layer_cache, h->ind0.p, h->ind1.p,
                      h->flip.p, h->dctx.p, R, d, H, T_MAX, st, s);
    GemvArgs o;
    o.R = R; o.st = st; o.x = h->dctx.p; o.w = w.ow; o.bias = w.ob; o.out = h->dx.p; o.ldo = d; o.N = d; o.K = d;
    o.epi = GV_RESID;
    gemv_run(o, s);
    // LN2 + cross-attention
    GemvArgs q;
    q.R = R; q.st = st; q.x = h->dx.p; q.ln_g = w.ln2g; q.ln_b = w.ln2b; q.w = w.cqw; q.bias = w.cqb; q.out = h->dq.p;
    q.ldo = d; q.N = d; q.K = d; q.epi = GV_STORE;
    gemv_run(q, s);
    const __half* kl = h->ckv.p + (static_cast<size_t>(i * 2 + 0) * c.B_total + c.u0) * head_block;
    const __half* vl = h->ckv.p + (static_cast<size_t>(i * 2 + 1) * c.B_total + c.u0) * head_block;
    dec_cross_attn_run(h->dq.p, kl, vl, h->dctx.p, c.n_utt, c.beam, d, H, s);
    GemvArgs co;
    co.R = R; co.st = st; co.x = h->dctx.p; co.w = w.cow; co.bias = w.cob; co.out = h->dx.p; co.ldo = d; co.N = d;
    co.K = d; co.epi = GV_RESID;
    gemv_run(co, s);
    // LN3 + MLP
    GemvArgs f1;
    f1.R = R; f1.st = st; f1.x = h->dx.p; f1.ln_g = w.ln3g; f1.ln_b = w.ln3b; f1.w = w.fc1w; f1.bias = w.fc1b;
    f1.out = h->dh.p; f1.ldo = 4 * d; f1.N = 4 * d; f1.K = d; f1.epi = GV_GELU;
    gemv_run(f1, s);
    GemvArgs f2;
    f2.R = R; f2.st = st; f2.x = h->dh.p; f2.w = w.fc2w; f2.bias = w.fc2b; f2.out = h->dx.p; f2.ldo = d; f2.N = d;
    f2.K = 4 * d; f2.epi = GV_RESID;
    gemv_run(f2, s);
    n += 8;
  }
  if (with_logits) {
    GemvArgs v;
    v.R = R; v.st = st; v.x = h->dx.p; v.ln_g = h->F("dec.ln.g"); v.ln_b = h->F("dec.ln.b"); v.w = h->H("dec.tok_emb");
    v.out = h->logits.p; v.ldo = dm.n_vocab_pad; v.N = dm.n_vocab; v.K = d; v.epi = GV_STORE;
    gemv_run(v, s);
    ++n;
  }
  return n;
}

void enqueue_prefill(wisb_handle* h, const DecodeCfg& c) {
  enqueue_decoder_forward(h, c, false);
  prefill_advance_run(h->tokens.p, h->prompt_dev.p, c.prompt_len, c.n_utt * c.beam, c.beam, h->st.p, h->stream);
}
void enqueue_step(wisb_handle* h, const DecodeCfg& c) {
  enqueue_decoder_forward(h, c, true);
  search_step_run(make_search_args(h, c), h->stream);
}

DecGraphs& get_graphs(wisb_handle* h, const DecodeCfg& c) {
  GraphKey key;
  memset(&key, 0, sizeof(key));
  key.n_utt = c.n_utt; key.beam = c.beam; key.prompt_len = c.prompt_len; key.max_new = c.max_new;
  key.max_hyp = c.max_hyp; key.lp = c.lp;
  key.u0 = c.u0; key.b_total = c.B_total;  // they move the cross-K/V base pointers baked into the graph
  key.ts_begin = c.ts_begin; key.max_init_ts = c.max_init_ts;  // baked into the search kernels' arguments
  auto it = h->graphs.find(key);
  if (it != h->graphs.end()) return it->second;
  if (h->graphs.size() > 64) {  // bound the cache
    for (auto& kv : h->graphs) {
      if (kv.second.prefill) cudaGraphExecDestroy(kv.second.prefill);
      if (kv.second.step) cudaGraphExecDestroy(kv.second.step);
    }
    h->graphs.clear();
  }
  DecGraphs g;
  cudaGraph_t graph;
  WISB_CUDA(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
  enqueue_prefill(h, c);
  WISB_CUDA(cudaStreamEndCapture(h->stream, &graph));
  WISB_CUDA(cudaGraphInstantiate(&g.prefill, graph, 0));
  WISB_CUDA(cudaGraphDestroy(graph));
  WISB_CUDA(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
  enqueue_step(h, c);
  WISB_CUDA(cudaStreamEndCapture(h->stream, &graph));
  WISB_CUDA(cudaGraphInstantiate(&g.step, graph, 0));
  WISB_CUDA(cudaGraphDestroy(graph));
  return h->graphs[key] = g;
}

void set_extra_suppress(wisb_handle* h, const int32_t* extra, int n_extra) {
  std::vector<int> want(extra ? extra : nullptr, extra ? extra + n_extra : nullptr);
  if (want == h->mask_extra) return;
  const Dims& dm = h->dims;
  for (int id : want) WISB_REQUIRE(id >= 0 && id < dm.n_vocab, "suppress token id outside the vocabulary");
  h->mask_extra.assign(1, -1);  // not a valid set: if anything below fails, the next call rebuilds the mask
  WISB_CUDA(cudaMemcpyAsync(h->mask_cur.p, h->mask_base.p, dm.n_vocab, cudaMemcpyDeviceToDevice, h->stream));
  if (!want.empty()) {
    std::vector<uint8_t> m(dm.n_vocab);
    WISB_CUDA(cudaMemcpyAsync(m.data(), h->mask_base.p, dm.n_vocab, cudaMemcpyDeviceToHost, h->stream));
    WISB_CUDA(cudaStreamSynchronize(h->stream));
    for (int id : want) m[id] |= 1;
    WISB_CUDA(cudaMemcpyAsync(h->mask_cur.p, m.data(), dm.n_vocab, cudaMemcpyHostToDevice, h->stream));
    WISB_CUDA(cudaStreamSynchronize(h->stream));
  }
  h->mask_extra = want;
}

// decode utterances [u0, u0 + n_utt) of the encoded batch; writes results to the host arrays
int decode_pass(wisb_handle* h, const DecodeCfg& c, const int32_t* prompts, int32_t* out_ids, int out_stride,
                int32_t* out_len, float* out_score) {
  cudaStream_t s = h->stream;
  const int R = c.n_utt * c.beam;
  int steps = 0;
  // prompts for this pass
  memcpy(h->pin_i.p + 4, prompts + static_cast<size_t>(c.u0) * c.prompt_len, sizeof(int) * c.n_utt * c.prompt_len);
  WISB_CUDA(cudaMemcpyAsync(h->prompt_dev.p, h->pin_i.p + 4, sizeof(int) * c.n_utt * c.prompt_len, cudaMemcpyHostToDevice, s));
  SearchArgs sa = make_search_args(h, c);
  // persistent-pass path: forward the prompt prefix of all utterances in one pass when it fits the 8-row kernel
  const int pf_rows = c.n_utt * (c.prompt_len - 1);
  const bool one_pass_prefill = h->decoder_mega && c.prompt_len > 1 && pf_rows <= DEC_MAX_ROWS && c.prompt_len - 1 <= MAX_BEAM;
  search_init_run(sa, h->prompt_dev.p, s, one_pass_prefill ? 1 : 0);
  if (h->decoder_mega) upload_mega_layers(h, c);
  if (c.max_new > 0) {
    // the persistent pass kernel is a handful of launches per step: no graph needed (and it is a cooperative launch)
    DecGraphs* g = (h->use_graphs && !h->decoder_mega) ? &get_graphs(h, c) : nullptr;
    if (one_pass_prefill) {
      enqueue_decoder_forward_mega(h, c, false, true);
      ++steps;
    } else {
      for (int p = 0; p + 1 < c.prompt_len; ++p) {
        if (g) WISB_CUDA(cudaGraphLaunch(g->prefill, s)); else enqueue_prefill(h, c);
        ++steps;
      }
    }
    const int fwd = h->decoder_mega ? 1 : 1 + 8 * h->dims.n_dec_layers + 1;
    const int per_step = fwd + 2;
    h->launches += (c.prompt_len - 1) * (fwd + 1);
    volatile int* flag = h->pin_i.p;
    flag[0] = flag[1] = 0;
    // persistent-pass path with a poll every step: step gs + 1 is enqueued BEFORE the host waits for step gs's `all_done`
    // word (the kernels of a step that turns out to be superfluous leave at once on the device flag), so neither the
    // launch latency of the cooperative kernel nor the host's wake-up sits between two steps
    const bool ahead = h->decoder_mega && h->decode_poll == 1;
    if (ahead && h->ev_flag[0] == nullptr) {
      WISB_CUDA(cudaEventCreateWithFlags(&h->ev_flag[0], cudaEventDisableTiming));
      WISB_CUDA(cudaEventCreateWithFlags(&h->ev_flag[1], cudaEventDisableTiming));
    }
    for (int gs = 0; gs < c.max_new; ++gs) {
      if (g) WISB_CUDA(cudaGraphLaunch(g->step, s)); else enqueue_step(h, c);
      ++steps;
      h->launches += per_step;
      if (ahead) {
        WISB_CUDA(cudaMemcpyAsync(const_cast<int*>(flag) + (gs & 1), &h->st.p->all_done, sizeof(int), cudaMemcpyDeviceToHost, s));
        WISB_CUDA(cudaEventRecord(h->ev_flag[gs & 1], s));
        if (gs >= 1) {
          WISB_CUDA(cudaEventSynchronize(h->ev_flag[(gs - 1) & 1]));
          if (flag[(gs - 1) & 1]) {
            --steps;  // the step just enqueued does nothing
            break;
          }
        }
        continue;
      }
      const bool poll = ((gs + 1) % h->decode_poll == 0) || gs + 1 == c.max_new;
      if (poll) {
        WISB_CUDA(cudaMemcpyAsync(const_cast<int*>(flag), &h->st.p->all_done, sizeof(int), cudaMemcpyDeviceToHost, s));
        WISB_CUDA(cudaStreamSynchronize(s));
        if (*flag) break;
      }
    }
  }
  // results
  int* lens = h->pin_i.p + 4;
  int* toks = lens + DEC_MAX_ROWS;
  WISB_CUDA(cudaMemcpyAsync(lens, h->best_len.p, sizeof(int) * c.n_utt, cudaMemcpyDeviceToHost, s));
  WISB_CUDA(cudaMemcpyAsync(toks, h->best_tokens.p, sizeof(int) * c.n_utt * (c.max_new > 0 ? c.max_new : 1), cudaMemcpyDeviceToHost, s));
  WISB_CUDA(cudaMemcpyAsync(h->pin_f.p, h->best_score.p, sizeof(float) * c.n_utt, cudaMemcpyDeviceToHost, s));
  WISB_CUDA(cudaStreamSynchronize(s));
  for (int u = 0; u < c.n_utt; ++u) {
    const int len = c.max_new > 0 ? lens[u] : 0;
    out_len[c.u0 + u] = len;
    for (int t = 0; t < len && t < out_stride; ++t) out_ids[static_cast<size_t>(c.u0 + u) * out_stride + t] = toks[u * c.max_new + t];
    if (out_score) out_score[c.u0 + u] = c.max_new > 0 ? h->pin_f.p[u] : 0.f;
  }
  (void)R;
  return steps;
}


// ------------------------------------------------------------------------------------------------- batched decoder pass
// tile width / split-K of one decoder GEMM for `M` rows: keep >= ~120 CTAs streaming the weight matrix
void plan_dec_gemm(wisb_handle* h, GemmPlan& p, const __half* a, long long lda, const __half* w, int M, int N, int K,
                   GemmEpi e, bool allow_split) {
  const int mt = M / 128;
  int bn = 256;
  while (bn > 64 && (N % bn != 0 || mt * (N / bn) < 120)) bn /= 2;
  int splits = 1;
  if (allow_split) {
    const int kb = K / 64;
    while (mt * (N / bn) * splits < 120 && splits < 8 && kb % (splits * 2) == 0 && kb / (splits * 2) >= 4) splits *= 2;
    e.mode = EPI_F32;
    e.split_stride = static_cast<long long>(M) * N;
  }
  gemm_plan(p, a, lda, w, M, N, K, e, h->num_sms, bn, 0, splits);
}

// workspaces + GEMM plans of the batched pass for `rows` rows and `t_need` text positions per cache slot
void ensure_batch(wisb_handle* h, int rows, int t_need) {
  const Dims& dm = h->dims;
  const int d = dm.d_model, L = dm.n_dec_layers;
  int Rp = round_up(rows, 128);
  int tc = round_up(t_need, 32);
  if (tc > T_MAX) tc = T_MAX;
  ensure_search(h, rows);
  // (the QKV epilogues hold the row_slot / row_pos pointers of the search state: a reallocation there stales the plans)
  if (Rp <= h->bd_rows && tc <= h->bd_tcap && h->bd_search_gen == h->search_gen) return;
  if (Rp < h->bd_rows) Rp = h->bd_rows;
  if (tc < h->bd_tcap) tc = h->bd_tcap;
  WISB_CUDA(cudaStreamSynchronize(h->stream));
  drop_graphs(h);
  const size_t M = static_cast<size_t>(Rp);
  h->bx.ensure(M * d, true);
  h->bq.ensure(M * d, true);
  h->bxn.ensure(M * d, true);    // rows beyond the live ones stay zero: finite GEMM inputs, outputs never stored
  h->bctx.ensure(M * d, true);
  h->bh.ensure(M * 4 * d, true);
  h->bpart.ensure(8 * M * d, true);
  h->blogits.ensure(M * dm.n_vocab_pad, true);
  const size_t layer_cache = M * tc * d;
  if (layer_cache * L > h->bkc.n) {  // (free first: the two caches are the largest buffers of the handle)
    h->bkc.release();
    h->bvc.release();
  }
  h->bkc.ensure(layer_cache * L, true);
  h->bvc.ensure(layer_cache * L, true);
  h->bd_layers.assign(L, BatchLayer());
  for (int i = 0; i < L; ++i) {
    const DecLayerW& w = h->dec_w[i];
    BatchLayer& b = h->bd_layers[i];
    b.kcache = h->bkc.p + layer_cache * i;
    b.vcache = h->bvc.p + layer_cache * i;
    b.ln1g = w.ln1g; b.ln1b = w.ln1b;
    b.ob = w.ob; b.ln2g = w.ln2g; b.ln2b = w.ln2b;
    b.cob = w.cob; b.ln3g = w.ln3g; b.ln3b = w.ln3b;
    b.fc2b = w.fc2b;
    b.next_g = (i + 1 < L) ? h->dec_w[i + 1].ln1g : h->F("dec.ln.g");
    b.next_b = (i + 1 < L) ? h->dec_w[i + 1].ln1b : h->F("dec.ln.b");
    GemmEpi e;
    e.mode = EPI_DEC_QKV;
    e.bias = w.qkvb;
    e.out = h->bq.p;
    e.ldo = d;
    e.aux = b.kcache;
    e.aux2 = b.vcache;
    e.d_model = d;
    e.row_slot = h->row_slot.p;
    e.row_pos = h->row_pos.p;
    e.t_cap = tc;
    plan_dec_gemm(h, b.qkv, h->bxn.p, d, w.qkvw, Rp, 3 * d, d, e, false);
    GemmEpi ep;  // split-K partials; bias / residual / LayerNorm happen in bd_resid_ln_kernel
    ep.out = h->bpart.p;
    ep.ldo = d;
    plan_dec_gemm(h, b.o, h->bctx.p, d, w.ow, Rp, d, d, ep, true);
    GemmEpi eq;
    eq.mode = EPI_F32;
    eq.bias = w.cqb;
    eq.out = h->bq.p;
    eq.ldo = d;
    plan_dec_gemm(h, b.cq, h->bxn.p, d, w.cqw, Rp, d, d, eq, false);
    plan_dec_gemm(h, b.co, h->bctx.p, d, w.cow, Rp, d, d, ep, true);
    GemmEpi e1;
    e1.mode = EPI_F16_GELU;
    e1.bias = w.fc1b;
    e1.out = h->bh.p;
    e1.ldo = 4 * d;
    plan_dec_gemm(h, b.fc1, h->bxn.p, d, w.fc1w, Rp, 4 * d, d, e1, false);
    plan_dec_gemm(h, b.fc2, h->bh.p, 4LL * d, w.fc2w, Rp, d, 4 * d, ep, true);
  }
  {
    GemmEpi ev;
    ev.mode = EPI_F32;
    ev.out = h->blogits.p;
    ev.ldo = dm.n_vocab_pad;
    plan_dec_gemm(h, h->bd_vocab, h->bxn.p, d, h->H("dec.tok_emb"), Rp, dm.n_vocab_pad, d, ev, false);
  }
  h->bd_rows = Rp;
  h->bd_tcap = tc;
  h->bd_search_gen = h->search_gen;
}

BatchArgs make_batch_args(wisb_handle* h, const DecodeCfg& c) {
  const Dims& dm = h->dims;
  BatchArgs a;
  a.d = dm.d_model;
  a.H = dm.n_heads;
  a.n_utt = c.n_utt;
  a.t_cap = h->bd_tcap;
  a.t_ind = T_MAX;
  a.pdl = h->batch_pdl;
  a.tokens = h->tokens.p;
  a.row_pos = h->row_pos.p;
  a.row_slot = h->row_slot.p;
  a.tok_emb = h->H("dec.tok_emb");
  a.pos_emb = h->F("dec.pos");
  a.x = h->bx.p;
  a.xn = h->bxn.p;
  a.q = h->bq.p;
  a.ctx = h->bctx.p;
  a.part = h->bpart.p;
  a.part_stride = static_cast<long long>(h->bd_rows) * dm.d_model;
  a.indir0 = h->ind0.p;
  a.indir1 = h->ind1.p;
  a.flip = h->flip.p;
  a.vocab = &h->bd_vocab;
  a.cross_tc = h->cross_tc;
  a.num_sms = h->num_sms;
  a.ckv_map = &h->ckv_map;
  a.ckv_base = h->ckv.p;
  if (h->profile) {
    a.prof = [](void* ctx, int cat, int begin) {
      wisb_handle* hh = static_cast<wisb_handle*>(ctx);
      if (begin) hh->prof_begin(cat); else hh->prof_end();
    };
    a.prof_ctx = h;
  }
  return a;
}

SearchArgs make_batch_search_args(wisb_handle* h, const DecodeCfg& c) {
  SearchArgs sa = make_search_args(h, c);
  sa.logits = h->blogits.p;
  return sa;
}

void enqueue_batch_step(wisb_handle* h, const DecodeCfg& c) {
  BatchArgs a = make_batch_args(h, c);
  a.R = c.n_utt * c.beam;
  a.rows_per_utt = c.beam;
  a.with_logits = 1;
  a.done = h->done.p;
  h->bd_launches_step = batch_pass_run(a, h->bd_layers.data(), h->dims.n_dec_layers, h->stream) + 2;
  search_step_run(make_batch_search_args(h, c), h->stream);
}

// decode utterances [u0, u0 + n_utt) of the encoded batch with ONE shared decoder pass per generated token
int decode_batch(wisb_handle* h, const DecodeCfg& c, const int32_t* prompts, const int* max_new_host, int32_t* out_ids,
                 int out_stride, int32_t* out_len, float* out_score) {
  const Dims& dm = h->dims;
  cudaStream_t s = h->stream;
  const int R = c.n_utt * c.beam;
  const int H = dm.n_heads;
  ensure_batch(h, R, c.prompt_len + c.max_new);
  // cross K/V of the utterances of this pass
  const size_t head_block = static_cast<size_t>(H) * T_ENC_PAD * HEAD_DIM;
  for (int i = 0; i < dm.n_dec_layers; ++i) {
    h->bd_layers[i].ck = h->ckv.p + (static_cast<size_t>(i * 2 + 0) * c.B_total + c.u0) * head_block;
    h->bd_layers[i].cv = h->ckv.p + (static_cast<size_t>(i * 2 + 1) * c.B_total + c.u0) * head_block;
  }
  int steps = 0;
  int* pin = h->pin_i.p + 4;
  memcpy(pin, prompts + static_cast<size_t>(c.u0) * c.prompt_len, sizeof(int) * c.n_utt * c.prompt_len);
  WISB_CUDA(cudaMemcpyAsync(h->prompt_dev.p, pin, sizeof(int) * c.n_utt * c.prompt_len, cudaMemcpyHostToDevice, s));
  int* pin_mx = pin + static_cast<size_t>(c.n_utt) * c.prompt_len;
  if (c.per_utt_max_new) {
    memcpy(pin_mx, max_new_host, sizeof(int) * c.n_utt);
    WISB_CUDA(cudaMemcpyAsync(h->max_new_u.p, pin_mx, sizeof(int) * c.n_utt, cudaMemcpyHostToDevice, s));
  }
  if (c.max_new > 0) {
    // ---- prompt prefix: every utterance's positions [0, prompt_len - 1) as rows of shared passes (<= 8 positions and
    //      <= the row capacity per pass), K/V into the slot of the utterance's first beam
    const int pf_len = c.prompt_len - 1;
    int chunk_max = h->bd_rows / c.n_utt;
    if (chunk_max > MAX_BEAM) chunk_max = MAX_BEAM;
    if (chunk_max < 1) chunk_max = 1;
    for (int p0 = 0; p0 < pf_len; p0 += chunk_max) {
      const int chunk = pf_len - p0 < chunk_max ? pf_len - p0 : chunk_max;
      prefill_rows_run(h->tokens.p, h->row_pos.p, h->row_slot.p, h->prompt_dev.p, c.prompt_len, c.n_utt, p0, chunk, c.beam, s);
      BatchArgs a = make_batch_args(h, c);
      a.R = c.n_utt * chunk;
      a.rows_per_utt = chunk;
      a.prefill = 1;
      h->launches += 1 + batch_pass_run(a, h->bd_layers.data(), dm.n_dec_layers, s);
      ++steps;
    }
    SearchArgs sa = make_batch_search_args(h, c);
    search_init_run(sa, h->prompt_dev.p, s, 1);
    DecGraphs* g = nullptr;
    if (h->use_graphs && !h->profile) {  // (the per-kernel timing hook needs eager launches)
      GraphKey key;
      memset(&key, 0, sizeof(key));
      key.n_utt = c.n_utt; key.beam = c.beam; key.prompt_len = c.prompt_len; key.max_new = c.max_new;
      key.max_hyp = c.max_hyp; key.lp = c.lp; key.u0 = c.u0; key.b_total = c.B_total;
      key.batched = 1 + c.per_utt_max_new;
      key.ts_begin = c.ts_begin; key.max_init_ts = c.max_init_ts;
      auto it = h->graphs.find(key);
      if (it == h->graphs.end()) {
        if (h->graphs.size() > 64) drop_graphs(h);
        DecGraphs ng;
        cudaGraph_t graph;
        WISB_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
        enqueue_batch_step(h, c);
        WISB_CUDA(cudaStreamEndCapture(s, &graph));
        WISB_CUDA(cudaGraphInstantiate(&ng.step, graph, 0));
        WISB_CUDA(cudaGraphDestroy(graph));
        it = h->graphs.emplace(key, ng).first;
      }
      g = &it->second;
    }
    volatile int* flag = h->pin_i.p;
    *flag = 0;
    for (int gs = 0; gs < c.max_new; ++gs) {
      if (g) WISB_CUDA(cudaGraphLaunch(g->step, s)); else enqueue_batch_step(h, c);
      ++steps;
      h->launches += h->bd_launches_step;
      const bool poll = ((gs + 1) % h->decode_poll == 0) || gs + 1 == c.max_new;
      if (poll) {
        WISB_CUDA(cudaMemcpyAsync(const_cast<int*>(flag), &h->st.p->all_done, sizeof(int), cudaMemcpyDeviceToHost, s));
        WISB_CUDA(cudaStreamSynchronize(s));
        if (*flag) break;
      }
    }
  }
  // results
  int* lens = h->pin_i.p + 4;
  int* toks = lens + c.n_utt;
  const int mn = c.max_new > 0 ? c.max_new : 1;
  WISB_CUDA(cudaMemcpyAsync(lens, h->best_len.p, sizeof(int) * c.n_utt, cudaMemcpyDeviceToHost, s));
  WISB_CUDA(cudaMemcpyAsync(toks, h->best_tokens.p, sizeof(int) * c.n_utt * mn, cudaMemcpyDeviceToHost, s));
  WISB_CUDA(cudaMemcpyAsync(h->pin_f.p, h->best_score.p, sizeof(float) * c.n_utt, cudaMemcpyDeviceToHost, s));
  WISB_CUDA(cudaStreamSynchronize(s));
  for (int u = 0; u < c.n_utt; ++u) {
    const int len = c.max_new > 0 ? lens[u] : 0;
    out_len[c.u0 + u] = len;
    for (int t = 0; t < len && t < out_stride; ++t) out_ids[static_cast<size_t>(c.u0 + u) * out_stride + t] = toks[u * mn + t];
    if (out_score) out_score[c.u0 + u] = c.max_new > 0 ? h->pin_f.p[u] : 0.f;
  }
  return steps;
}

template <typename Fn>
int guarded(wisb_handle* h, Fn&& fn) {
  try {
    if (h == nullptr) throw Error(1, "null handle");
    std::lock_guard<std::mutex> lock(h->mu);
    WISB_CUDA(cudaSetDevice(h->device));
    fn();
    return 0;
  } catch (const Error& e) {
    g_last_error = e.what();
    if (h && h->stream) {  // leave no dangling capture / sticky state behind
      cudaStreamCaptureStatus cs;
      if (cudaStreamIsCapturing(h->stream, &cs) == cudaSuccess && cs != cudaStreamCaptureStatusNone) {
        cudaGraph_t g = nullptr;
        cudaStreamEndCapture(h->stream, &g);
        if (g) cudaGraphDestroy(g);
      }
      cudaGetLastError();
    }
    return e.code;
  } catch (const std::exception& e) {
    g_last_error = e.what();
    return 2;
  }
}

int create_common(wisb_handle** out, int device, const std::function<void(wisb_handle*)>& load) {
  if (out == nullptr) {
    g_last_error = "out handle pointer is NULL";
    return 1;
  }
  *out = nullptr;
  std::unique_ptr<wisb_handle> h(new wisb_handle());
  try {
    int n_dev = 0;
    cudaError_t e = cudaGetDeviceCount(&n_dev);
    if (e != cudaSuccess || n_dev == 0)
      throw Error(2, std::string("no CUDA device available (libwisb200 has no CPU fallback): ") + cudaGetErrorString(e));
    WISB_REQUIRE(device >= 0 && device < n_dev, "device index out of range");
    h->device = device;
    WISB_CUDA(cudaSetDevice(device));
    load(h.get());
    finish_create(h.get());
    *out = h.release();
    return 0;
  } catch (const Error& e) {
    g_last_error = e.what();
    return e.code;
  } catch (const std::exception& e) {
    g_last_error = e.what();
    return 2;
  }
}

}  // namespace

// ===================================================================================================================== C ABI
extern "C" {

int wisb_abi_version(void) { return WISB_ABI_VERSION; }
const char* wisb_last_error(void) { return g_last_error.c_str(); }

int wisb_create_from_host(const void* blob, size_t nbytes, int device, wisb_handle** out) {
  return create_common(out, device, [&](wisb_handle* h) {
    WISB_REQUIRE(blob != nullptr && nbytes >= 256, "weight blob is NULL or too small");
    h->blob_bytes = nbytes;
    h->own_blob = true;
    WISB_CUDA(cudaMalloc(&h->blob, nbytes));
    WISB_CUDA(cudaMemcpy(h->blob, blob, nbytes, cudaMemcpyHostToDevice));
    const uint8_t* b = static_cast<const uint8_t*>(blob);
    uint32_t n_tensors = 0;
    memcpy(&n_tensors, b + 12, 4);
    const size_t head = 256 + 96ull * n_tensors;
    WISB_REQUIRE(head <= nbytes, "truncated weight blob");
    parse_blob(h, std::vector<uint8_t>(b, b + head));
  });
}

int wisb_create(const char* weights_path, int device, wisb_handle** out) {
  if (weights_path == nullptr) {
    g_last_error = "weights_path is NULL";
    return 1;
  }
  FILE* f = fopen(weights_path, "rb");
  if (!f) {
    g_last_error = std::string("cannot open weight blob '") + weights_path + "'";
    return 1;
  }
  fseek(f, 0, SEEK_END);
  const long long sz = ftell(f);
  fseek(f, 0, SEEK_SET);
  std::vector<uint8_t> buf(static_cast<size_t>(sz > 0 ? sz : 0));
  const size_t got = buf.empty() ? 0 : fread(buf.data(), 1, buf.size(), f);
  fclose(f);
  if (got != buf.size()) {
    g_last_error = "short read on the weight blob";
    return 1;
  }
  return wisb_create_from_host(buf.data(), buf.size(), device, out);
}

int wisb_create_from_device(const void* device_blob, size_t nbytes, int device, wisb_handle** out) {
  return create_common(out, device, [&](wisb_handle* h) {
    WISB_REQUIRE(device_blob != nullptr && nbytes >= 256, "weight blob is NULL or too small");
    h->blob_bytes = nbytes;
    h->own_blob = false;
    h->blob = const_cast<uint8_t*>(static_cast<const uint8_t*>(device_blob));
    std::vector<uint8_t> head(256);
    WISB_CUDA(cudaMemcpy(head.data(), h->blob, 256, cudaMemcpyDeviceToHost));
    uint32_t n_tensors = 0;
    memcpy(&n_tensors, head.data() + 12, 4);
    const size_t hb = 256 + 96ull * n_tensors;
    WISB_REQUIRE(hb <= nbytes, "truncated weight blob");
    head.resize(hb);
    WISB_CUDA(cudaMemcpy(head.data(), h->blob, hb, cudaMemcpyDeviceToHost));
    parse_blob(h, head);
  });
}

int wisb_create_frontend(int device, wisb_handle** out) {
  return create_common(out, device, [&](wisb_handle*) {});
}

int wisb_destroy(wisb_handle* h) {
  if (h == nullptr) return 0;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  for (auto& kv : h->graphs) {
    if (kv.second.prefill) cudaGraphExecDestroy(kv.second.prefill);
    if (kv.second.step) cudaGraphExecDestroy(kv.second.step);
  }
  for (auto& e : h->ev)
    if (e) cudaEventDestroy(e);
  for (auto& e : h->prof_ev) cudaEventDestroy(e);
  if (h->own_blob && h->blob) cudaFree(h->blob);
  for (cudaEvent_t ev : h->ev_flag)
    if (ev) cudaEventDestroy(ev);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
  return 0;
}

int wisb_get_dims(wisb_handle* h, int32_t* dims) {
  return guarded(h, [&] {
    WISB_REQUIRE(dims != nullptr, "dims is NULL");
    memcpy(dims, &h->dims, sizeof(Dims));
  });
}

int wisb_set_option(wisb_handle* h, const char* key, int value) {
  return guarded(h, [&] {
    WISB_REQUIRE(key != nullptr, "key is NULL");
    const std::string k(key);
    if (k == "use_graphs") h->use_graphs = value;
    else if (k == "attn_v_mn_major") h->attn_v_mn = value;
    else if (k == "attn_ref") h->attn_ref = value;
    else if (k == "decode_poll") h->decode_poll = value < 1 ? 1 : value;
    else if (k == "profile") h->profile = value;
    else if (k == "decoder_mega") h->decoder_mega = value;
    else if (k == "encoder_cache") {
      h->encoder_cache = value ? 1 : 0;
      h->enc_valid = false;
    }
    else if (k == "mega_trace") h->mega_trace_on = value;
    else if (k == "mega_dbg") h->mega_dbg = value;
    else if (k == "enc_pdl") h->enc_pdl = value ? 1 : 0;
    else if (k == "mega_trace_cta") h->mega_trace_cta = value;
    else if (k == "mega_trace_layer") h->mega_trace_layer = value;
    else if (k == "batch_rows") {
      WISB_REQUIRE(value >= 8 && value <= 1024, "batch_rows must be in [8, 1024]");
      h->batch_rows = value;
    }
    else if (k == "batch_pdl") h->batch_pdl = value ? 1 : 0;
    else if (k == "mega_barrier") h->mega_barrier = value ? 1 : 0;
    else if (k == "debug_chunk") h->debug_chunk = value;
    else if (k == "mega_tc" || k == "mega_mma") {  // 1: GEMV phases of the persistent pass on the warp-level tensor path, 0: the SIMT pass
      WISB_REQUIRE(!value || h->mega_img.p != nullptr, "mega_mma needs d_model <= 1280 and a multiple of 64");
      h->mega_tc = value ? 1 : 0;
    }
    else if (k == "cross_tc") {  // 1: tcgen05 cross-attention in the batched pass, 0: the SIMT cluster kernel (cross-check)
      h->cross_tc = value ? 1 : 0;
      drop_graphs(h);
    }
    else if (k == "decoder_batch") h->decoder_batch = value;  // 2 = use the batched pass even for <= 8 rows (tests)
    else throw Error(1, "unknown option '" + k + "'");
  });
}

int wisb_get_timing(wisb_handle* h, float* out16) {
  return guarded(h, [&] {
    WISB_REQUIRE(out16 != nullptr, "out is NULL");
    memcpy(out16, h->timing, sizeof(h->timing));
  });
}

int wisb_logmel(wisb_handle* h, const void* pcm, int pcm_dtype, int pcm_on_device, const int64_t* offsets,
                const int32_t* n_samples, int B, float* mel_out, int keep_on_device) {
  return guarded(h, [&] {
    WISB_REQUIRE(pcm != nullptr && offsets != nullptr && n_samples != nullptr, "pcm / offsets / n_samples is NULL");
    WISB_REQUIRE(B >= 1 && B <= 4096, "B out of range");
    WISB_REQUIRE(pcm_dtype == WISB_PCM_F32 || pcm_dtype == WISB_PCM_S16, "pcm_dtype must be WISB_PCM_F32 or WISB_PCM_S16");
    const size_t esz = pcm_dtype == WISB_PCM_S16 ? 2 : 4;
    long long total = 0;
    for (int b = 0; b < B; ++b) {
      WISB_REQUIRE(n_samples[b] >= 0 && offsets[b] >= 0, "negative n_samples / offset");
      const long long end = offsets[b] + n_samples[b];
      if (end > total) total = end;
    }
    cudaStream_t s = h->stream;
    ensure_mel(h, B);
    h->pcm_off.ensure(B);
    h->pcm_n.ensure(B);
    WISB_CUDA(cudaEventRecord(h->ev[0], s));
    const void* pcm_d = pcm;
    if (!pcm_on_device) {
      h->pcm_dev.ensure(static_cast<size_t>(total > 0 ? total : 1) * esz);
      if (total > 0) WISB_CUDA(cudaMemcpyAsync(h->pcm_dev.p, pcm, static_cast<size_t>(total) * esz, cudaMemcpyHostToDevice, s));
      pcm_d = h->pcm_dev.p;
    }
    static_assert(sizeof(long long) == sizeof(int64_t), "offset type");
    WISB_CUDA(cudaMemcpyAsync(h->pcm_off.p, offsets, sizeof(int64_t) * B, cudaMemcpyHostToDevice, s));
    WISB_CUDA(cudaMemcpyAsync(h->pcm_n.p, n_samples, sizeof(int32_t) * B, cudaMemcpyHostToDevice, s));
    logmel_run(pcm_d, pcm_dtype == WISB_PCM_S16, h->pcm_off.p, h->pcm_n.p, B, h->lm_tables.p, h->mel.p, h->lm_max.p, s);
    if (mel_out != nullptr)
      WISB_CUDA(cudaMemcpyAsync(mel_out, h->mel.p, static_cast<size_t>(B) * N_MELS * N_FRAMES * sizeof(float), cudaMemcpyDeviceToHost, s));
    WISB_CUDA(cudaEventRecord(h->ev[1], s));
    WISB_CUDA(cudaStreamSynchronize(s));
    WISB_CUDA(cudaEventElapsedTime(&h->timing[0], h->ev[0], h->ev[1]));
    h->mel_B = keep_on_device ? B : 0;
    h->enc_valid = false;  // the device feature buffer was rewritten
    h->mel_cache_B = 0;
  });
}

// wisb_generate_ex (timestamps == 0) and wisb_generate_ts (timestamps != 0)
static int generate_common(wisb_handle* h, const float* mel, int B, const int32_t* prompts, int prompt_len, int beam_size,
                           float patience, float length_penalty, int max_length, const int32_t* max_length_per_utt,
                           const int32_t* extra_suppress, int n_extra, int timestamps, int max_initial_timestamp_index,
                           int32_t* out_ids, int out_stride, int32_t* out_len, float* out_score) {
  return guarded(h, [&] {
    const Dims& dm = h->dims;
    WISB_REQUIRE(h->blob != nullptr, "handle has no model (created by wisb_create_frontend)");
    WISB_REQUIRE(B >= 1 && B <= 4096, "B out of range");
    WISB_REQUIRE(prompts != nullptr && out_ids != nullptr && out_len != nullptr, "prompts / out_ids / out_len is NULL");
    WISB_REQUIRE(beam_size >= 1 && beam_size <= MAX_BEAM, "beam_size must be in [1, 8]");
    WISB_REQUIRE(prompt_len >= 1 && prompt_len <= dm.n_text_ctx, "prompt length out of range");
    WISB_REQUIRE(max_length >= 1 && max_length <= dm.n_text_ctx, "max_length must be in [1, n_text_ctx]");
    WISB_REQUIRE(patience > 0.f, "patience must be positive");
    WISB_REQUIRE(n_extra >= 0 && (n_extra == 0 || extra_suppress != nullptr), "bad extra_suppress");
    for (long long i = 0; i < static_cast<long long>(B) * prompt_len; ++i)
      WISB_REQUIRE(prompts[i] >= 0 && prompts[i] < dm.n_vocab, "prompt token outside the vocabulary");
    const int ts_begin = timestamps ? dm.no_timestamps + 1 : -1;
    if (timestamps) {
      WISB_REQUIRE(ts_begin > dm.eot && ts_begin < dm.n_vocab, "the model's vocabulary has no timestamp tokens");
      WISB_REQUIRE(max_initial_timestamp_index >= 0 && max_initial_timestamp_index <= dm.n_vocab - ts_begin - 1,
                   "max_initial_timestamp_index must be in [0, number of timestamp tokens - 1]");
      for (long long i = 0; i < static_cast<long long>(B) * prompt_len; ++i)
        WISB_REQUIRE(prompts[i] != dm.no_timestamps, "timestamp decoding: the prompt must not contain <|notimestamps|>");
    }
    auto new_tokens = [&](int ml) {  // CTranslate2: at most max_length / 2 new tokens, max_length in total
      int v = ml / 2 < ml - prompt_len ? ml / 2 : ml - prompt_len;
      return v < 0 ? 0 : v;
    };
    int max_new = new_tokens(max_length);
    std::vector<int> per_utt;
    if (max_length_per_utt != nullptr) {
      per_utt.resize(B);
      max_new = 0;
      for (int b = 0; b < B; ++b) {
        WISB_REQUIRE(max_length_per_utt[b] >= 1 && max_length_per_utt[b] <= dm.n_text_ctx, "per-utterance max_length out of range");
        per_utt[b] = new_tokens(max_length_per_utt[b]);
        if (per_utt[b] > max_new) max_new = per_utt[b];
      }
    }
    WISB_REQUIRE(out_stride >= max_new, "out_stride smaller than the maximum number of generated tokens");
    cudaStream_t s = h->stream;
    h->launches = 0;
    for (int i = 1; i <= 5; ++i) h->timing[i] = 0.f;
    WISB_CUDA(cudaEventRecord(h->ev[0], s));
    bool reuse = upload_mel(h, mel, B);
    h->ckv_sw = want_ckv_swizzle(h, B * beam_size) ? 1 : 0;
    if (reuse && h->ckv_is_sw != h->ckv_sw) reuse = false;  // cached cross K/V is in the other pass's layout (the features are still on the device)
    set_extra_suppress(h, extra_suppress, n_extra);
    WISB_CUDA(cudaEventRecord(h->ev[2], s));
    WISB_CUDA(cudaEventSynchronize(h->ev[2]));
    WISB_CUDA(cudaEventElapsedTime(&h->timing[1], h->ev[0], h->ev[2]));
    DecodeCfg c;
    c.beam = beam_size;
    c.prompt_len = prompt_len;
    c.max_hyp = static_cast<int>(beam_size * patience + 0.5f);
    if (c.max_hyp < 1) c.max_hyp = 1;
    c.lp = length_penalty;
    c.ts_begin = ts_begin;
    c.max_init_ts = timestamps ? max_initial_timestamp_index : 0;
    // Utterances are encoded and decoded in groups that share every decoder pass: the group's rows (utterances x beams)
    // are the M dimension of the batched pass, so the decoder weights stream once per generated token for the whole
    // group.  The group size only bounds the workspaces (cross K/V: 252 MB per large-v2 utterance).
    const bool mega = B * beam_size <= DEC_MAX_ROWS && h->decoder_batch != 2;
    int group = mega ? B : h->batch_rows / beam_size;
    if (group < 1) group = 1;
    int steps = 0;
    for (int g0 = 0; g0 < B; g0 += group) {
      const int n = B - g0 < group ? B - g0 : group;
      WISB_CUDA(cudaEventRecord(h->ev[2], s));
      if (reuse) {
        WISB_CUDA(cudaEventRecord(h->ev[3], s));
      } else {
        run_encoder(h, n, -1, true, g0);
        h->enc_valid = h->encoder_cache != 0 && h->mel_cache_B == B && n == B;
      }
      WISB_CUDA(cudaEventRecord(h->ev[4], s));
      c.u0 = 0;
      c.n_utt = n;
      c.B_total = n;
      c.max_new = max_new;
      c.per_utt_max_new = 0;
      if (!per_utt.empty()) {
        c.per_utt_max_new = 1;
        c.max_new = 0;
        for (int u = 0; u < n; ++u) c.max_new = per_utt[g0 + u] > c.max_new ? per_utt[g0 + u] : c.max_new;
      }
      const int32_t* gp = prompts + static_cast<size_t>(g0) * prompt_len;
      int32_t* gi = out_ids + static_cast<size_t>(g0) * out_stride;
      if (mega) {
        WISB_REQUIRE(per_utt.empty() || c.max_new == max_new, "internal: per-utterance limits on the small path");
        if (!per_utt.empty()) {  // small path: the search kernels read the per-utterance caps from the same buffer
          WISB_CUDA(cudaMemcpyAsync(h->max_new_u.p, per_utt.data() + g0, sizeof(int) * n, cudaMemcpyHostToDevice, s));
          WISB_CUDA(cudaStreamSynchronize(s));
        }
        steps += decode_pass(h, c, gp, gi, out_stride, out_len + g0, out_score ? out_score + g0 : nullptr);
      } else {
        steps += decode_batch(h, c, gp, per_utt.empty() ? nullptr : per_utt.data() + g0, gi, out_stride, out_len + g0,
                              out_score ? out_score + g0 : nullptr);
      }
      WISB_CUDA(cudaEventRecord(h->ev[5], s));
      WISB_CUDA(cudaStreamSynchronize(s));
      float t;
      WISB_CUDA(cudaEventElapsedTime(&t, h->ev[2], h->ev[3]));
      h->timing[2] += t;
      WISB_CUDA(cudaEventElapsedTime(&t, h->ev[3], h->ev[4]));
      h->timing[3] += t;
      WISB_CUDA(cudaEventElapsedTime(&t, h->ev[4], h->ev[5]));
      h->timing[4] += t;
    }
    WISB_CUDA(cudaEventElapsedTime(&h->timing[5], h->ev[0], h->ev[5]));
    h->timing[6] = static_cast<float>(steps);
    h->timing[7] = static_cast<float>(h->launches);
    h->prof_collect();
  });
}

int wisb_generate_ex(wisb_handle* h, const float* mel, int B, const int32_t* prompts, int prompt_len, int beam_size,
                     float patience, float length_penalty, int max_length, const int32_t* max_length_per_utt,
                     const int32_t* extra_suppress, int n_extra, int32_t* out_ids, int out_stride, int32_t* out_len,
                     float* out_score) {
  return generate_common(h, mel, B, prompts, prompt_len, beam_size, patience, length_penalty, max_length,
                         max_length_per_utt, extra_suppress, n_extra, 0, 0, out_ids, out_stride, out_len, out_score);
}

int wisb_generate_ts(wisb_handle* h, const float* mel, int B, const int32_t* prompts, int prompt_len, int beam_size,
                     float patience, float length_penalty, int max_length, const int32_t* max_length_per_utt,
                     const int32_t* extra_suppress, int n_extra, int max_initial_timestamp_index, int32_t* out_ids,
                     int out_stride, int32_t* out_len, float* out_score) {
  return generate_common(h, mel, B, prompts, prompt_len, beam_size, patience, length_penalty, max_length,
                         max_length_per_utt, extra_suppress, n_extra, 1, max_initial_timestamp_index, out_ids, out_stride,
                         out_len, out_score);
}

int wisb_generate(wisb_handle* h, const float* mel, int B, const int32_t* prompts, int prompt_len, int beam_size,
                  float patience, float length_penalty, int max_length, const int32_t* extra_suppress, int n_extra,
                  int32_t* out_ids, int out_stride, int32_t* out_len, float* out_score) {
  return wisb_generate_ex(h, mel, B, prompts, prompt_len, beam_size, patience, length_penalty, max_length, nullptr,
                          extra_suppress, n_extra, out_ids, out_stride, out_len, out_score);
}

int wisb_detect_language(wisb_handle* h, const float* mel, int B, int32_t* lang_ids_out, float* probs_out) {
  return guarded(h, [&] {
    const Dims& dm = h->dims;
    WISB_REQUIRE(h->blob != nullptr, "handle has no model (created by wisb_create_frontend)");
    WISB_REQUIRE(B >= 1 && B <= 4096, "B out of range");
    WISB_REQUIRE(lang_ids_out != nullptr && probs_out != nullptr, "output pointer is NULL");
    cudaStream_t s = h->stream;
    bool reuse = upload_mel(h, mel, B);
    h->ckv_sw = (h->decoder_mega && h->mega_tc) ? 1 : 0;  // language detection always runs the <= 8-row pass
    if (reuse && h->ckv_is_sw != h->ckv_sw) reuse = false;
    encode_for_decode(h, B, reuse);
    const int nl = dm.n_langs;
    h->lang_ids.ensure(nl);
    std::vector<int> ids(nl);
    for (int i = 0; i < nl; ++i) ids[i] = dm.lang_first + i;
    WISB_CUDA(cudaMemcpyAsync(h->lang_ids.p, ids.data(), sizeof(int) * nl, cudaMemcpyHostToDevice, s));
    WISB_CUDA(cudaStreamSynchronize(s));
    std::vector<int32_t> sot(DEC_MAX_ROWS, dm.sot);
    for (int u0 = 0; u0 < B; u0 += DEC_MAX_ROWS) {
      DecodeCfg c;
      c.u0 = u0;
      c.n_utt = (B - u0 < DEC_MAX_ROWS) ? B - u0 : DEC_MAX_ROWS;
      c.B_total = B;
      c.beam = 1;
      c.prompt_len = 1;
      c.max_new = 1;
      c.max_hyp = 1;
      c.lp = 1.f;
      memcpy(h->pin_i.p + 4, sot.data(), sizeof(int) * c.n_utt);
      WISB_CUDA(cudaMemcpyAsync(h->prompt_dev.p, h->pin_i.p + 4, sizeof(int) * c.n_utt, cudaMemcpyHostToDevice, s));
      search_init_run(make_search_args(h, c), h->prompt_dev.p, s);
      if (h->decoder_mega) upload_mega_layers(h, c);
      enqueue_decoder_forward(h, c, true);
      lang_probs_run(h->logits.p, dm.n_vocab_pad, h->lang_ids.p, nl, c.n_utt, 1, h->lang_probs.p, s);
      WISB_CUDA(cudaMemcpyAsync(h->pin_f.p, h->lang_probs.p, sizeof(float) * c.n_utt * nl, cudaMemcpyDeviceToHost, s));
      WISB_CUDA(cudaStreamSynchronize(s));
      for (int u = 0; u < c.n_utt; ++u) {
        std::vector<int> order(nl);
        for (int i = 0; i < nl; ++i) order[i] = i;
        const float* p = h->pin_f.p + u * nl;
        std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return p[a] > p[b]; });
        for (int i = 0; i < nl; ++i) {
          lang_ids_out[static_cast<size_t>(u0 + u) * nl + i] = ids[order[i]];
          probs_out[static_cast<size_t>(u0 + u) * nl + i] = p[order[i]];
        }
      }
    }
  });
}

// --------------------------------------------------------------------------------------------------------------------- diagnostics
int wisb_debug_gemm(wisb_handle* h, const uint16_t* a, const uint16_t* w, float* c, int M, int N, int K, int impl, int bn) {
  return guarded(h, [&] {
    WISB_REQUIRE(a && w && c, "NULL pointer");
    cudaStream_t s = h->stream;
    DevBuf<__half> da, dw;
    DevBuf<float> dc;
    da.ensure(static_cast<size_t>(M) * K);
    dw.ensure(static_cast<size_t>(N) * K);
    dc.ensure(static_cast<size_t>(M) * N, true);
    WISB_CUDA(cudaMemcpyAsync(da.p, a, sizeof(__half) * M * K, cudaMemcpyHostToDevice, s));
    WISB_CUDA(cudaMemcpyAsync(dw.p, w, sizeof(__half) * N * K, cudaMemcpyHostToDevice, s));
    if (impl == 1) {
      gemm_ref_run(da.p, K, dw.p, dc.p, M, N, K, s);
    } else {
      GemmPlan p;
      GemmEpi e;
      e.mode = EPI_F32;
      e.out = dc.p;
      e.ldo = N;
      gemm_plan(p, da.p, K, dw.p, M, N, K, e, h->num_sms, bn);
      gemm_run(p, s);
    }
    WISB_CUDA(cudaMemcpyAsync(c, dc.p, sizeof(float) * M * N, cudaMemcpyDeviceToHost, s));
    WISB_CUDA(cudaStreamSynchronize(s));
  });
}

int wisb_debug_gemv_tc(wisb_handle* h, const float* x, const uint16_t* w, const float* bias, float* out, int R, int N, int K,
                       int iters, float* avg_us) {
  return guarded(h, [&] {
    WISB_REQUIRE(x && w && out, "NULL pointer");
    cudaStream_t s = h->stream;
    DevBuf<float> dx, db, dout;
    DevBuf<__half> dw;
    dx.ensure(static_cast<size_t>(R) * K);
    dw.ensure(static_cast<size_t>(N) * K);
    db.ensure(static_cast<size_t>(N));
    dout.ensure(static_cast<size_t>(R) * N, true);
    WISB_CUDA(cudaMemcpyAsync(dx.p, x, sizeof(float) * R * K, cudaMemcpyHostToDevice, s));
    WISB_CUDA(cudaMemcpyAsync(dw.p, w, sizeof(__half) * static_cast<size_t>(N) * K, cudaMemcpyHostToDevice, s));
    if (bias) WISB_CUDA(cudaMemcpyAsync(db.p, bias, sizeof(float) * N, cudaMemcpyHostToDevice, s));
    const float us = gemv_tc_debug_run(dx.p, dw.p, bias ? db.p : nullptr, dout.p, R, N, K, h->num_sms, iters, s);
    if (avg_us) *avg_us = us;
    WISB_CUDA(cudaMemcpyAsync(out, dout.p, sizeof(float) * R * N, cudaMemcpyDeviceToHost, s));
    WISB_CUDA(cudaStreamSynchronize(s));
  });
}

int wisb_debug_read_trace(wisb_handle* h, unsigned long long* out, int n) {
  return guarded(h, [&] {
    WISB_REQUIRE(out != nullptr && n > 0 && n <= 2048 + 160 * 264, "trace: at most 2048 + 160 * 264 words");
    h->mega_trace.ensure(2048 + 160 * 264, true);
    WISB_CUDA(cudaMemcpy(out, h->mega_trace.p, sizeof(unsigned long long) * n, cudaMemcpyDeviceToHost));
  });
}

int wisb_debug_encode(wisb_handle* h, const float* mel, int B, float* enc_out, int n_layers) {
  return guarded(h, [&] {
    WISB_REQUIRE(h->blob != nullptr && enc_out != nullptr && B >= 1, "bad arguments");
    const int d = h->dims.d_model;
    cudaStream_t s = h->stream;
    upload_mel(h, mel, B);
    run_encoder(h, B, n_layers, false);
    std::vector<__half> tmp(static_cast<size_t>(B) * T_ENC_PAD * d);
    WISB_CUDA(cudaMemcpyAsync(tmp.data(), h->enc_out.p, tmp.size() * sizeof(__half), cudaMemcpyDeviceToHost, s));
    WISB_CUDA(cudaStreamSynchronize(s));
    for (int b = 0; b < B; ++b)
      for (int t = 0; t < T_ENC; ++t)
        for (int e = 0; e < d; ++e)
          enc_out[(static_cast<size_t>(b) * T_ENC + t) * d + e] = __half2float(tmp[(static_cast<size_t>(b) * T_ENC_PAD + t) * d + e]);
  });
}

int wisb_debug_forced_logits(wisb_handle* h, const float* mel, const int32_t* tokens, int n_tokens, float* logits_out) {
  return guarded(h, [&] {
    const Dims& dm = h->dims;
    WISB_REQUIRE(h->blob != nullptr && tokens != nullptr && logits_out != nullptr && n_tokens >= 1 && n_tokens <= dm.n_text_ctx, "bad arguments");
    cudaStream_t s = h->stream;
    upload_mel(h, mel, 1);
    h->ckv_sw = want_ckv_swizzle(h, 1) ? 1 : 0;
    run_encoder(h, 1, -1, true);
    DecodeCfg c;
    c.u0 = 0; c.n_utt = 1; c.B_total = 1; c.beam = 1; c.prompt_len = n_tokens; c.max_new = 1; c.max_hyp = 1; c.lp = 1.f;
    memcpy(h->pin_i.p + 4, tokens, sizeof(int) * n_tokens);
    WISB_CUDA(cudaMemcpyAsync(h->prompt_dev.p, h->pin_i.p + 4, sizeof(int) * n_tokens, cudaMemcpyHostToDevice, s));
    if (h->decoder_batch == 2) {  // the batched pass, one row: position p of the token list per pass
      ensure_batch(h, MAX_BEAM, n_tokens);
      const size_t head_block = static_cast<size_t>(dm.n_heads) * T_ENC_PAD * HEAD_DIM;
      for (int i = 0; i < dm.n_dec_layers; ++i) {
        h->bd_layers[i].ck = h->ckv.p + static_cast<size_t>(i * 2 + 0) * head_block;
        h->bd_layers[i].cv = h->ckv.p + static_cast<size_t>(i * 2 + 1) * head_block;
      }
      // `debug_chunk` positions per pass (1..8): > 1 feeds consecutive positions as rows of one pass, the way the prompt
      // prefix is prefilled (exercises the multi-row paths of the attention kernels under teacher forcing)
      const int chunk_max = h->debug_chunk < 1 ? 1 : (h->debug_chunk > MAX_BEAM ? MAX_BEAM : h->debug_chunk);
      for (int p = 0; p < n_tokens; p += chunk_max) {
        const int chunk = n_tokens - p < chunk_max ? n_tokens - p : chunk_max;
        prefill_rows_run(h->tokens.p, h->row_pos.p, h->row_slot.p, h->prompt_dev.p, n_tokens, 1, p, chunk, 1, s);
        BatchArgs a = make_batch_args(h, c);
        a.R = chunk;
        a.rows_per_utt = chunk;
        a.prefill = 1;
        a.with_logits = 1;
        batch_pass_run(a, h->bd_layers.data(), dm.n_dec_layers, s);
        WISB_CUDA(cudaMemcpy2DAsync(logits_out + static_cast<size_t>(p) * dm.n_vocab, sizeof(float) * dm.n_vocab, h->blogits.p,
                                    sizeof(float) * dm.n_vocab_pad, sizeof(float) * dm.n_vocab, chunk, cudaMemcpyDeviceToHost, s));
      }
      WISB_CUDA(cudaStreamSynchronize(s));
      return;
    }
    search_init_run(make_search_args(h, c), h->prompt_dev.p, s);
    if (h->decoder_mega) upload_mega_layers(h, c);
    for (int p = 0; p < n_tokens; ++p) {
      enqueue_decoder_forward(h, c, true);
      WISB_CUDA(cudaMemcpyAsync(logits_out + static_cast<size_t>(p) * dm.n_vocab, h->logits.p, sizeof(float) * dm.n_vocab, cudaMemcpyDeviceToHost, s));
      if (p + 1 < n_tokens) prefill_advance_run(h->tokens.p, h->prompt_dev.p, n_tokens, 1, 1, h->st.p, s);
    }
    WISB_CUDA(cudaStreamSynchronize(s));
  });
}

}  // extern "C"
