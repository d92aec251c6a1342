// dcb200 engine: C-ABI implementation (include/dcb200.h) -- configuration, weight packing into
// the device operand images, workspace management and the per-chunk launch sequence.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <functional>
#include <map>
#include <string>
#include <vector>

#include "../../include/dcb200.h"
#include "../../include/dcb200_debug.h"
#include "kernels.h"

#ifndef DCB_FUSE_HEAD_DEFAULT
#define DCB_FUSE_HEAD_DEFAULT 1
#endif

using namespace dcb;

namespace {

thread_local std::string g_create_error;

struct LayerDev {
  __nv_bfloat16* wqkv = nullptr;  // 2 groups x [36][432][8]
  uint8_t* wq3 = nullptr;         // stack kernel: per (head, rank, q|k|v) [36][72][8]
  uint8_t* wqa = nullptr;         // fused QKV+attention: per (head, rank) [36][216][8], rows = q|k|v halves
  __nv_bfloat16* wo = nullptr;    // [36][288][8]
  uint8_t* wffn2 = nullptr;       // CTA-pair image: per (chunk, rank): [36][64][8] then [16][144][8]
  float b2_mean = 0.f;            // mean of b2 over its 280 columns (stack kernel, deferred LayerNorm)
  uint8_t* wffn2s = nullptr;      // the stack kernel's copy: b1 / deferred-LayerNorm terms in the padding rows (common.h, StackParams)
  uint8_t* wo2 = nullptr;         // CTA-pair out-proj image: per rank [36][144][8]
  float* b1 = nullptr;            // [ff]
  float* b2 = nullptr;            // [288] (gain folded)
  float* ln_g[2] = {nullptr, nullptr};  // pre-norm gamma/beta of the attention / FFN sub-layer
  float* ln_b[2] = {nullptr, nullptr};
};

}  // namespace

struct dcb_engine {
  dcb_config cfg{};
  std::string err;
  int R = 0, L = 0, Lw = 0, E = 0, Epad = 0, echunks = 0;   // Lw: tokens per window in the layout (>= L)
  PackedLayout pl{};
  int chunk_tiles = 0, chunk_windows = 0;
  int num_sms = 148;
  cudaStream_t stream = nullptr;        // compute (+ result D2H)
  cudaStream_t copy_stream = nullptr;   // H2D of the rows of the NEXT submission, overlapping the kernels of the current one
  cudaStream_t out_stream = nullptr;    // D2H of the results of the PREVIOUS submission, off the compute stream
  // Two-deep submission pipeline (dcb_submit / dcb_wait): only the input rows and the status word are per slot; every
  // other buffer is reused in stream order.
  struct Slot {
    float* d_rows = nullptr;
    uint8_t* d_packed = nullptr;        // packed rows of a dcb_submit_packed call (allocated on first use)
    uint8_t *d_bases = nullptr, *d_quals = nullptr;   // per slot: the results of batch i are copied out on `out_stream`
    float *d_probs = nullptr, *d_logits = nullptr;    // while the kernels of batch i+1 already write the other slot's
    int* d_status = nullptr;
    int* h_status = nullptr;            // pinned
    cudaEvent_t rows_ready = nullptr, ev0 = nullptr, ev1 = nullptr, done = nullptr;
    bool busy = false, used = false;
    int64_t ticket = -1;
    int launches = 0;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> prof_events;  // around every launch when profiling
    std::vector<int> prof_kind;                                    // kernel class of each event pair
    size_t prof_used = 0;
  } slots[2];
  int64_t next_ticket = 0;
  bool weights_loaded = false;
  bool debug = false;
  bool fuse_oproj = true;
  bool fuse_embed = true;
  bool fuse_qa = true;
  bool fuse_head = DCB_FUSE_HEAD_DEFAULT != 0;   // head in the tail of the stack kernel (one pipelined pass over the row, the
                           // gamma * Wfc table in the idle staging area): +1.7 % against the separate head_kernel, and the
                           // residual image is never written back.  DCB_FUSE_HEAD=0 (developer build): head_kernel
  bool stack = true;   // whole encoder stack in one launch (stack_pair_kernel) when the configuration allows it
  bool fused_last = false;
  bool stack_last = false;
  bool profile = false;
  float prof_ms[6] = {0, 0, 0, 0, 0, 0};   // embed, gemm_row, qkv, attention, ffn(+out-proj), head
  int prof_n[6] = {0, 0, 0, 0, 0, 0};
  float prof_ffn_ms = 0.f;
  int prof_ffn_launches = 0;
  long long prof_ffn_tokens = 0;
  float last_ms = 0.f;
  int last_launches = 0;
  int last_chunk_tokens = 0;
  // model
  EmbedCol* d_cols = nullptr;
  EmbedRow* d_rowmeta = nullptr;
  int table_elems = 0;
  __nv_bfloat16* d_tables = nullptr;
  __nv_bfloat16* d_wc = nullptr;
  float* d_pe = nullptr;
  float* d_pe_img = nullptr;   // same table in residual-image order (window-aligned layout only)
  std::vector<LayerDev> layers;
  float *d_fln_g = nullptr, *d_fln_b = nullptr, *d_wfc = nullptr, *d_bfc = nullptr;
  float *d_head_gw8 = nullptr, *d_head_ab = nullptr;   // head_kernel: gamma * Wfc (padded to 8) and the A / B sums
  // workspace
  __nv_bfloat16* d_embqkv = nullptr;
  float* d_x = nullptr;
  __nv_bfloat16* d_xb = nullptr;
  __nv_bfloat16* d_att = nullptr;
  // stitch scratch (grown on demand)
  uint8_t *d_st_in = nullptr, *d_st_out = nullptr;   // [2][cap] each: bases|quals, seq|qual
  int32_t *d_st_start = nullptr, *d_st_len = nullptr;
  int64_t* d_st_off = nullptr;                        // byte offset of every read (n_zmw + 1)
  size_t st_cap = 0, st_zcap = 0;
  // post-model stage scratch (dcb_stitch_fastq / dcb_skip_mask / dcb_fill_skipped), grown on demand
  double* d_p10 = nullptr;           // 10^(-q/10), q = 0..255 (host libm pow, as NumPy)
  struct Scratch { void* p = nullptr; size_t cap = 0; } sc_pos, sc_names, sc_nameoff, sc_outcome, sc_avg, sc_recoff, sc_fastq,
      sc_bq, sc_mask, sc_ids, sc_dst, sc_tmpb, sc_tmpq;
  float* d_dbg = nullptr;  // [stages][chunk_tiles * x_image]
  // strict-fp32 path (strict_kernels.cu): float32 copies of every variable in the reference's own shapes, and a
  // row-major workspace allocated on the first strict call
  struct StrictLayer {
    float *wq = nullptr, *wk = nullptr, *wv = nullptr, *wo = nullptr, *w1 = nullptr, *b1 = nullptr, *w2 = nullptr, *b2 = nullptr;
    float *ln_g[2] = {nullptr, nullptr}, *ln_b[2] = {nullptr, nullptr};
    float alpha[2] = {1.f, 1.f};
  };
  struct Strict {
    StrictEmbedRow* meta = nullptr;
    float *tables = nullptr, *wc = nullptr, *pe = nullptr;
    float *fln_g = nullptr, *fln_b = nullptr;
    std::vector<StrictLayer> layers;
    float *emb = nullptr, *x = nullptr, *y = nullptr, *q = nullptr, *k = nullptr, *v = nullptr, *att = nullptr, *hid = nullptr;
    int chunk_windows = 0;
  } strict;
  std::vector<void*> owned;
};

namespace {

int fail(dcb_engine* e, int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (e) e->err = buf; else g_create_error = buf;
  return code;
}

#define CU(e, call)                                                                     \
  do {                                                                                  \
    cudaError_t _st = (call);                                                           \
    if (_st != cudaSuccess)                                                             \
      return fail(e, DCB_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_st), \
                  __FILE__, __LINE__);                                                  \
  } while (0)

template <typename T>
int dev_alloc(dcb_engine* e, T** p, size_t n) {
  CU(e, cudaMalloc(reinterpret_cast<void**>(p), n * sizeof(T)));
  CU(e, cudaMemset(*p, 0, n * sizeof(T)));
  e->owned.push_back(*p);
  return DCB_OK;
}

template <typename T>
int upload(dcb_engine* e, T** p, const std::vector<T>& h) {
  int rc = dev_alloc(e, p, h.size());
  if (rc) return rc;
  CU(e, cudaMemcpy(*p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
  return DCB_OK;
}

// B-operand image [K/8][N][8] bf16 from a getter W(k, n) (zero outside the real extents).
std::vector<__nv_bfloat16> pack_b(int kpad, int n, const std::function<float(int, int)>& w) {
  std::vector<__nv_bfloat16> img((size_t)kpad * n);
  for (int kc = 0; kc < kpad / 8; ++kc)
    for (int r = 0; r < n; ++r)
      for (int j = 0; j < 8; ++j)
        img[((size_t)kc * n + r) * 8 + j] = __float2bfloat16(w(kc * 8 + j, r));
  return img;
}

struct TensorMap {
  std::map<std::string, const dcb_tensor*> m;
  dcb_engine* e;
  const float* get(const std::string& name, std::initializer_list<int64_t> shape, int* rc) {
    auto it = m.find(name);
    if (it == m.end()) {
      *rc = fail(e, DCB_ERR_WEIGHTS, "missing variable %s", name.c_str());
      return nullptr;
    }
    const dcb_tensor* t = it->second;
    bool ok = t->ndim == (int)shape.size() && t->data != nullptr;
    int i = 0;
    for (int64_t s : shape) { if (ok && t->shape[i] != s) ok = false; ++i; }
    if (!ok) {
      *rc = fail(e, DCB_ERR_WEIGHTS, "variable %s has the wrong shape/ndim", name.c_str());
      return nullptr;
    }
    return t->data;
  }
};

std::vector<float> pad288(const float* src, float scale = 1.f) {
  std::vector<float> v(kDP, 0.f);
  for (int i = 0; i < kD; ++i) v[i] = src[i] * scale;
  return v;
}

}  // namespace

extern "C" {

const char* dcb_version(void) { return "dcb200 0.1.0 (sm_100a)"; }

const char* dcb_last_error(const dcb_engine* e) { return e ? e->err.c_str() : g_create_error.c_str(); }

int dcb_create(const dcb_config* cfg, dcb_engine** out) {
  if (!cfg || !out) return fail(nullptr, DCB_ERR_INVALID, "null argument");
  if (cfg->struct_size != (int32_t)sizeof(dcb_config))
    return fail(nullptr, DCB_ERR_INVALID, "dcb_config size mismatch: got %d, built with %zu",
                cfg->struct_size, sizeof(dcb_config));
  if (cfg->hidden_size != kD || cfg->num_heads != kHeads)
    return fail(nullptr, DCB_ERR_INVALID, "unsupported model: hidden_size=%d num_heads=%d (engine is built for %d/%d)",
                cfg->hidden_size, cfg->num_heads, kD, kHeads);
  if (!cfg->condense_transformer_input)
    return fail(nullptr, DCB_ERR_INVALID, "condense_transformer_input must be true");
  if (cfg->filter_size <= 0 || cfg->filter_size % kFFChunk || cfg->filter_size > 2048)
    return fail(nullptr, DCB_ERR_INVALID, "filter_size must be a multiple of %d and <= 2048", kFFChunk);
  if (cfg->max_passes <= 0 || cfg->max_length <= 0 || cfg->max_length > 256 || cfg->num_hidden_layers <= 0 ||
      cfg->max_batch <= 0)
    return fail(nullptr, DCB_ERR_INVALID, "bad max_passes/max_length(<=256)/num_hidden_layers/max_batch");
  if (cfg->precision != DCB_PRECISION_BF16 && cfg->precision != DCB_PRECISION_FP32)
    return fail(nullptr, DCB_ERR_INVALID, "precision must be DCB_PRECISION_BF16 or DCB_PRECISION_FP32");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(nullptr, DCB_ERR_CUDA, "no CUDA device available (the dcb200 engine has no CPU fallback)");
  if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, DCB_ERR_INVALID, "bad device ordinal %d", cfg->device);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, cfg->device) != cudaSuccess || prop.major != 10)
    return fail(nullptr, DCB_ERR_CUDA, "device %d is not an sm_100 GPU (compute capability %d.%d)", cfg->device,
                prop.major, prop.minor);

  dcb_engine* e = new dcb_engine();
  e->cfg = *cfg;
  e->num_sms = prop.multiProcessorCount;
  e->L = cfg->max_length;
  e->Lw = e->L;
  bool align = true;
  int ct = cfg->chunk_tiles;
#ifdef DCB_DEV_SWITCHES
  // Developer build only (libdcb200_dev.so, csrc/build.sh): environment switches that select the measured
  // alternative kernel paths.  The product library ignores the environment.
  if (const char* env = getenv("DCB_ALIGN")) align = atoi(env) != 0;
  if (const char* env = getenv("DCB_FUSE_OPROJ")) e->fuse_oproj = atoi(env) != 0;
  if (const char* env = getenv("DCB_FUSE_EMBED")) e->fuse_embed = atoi(env) != 0;
  if (const char* env = getenv("DCB_FUSE_QA")) e->fuse_qa = atoi(env) != 0;
  if (const char* env = getenv("DCB_STACK")) e->stack = atoi(env) != 0;
  if (const char* env = getenv("DCB_FUSE_HEAD")) e->fuse_head = atoi(env) != 0;
  if (const char* env = getenv("DCB_CHUNK_TILES")) ct = atoi(env);
#endif
  // window-aligned tiling: one window per 128-token tile when it fits (lets QKV + attention fuse);
  // otherwise windows are packed back to back
  if (align && e->L <= kTileM) e->Lw = kTileM;
  // 128 < L <= 256: one window per tile PAIR, so that the one-kernel stack (a CTA pair per window, attention halo
  // across the pair) applies -- when the rest of its conditions hold
  else if (align && e->L <= 2 * kTileM && e->stack && cfg->attn_win_size > 0 && cfg->attn_win_size <= 16 &&
           cfg->num_hidden_layers <= kMaxLayers)
    e->Lw = 2 * kTileM;
  e->R = 4 * cfg->max_passes + (cfg->use_ccs_bq ? 6 : 5);  // data_providers.py:61-78
  e->pl = make_packed_layout(cfg->max_passes, cfg->max_length, cfg->use_ccs_bq ? 1 : 0);
  e->E = cfg->max_passes * (cfg->per_base_hidden_size + cfg->pw_hidden_size + cfg->ip_hidden_size +
                            cfg->strand_hidden_size) +
         cfg->per_base_hidden_size + (cfg->use_ccs_bq ? cfg->ccs_bq_hidden_size : 0) +
         4 * cfg->sn_hidden_size;
  e->Epad = (e->E + 15) / 16 * 16;
  e->echunks = e->Epad / 8;
  if (ct <= 0) ct = 8 * e->num_sms;   // measured: larger chunks win (kernels are not DRAM-bound)
  const int max_tiles = (int)(((int64_t)cfg->max_batch * e->Lw + kTileM - 1) / kTileM);
  e->chunk_windows = std::max(1, std::min(cfg->max_batch, ct * kTileM / e->Lw));
  e->chunk_tiles = std::min(max_tiles, (e->chunk_windows * e->Lw + kTileM - 1) / kTileM);

  auto bail = [&](int rc) { std::string m = e->err; dcb_destroy(e); g_create_error = m; return rc; };
#define TRY(x) do { int _rc = (x); if (_rc) return bail(_rc); } while (0)
#define CUC(call) do { cudaError_t _s = (call); if (_s != cudaSuccess) { fail(e, DCB_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(_s)); return bail(DCB_ERR_CUDA); } } while (0)
  CUC(cudaSetDevice(cfg->device));
  CUC(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
  CUC(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
  CUC(cudaStreamCreateWithFlags(&e->out_stream, cudaStreamNonBlocking));
  for (auto& sl : e->slots) {
    CUC(cudaEventCreateWithFlags(&sl.rows_ready, cudaEventDisableTiming));
    CUC(cudaEventCreate(&sl.ev0));
    CUC(cudaEventCreate(&sl.ev1));
    CUC(cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming));
    CUC(cudaMallocHost(reinterpret_cast<void**>(&sl.h_status), sizeof(int)));
  }
  CUC(kernels_init());
  {
    std::vector<double> p10(256);
    for (int q = 0; q < 256; ++q) p10[q] = pow(10.0, (double)q / -10.0);    // utils.py:103: 10 ** (q / -10.0)
    TRY(upload(e, &e->d_p10, p10));
  }
  const size_t T = e->chunk_tiles;
  for (auto& sl : e->slots) {
    TRY(dev_alloc(e, &sl.d_rows, (size_t)cfg->max_batch * e->R * e->L));
    TRY(dev_alloc(e, &sl.d_status, 1));
  }
  TRY(dev_alloc(e, &e->d_embqkv, T * kTileM * (size_t)std::max(e->Epad, kQKVN)));
  TRY(dev_alloc(e, &e->d_x, T * x_image_elems()));
  TRY(dev_alloc(e, &e->d_xb, T * act_image_elems(kDP)));
  TRY(dev_alloc(e, &e->d_att, T * act_image_elems(kDP)));
  const size_t mtok = (size_t)cfg->max_batch * e->L;
  for (auto& sl : e->slots) {
    TRY(dev_alloc(e, &sl.d_bases, mtok));
    TRY(dev_alloc(e, &sl.d_quals, mtok));
  }
#undef TRY
#undef CUC
  *out = e;
  return DCB_OK;
}

void dcb_destroy(dcb_engine* e) {
  if (!e) return;
  cudaSetDevice(e->cfg.device);
  if (e->copy_stream) cudaStreamSynchronize(e->copy_stream);
  if (e->stream) cudaStreamSynchronize(e->stream);
  if (e->out_stream) cudaStreamSynchronize(e->out_stream);
  for (void* p : e->owned) cudaFree(p);
  if (e->d_st_in) cudaFree(e->d_st_in);
  if (e->d_st_out) cudaFree(e->d_st_out);
  if (e->d_st_start) cudaFree(e->d_st_start);
  if (e->d_st_len) cudaFree(e->d_st_len);
  if (e->d_st_off) cudaFree(e->d_st_off);
  for (dcb_engine::Scratch* sc : {&e->sc_pos, &e->sc_names, &e->sc_nameoff, &e->sc_outcome, &e->sc_avg, &e->sc_recoff,
                                  &e->sc_fastq, &e->sc_bq, &e->sc_mask, &e->sc_ids, &e->sc_dst, &e->sc_tmpb, &e->sc_tmpq})
    if (sc->p) cudaFree(sc->p);
  for (auto& sl : e->slots)
    for (auto& pr : sl.prof_events) { cudaEventDestroy(pr.first); cudaEventDestroy(pr.second); }
  if (e->copy_stream) cudaStreamSynchronize(e->copy_stream);
  for (auto& sl : e->slots) {
    if (sl.rows_ready) cudaEventDestroy(sl.rows_ready);
    if (sl.ev0) cudaEventDestroy(sl.ev0);
    if (sl.ev1) cudaEventDestroy(sl.ev1);
    if (sl.done) cudaEventDestroy(sl.done);
    if (sl.h_status) cudaFreeHost(sl.h_status);
  }
  if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
  if (e->out_stream) cudaStreamDestroy(e->out_stream);
  if (e->stream) cudaStreamDestroy(e->stream);
  delete e;
}

int dcb_load_weights(dcb_engine* e, const dcb_tensor* tensors, int32_t n) {
  if (!e || !tensors) return fail(e, DCB_ERR_INVALID, "null argument");
  CU(e, cudaSetDevice(e->cfg.device));
  const dcb_config& c = e->cfg;
  TensorMap tm;
  tm.e = e;
  for (int i = 0; i < n; ++i)
    if (tensors[i].name) tm.m[tensors[i].name] = &tensors[i];
  int rc = DCB_OK;

  // ---- embedding tables (networks.py:375-421), pre-scaled by sqrt(width), row 0 zeroed
  //      (ModifiedOnDeviceEmbedding, networks.py:42-63)
  struct Tab { const char* layer; int vocab, width; int off; const float* data; };
  std::vector<Tab> tabs = {
      {"bases_embedding_layer", kVocab, c.per_base_hidden_size, 0, nullptr},
      {"pw_embedding_layer", c.pw_max + 1, c.pw_hidden_size, 0, nullptr},
      {"ip_embedding_layer", c.ip_max + 1, c.ip_hidden_size, 0, nullptr},
      {"strand_embedding_layer", c.strand_max + 1, c.strand_hidden_size, 0, nullptr},
      {"ccs_base_quality_scores_embedding_layer", c.ccs_bq_max, c.ccs_bq_hidden_size, 0, nullptr},
      {"sn_embedding_layer", c.sn_max + 1, c.sn_hidden_size, 0, nullptr},
  };
  std::vector<__nv_bfloat16> blob;
  for (size_t t = 0; t < tabs.size(); ++t) {
    if (t == 4 && !c.use_ccs_bq) continue;
    Tab& tb = tabs[t];
    tb.data = tm.get(std::string("model/") + tb.layer + "/embeddings", {tb.vocab, tb.width}, &rc);
    if (rc) return rc;
    while (blob.size() % 8) blob.push_back(__float2bfloat16(0.f));   // 16-byte aligned table rows (width-8 fast path)
    tb.off = (int)blob.size();
    const float scale = sqrtf((float)tb.width);
    for (int v = 0; v < tb.vocab; ++v)
      for (int j = 0; j < tb.width; ++j)
        blob.push_back(__float2bfloat16(v == 0 ? 0.f : tb.data[v * tb.width + j] * scale));
  }
  // ---- per-column gather descriptors in concat order (networks.py:457-506)
  std::vector<EmbedCol> cols(e->Epad);
  for (auto& cc : cols) { cc = EmbedCol{}; cc.src_row = -1; }
  {
    const int P = c.max_passes;
    int eoff = 0;
    auto add_rows = [&](int tab, int row0, int nrows, float clip, int shift) {
      for (int r = 0; r < nrows; ++r)
        for (int j = 0; j < tabs[tab].width; ++j) {
          EmbedCol& cc = cols[eoff++];
          cc.src_row = (int16_t)(row0 + r);
          cc.width = (int16_t)tabs[tab].width;
          cc.col = (int16_t)j;
          cc.shift = (int16_t)shift;
          cc.table_off = tabs[tab].off;
          cc.vocab = tabs[tab].vocab;
          cc.clip_hi = clip;
        }
    };
    add_rows(0, 0, P, 0.f, 0);                                  // bases
    add_rows(1, P, P, (float)c.pw_max, 0);                      // pw   (clip: data_providers.py:151-154)
    add_rows(2, 2 * P, P, (float)c.ip_max, 0);                  // ip   (:155-158)
    add_rows(3, 3 * P, P, 0.f, 0);                              // strand
    add_rows(0, 4 * P, 1, 0.f, 0);                              // ccs shares the bases table (networks.py:485-489)
    int next = 4 * P + 1;
    if (c.use_ccs_bq) { add_rows(4, next, 1, 0.f, 1); ++next; }  // +1 shift (networks.py:495)
    add_rows(5, next, 4, (float)c.sn_max, 0);                   // sn   (:159-162)
    if (eoff != e->E) return fail(e, DCB_ERR_INVALID, "internal: embedding width %d != %d", eoff, e->E);
  }
  {
    std::vector<EmbedRow> meta(e->R, EmbedRow{0.f, 0, 1});
    for (const EmbedCol& cc : cols)
      if (cc.src_row >= 0) meta[cc.src_row] = EmbedRow{cc.clip_hi, cc.shift, cc.vocab};
    if ((rc = upload(e, &e->d_rowmeta, meta))) return rc;
    e->table_elems = (int)blob.size();
    if (embed_smem_bytes(e->R, e->echunks, e->table_elems) > 160 * 1024)
      return fail(e, DCB_ERR_INVALID, "embedding tables + ids do not fit the embed kernel's shared memory");
  }
  if ((rc = upload(e, &e->d_tables, blob))) return rc;
  if ((rc = upload(e, &e->d_cols, cols))) return rc;

  // ---- condenser (networks.py:426-434): B image [Epad/8][288][8]
  {
    const float* wc = tm.get("model/transformer_input_condenser/kernel", {e->E, kD}, &rc);
    if (rc) return rc;
    const int E = e->E;
    auto img = pack_b(e->Epad, kDP, [&](int k, int nn) { return (k < E && nn < kD) ? wc[(size_t)k * kD + nn] : 0.f; });
    if ((rc = upload(e, &e->d_wc, img))) return rc;
  }
  // ---- positional encoding table [L][288] (tf-models RelativePositionEmbedding; networks.py:301-323)
  {
    std::vector<float> pe((size_t)e->Lw * kDP, 0.f);
    if (c.add_pos_encoding) {
      const int nt = kD / 2;
      const float inc = (float)(log(1e4 / 1.0) / (double)(nt - 1));
      for (int l = 0; l < e->L; ++l)
        for (int k = 0; k < nt; ++k) {
          const float inv = expf((float)k * -inc);
          const float sc = (float)l * inv;
          pe[(size_t)l * kDP + k] = sinf(sc);
          pe[(size_t)l * kDP + nt + k] = cosf(sc);
        }
    }
    if ((rc = upload(e, &e->d_pe, pe))) return rc;
    if (e->Lw == kTileM) {
      // window-aligned layout: every tile sees positions 0..127, so the table can also be laid out like the residual
      // image [72][128][4] -- a warp of the row epilogue then reads 512 contiguous bytes instead of 32 scattered rows
      std::vector<float> img((size_t)kTileM * kDP, 0.f);
      for (int l = 0; l < kTileM; ++l)
        for (int col = 0; col < kDP; ++col) img[((size_t)(col / 4) * kTileM + l) * 4 + (col & 3)] = pe[(size_t)l * kDP + col];
      if ((rc = upload(e, &e->d_pe_img, img))) return rc;
    }
  }
  // ---- encoder layers
  const int ff = c.filter_size;
  e->layers.assign(c.num_hidden_layers, LayerDev());
  std::vector<float> last_b2(kD, 0.f);   // output bias of the last layer's FFN (ReZero gain folded in), for the fused head
  for (int n_ = 0; n_ < c.num_hidden_layers; ++n_) {
    LayerDev& ld = e->layers[n_];
    char pre[128];
    snprintf(pre, sizeof pre, "model/encoder_stack/layers/%d", n_);
    const std::string P0 = std::string(pre) + "/0", P1 = std::string(pre) + "/1";
    float alpha0 = 1.f, alpha1 = 1.f;
    const float *gam[2] = {nullptr, nullptr}, *bet[2] = {nullptr, nullptr};   // pre-LN gamma / beta of the two sub-layers
    // Padding rows 280..287 of a stack-kernel [kDP/8][n][8] image (common.h, StackParams).  beta != null: deferred
    // LayerNorm, rows 0..279 hold bf16(gamma * W), wcol(k, nn) = the unfolded weight, extra(nn) = a bias that joins
    // beta^T W.  beta == null (ReZero): only the bias rows.
    auto deferred_rows = [&](std::vector<__nv_bfloat16>& part, int n, const float* beta,
                             const std::function<float(int, int)>& wcol, const std::function<float(int)>& extra) {
      for (int nn = 0; nn < n; ++nn) {
        float cs = 0.f, bw = extra(nn);
        for (int k = 0; beta && k < kD; ++k) {
          cs += __bfloat162float(part[((size_t)(k / 8) * n + nn) * 8 + k % 8]);
          bw += beta[k] * wcol(k, nn);
        }
        const __nv_bfloat16 ch = __float2bfloat16(cs), cl = __float2bfloat16(cs - __bfloat162float(ch));
        const __nv_bfloat16 bh = __float2bfloat16(bw), bl = __float2bfloat16(bw - __bfloat162float(bh));
        __nv_bfloat16* row = &part[((size_t)(kD / 8) * n + nn) * 8];
        row[0] = ch; row[1] = cl; row[2] = ch; row[3] = cl;
        row[4] = bh; row[5] = bl; row[6] = bh; row[7] = bl;
      }
    };
    static_assert(kDP - kD == 8 && kD % 8 == 0, "deferred LayerNorm uses the eight padding rows of the operand tile");
    if (c.rezero) {
      const float* a0 = tm.get(P0 + "/alpha", std::initializer_list<int64_t>{}, &rc); if (rc) return rc;
      const float* a1 = tm.get(P1 + "/alpha", std::initializer_list<int64_t>{}, &rc); if (rc) return rc;
      alpha0 = *a0; alpha1 = *a1;
    } else {
      for (int s = 0; s < 2; ++s) {
        const std::string P = s ? P1 : P0;
        const float* g = tm.get(P + "/layer_norm/gamma", {kD}, &rc); if (rc) return rc;
        const float* b = tm.get(P + "/layer_norm/beta", {kD}, &rc); if (rc) return rc;
        gam[s] = g; bet[s] = b;
        if ((rc = upload(e, &ld.ln_g[s], pad288(g)))) return rc;
        if ((rc = upload(e, &ld.ln_b[s], pad288(b)))) return rc;
      }
    }
    const float* wq = tm.get(P0 + "/layer/query_dense_layer/kernel", {kD, kHeads, kDH}, &rc); if (rc) return rc;
    const float* wk = tm.get(P0 + "/layer/key_dense_layer/kernel", {kD, kHeads, kDH}, &rc); if (rc) return rc;
    const float* wv = tm.get(P0 + "/layer/value_dense_layer/kernel", {kD, kHeads, kDH}, &rc); if (rc) return rc;
    const float* wo = tm.get(P0 + "/layer/output_dense_layer/kernel", {kHeads, kDH, kD}, &rc); if (rc) return rc;
    const float qscale = 1.0f / sqrtf((float)kDH);  // query *= depth**-0.5 (attention_layer.py:196-197)
    {
      // two n-groups of 432 columns: [q_h0 q_h1 k_h0 | k_h1 v_h0 v_h1], each slot 144 wide (140 + 4 zero)
      std::vector<__nv_bfloat16> img;
      for (int grp = 0; grp < 2; ++grp) {
        auto part = pack_b(kDP, 3 * kNC, [&](int k, int nn) {
          const int colg = grp * 3 * kNC + nn;
          const int slot = colg / kDHP, dd = colg % kDHP;
          if (k >= kD || dd >= kDH) return 0.f;
          const int proj = slot / kHeads, head = slot % kHeads;
          const float* w = proj == 0 ? wq : (proj == 1 ? wk : wv);
          const float v = w[((size_t)k * kHeads + head) * kDH + dd];
          return proj == 0 ? v * qscale : v;
        });
        img.insert(img.end(), part.begin(), part.end());
      }
      if ((rc = upload(e, &ld.wqkv, img))) return rc;
      // fused QKV + attention (CTA pairs): for head h and rank rk the 216 rows of a k-step are
      // [q_h | k_h | v_h], each the rk-th half (72 columns) of that 144-wide matrix
      std::vector<__nv_bfloat16> imga;
      for (int h = 0; h < kHeads; ++h)
        for (int rk = 0; rk < 2; ++rk) {
          auto part = pack_b(kDP, 3 * (kDHP / 2), [&](int k, int nn) {
            const int m = nn / (kDHP / 2), dd = rk * (kDHP / 2) + nn % (kDHP / 2);
            if (k >= kD || dd >= kDH) return 0.f;
            const float* w = m == 0 ? wq : (m == 1 ? wk : wv);
            const float v = w[((size_t)k * kHeads + h) * kDH + dd];
            return m == 0 ? v * qscale : v;
          });
          imga.insert(imga.end(), part.begin(), part.end());
        }
      __nv_bfloat16* dptr2 = nullptr;
      if ((rc = upload(e, &dptr2, imga))) return rc;
      ld.wqa = reinterpret_cast<uint8_t*>(dptr2);
      // stack kernel: one [36][72][8] block per (head, rank, q|k|v), consumed as three 6-k-step stages
      std::vector<__nv_bfloat16> img3;
      for (int h = 0; h < kHeads; ++h)
        for (int rk = 0; rk < 2; ++rk)
          for (int m = 0; m < 3; ++m) {
            auto wval = [&](int k, int nn) {
              const int dd = rk * (kDHP / 2) + nn;
              if (k >= kD || dd >= kDH) return 0.f;
              const float* w = m == 0 ? wq : (m == 1 ? wk : wv);
              const float v = w[((size_t)k * kHeads + h) * kDH + dd];
              return m == 0 ? v * qscale : v;
            };
            auto part = pack_b(kDP, kDHP / 2, [&](int k, int nn) {
              return (gam[0] && k < kD) ? gam[0][k] * wval(k, nn) : wval(k, nn);     // pre-LN: gamma_0 folded into the rows
            });
            if (gam[0]) deferred_rows(part, kDHP / 2, bet[0], wval, [](int) { return 0.f; });
            img3.insert(img3.end(), part.begin(), part.end());
          }
      __nv_bfloat16* dptr3 = nullptr;
      if ((rc = upload(e, &dptr3, img3))) return rc;
      ld.wq3 = reinterpret_cast<uint8_t*>(dptr3);
    }
    {
      // out-proj: K index = head*144 + dd, N = e; ReZero alpha folded in (encoder_stack.py:88-90)
      auto img = pack_b(kDP, kDP, [&](int k, int nn) {
        const int head = k / kDHP, dd = k % kDHP;
        if (dd >= kDH || nn >= kD) return 0.f;
        return wo[((size_t)head * kDH + dd) * kD + nn] * alpha0;
      });
      if ((rc = upload(e, &ld.wo, img))) return rc;
      // CTA-pair halves: rank r holds, for each 144-wide N chunk j, output rows j*144 + r*72 + [0,72)
      std::vector<__nv_bfloat16> img2;
      for (int rk = 0; rk < 2; ++rk) {
        auto part = pack_b(kDP, kDP / 2, [&](int k, int nn) {
          const int col = (nn / (kNC / 2)) * kNC + rk * (kNC / 2) + nn % (kNC / 2);
          const int head = k / kDHP, dd = k % kDHP;
          if (dd >= kDH || col >= kD) return 0.f;
          return wo[((size_t)head * kDH + dd) * kD + col] * alpha0;
        });
        img2.insert(img2.end(), part.begin(), part.end());
      }
      __nv_bfloat16* dptr = nullptr;
      if ((rc = upload(e, &dptr, img2))) return rc;
      ld.wo2 = reinterpret_cast<uint8_t*>(dptr);
    }
    const float* w1 = tm.get(P1 + "/layer/filter_dense_layer/kernel", {kD, ff}, &rc); if (rc) return rc;
    const float* b1 = tm.get(P1 + "/layer/filter_dense_layer/bias", {ff}, &rc); if (rc) return rc;
    const float* w2 = tm.get(P1 + "/layer/output_dense_layer/kernel", {ff, kD}, &rc); if (rc) return rc;
    const float* b2 = tm.get(P1 + "/layer/output_dense_layer/bias", {kD}, &rc); if (rc) return rc;
    {
      // CTA-pair image: rank r holds hidden units c*128 + r*64 + [0,64) of W1 and, for each 144-wide
      // N chunk j of W2, output rows j*144 + r*72 + [0,72)
      std::vector<__nv_bfloat16> img;
      img.reserve((size_t)ff * kDP * 2);
      for (int ch = 0; ch < ff / kFFChunk; ++ch)
        for (int rk = 0; rk < 2; ++rk) {
          auto p1 = pack_b(kDP, kFFChunk / 2, [&](int k, int nn) {
            return k < kD ? w1[(size_t)k * ff + ch * kFFChunk + rk * (kFFChunk / 2) + nn] : 0.f;
          });
          auto p2 = pack_b(kFFChunk, kDP / 2, [&](int k, int nn) {
            const int col = (nn / (kNC / 2)) * kNC + rk * (kNC / 2) + nn % (kNC / 2);
            return col < kD ? w2[(size_t)(ch * kFFChunk + k) * kD + col] * alpha1 : 0.f;
          });
          img.insert(img.end(), p1.begin(), p1.end());
          img.insert(img.end(), p2.begin(), p2.end());
        }
      __nv_bfloat16* dptr = nullptr;
      if ((rc = upload(e, &dptr, img))) return rc;
      ld.wffn2 = reinterpret_cast<uint8_t*>(dptr);
      {
        // the stack kernel's copy: b1 in the padding rows of W1; pre-LN models: gamma_1 folded in, deferred-LayerNorm rows
        std::vector<__nv_bfloat16> imgs;
        imgs.reserve(img.size());
        for (int ch = 0; ch < ff / kFFChunk; ++ch)
          for (int rk = 0; rk < 2; ++rk) {
            const int c0 = ch * kFFChunk + rk * (kFFChunk / 2);
            auto w1col = [&](int k, int nn) { return k < kD ? w1[(size_t)k * ff + c0 + nn] : 0.f; };
            auto p1 = pack_b(kDP, kFFChunk / 2, [&](int k, int nn) { return (gam[1] && k < kD) ? gam[1][k] * w1col(k, nn) : w1col(k, nn); });
            deferred_rows(p1, kFFChunk / 2, bet[1], w1col, [&](int nn) { return b1[c0 + nn]; });
            auto p2 = pack_b(kFFChunk, kDP / 2, [&](int k, int nn) {
              const int col = (nn / (kNC / 2)) * kNC + rk * (kNC / 2) + nn % (kNC / 2);
              return col < kD ? w2[(size_t)(ch * kFFChunk + k) * kD + col] * alpha1 : 0.f;
            });
            imgs.insert(imgs.end(), p1.begin(), p1.end());
            imgs.insert(imgs.end(), p2.begin(), p2.end());
          }
        __nv_bfloat16* dps = nullptr;
        if ((rc = upload(e, &dps, imgs))) return rc;
        ld.wffn2s = reinterpret_cast<uint8_t*>(dps);
      }
    }
    if ((rc = upload(e, &ld.b1, std::vector<float>(b1, b1 + ff)))) return rc;
    if ((rc = upload(e, &ld.b2, pad288(b2, alpha1)))) return rc;
    last_b2.assign(kD, 0.f);
    for (int k = 0; k < kD; ++k) last_b2[k] = b2[k] * alpha1;      // what the stack kernel adds to Y after this layer
    ld.b2_mean = 0.f;
    for (int k = 0; k < kD; ++k) ld.b2_mean += last_b2[k];
    ld.b2_mean /= (float)kD;
  }
  // ---- head
  {
    const float* g = tm.get("model/encoder_stack/output_normalization/gamma", {kD}, &rc); if (rc) return rc;
    const float* b = tm.get("model/encoder_stack/output_normalization/beta", {kD}, &rc); if (rc) return rc;
    const float* w = tm.get("model/fc1/kernel", {kD, kVocab}, &rc); if (rc) return rc;
    const float* bb = tm.get("model/fc1/bias", {kVocab}, &rc); if (rc) return rc;
    if ((rc = upload(e, &e->d_fln_g, pad288(g)))) return rc;
    if ((rc = upload(e, &e->d_fln_b, pad288(b)))) return rc;
    if ((rc = upload(e, &e->d_wfc, std::vector<float>(w, w + kD * kVocab)))) return rc;
    if ((rc = upload(e, &e->d_bfc, std::vector<float>(bb, bb + kVocab)))) return rc;
    // head_kernel folds the final LayerNorm into the fc1 sums (one pass over the row): logits_j = rstd * (sum_c y_c g_c W_cj
    // - mean_y * A_j) + B_j + bfc_j.  The products are formed here once, in float32 in the same order the kernel used to.
    // The fused tail of the stack kernel works on Y = x - b2 (b2 of the last layer joins here): column 5 of the table and
    // H_j, sum b2, sum b2^2 carry it (stack_kernel.cuh, fused head).
    std::vector<float> gw8((size_t)kD * 8, 0.f), ab(32, 0.f);
    for (int cc = 0; cc < kD; ++cc) {
      for (int j = 0; j < kVocab; ++j) gw8[(size_t)cc * 8 + j] = g[cc] * w[cc * kVocab + j];
      gw8[(size_t)cc * 8 + 5] = last_b2[cc];
    }
    for (int j = 0; j < kVocab; ++j) {
      float a = 0.f, bsum = 0.f, h = 0.f;
      for (int cc = 0; cc < kD; ++cc) {
        a += g[cc] * w[cc * kVocab + j]; bsum += b[cc] * w[cc * kVocab + j];
        h += last_b2[cc] * (g[cc] * w[cc * kVocab + j]);
      }
      ab[j] = a; ab[8 + j] = bsum; ab[16 + j] = h;
    }
    for (int cc = 0; cc < kD; ++cc) { ab[24] += last_b2[cc]; ab[25] += last_b2[cc] * last_b2[cc]; }
    if ((rc = upload(e, &e->d_head_gw8, gw8))) return rc;
    if ((rc = upload(e, &e->d_head_ab, ab))) return rc;
  }
  // ---- strict-fp32 path: every variable once more as float32, in the reference's own shapes
  {
    dcb_engine::Strict& S = e->strict;
    std::vector<float> fblob;
    std::vector<int> foff(tabs.size(), 0);
    for (size_t t = 0; t < tabs.size(); ++t) {
      if (t == 4 && !c.use_ccs_bq) continue;
      const Tab& tb = tabs[t];
      foff[t] = (int)fblob.size();
      const float scale = sqrtf((float)tb.width);          // networks.py:54
      for (int v = 0; v < tb.vocab; ++v)
        for (int j = 0; j < tb.width; ++j) fblob.push_back(v == 0 ? 0.f : tb.data[v * tb.width + j] * scale);   // :58-63
    }
    std::vector<StrictEmbedRow> meta(e->R);
    {
      const int P = c.max_passes;
      int col = 0, row = 0;
      auto add = [&](int tab, int nrows, float clip, int shift) {
        for (int r = 0; r < nrows; ++r) {
          meta[row++] = StrictEmbedRow{clip, shift, tabs[tab].vocab, tabs[tab].width, col, foff[tab]};
          col += tabs[tab].width;
        }
      };
      add(0, P, 0.f, 0); add(1, P, (float)c.pw_max, 0); add(2, P, (float)c.ip_max, 0); add(3, P, 0.f, 0);
      add(0, 1, 0.f, 0);
      if (c.use_ccs_bq) add(4, 1, 0.f, 1);
      add(5, 4, (float)c.sn_max, 0);
      if (row != e->R || col != e->E) return fail(e, DCB_ERR_INVALID, "internal: strict embedding layout %d/%d", row, col);
    }
    if ((rc = upload(e, &S.meta, meta))) return rc;
    if ((rc = upload(e, &S.tables, fblob))) return rc;
    const float* wc = tm.get("model/transformer_input_condenser/kernel", {e->E, kD}, &rc); if (rc) return rc;
    if ((rc = upload(e, &S.wc, std::vector<float>(wc, wc + (size_t)e->E * kD)))) return rc;
    {
      std::vector<float> pe((size_t)e->L * kD, 0.f);
      if (c.add_pos_encoding) {
        const int nt = kD / 2;
        const float inc = (float)(log(1e4 / 1.0) / (double)(nt - 1));
        for (int l = 0; l < e->L; ++l)
          for (int k = 0; k < nt; ++k) {
            const float sc = (float)l * expf((float)k * -inc);
            pe[(size_t)l * kD + k] = sinf(sc);
            pe[(size_t)l * kD + nt + k] = cosf(sc);
          }
      }
      if ((rc = upload(e, &S.pe, pe))) return rc;
    }
    S.layers.assign(c.num_hidden_layers, dcb_engine::StrictLayer());
    for (int n_ = 0; n_ < c.num_hidden_layers; ++n_) {
      dcb_engine::StrictLayer& sl = S.layers[n_];
      char pre[128];
      snprintf(pre, sizeof pre, "model/encoder_stack/layers/%d", n_);
      const std::string P0 = std::string(pre) + "/0", P1 = std::string(pre) + "/1";
      auto up = [&](float** dst, const std::string& name, std::initializer_list<int64_t> shape, size_t count) {
        const float* src = tm.get(name, shape, &rc);
        if (rc) return rc;
        return rc = upload(e, dst, std::vector<float>(src, src + count));
      };
      if (c.rezero) {
        sl.alpha[0] = *tm.get(P0 + "/alpha", std::initializer_list<int64_t>{}, &rc); if (rc) return rc;
        sl.alpha[1] = *tm.get(P1 + "/alpha", std::initializer_list<int64_t>{}, &rc); if (rc) return rc;
      } else {
        for (int sidx = 0; sidx < 2; ++sidx) {
          const std::string PP = sidx ? P1 : P0;
          if (up(&sl.ln_g[sidx], PP + "/layer_norm/gamma", {kD}, kD)) return rc;
          if (up(&sl.ln_b[sidx], PP + "/layer_norm/beta", {kD}, kD)) return rc;
        }
      }
      if (up(&sl.wq, P0 + "/layer/query_dense_layer/kernel", {kD, kHeads, kDH}, (size_t)kD * kD)) return rc;
      if (up(&sl.wk, P0 + "/layer/key_dense_layer/kernel", {kD, kHeads, kDH}, (size_t)kD * kD)) return rc;
      if (up(&sl.wv, P0 + "/layer/value_dense_layer/kernel", {kD, kHeads, kDH}, (size_t)kD * kD)) return rc;
      if (up(&sl.wo, P0 + "/layer/output_dense_layer/kernel", {kHeads, kDH, kD}, (size_t)kD * kD)) return rc;
      if (up(&sl.w1, P1 + "/layer/filter_dense_layer/kernel", {kD, ff}, (size_t)kD * ff)) return rc;
      if (up(&sl.b1, P1 + "/layer/filter_dense_layer/bias", {ff}, (size_t)ff)) return rc;
      if (up(&sl.w2, P1 + "/layer/output_dense_layer/kernel", {ff, kD}, (size_t)ff * kD)) return rc;
      if (up(&sl.b2, P1 + "/layer/output_dense_layer/bias", {kD}, (size_t)kD)) return rc;
    }
  }
  CU(e, cudaDeviceSynchronize());
  e->weights_loaded = true;
  return DCB_OK;
}

// One chunk of the strict-fp32 forward (strict_kernels.cu): rows [bw, R, L] -> outputs via hp.  Returns launches.
static int strict_forward_chunk(dcb_engine* e, const float* rows_chunk, int bw, const HeadParams& hp, int* d_status,
                                cudaStream_t st) {
  const dcb_config& c = e->cfg;
  dcb_engine::Strict& S = e->strict;
  const int L = e->L, M = bw * L, ff = c.filter_size;
  int launches = 0;
  launch_strict_embed(rows_chunk, e->R, L, e->E, bw, S.meta, S.tables, S.emb, d_status, st); ++launches;
  {
    StrictEpi ep;
    if (c.add_pos_encoding) { ep.pe = S.pe; ep.pe_L = L; }
    launch_strict_gemm(S.emb, S.wc, S.x, M, kD, e->E, ep, st); ++launches;            // networks.py:509-516, :319-323
  }
  const float qscale = 1.0f / sqrtf((float)kDH);                                       // attention_layer.py:196-197
  for (int n_ = 0; n_ < c.num_hidden_layers; ++n_) {
    const dcb_engine::StrictLayer& sl = S.layers[n_];
    const float* yin = S.x;
    if (!c.rezero) { launch_strict_layernorm(S.x, S.y, M, sl.ln_g[0], sl.ln_b[0], st); ++launches; yin = S.y; }
    StrictEpi eq; eq.scale = qscale;
    launch_strict_gemm(yin, sl.wq, S.q, M, kD, kD, eq, st);
    launch_strict_gemm(yin, sl.wk, S.k, M, kD, kD, StrictEpi(), st);
    launch_strict_gemm(yin, sl.wv, S.v, M, kD, kD, StrictEpi(), st);
    launch_strict_attention(S.q, S.k, S.v, S.att, bw, L, c.attn_win_size, st);
    StrictEpi eo; eo.residual = S.x; eo.scale = c.rezero ? sl.alpha[0] : 1.f;         // encoder_stack.py:88-92
    launch_strict_gemm(S.att, sl.wo, S.x, M, kD, kD, eo, st);
    launches += 5;
    yin = S.x;
    if (!c.rezero) { launch_strict_layernorm(S.x, S.y, M, sl.ln_g[1], sl.ln_b[1], st); ++launches; yin = S.y; }
    StrictEpi e1; e1.bias = sl.b1; e1.relu = 1;                                        // ffn_layer.py:83-86
    launch_strict_gemm(yin, sl.w1, S.hid, M, ff, kD, e1, st);
    StrictEpi e2; e2.bias = sl.b2; e2.residual = S.x; e2.scale = c.rezero ? sl.alpha[1] : 1.f;
    launch_strict_gemm(S.hid, sl.w2, S.x, M, kD, ff, e2, st);
    launches += 2;
  }
  HeadParams h = hp;
  h.x = S.x; h.M = M; h.L = L; h.Lw = L;
  launch_strict_head(S.x, M, h, st); ++launches;
  return launches;
}

int dcb_set_debug(dcb_engine* e, int32_t enabled) {
  if (!e) return DCB_ERR_INVALID;
  e->debug = enabled != 0;
  if (e->debug && !e->d_dbg) {
    CU(e, cudaSetDevice(e->cfg.device));
    const size_t stages = 1 + 2 * (size_t)e->cfg.num_hidden_layers;
    int rc = dev_alloc(e, &e->d_dbg, stages * e->chunk_tiles * x_image_elems());
    if (rc) return rc;
  }
  return DCB_OK;
}

static int submit_impl(dcb_engine* e, const float* rows, const uint8_t* packed, int32_t batch, uint32_t flags,
                       uint8_t* bases_out, uint8_t* quals_out, float* probs_out, float* logits_out, int64_t* ticket_out) {
  if (!e || !ticket_out) return DCB_ERR_INVALID;
  if (!e->weights_loaded) return fail(e, DCB_ERR_STATE, "dcb_forward before dcb_load_weights");
  // any free slot (preferring the alternating one): a blocking dcb_forward between two submissions must not collide
  // with the slot of the one still outstanding
  int si = (int)(e->next_ticket & 1);
  if (e->slots[si].busy) si ^= 1;
  dcb_engine::Slot& sl = e->slots[si];
  if (sl.busy) return fail(e, DCB_ERR_STATE, "two submissions in flight: dcb_wait(ticket %lld) first",
                           (long long)std::min(e->slots[0].ticket, e->slots[1].ticket));
  if (batch < 0 || batch > e->cfg.max_batch) return fail(e, DCB_ERR_INVALID, "batch %d outside [0, max_batch=%d]", batch, e->cfg.max_batch);
  sl.launches = 0;
  sl.ticket = e->next_ticket;
  if (batch == 0) { sl.busy = true; sl.used = false; *ticket_out = e->next_ticket++; return DCB_OK; }
  if ((!rows && !packed) || !bases_out || !quals_out) return fail(e, DCB_ERR_INVALID, "null rows / output buffer");
  CU(e, cudaSetDevice(e->cfg.device));
  const dcb_config& c = e->cfg;
  if (packed && (c.pw_max > 255 || c.ip_max > 255)) return fail(e, DCB_ERR_INVALID, "packed rows need PW_MAX, IP_MAX <= 255");
  const int L = e->L, R = e->R;
  const size_t mtok = (size_t)c.max_batch * L;
  if (probs_out && !sl.d_probs) { int rc = dev_alloc(e, &sl.d_probs, mtok * kVocab); if (rc) return rc; }
  if (logits_out && !sl.d_logits) { int rc = dev_alloc(e, &sl.d_logits, mtok * kVocab); if (rc) return rc; }
  const bool rows_dev = flags & DCB_ROWS_ON_DEVICE;
  const bool out_dev = flags & DCB_OUT_ON_DEVICE;
  if ((flags & DCB_STRICT_FP32) && (flags & DCB_FAST_BF16)) return fail(e, DCB_ERR_INVALID, "DCB_STRICT_FP32 and DCB_FAST_BF16 are exclusive");
  const bool strict = (flags & DCB_STRICT_FP32) || (c.precision == DCB_PRECISION_FP32 && !(flags & DCB_FAST_BF16));
  if (rows_dev && ((reinterpret_cast<uintptr_t>(rows) | reinterpret_cast<uintptr_t>(packed)) & 15))
    return fail(e, DCB_ERR_INVALID, "device-resident rows must be 16-byte aligned");
  if (strict && !e->strict.emb) {
    // workspace of the strict path, on first use: ~16 k tokens per chunk
    dcb_engine::Strict& S = e->strict;
    S.chunk_windows = std::max(1, std::min(c.max_batch, 16384 / L));
    const size_t Mc = (size_t)S.chunk_windows * L;
    int rc = 0;
    if ((rc = dev_alloc(e, &S.emb, Mc * e->E)) || (rc = dev_alloc(e, &S.x, Mc * kD)) || (rc = dev_alloc(e, &S.y, Mc * kD)) ||
        (rc = dev_alloc(e, &S.q, Mc * kD)) || (rc = dev_alloc(e, &S.k, Mc * kD)) || (rc = dev_alloc(e, &S.v, Mc * kD)) ||
        (rc = dev_alloc(e, &S.att, Mc * kD)) || (rc = dev_alloc(e, &S.hid, Mc * c.filter_size)))
      return rc;
  }
  cudaStream_t st = e->stream;
  if (packed && !rows_dev && !sl.d_packed) {
    int rc = dev_alloc(e, &sl.d_packed, (size_t)c.max_batch * e->pl.stride);
    if (rc) return rc;
  }
  if (!rows_dev) {
    // The slot's previous forward (two submissions ago) was waited for before the slot was handed out again, so its
    // rows buffer is free; the copy overlaps whatever the compute stream is still running for the other slot.
    if (packed) CU(e, cudaMemcpyAsync(sl.d_packed, packed, (size_t)batch * e->pl.stride, cudaMemcpyHostToDevice, e->copy_stream));
    else CU(e, cudaMemcpyAsync(sl.d_rows, rows, (size_t)batch * R * L * sizeof(float), cudaMemcpyHostToDevice, e->copy_stream));
    CU(e, cudaEventRecord(sl.rows_ready, e->copy_stream));
    CU(e, cudaStreamWaitEvent(st, sl.rows_ready, 0));
  }
  const uint8_t* packed_base = packed ? (rows_dev ? packed : sl.d_packed) : nullptr;
  // the embedding kernel reads packed rows directly on the window-aligned fast path; every other path gets the float32
  // rows they stand for
  const bool packed_direct = packed_base && !strict && e->fuse_embed && embed_condense_reads_packed(L, e->Lw) &&
                             embed_condense_smem_bytes(R, e->echunks, e->table_elems, e->pl.stride) <= 225 * 1024;
  if (packed_base && !packed_direct) launch_unpack_rows(packed_base, e->pl, batch, sl.d_rows, st);
  const float* rows_base = packed ? sl.d_rows : (rows_dev ? rows : sl.d_rows);
  CU(e, cudaMemsetAsync(sl.d_status, 0, sizeof(int), st));
  CU(e, cudaEventRecord(sl.ev0, st));
  int launches = (packed_base && !packed_direct) ? 1 : 0;
  const size_t ximg = x_image_elems();
  bool prof_err = false;
  auto pbegin = [&](int kind) {
    if (!e->profile) return;
    if (sl.prof_used == sl.prof_events.size()) {
      cudaEvent_t a, b;
      if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) { prof_err = true; return; }
      sl.prof_events.emplace_back(a, b);
    }
    if (sl.prof_kind.size() <= sl.prof_used) sl.prof_kind.resize(sl.prof_used + 1);
    sl.prof_kind[sl.prof_used] = kind;
    cudaEventRecord(sl.prof_events[sl.prof_used].first, st);
  };
  auto pend = [&]() {
    if (!e->profile || prof_err) return;
    cudaEventRecord(sl.prof_events[sl.prof_used].second, st);
    ++sl.prof_used;
  };
  auto make_head_at = [&](int w0) {
    HeadParams hp{};
    hp.x = e->d_x; hp.ln_g = e->d_fln_g; hp.ln_b = e->d_fln_b; hp.wfc = e->d_wfc; hp.bfc = e->d_bfc;
    hp.gw8 = e->d_head_gw8; hp.ab = e->d_head_ab;
    const size_t t0 = (size_t)w0 * L;
    hp.bases = (out_dev ? bases_out : sl.d_bases) + t0;
    hp.quals = (out_dev ? quals_out : sl.d_quals) + t0;
    hp.probs = probs_out ? ((out_dev ? probs_out : sl.d_probs) + t0 * kVocab) : nullptr;
    hp.logits = logits_out ? ((out_dev ? logits_out : sl.d_logits) + t0 * kVocab) : nullptr;
    hp.calib_enabled = c.calibration_enabled;
    hp.calib_thr = (float)c.calibration_threshold; hp.calib_w = (float)c.calibration_w; hp.calib_b = (float)c.calibration_b;
    hp.calib_thr64 = c.calibration_threshold; hp.calib_w64 = c.calibration_w; hp.calib_b64 = c.calibration_b;
    hp.max_q = (float)c.max_base_quality;
    return hp;
  };
  if (strict) {
    for (int w0 = 0; w0 < batch; w0 += e->strict.chunk_windows) {
      const int bw = std::min(e->strict.chunk_windows, batch - w0);
      launches += strict_forward_chunk(e, rows_base + (size_t)w0 * R * L, bw, make_head_at(w0), sl.d_status, st);
    }
    e->stack_last = false;
  }
  for (int w0 = 0; !strict && w0 < batch; w0 += e->chunk_windows) {
    const int bw = std::min(e->chunk_windows, batch - w0);
    const int Lw = e->Lw;
    const int M = bw * Lw;          // tokens in the (possibly window-aligned) layout
    const int T = (M + kTileM - 1) / kTileM;
    const float* rows_chunk = rows_base + (size_t)w0 * R * L;
    int stage = 0;
    auto snap = [&]() {
      if (e->debug) cudaMemcpyAsync(e->d_dbg + (size_t)stage * e->chunk_tiles * ximg, e->d_x, (size_t)T * ximg * sizeof(float), cudaMemcpyDeviceToDevice, st);
      ++stage;
    };
    auto make_head = [&]() {
      HeadParams hp = make_head_at(w0);
      hp.M = M; hp.L = L; hp.Lw = Lw;
      return hp;
    };
    const bool use_stack = e->stack && e->fuse_qa && e->fuse_oproj && e->fuse_embed && !e->debug &&
                           (Lw == kTileM || (Lw == 2 * kTileM && L > kTileM)) &&
                           c.attn_win_size > 0 && c.attn_win_size <= 16 && c.num_hidden_layers <= kMaxLayers;
    {
      RowEpi epi{};
      // the one-kernel stack builds every operand tile from the residual in TMEM: no bf16 operand image needed
      epi.x = e->d_x; epi.xb = use_stack ? nullptr : e->d_xb; epi.bias = nullptr;
      epi.pe = c.add_pos_encoding ? e->d_pe : nullptr;
      epi.pe_img = c.add_pos_encoding ? e->d_pe_img : nullptr;
      epi.ln_g = (c.rezero || use_stack) ? nullptr : e->layers[0].ln_g[0];
      epi.ln_b = (c.rezero || use_stack) ? nullptr : e->layers[0].ln_b[0];
      epi.has_xold = 0; epi.L = Lw;
      bool fused_embed = false;
      if (e->fuse_embed) {
        pbegin(1);
        fused_embed = launch_embed_condense(rows_chunk, packed_direct ? packed_base + (size_t)w0 * e->pl.stride : nullptr, e->pl,
                                            R, L, Lw, M, T, e->echunks, e->d_cols, e->d_rowmeta, e->d_tables,
                                            e->table_elems, e->d_wc, epi, sl.d_status, st);
        if (!fused_embed && packed_direct) return fail(e, DCB_ERR_INVALID, "internal: packed rows on a path that cannot read them");
        pend();
        if (fused_embed) ++launches;
      }
      if (!fused_embed) {
        pbegin(0);
        launch_embed(rows_chunk, R, L, Lw, M, T, e->echunks, e->d_cols, e->d_rowmeta, e->d_tables, e->table_elems, e->d_embqkv, sl.d_status, st);
        pend();
        pbegin(1);
        launch_gemm_row(e->d_embqkv, e->d_wc, e->Epad / 16, T, epi, st);
        pend();
        launches += 2;
      }
      snap();
    }
    if (use_stack) {
      StackParams sp{};
      sp.num_layers = c.num_hidden_layers;
      sp.ff = c.filter_size;
      sp.deferred_ln = c.rezero ? 0 : 1;
      for (int n_ = 0; n_ < c.num_hidden_layers; ++n_) {
        const LayerDev& ld = e->layers[n_];
        sp.wq3[n_] = ld.wq3; sp.wo2[n_] = ld.wo2; sp.wffn2[n_] = ld.wffn2s;
        sp.b2[n_] = ld.b2; sp.b2_mean[n_] = ld.b2_mean;
      }
      HeadParams hs{};
      if (e->fuse_head) { hs = make_head(); }
      pbegin(4);
      launch_stack(e->d_x, T, L, c.attn_win_size, sp, hs, st);
      pend();
      if (e->profile) e->prof_ffn_tokens += (long long)bw * L;
      e->fused_last = true;
      e->stack_last = true;
      ++launches;
    } else e->stack_last = false;
    for (int n_ = 0; !use_stack && n_ < c.num_hidden_layers; ++n_) {
      const LayerDev& ld = e->layers[n_];
      const bool last = n_ + 1 == c.num_hidden_layers;
      if (e->fuse_qa && Lw == kTileM) {
        pbegin(2);
        launch_qkv_attn(e->d_xb, ld.wqa, T, L, c.attn_win_size, e->d_att, st);
        pend();
        --launches;   // one launch instead of two (3 per layer are added below)
      } else {
        pbegin(2);
        launch_gemm_qkv(e->d_xb, ld.wqkv, T, e->d_embqkv, st);
        pend();
        pbegin(3);
        launch_attention(e->d_embqkv, e->d_att, L, Lw, c.attn_win_size, bw, st);
        pend();
      }
      // attention out-proj + FFN: fused into one CTA-pair kernel unless debugging the intermediate
      const bool fused = e->fuse_oproj && !e->debug;
      RowEpi ef{};
      ef.x = e->d_x; ef.xb = last ? nullptr : e->d_xb; ef.bias = ld.b2; ef.pe = nullptr;
      ef.ln_g = (c.rezero || last) ? nullptr : e->layers[n_ + 1].ln_g[0];
      ef.ln_b = (c.rezero || last) ? nullptr : e->layers[n_ + 1].ln_b[0];
      ef.has_xold = 1; ef.L = Lw;
      if (!fused) {
        RowEpi ea{};
        ea.x = e->d_x; ea.xb = e->d_xb; ea.bias = nullptr; ea.pe = nullptr;
        ea.ln_g = c.rezero ? nullptr : ld.ln_g[1];
        ea.ln_b = c.rezero ? nullptr : ld.ln_b[1];
        ea.has_xold = 1; ea.L = Lw;
        pbegin(1);
        launch_gemm_row(e->d_att, ld.wo, kDP / 16, T, ea, st);
        pend();
        ++launches;
        snap();
      }
      pbegin(4);
      if (fused)
        launch_ffn_pair(e->d_att, ld.wffn2, ld.b1, c.filter_size, T, ef, st, ld.wo2,
                        c.rezero ? nullptr : ld.ln_g[1], c.rezero ? nullptr : ld.ln_b[1]);
      else
        launch_ffn_pair(e->d_xb, ld.wffn2, ld.b1, c.filter_size, T, ef, st);
      pend();
      if (e->profile) e->prof_ffn_tokens += (long long)bw * L;   // valid tokens (layout padding is not algorithmic work)
      if (!fused) snap();
      e->fused_last = fused;
      launches += 3;
    }
    const bool head_done = use_stack && e->fuse_head;
    if (!head_done) {
      pbegin(5);
      launch_head(make_head(), T, st);
      pend();
      ++launches;
    }
    e->last_chunk_tokens = M;
  }
  CU(e, cudaEventRecord(sl.ev1, st));
  // results and status go back on their own stream: the compute stream is free for the next submission's kernels
  cudaStream_t os = e->out_stream;
  CU(e, cudaStreamWaitEvent(os, sl.ev1, 0));
  if (!out_dev) {
    const size_t ntok = (size_t)batch * L;
    CU(e, cudaMemcpyAsync(bases_out, sl.d_bases, ntok, cudaMemcpyDeviceToHost, os));
    CU(e, cudaMemcpyAsync(quals_out, sl.d_quals, ntok, cudaMemcpyDeviceToHost, os));
    if (probs_out) CU(e, cudaMemcpyAsync(probs_out, sl.d_probs, ntok * kVocab * sizeof(float), cudaMemcpyDeviceToHost, os));
    if (logits_out) CU(e, cudaMemcpyAsync(logits_out, sl.d_logits, ntok * kVocab * sizeof(float), cudaMemcpyDeviceToHost, os));
  }
  CU(e, cudaMemcpyAsync(sl.h_status, sl.d_status, sizeof(int), cudaMemcpyDeviceToHost, os));
  CU(e, cudaEventRecord(sl.done, os));
  CU(e, cudaGetLastError());
  sl.launches = launches;
  sl.busy = true;
  sl.used = true;
  *ticket_out = e->next_ticket++;
  return DCB_OK;
}

int dcb_submit(dcb_engine* e, const float* rows, int32_t batch, uint32_t flags, uint8_t* bases_out,
               uint8_t* quals_out, float* probs_out, float* logits_out, int64_t* ticket_out) {
  return submit_impl(e, rows, nullptr, batch, flags, bases_out, quals_out, probs_out, logits_out, ticket_out);
}

int dcb_submit_packed(dcb_engine* e, const uint8_t* packed, int32_t batch, uint32_t flags, uint8_t* bases_out,
                      uint8_t* quals_out, float* probs_out, float* logits_out, int64_t* ticket_out) {
  return submit_impl(e, nullptr, packed, batch, flags, bases_out, quals_out, probs_out, logits_out, ticket_out);
}

int dcb_forward_packed(dcb_engine* e, const uint8_t* packed, int32_t batch, uint32_t flags, uint8_t* bases_out,
                       uint8_t* quals_out, float* probs_out, float* logits_out) {
  int64_t ticket = -1;
  int rc = dcb_submit_packed(e, packed, batch, flags, bases_out, quals_out, probs_out, logits_out, &ticket);
  if (rc) return rc;
  return dcb_wait(e, ticket);
}

size_t dcb_packed_window_bytes(const dcb_config* cfg) {
  if (!cfg || cfg->max_passes <= 0 || cfg->max_length <= 0) return 0;
  return (size_t)make_packed_layout(cfg->max_passes, cfg->max_length, cfg->use_ccs_bq ? 1 : 0).stride;
}

// float32 rows [B, R, L] -> packed rows (include/dcb200.h).  Host code (no GPU, no engine): the producer side of the path.
int dcb_pack_rows(const dcb_config* cfg, const float* rows, int32_t batch, uint8_t* out) {
  if (!cfg || !rows || !out || batch < 0 || cfg->max_passes <= 0 || cfg->max_length <= 0)
    return fail(nullptr, DCB_ERR_INVALID, "dcb_pack_rows: bad argument");
  const dcb_config& c = *cfg;
  dcb_engine* e = nullptr;   // messages go to the engine-less error slot (dcb_last_error(NULL))
  if (c.pw_max > 255 || c.ip_max > 255) return fail(e, DCB_ERR_INVALID, "packed rows need PW_MAX, IP_MAX <= 255");
  const PackedLayout pl = make_packed_layout(c.max_passes, c.max_length, c.use_ccs_bq ? 1 : 0);
  const int P = pl.P, L = pl.L, R = pl.R;
  bool bad = false;
  auto trunc_clip = [](float v, int hi, bool* flag) {   // clip to [0, hi] as format_rows, then truncate as tf.cast
    if (!(v >= 0.f)) { if (v < 0.f || v != v) { if (flag) *flag = true; } return 0; }
    if (v > (float)hi) { if (flag) *flag = true; return hi; }
    return (int)v;
  };
  for (int b = 0; b < batch; ++b) {
    const float* w = rows + (size_t)b * R * L;
    uint8_t* o = out + (size_t)b * pl.stride;
    memset(o, 0, pl.stride);
    for (int p_ = 0; p_ < P; ++p_)
      for (int l = 0; l < L; ++l) {
        const int base = trunc_clip(w[(size_t)p_ * L + l], kVocab - 1, &bad);               // outside 0..4: TF raises
        const int strand = trunc_clip(w[(size_t)(3 * P + p_) * L + l], c.strand_max, &bad);
        o[p_ * L + l] = (uint8_t)(base | (strand << 3));
        o[(P + p_) * L + l] = (uint8_t)trunc_clip(w[(size_t)(P + p_) * L + l], 255, nullptr);       // clip, not an error
        o[(2 * P + p_) * L + l] = (uint8_t)trunc_clip(w[(size_t)(2 * P + p_) * L + l], 255, nullptr);
      }
    for (int l = 0; l < L; ++l) o[3 * P * L + l] = (uint8_t)trunc_clip(w[(size_t)4 * P * L + l], kVocab - 1, &bad);
    if (pl.bq)
      for (int l = 0; l < L; ++l)
        o[(3 * P + 1) * L + l] = (uint8_t)trunc_clip(w[(size_t)(4 * P + 1) * L + l] + 1.f, c.ccs_bq_max - 1, &bad);
    float* sn = reinterpret_cast<float*>(o + pl.sn_off);
    for (int i = 0; i < 4; ++i) {
      const float* row = w + (size_t)(R - 4 + i) * L;
      sn[i] = row[0];
      for (int l = 1; l < L; ++l)
        if (row[l] != row[0]) bad = true;
    }
  }
  if (bad) return fail(e, DCB_ERR_INPUT_RANGE, "dcb_pack_rows: value outside its vocabulary (clamped) or SN row not constant");
  return DCB_OK;
}

int dcb_wait(dcb_engine* e, int64_t ticket) {
  if (!e) return DCB_ERR_INVALID;
  int si = -1;
  for (int i = 0; i < 2; ++i)
    if (e->slots[i].busy && e->slots[i].ticket == ticket) si = i;
  if (ticket < 0 || si < 0) return fail(e, DCB_ERR_STATE, "dcb_wait: ticket %lld is not in flight", (long long)ticket);
  dcb_engine::Slot& sl = e->slots[si];
  sl.busy = false;
  if (!sl.used) { e->last_ms = 0.f; e->last_launches = 0; return DCB_OK; }   // empty batch
  CU(e, cudaSetDevice(e->cfg.device));
  CU(e, cudaEventSynchronize(sl.done));
  CU(e, cudaGetLastError());
  CU(e, cudaEventElapsedTime(&e->last_ms, sl.ev0, sl.ev1));
  e->last_launches = sl.launches;
  const int status = *sl.h_status;
  {
    for (size_t i = 0; i < sl.prof_used; ++i) {
      float ms = 0.f;
      CU(e, cudaEventElapsedTime(&ms, sl.prof_events[i].first, sl.prof_events[i].second));
      const int kind = sl.prof_kind[i];
      e->prof_ms[kind] += ms;
      ++e->prof_n[kind];
      if (kind == 4) { e->prof_ffn_ms += ms; ++e->prof_ffn_launches; }
    }
    sl.prof_used = 0;
  }
  if (status & 1) return fail(e, DCB_ERR_INPUT_RANGE, "embedding id out of range in the input rows (clamped)");
  return DCB_OK;
}

int dcb_forward(dcb_engine* e, const float* rows, int32_t batch, uint32_t flags, uint8_t* bases_out,
                uint8_t* quals_out, float* probs_out, float* logits_out) {
  int64_t ticket = -1;
  int rc = dcb_submit(e, rows, batch, flags, bases_out, quals_out, probs_out, logits_out, &ticket);
  if (rc) return rc;
  return dcb_wait(e, ticket);
}

int dcb_last_forward_ms(dcb_engine* e, float* ms) {
  if (!e || !ms) return DCB_ERR_INVALID;
  *ms = e->last_ms;
  return DCB_OK;
}

int dcb_last_forward_launches(dcb_engine* e, int32_t* n) {
  if (!e || !n) return DCB_ERR_INVALID;
  *n = e->last_launches;
  return DCB_OK;
}

int dcb_set_profile(dcb_engine* e, int32_t enabled) {
  if (!e) return DCB_ERR_INVALID;
  e->profile = enabled != 0;
  e->prof_ffn_ms = 0.f;
  e->prof_ffn_launches = 0;
  e->prof_ffn_tokens = 0;
  for (auto& sl : e->slots) sl.prof_used = 0;
  for (int i = 0; i < 6; ++i) { e->prof_ms[i] = 0.f; e->prof_n[i] = 0; }
  return DCB_OK;
}

int dcb_get_profile(dcb_engine* e, float* ffn_ms_total, int32_t* ffn_launches, int64_t* ffn_tokens) {
  if (!e || !ffn_ms_total || !ffn_launches || !ffn_tokens) return DCB_ERR_INVALID;
  *ffn_ms_total = e->prof_ffn_ms;
  *ffn_launches = e->prof_ffn_launches;
  *ffn_tokens = e->prof_ffn_tokens;
  return DCB_OK;
}

int dcb_get_profile_kernels(dcb_engine* e, float* ms6, int32_t* n6, int32_t* fused_oproj) {
  if (!e || !ms6 || !n6 || !fused_oproj) return DCB_ERR_INVALID;
  for (int i = 0; i < 6; ++i) { ms6[i] = e->prof_ms[i]; n6[i] = e->prof_n[i]; }
  *fused_oproj = e->stack_last ? 2 : (e->fused_last ? 1 : 0);   // 2: whole stack in one kernel
  return DCB_OK;
}

int dcb_debug_residual(dcb_engine* e, int32_t stage, float* out, int64_t out_elems) {
  if (!e || !out) return DCB_ERR_INVALID;
  if (!e->debug || !e->d_dbg) return fail(e, DCB_ERR_STATE, "debug capture not enabled");
  const int stages = 1 + 2 * e->cfg.num_hidden_layers;
  if (stage < 0 || stage >= stages) return fail(e, DCB_ERR_INVALID, "stage %d outside [0,%d)", stage, stages);
  const int Mlay = e->last_chunk_tokens;               // tokens in the layout
  const int M = Mlay / e->Lw * e->L;                   // valid tokens
  if (out_elems < (int64_t)M * kD) return fail(e, DCB_ERR_INVALID, "output too small: need %lld", (long long)M * kD);
  CU(e, cudaSetDevice(e->cfg.device));
  const int T = (Mlay + kTileM - 1) / kTileM;
  std::vector<float> img((size_t)T * x_image_elems());
  CU(e, cudaMemcpy(img.data(), e->d_dbg + (size_t)stage * e->chunk_tiles * x_image_elems(), img.size() * sizeof(float), cudaMemcpyDeviceToHost));
  for (int t = 0; t < M; ++t) {
    const int tl = t / e->L * e->Lw + t % e->L;        // position of valid token t in the layout
    const int tile = tl / kTileM, r = tl % kTileM;
    for (int col = 0; col < kD; ++col)
      out[(size_t)t * kD + col] = img[(((size_t)tile * kXChunks + col / 4) * kTileM + r) * 4 + col % 4];
  }
  return DCB_OK;
}

namespace {
int stitch_spans(dcb_engine* e, const uint8_t* bases, const uint8_t* quals, size_t nbytes, const int64_t* read_off,
                 const int32_t* zmw_start, int32_t n_zmw, uint32_t flags, uint8_t* seq_out, uint8_t* qual_out,
                 int32_t* len_out);
}  // namespace

int dcb_stitch(dcb_engine* e, const uint8_t* bases, const uint8_t* quals, int32_t n_windows, int32_t L,
               const int32_t* zmw_start, int32_t n_zmw, uint32_t flags,
               uint8_t* seq_out, uint8_t* qual_out, int32_t* len_out) {
  if (!e) return DCB_ERR_INVALID;
  if (n_windows < 0 || L <= 0 || n_zmw < 0) return fail(e, DCB_ERR_INVALID, "dcb_stitch: negative size");
  if (n_zmw == 0 || n_windows == 0) return DCB_OK;
  if (!bases || !quals || !zmw_start || !seq_out || !qual_out || !len_out) return fail(e, DCB_ERR_INVALID, "dcb_stitch: null pointer");
  if (zmw_start[0] < 0 || zmw_start[n_zmw] > n_windows) return fail(e, DCB_ERR_INVALID, "dcb_stitch: zmw_start outside [0, n_windows]");
  for (int z = 0; z < n_zmw; ++z)
    if (zmw_start[z + 1] < zmw_start[z]) return fail(e, DCB_ERR_INVALID, "dcb_stitch: zmw_start must be non-decreasing");
  std::vector<int64_t> read_off((size_t)n_zmw + 1);
  for (int z = 0; z <= n_zmw; ++z) read_off[z] = (int64_t)zmw_start[z] * L;
  return stitch_spans(e, bases, quals, (size_t)n_windows * L, read_off.data(), zmw_start, n_zmw, flags, seq_out, qual_out,
                      len_out);
}

namespace {
// dcb_stitch on byte spans: read z is bytes [read_off[z], read_off[z + 1]) of bases / quals (nbytes in all; host int64
// offsets) and is written at the same offsets of seq_out / qual_out.  zmw_start is left in d_st_start, read_off in d_st_off.
int stitch_spans(dcb_engine* e, const uint8_t* bases, const uint8_t* quals, size_t nbytes, const int64_t* read_off,
                 const int32_t* zmw_start, int32_t n_zmw, uint32_t flags, uint8_t* seq_out, uint8_t* qual_out,
                 int32_t* len_out) {
  for (int z = 0; z < n_zmw; ++z)
    if (read_off[z + 1] - read_off[z] > INT32_MAX) return fail(e, DCB_ERR_INVALID, "dcb_stitch: read %d spans 2^31 bytes or more", z);
  CU(e, cudaSetDevice(e->cfg.device));
  const bool in_dev = flags & DCB_ROWS_ON_DEVICE, out_dev = flags & DCB_OUT_ON_DEVICE;
  cudaStream_t st = e->stream;
  if (nbytes > e->st_cap) {
    CU(e, cudaStreamSynchronize(st));
    if (e->d_st_in) cudaFree(e->d_st_in);
    if (e->d_st_out) cudaFree(e->d_st_out);
    e->d_st_in = e->d_st_out = nullptr;
    e->st_cap = 0;
    CU(e, cudaMalloc(reinterpret_cast<void**>(&e->d_st_in), 2 * nbytes));
    CU(e, cudaMalloc(reinterpret_cast<void**>(&e->d_st_out), 2 * nbytes));
    e->st_cap = nbytes;
  }
  if ((size_t)n_zmw + 1 > e->st_zcap) {
    CU(e, cudaStreamSynchronize(st));
    if (e->d_st_start) cudaFree(e->d_st_start);
    if (e->d_st_len) cudaFree(e->d_st_len);
    if (e->d_st_off) cudaFree(e->d_st_off);
    e->d_st_start = e->d_st_len = nullptr;
    e->d_st_off = nullptr;
    e->st_zcap = 0;
    CU(e, cudaMalloc(reinterpret_cast<void**>(&e->d_st_start), ((size_t)n_zmw + 1) * sizeof(int32_t)));
    CU(e, cudaMalloc(reinterpret_cast<void**>(&e->d_st_len), ((size_t)n_zmw + 1) * sizeof(int32_t)));
    CU(e, cudaMalloc(reinterpret_cast<void**>(&e->d_st_off), ((size_t)n_zmw + 1) * sizeof(int64_t)));
    e->st_zcap = (size_t)n_zmw + 1;
  }
  const uint8_t *db = bases, *dq = quals;
  if (!in_dev) {
    CU(e, cudaMemcpyAsync(e->d_st_in, bases, nbytes, cudaMemcpyHostToDevice, st));
    CU(e, cudaMemcpyAsync(e->d_st_in + e->st_cap, quals, nbytes, cudaMemcpyHostToDevice, st));
    db = e->d_st_in; dq = e->d_st_in + e->st_cap;
  }
  CU(e, cudaMemcpyAsync(e->d_st_start, zmw_start, ((size_t)n_zmw + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  CU(e, cudaMemcpyAsync(e->d_st_off, read_off, ((size_t)n_zmw + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
  uint8_t* ds = out_dev ? seq_out : e->d_st_out;
  uint8_t* dqo = out_dev ? qual_out : e->d_st_out + e->st_cap;
  int32_t* dl = out_dev ? len_out : e->d_st_len;
  launch_stitch(db, dq, e->d_st_off, n_zmw, ds, dqo, dl, st);
  if (!out_dev) {
    CU(e, cudaMemcpyAsync(seq_out, ds, nbytes, cudaMemcpyDeviceToHost, st));
    CU(e, cudaMemcpyAsync(qual_out, dqo, nbytes, cudaMemcpyDeviceToHost, st));
    CU(e, cudaMemcpyAsync(len_out, dl, (size_t)n_zmw * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  }
  CU(e, cudaStreamSynchronize(st));
  CU(e, cudaGetLastError());
  return DCB_OK;
}

// grow-on-demand device scratch; contents are not preserved
int ensure(dcb_engine* e, dcb_engine::Scratch& sc, size_t bytes) {
  if (bytes <= sc.cap) return DCB_OK;
  CU(e, cudaStreamSynchronize(e->stream));
  if (sc.p) cudaFree(sc.p);
  sc.p = nullptr; sc.cap = 0;
  CU(e, cudaMalloc(&sc.p, bytes));
  sc.cap = bytes;
  return DCB_OK;
}
}  // namespace

int dcb_stitch_fastq(dcb_engine* e, const uint8_t* bases, const uint8_t* quals, int32_t n_windows, int32_t L,
                     const int32_t* zmw_start, int32_t n_zmw, const int32_t* window_pos, const uint8_t* names,
                     const int32_t* name_off, double min_quality, int32_t min_length, uint32_t flags, uint8_t* fastq_out,
                     int64_t fastq_cap, int64_t* rec_off, int32_t* outcome, double* avg_q) {
  if (!e) return DCB_ERR_INVALID;
  if (n_windows < 0 || L <= 0) return fail(e, DCB_ERR_INVALID, "dcb_stitch_fastq: negative size");
  std::vector<int64_t> window_off((size_t)n_windows + 1);
  for (int w = 0; w <= n_windows; ++w) window_off[w] = (int64_t)w * L;
  return dcb_stitch_fastq_ragged(e, bases, quals, n_windows, window_off.data(), L, zmw_start, n_zmw, window_pos, names,
                                 name_off, min_quality, min_length, flags, fastq_out, fastq_cap, rec_off, outcome, avg_q);
}

int dcb_stitch_fastq_ragged(dcb_engine* e, const uint8_t* bases, const uint8_t* quals, int32_t n_windows,
                            const int64_t* window_off, int32_t L, const int32_t* zmw_start, int32_t n_zmw,
                            const int32_t* window_pos, const uint8_t* names, const int32_t* name_off, double min_quality,
                            int32_t min_length, uint32_t flags, uint8_t* fastq_out, int64_t fastq_cap, int64_t* rec_off,
                            int32_t* outcome, double* avg_q) {
  if (!e) return DCB_ERR_INVALID;
  if (n_windows < 0 || L <= 0 || n_zmw < 0 || fastq_cap < 0) return fail(e, DCB_ERR_INVALID, "dcb_stitch_fastq: negative size");
  if (!rec_off) return fail(e, DCB_ERR_INVALID, "dcb_stitch_fastq: null pointer");
  if (n_zmw == 0) { rec_off[0] = 0; return DCB_OK; }
  if (!bases || !quals || !window_off || !zmw_start || !window_pos || !names || !name_off || !fastq_out || !outcome || !avg_q)
    return fail(e, DCB_ERR_INVALID, "dcb_stitch_fastq: null pointer");
  if (name_off[0] != 0) return fail(e, DCB_ERR_INVALID, "dcb_stitch_fastq: name_off[0] must be 0");
  for (int z = 0; z < n_zmw; ++z)
    if (name_off[z + 1] < name_off[z]) return fail(e, DCB_ERR_INVALID, "dcb_stitch_fastq: name_off must be non-decreasing");
  if (zmw_start[0] < 0 || zmw_start[n_zmw] > n_windows) return fail(e, DCB_ERR_INVALID, "dcb_stitch_fastq: zmw_start outside [0, n_windows]");
  for (int z = 0; z < n_zmw; ++z)
    if (zmw_start[z + 1] < zmw_start[z]) return fail(e, DCB_ERR_INVALID, "dcb_stitch_fastq: zmw_start must be non-decreasing");
  if (window_off[0] < 0) return fail(e, DCB_ERR_INVALID, "dcb_stitch_fastq: negative window offset");
  for (int w = 0; w < n_windows; ++w)
    if (window_off[w + 1] < window_off[w]) return fail(e, DCB_ERR_INVALID, "dcb_stitch_fastq: window_off must be non-decreasing");
  std::vector<int64_t> read_off((size_t)n_zmw + 1);
  for (int z = 0; z <= n_zmw; ++z) read_off[z] = window_off[zmw_start[z]];
  const size_t nbytes = (size_t)window_off[n_windows];
  // stage 1: concatenation + gap compaction (dcb_stitch), results stay on the device
  CU(e, cudaSetDevice(e->cfg.device));
  cudaStream_t st = e->stream;
  int rc;
  // reuse dcb_stitch with device-side outputs into our own scratch
  if ((rc = ensure(e, e->sc_tmpb, nbytes ? nbytes : 1)) || (rc = ensure(e, e->sc_tmpq, nbytes ? nbytes : 1)) ||
      (rc = ensure(e, e->sc_dst, ((size_t)n_zmw + 1) * sizeof(int32_t))))
    return rc;
  uint8_t* d_seq = static_cast<uint8_t*>(e->sc_tmpb.p);
  uint8_t* d_qual = static_cast<uint8_t*>(e->sc_tmpq.p);
  int32_t* d_len = static_cast<int32_t*>(e->sc_dst.p);
  if (nbytes > 0) {
    rc = stitch_spans(e, bases, quals, nbytes, read_off.data(), zmw_start, n_zmw, (flags & DCB_ROWS_ON_DEVICE) | DCB_OUT_ON_DEVICE,
                      d_seq, d_qual, d_len);
    if (rc) return rc;
  } else {
    CU(e, cudaMemsetAsync(d_len, 0, ((size_t)n_zmw + 1) * sizeof(int32_t), st));
  }
  const size_t names_bytes = (size_t)name_off[n_zmw];
  const size_t cap = (size_t)fastq_cap;
  if ((rc = ensure(e, e->sc_pos, (n_windows ? (size_t)n_windows : 1) * sizeof(int32_t))) ||
      (rc = ensure(e, e->sc_names, names_bytes ? names_bytes : 1)) ||
      (rc = ensure(e, e->sc_nameoff, ((size_t)n_zmw + 1) * sizeof(int32_t))) ||
      (rc = ensure(e, e->sc_outcome, (size_t)n_zmw * sizeof(int32_t))) || (rc = ensure(e, e->sc_avg, (size_t)n_zmw * sizeof(double))) ||
      (rc = ensure(e, e->sc_recoff, ((size_t)n_zmw + 1) * sizeof(int64_t))) || (rc = ensure(e, e->sc_fastq, cap ? cap : 1)))
    return rc;
  // stitch_spans left zmw_start / read_off in its own scratch (d_st_start / d_st_off)
  if (nbytes == 0) {
    if ((size_t)n_zmw + 1 > e->st_zcap) {
      if (e->d_st_start) cudaFree(e->d_st_start);
      if (e->d_st_len) cudaFree(e->d_st_len);
      if (e->d_st_off) cudaFree(e->d_st_off);
      e->d_st_start = e->d_st_len = nullptr; e->d_st_off = nullptr; e->st_zcap = 0;
      CU(e, cudaMalloc(reinterpret_cast<void**>(&e->d_st_start), ((size_t)n_zmw + 1) * sizeof(int32_t)));
      CU(e, cudaMalloc(reinterpret_cast<void**>(&e->d_st_len), ((size_t)n_zmw + 1) * sizeof(int32_t)));
      CU(e, cudaMalloc(reinterpret_cast<void**>(&e->d_st_off), ((size_t)n_zmw + 1) * sizeof(int64_t)));
      e->st_zcap = (size_t)n_zmw + 1;
    }
    CU(e, cudaMemcpyAsync(e->d_st_start, zmw_start, ((size_t)n_zmw + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    CU(e, cudaMemcpyAsync(e->d_st_off, read_off.data(), ((size_t)n_zmw + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
  }
  if (n_windows > 0) CU(e, cudaMemcpyAsync(e->sc_pos.p, window_pos, (size_t)n_windows * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  if (names_bytes) CU(e, cudaMemcpyAsync(e->sc_names.p, names, names_bytes, cudaMemcpyHostToDevice, st));
  CU(e, cudaMemcpyAsync(e->sc_nameoff.p, name_off, ((size_t)n_zmw + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  int32_t* d_out = static_cast<int32_t*>(e->sc_outcome.p);
  double* d_avg = static_cast<double*>(e->sc_avg.p);
  int64_t* d_rec = static_cast<int64_t*>(e->sc_recoff.p);
  launch_read_outcome(d_qual, d_len, e->d_st_off, e->d_st_start, static_cast<const int32_t*>(e->sc_pos.p), L, n_zmw, e->d_p10,
                      min_quality, min_length, d_out, d_avg, st);
  launch_fastq(d_seq, d_qual, d_len, e->d_st_off, n_zmw, d_out, static_cast<const uint8_t*>(e->sc_names.p),
               static_cast<const int32_t*>(e->sc_nameoff.p), d_rec, static_cast<uint8_t*>(e->sc_fastq.p), fastq_cap, st);
  CU(e, cudaMemcpyAsync(rec_off, d_rec, ((size_t)n_zmw + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  CU(e, cudaMemcpyAsync(outcome, d_out, (size_t)n_zmw * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CU(e, cudaMemcpyAsync(avg_q, d_avg, (size_t)n_zmw * sizeof(double), cudaMemcpyDeviceToHost, st));
  CU(e, cudaStreamSynchronize(st));
  if (rec_off[n_zmw] > fastq_cap) return fail(e, DCB_ERR_INVALID, "dcb_stitch_fastq: fastq_out too small: need %lld bytes", (long long)rec_off[n_zmw]);
  if (rec_off[n_zmw] > 0) CU(e, cudaMemcpy(fastq_out, e->sc_fastq.p, (size_t)rec_off[n_zmw], cudaMemcpyDeviceToHost));
  CU(e, cudaGetLastError());
  return DCB_OK;
}

int dcb_skip_mask(dcb_engine* e, const int16_t* ccs_bq, int32_t n_windows, int32_t L, double skip_windows_above,
                  uint8_t* mask_out, double* avg_out) {
  if (!e) return DCB_ERR_INVALID;
  if (n_windows < 0 || L <= 0) return fail(e, DCB_ERR_INVALID, "dcb_skip_mask: negative size");
  if (n_windows == 0) return DCB_OK;
  if (!ccs_bq || !mask_out) return fail(e, DCB_ERR_INVALID, "dcb_skip_mask: null pointer");
  CU(e, cudaSetDevice(e->cfg.device));
  cudaStream_t st = e->stream;
  const size_t n = (size_t)n_windows * L;
  int rc;
  if ((rc = ensure(e, e->sc_bq, n * sizeof(int16_t))) || (rc = ensure(e, e->sc_mask, (size_t)n_windows)) ||
      (rc = ensure(e, e->sc_avg, (size_t)n_windows * sizeof(double))))
    return rc;
  CU(e, cudaMemcpyAsync(e->sc_bq.p, ccs_bq, n * sizeof(int16_t), cudaMemcpyHostToDevice, st));
  launch_skip_mask(static_cast<const int16_t*>(e->sc_bq.p), n_windows, L, e->d_p10, skip_windows_above,
                   static_cast<uint8_t*>(e->sc_mask.p), static_cast<double*>(e->sc_avg.p), st);
  CU(e, cudaMemcpyAsync(mask_out, e->sc_mask.p, (size_t)n_windows, cudaMemcpyDeviceToHost, st));
  if (avg_out) CU(e, cudaMemcpyAsync(avg_out, e->sc_avg.p, (size_t)n_windows * sizeof(double), cudaMemcpyDeviceToHost, st));
  CU(e, cudaStreamSynchronize(st));
  CU(e, cudaGetLastError());
  return DCB_OK;
}

int dcb_fill_skipped(dcb_engine* e, const uint8_t* ccs_ids, const int16_t* ccs_bq, const int32_t* dst_window, int32_t k,
                     int32_t L, int32_t calibration_enabled, double calibration_threshold, double calibration_w,
                     double calibration_b, uint32_t flags, uint8_t* bases, uint8_t* quals) {
  if (!e) return DCB_ERR_INVALID;
  if (k < 0 || L <= 0) return fail(e, DCB_ERR_INVALID, "dcb_fill_skipped: negative size");
  if (k == 0) return DCB_OK;
  if (!ccs_ids || !ccs_bq || !dst_window || !bases || !quals) return fail(e, DCB_ERR_INVALID, "dcb_fill_skipped: null pointer");
  for (int j = 0; j < k; ++j)
    if (dst_window[j] < 0) return fail(e, DCB_ERR_INVALID, "dcb_fill_skipped: negative destination window");
  std::vector<int64_t> src_off((size_t)k + 1), dst_off((size_t)k);
  for (int j = 0; j <= k; ++j) src_off[j] = (int64_t)j * L;
  for (int j = 0; j < k; ++j) dst_off[j] = (int64_t)dst_window[j] * L;
  return dcb_fill_skipped_ragged(e, ccs_ids, ccs_bq, src_off.data(), dst_off.data(), k, calibration_enabled,
                                 calibration_threshold, calibration_w, calibration_b, flags, bases, quals);
}

int dcb_fill_skipped_ragged(dcb_engine* e, const uint8_t* ccs_ids, const int16_t* ccs_bq, const int64_t* src_off,
                            const int64_t* dst_off, int32_t k, int32_t calibration_enabled, double calibration_threshold,
                            double calibration_w, double calibration_b, uint32_t flags, uint8_t* bases, uint8_t* quals) {
  if (!e) return DCB_ERR_INVALID;
  if (k < 0) return fail(e, DCB_ERR_INVALID, "dcb_fill_skipped: negative size");
  if (k == 0) return DCB_OK;
  if (!ccs_ids || !ccs_bq || !src_off || !dst_off || !bases || !quals) return fail(e, DCB_ERR_INVALID, "dcb_fill_skipped: null pointer");
  if (src_off[0] != 0) return fail(e, DCB_ERR_INVALID, "dcb_fill_skipped: src_off[0] must be 0");
  for (int j = 0; j < k; ++j)
    if (src_off[j + 1] < src_off[j] || dst_off[j] < 0)
      return fail(e, DCB_ERR_INVALID, "dcb_fill_skipped: src_off must be non-decreasing, dst_off non-negative");
  CU(e, cudaSetDevice(e->cfg.device));
  cudaStream_t st = e->stream;
  const size_t n = (size_t)src_off[k];
  const bool out_dev = flags & DCB_OUT_ON_DEVICE;
  int rc;
  if ((rc = ensure(e, e->sc_ids, n ? n : 1)) || (rc = ensure(e, e->sc_bq, (n ? n : 1) * sizeof(int16_t))) ||
      (rc = ensure(e, e->sc_dst, (2 * (size_t)k + 1) * sizeof(int64_t))) || (rc = ensure(e, e->sc_mask, sizeof(int))))
    return rc;
  if (!out_dev && ((rc = ensure(e, e->sc_tmpb, n ? n : 1)) || (rc = ensure(e, e->sc_tmpq, n ? n : 1)))) return rc;
  int64_t* d_src = static_cast<int64_t*>(e->sc_dst.p);
  int64_t* d_dst = d_src + k + 1;
  CU(e, cudaMemcpyAsync(e->sc_ids.p, ccs_ids, n, cudaMemcpyHostToDevice, st));
  CU(e, cudaMemcpyAsync(e->sc_bq.p, ccs_bq, n * sizeof(int16_t), cudaMemcpyHostToDevice, st));
  CU(e, cudaMemcpyAsync(d_src, src_off, ((size_t)k + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
  // host outputs: a dense temporary laid out like the source, scattered on the host below
  CU(e, cudaMemcpyAsync(d_dst, out_dev ? dst_off : src_off, (size_t)k * sizeof(int64_t), cudaMemcpyHostToDevice, st));
  CU(e, cudaMemsetAsync(e->sc_mask.p, 0, sizeof(int), st));
  uint8_t* db = out_dev ? bases : static_cast<uint8_t*>(e->sc_tmpb.p);
  uint8_t* dq = out_dev ? quals : static_cast<uint8_t*>(e->sc_tmpq.p);
  launch_fill_skipped(static_cast<const uint8_t*>(e->sc_ids.p), static_cast<const int16_t*>(e->sc_bq.p), d_src, d_dst, k,
                      calibration_enabled, calibration_threshold, calibration_w, calibration_b, e->cfg.max_base_quality,
                      db, dq, static_cast<int*>(e->sc_mask.p), st);
  int status = 0;
  CU(e, cudaMemcpyAsync(&status, e->sc_mask.p, sizeof(int), cudaMemcpyDeviceToHost, st));
  if (!out_dev) {
    std::vector<uint8_t> hb(n), hq(n);
    CU(e, cudaMemcpyAsync(hb.data(), db, n, cudaMemcpyDeviceToHost, st));
    CU(e, cudaMemcpyAsync(hq.data(), dq, n, cudaMemcpyDeviceToHost, st));
    CU(e, cudaStreamSynchronize(st));
    for (int j = 0; j < k; ++j) {
      memcpy(bases + dst_off[j], hb.data() + src_off[j], (size_t)(src_off[j + 1] - src_off[j]));
      memcpy(quals + dst_off[j], hq.data() + src_off[j], (size_t)(src_off[j + 1] - src_off[j]));
    }
  } else {
    CU(e, cudaStreamSynchronize(st));
  }
  CU(e, cudaGetLastError());
  if (status & 1) return fail(e, DCB_ERR_INPUT_RANGE, "dcb_fill_skipped: CCS base id outside 0..4 (clamped)");
  return DCB_OK;
}

int dcb_debug_trace(uint64_t* out, int32_t n) {
  return read_ffn_trace(reinterpret_cast<unsigned long long*>(out), n) ? DCB_ERR_CUDA : DCB_OK;
}

int dcb_alloc_host(size_t bytes, void** out) {
  if (!out) return DCB_ERR_INVALID;
  return cudaMallocHost(out, bytes) == cudaSuccess ? DCB_OK : DCB_ERR_CUDA;
}
int dcb_free_host(void* p) { return cudaFreeHost(p) == cudaSuccess ? DCB_OK : DCB_ERR_CUDA; }

int dcb_alloc_device(dcb_engine* e, size_t bytes, void** out) {
  if (!e || !out) return DCB_ERR_INVALID;
  CU(e, cudaSetDevice(e->cfg.device));
  CU(e, cudaMalloc(out, bytes));
  return DCB_OK;
}
int dcb_free_device(dcb_engine* e, void* p) {
  if (!e) return DCB_ERR_INVALID;
  CU(e, cudaSetDevice(e->cfg.device));
  CU(e, cudaFree(p));
  return DCB_OK;
}
int dcb_memcpy_h2d(dcb_engine* e, void* dst, const void* src, size_t bytes) {
  if (!e) return DCB_ERR_INVALID;
  CU(e, cudaSetDevice(e->cfg.device));
  CU(e, cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice));
  return DCB_OK;
}
int dcb_memcpy_d2h(dcb_engine* e, void* dst, const void* src, size_t bytes) {
  if (!e) return DCB_ERR_INVALID;
  CU(e, cudaSetDevice(e->cfg.device));
  CU(e, cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
  return DCB_OK;
}
int dcb_synchronize(dcb_engine* e) {
  if (!e) return DCB_ERR_INVALID;
  CU(e, cudaSetDevice(e->cfg.device));
  CU(e, cudaDeviceSynchronize());
  return DCB_OK;
}

}  // extern "C"
