// Whole-path plan: forward / backward of the LSTUR training graph on one stream.
//
// Mirrors Seq2VecPaperSoftmaxId._build_model (task/paper.py:635-665): TimeDistributed news
// encoder over the B*W clicked titles and the B*C candidates, ComputeMasking multiply, user
// encoder (user-ID embedding + masked GRU), dot scorer, softmax + categorical cross-entropy.
// Host-side code only sequences kernels and carves the caller-provided workspace; all arithmetic
// is in the kernels of this directory.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "common.cuh"

namespace lstur {

static thread_local char g_err[512] = "";
unsigned long long g_launch_count = 0;
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// Workspace regions of a plan as (element type, name), in carve order.  lstur_plan_create carves the ones its
// configuration uses; lstur_plan_view serves them by name.
#define LSTUR_WS_REGIONS(X)                                                                                             \
  X(int, tokens) X(float, Xp) X(float, Cp) X(void, emb_bf16) X(void, wimg) X(void, C16) X(void, xmask)                 \
  X(int, title_flags) X(int, live_idx) X(int, n_live) X(int, tokens_c) X(float, att_a) X(float, att_w)                 \
  X(float, pooled) X(float, doc_vec) X(int, title_vert) X(int, title_subvert) X(float, vert_grad_ws)                   \
  X(float, hist_mask) X(float, gru_mask) X(float, u0) X(int, hist_live_idx) X(int, n_hist_live)                        \
  X(int, hist_live_scratch) X(int, hist_live_dummy) X(float, XW) X(float, hT) X(int, gru_key) X(int, gru_order)         \
  X(int, gru_sort_scratch) X(float, Z) X(float, R) X(float, HH) X(float, HP) X(float, RH) X(float, LI) X(float, LF)    \
  X(float, LG) X(float, LO) X(float, LCP) X(float, LHP) X(float, LTC) X(float, ua_a) X(float, ua_w)                    \
  X(float, ua_partial) X(float, seq2) X(float, mask2) X(float, d_seq2) X(float, d_hT) X(float, d_uh)                   \
  X(float, alpha_partial) X(float, cat) X(float, user_vec) X(float, sc_cat) X(float, sc_hid) X(float, sc_raw)           \
  X(float, sc_ones) X(float, sc_uh) X(float, sc_dh) X(int, vs_label) X(float, vs_hid) X(float, vs_logit)               \
  X(float, vs_probs) X(float, vs_loss_rows) X(float, vs_loss) X(float, vs_dlogit) X(float, vs_dhid) X(float, vs_ddoc)  \
  X(int, vc_label) X(float, vc_logit) X(float, vc_probs) X(float, vc_loss_rows) X(float, vc_loss) X(float, vc_dlogit)  \
  X(float, logits) X(float, probs) X(float, loss_rows) X(float, loss) X(float, d_user_vec) X(float, d_logits)          \
  X(float, d_doc_vec) X(float, d_pooled) X(float, dPre) X(void, dpre_img) X(void, wgrad_partial) X(void, wimg_d)       \
  X(void, dx16) X(float, dXp) X(void, wg_ws) X(float, attn_partials) X(float, WhT) X(float, gru_db_partial)            \
  X(float, dA) X(float, dh0) X(float, d_cat) X(float, sc_dhid) X(float, sc_whid) X(float, sc_dcat)                     \
  X(float, sc_dlogit) X(float, sc_scratch) X(float, sc_duh) X(float, sc_ddh) X(int, sorted_pos) X(int, user_rows)      \
  X(int, seg_start) X(int, inverse) X(int, n_user_rows) X(float, d_user_rows) X(float, d_u0) X(int, ev_user)           \
  X(float, ev_scale) X(float, ev_scale2) X(int, ev_off) X(int, ev_pair_row) X(void, gemm_ws) X(float, colsum_ws)

// Tensors of the dense-parameter arena, in layout order; lstur_plan_dense_offset serves them by name.
#define LSTUR_DENSE_TENSORS(X)                                                                                          \
  X(conv_w) X(conv_b) X(att_w) X(att_b) X(dense_w) X(dense_b) X(vert_emb) X(subvert_emb) X(gru_wx) X(gru_wh) X(gru_b)   \
  X(lstm_wx) X(lstm_wh) X(lstm_b) X(uatt_w) X(uatt_b) X(alpha) X(con_w) X(con_b) X(sh_w) X(sh_b) X(so_w) X(so_b)       \
  X(su_w) X(su_b) X(sd_w) X(sd_b) X(vs_w1) X(vs_b1) X(vs_w2) X(vs_b2) X(vcls_w) X(vcls_b)

struct Region {
  size_t off = 0;         // bytes into the workspace / floats into the dense arena
  long long count = 0;    // elements (4-byte)
  bool carved = false;    // part of this configuration; a region that is not yields nullptr (kernels take it as "absent")
  size_t bytes() const { return (size_t)count * 4; }
};
template <typename T>
struct WsRegion : Region {
  T* operator()(void* ws) const { return carved ? (T*)((char*)ws + off) : nullptr; }
};
struct DenseTensor : Region {
  const float* operator()(const float* arena) const { return carved ? arena + off : nullptr; }
  float* operator()(float* arena) const { return carved ? arena + off : nullptr; }
};
struct WsLayout {
#define X(T, name) WsRegion<T> name;
  LSTUR_WS_REGIONS(X)
#undef X
};
struct DenseLayout {
#define X(name) DenseTensor name;
  LSTUR_DENSE_TENSORS(X)
#undef X
};

}  // namespace lstur

struct lstur_plan {
  lstur_config c;
  int N, Nh, Nc, Lp, D;
  lstur::WsLayout ws;
  lstur::DenseLayout dense;
  size_t ws_bytes = 0;
  long long dense_count = 0;
  size_t gemm_ws_bytes = 0;
  // code paths of the step, decided by lstur_plan_create
  bool tc_prec = false;         // tensor-core precision: tcgen05 news encoder and dense GEMMs
  bool compact_titles = false;  // the news encoder runs over the compacted list of live titles (live_idx, n_live)
  bool live_hist_rows = false;  // list of the unmasked (user, step) rows for the GRU-side GEMMs (hist_live_idx, n_hist_live)
  bool gru_sort = false;        // the recurrence takes the batch rows sorted by history length (gru_order)
  bool tc_gru = false;          // the GRU recurrence runs on tcgen05 (gru_tc.cu): tensor-core precision, lstur_gru_tc_supported
  bool cat_head = false;        // the user vector is built from [GRU output ‖ id vector] (cat)
  // optional CUDA events recorded around one kernel of the step (bench.py roofline probe)
  int probe_id = 0;
  cudaEvent_t probe_start = nullptr, probe_stop = nullptr;
  // the 16-bit copy of the (frozen) word table in the workspace is re-packed only when its source / destination
  // changes or lstur_plan_invalidate_tables() was called (the table was written)
  const void* emb16_src = nullptr;
  void* emb16_dst = nullptr;
  // data-parallel overlap: recorded by lstur_backward once every gradient except the title-encoder bucket (conv_w, conv_b,
  // att_w, att_b = the first dense_head floats of the arena) and the user-row gradients are final
  cudaEvent_t ev_tail_ready = nullptr;
  long long dense_head = 0;
  unsigned last_seed = 0;   // seed / mode of the last forward (backward replays its dropout streams)
  int last_training = 0;
  int last_aux = 0;        // the last forward ran the auxiliary vertical classifier (labels were given)
  int last_cls_n = 0;      // titles of the last lstur_title_cls_forward
};

#define PROBE_BEGIN(p, id, st) do { if ((p)->probe_id == (id) && (p)->probe_start) cudaEventRecord((p)->probe_start, st); } while (0)
#define PROBE_END(p, id, st) do { if ((p)->probe_id == (id) && (p)->probe_stop) cudaEventRecord((p)->probe_stop, st); } while (0)

#define RC(x)              \
  do {                     \
    int rc__ = (x);        \
    if (rc__) return rc__; \
  } while (0)

using namespace lstur;

extern "C" const char* lstur_last_error(void) { return g_err; }
extern "C" const char* lstur_version(void) { return "lstur_b200 0.1 (sm_100a)"; }
extern "C" unsigned long long lstur_launch_count(void) { return g_launch_count; }
extern "C" int lstur_plan_set_probe(lstur_plan* plan, int probe_id, void* start_event, void* stop_event) {
  LSTUR_REQUIRE(plan != nullptr, "lstur_plan_set_probe");
  plan->probe_id = probe_id;
  plan->probe_start = (cudaEvent_t)start_event;
  plan->probe_stop = (cudaEvent_t)stop_event;
  return LSTUR_OK;
}
extern "C" int lstur_plan_set_event(lstur_plan* plan, int which, void* event) {
  LSTUR_REQUIRE(plan != nullptr && which == LSTUR_EVENT_TAIL_GRADS_READY, "lstur_plan_set_event");
  plan->ev_tail_ready = (cudaEvent_t)event;
  return LSTUR_OK;
}
extern "C" long long lstur_plan_dense_head_count(const lstur_plan* plan) { return plan ? plan->dense_head : 0; }
extern "C" int lstur_stream_wait_event(cudaStream_t stream, void* event) {
  cudaError_t e = cudaStreamWaitEvent(stream, (cudaEvent_t)event, 0);
  if (e != cudaSuccess) { set_error("cudaStreamWaitEvent: %s", cudaGetErrorString(e)); return LSTUR_ERR_CUDA; }
  return LSTUR_OK;
}
extern "C" int lstur_event_record(void* event, cudaStream_t stream) {
  cudaError_t e = cudaEventRecord((cudaEvent_t)event, stream);
  if (e != cudaSuccess) { set_error("cudaEventRecord: %s", cudaGetErrorString(e)); return LSTUR_ERR_CUDA; }
  return LSTUR_OK;
}
extern "C" int lstur_event_create(void** ev) {
  LSTUR_REQUIRE(ev != nullptr, "lstur_event_create");
  cudaEvent_t e;
  if (cudaEventCreate(&e) != cudaSuccess) { set_error("cudaEventCreate failed"); return LSTUR_ERR_CUDA; }
  *ev = (void*)e;
  return LSTUR_OK;
}
extern "C" int lstur_event_destroy(void* ev) { return cudaEventDestroy((cudaEvent_t)ev) == cudaSuccess ? LSTUR_OK : LSTUR_ERR_CUDA; }
extern "C" int lstur_event_elapsed_ms(void* a, void* b, float* ms) {
  cudaError_t e = cudaEventElapsedTime(ms, (cudaEvent_t)a, (cudaEvent_t)b);
  if (e != cudaSuccess) { set_error("cudaEventElapsedTime: %s", cudaGetErrorString(e)); return LSTUR_ERR_CUDA; }
  return LSTUR_OK;
}

namespace {

void add_ws(lstur_plan* p, Region& r, long long count) {
  size_t off = (p->ws_bytes + 255) & ~(size_t)255;
  r = Region{off, count, true};
  p->ws_bytes = off + (size_t)count * 4;
}
void add_dense(lstur_plan* p, Region& r, long long count) {
  long long off = (p->dense_count + 3) & ~3LL;
  r = Region{(size_t)off, count, true};
  p->dense_count = off + count;
}
// the carved region / tensor called `name`; nullptr if no region of that name is carved in this configuration
const Region* ws_region(const lstur_plan* p, const char* name) {
#define X(T, n) if (!strcmp(name, #n)) return p->ws.n.carved ? &p->ws.n : nullptr;
  LSTUR_WS_REGIONS(X)
#undef X
  return nullptr;
}
const Region* dense_tensor(const lstur_plan* p, const char* name) {
#define X(n) if (!strcmp(name, #n)) return p->dense.n.carved ? &p->dense.n : nullptr;
  LSTUR_DENSE_TENSORS(X)
#undef X
  return nullptr;
}
void track_gemm(lstur_plan* p, int M, int N, int K) {
  size_t b = lstur_gemm_f32_workspace_bytes(M, N, K, nullptr);
  size_t b2 = lstur_gemm_tc_workspace_bytes(M, N, K);
  if (b2 > b) b = b2;
  if (b > p->gemm_ws_bytes) p->gemm_ws_bytes = b;
}
typedef int (*gemm_fn)(int, int, int, int, int, const float*, long long, const float*, long long, float*, long long,
                       const float*, int, void*, size_t, cudaStream_t);
// user-encoder architecture classes
inline bool arch_has_gru(int a) {
  return a == LSTUR_ARCH_INI || a == LSTUR_ARCH_CON_DENSE || a == LSTUR_ARCH_CON_CAT || a == LSTUR_ARCH_NOID ||
         a == LSTUR_ARCH_ADD || a == LSTUR_ARCH_INI_CAT || a == LSTUR_ARCH_INI_CON || a == LSTUR_ARCH_INI_ADD ||
         a == LSTUR_ARCH_ATT_PAIR || a == LSTUR_ARCH_ALPHA;
}
inline bool arch_has_lstm(int a) { return a == LSTUR_ARCH_LSTM_CAT; }
inline bool arch_has_user(int a) { return a != LSTUR_ARCH_NOID && a != LSTUR_ARCH_AVG && a != LSTUR_ARCH_ATT; }
inline bool arch_hist_avg(int a) { return a == LSTUR_ARCH_AVG || a == LSTUR_ARCH_AVG_CAT; }
inline bool arch_hist_att(int a) { return a == LSTUR_ARCH_ATT || a == LSTUR_ARCH_ATT_CAT; }
// width of the user-embedding part that joins a concat / add ('iigru', 'inigru', 'inagru': the second table = columns G..)
inline int arch_uc(const lstur_config& c) {
  return (c.arch == LSTUR_ARCH_INI_CON || c.arch == LSTUR_ARCH_INI_CAT || c.arch == LSTUR_ARCH_INI_ADD) ? c.Ue - c.G : c.Ue;
}
// the tensor-core precision modes (tcgen05 news encoder, dense GEMMs and, where it fits, GRU recurrence)
inline bool prec_tc(const lstur_config& c) { return c.precision == LSTUR_PREC_BF16_TC || c.precision == LSTUR_PREC_FP16_TC; }
inline gemm_fn pick_gemm(const lstur_plan* p) { return p->tc_prec ? lstur_gemm_tc : lstur_gemm_f32; }

// C = A . op(B) (+ bias) over all M rows of A or, when `listed`, over the rows rows[0..*n_rows) only (the other rows of C
// are left untouched): the plan's dense GEMM, or lstur_gemm_tc_mrows on one of the plan's row lists.
int gemm_mrows(const lstur_plan* p, void* ws, bool listed, const int* rows, const int* n_rows, int transB, int M, int N,
               int K, const float* A, long long lda, const float* B, long long ldb, float* C, long long ldc,
               const float* bias, int flags, cudaStream_t st) {
  void* gws = p->ws.gemm_ws(ws);
  if (listed)
    return lstur_gemm_tc_mrows(transB, M, N, K, A, lda, B, ldb, C, ldc, bias, flags, rows, n_rows, gws, p->gemm_ws_bytes, st);
  return pick_gemm(p)(0, transB, M, N, K, A, lda, B, ldb, C, ldc, bias, flags, gws, p->gemm_ws_bytes, st);
}
// C[M,N] = A^T B summed over all K rows of A and B (stored [K,.]) or, when `listed`, over the rows rows[0..*n_rows) only.
int gemm_tn_rows(const lstur_plan* p, void* ws, bool listed, const int* rows, const int* n_rows, int M, int N, int K,
                 const float* A, long long lda, const float* B, long long ldb, float* C, long long ldc, cudaStream_t st) {
  void* gws = p->ws.gemm_ws(ws);
  if (listed) return lstur_gemm_tc_tn_rows(M, N, K, A, lda, B, ldb, C, ldc, rows, n_rows, gws, p->gemm_ws_bytes, st);
  return pick_gemm(p)(1, 0, M, N, K, A, lda, B, ldb, C, ldc, nullptr, 0, gws, p->gemm_ws_bytes, st);
}

// End of an entry point: report an error left by any launch or copy it enqueued.  Unlike LSTUR_CHECK_LAUNCH it counts
// no kernel launch.
int cuda_status(const char* entry) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: %s", entry, cudaGetErrorString(e));
    return LSTUR_ERR_CUDA;
  }
  return LSTUR_OK;
}

}  // namespace

extern "C" int lstur_plan_create(const lstur_config* cfg, lstur_plan** out) {
  LSTUR_REQUIRE(cfg && out, "lstur_plan_create");
  const lstur_config& c = *cfg;
  LSTUR_REQUIRE(c.B > 0 && c.W > 0 && c.C >= 1 && c.C <= 32 && c.L > 0 && c.L <= 256, "lstur_plan_create");
  LSTUR_REQUIRE(c.E > 0 && c.F > 0 && c.KS >= 1 && c.KS <= c.L, "lstur_plan_create");
  LSTUR_REQUIRE(c.dropout >= 0.f && c.dropout < 1.f, "lstur_plan_create");
  if (c.score_model < LSTUR_SCORE_DOT || c.score_model > LSTUR_SCORE_DDOT_LINEAR) {
    set_error("lstur_plan_create: score_model %d not implemented (NotImplementedError, task/paper.py:457)", c.score_model);
    return LSTUR_ERR_UNSUPPORTED;
  }
  if (c.arch < LSTUR_ARCH_INI || c.arch > LSTUR_ARCH_LSTM_CAT) {
    set_error("lstur_plan_create: Unsupport user model (task/paper.py:630)");
    return LSTUR_ERR_UNSUPPORTED;
  }
  LSTUR_REQUIRE(c.dv >= 0 && c.ds >= 0 && (c.dv == 0 || c.n_vert > 0) && (c.ds == 0 || c.n_subvert > 0), "lstur_plan_create");
  const int Dd = c.use_dense ? c.Dd : c.F;
  const int D = Dd + c.dv + c.ds;
  const bool has_gru = arch_has_gru(c.arch), has_lstm = arch_has_lstm(c.arch), has_rnn = has_gru || has_lstm;
  const bool has_user = arch_has_user(c.arch);
  const int NG = has_lstm ? 4 : 3;   // gates of the recurrent layer
  const bool dot = c.score_model == LSTUR_SCORE_DOT, dnn = c.score_model == LSTUR_SCORE_DNN, ddot = !dot && !dnn;
  LSTUR_REQUIRE(dot || c.Hs > 0, "lstur_plan_create('dnn' / 'ddot' scorers need Hs)");
  const bool bce = c.loss_model == LSTUR_LOSS_WEIGHTED_BCE;
  LSTUR_REQUIRE(c.loss_model == LSTUR_LOSS_SOFTMAX_CE || bce, "lstur_plan_create(loss_model)");
  LSTUR_REQUIRE(!bce || (c.C == 1 && c.bce_neg >= 1 && c.gain > 0.f), "lstur_plan_create(weighted BCE: C == 1, bce_neg >= 1, gain > 0)");
  LSTUR_REQUIRE(!has_rnn || (c.G > 0 && c.G <= 1024), "lstur_plan_create");
  LSTUR_REQUIRE(!has_user || (c.Ue > 0 && c.n_users > 0), "lstur_plan_create");
  // user-vector dim implied by the architecture
  int U = c.arch == LSTUR_ARCH_INI ? c.G : (c.arch == LSTUR_ARCH_CON_DENSE || c.arch == LSTUR_ARCH_INI_CON) ? c.U
          : c.arch == LSTUR_ARCH_CON_CAT ? c.G + c.Ue : c.arch == LSTUR_ARCH_INI_CAT ? c.Ue
          : c.arch == LSTUR_ARCH_NOID ? c.G : c.arch == LSTUR_ARCH_ADD ? c.G : c.arch == LSTUR_ARCH_AVG ? D
          : c.arch == LSTUR_ARCH_AVG_CAT ? D + c.Ue : c.arch == LSTUR_ARCH_ATT ? D : c.arch == LSTUR_ARCH_ATT_CAT ? D + c.Ue
          : c.arch == LSTUR_ARCH_ATT_PAIR ? 1     // 'atgru' pools 2G one-feature steps into one scalar (task/cook.py:184-190)
          : (c.arch == LSTUR_ARCH_INI_ADD || c.arch == LSTUR_ARCH_ALPHA) ? c.G
          : c.arch == LSTUR_ARCH_LSTM_CAT ? c.G + c.Ue : c.Ue;
  LSTUR_REQUIRE(U == c.U, "lstur_plan_create(U inconsistent with arch)");
  LSTUR_REQUIRE(c.arch != LSTUR_ARCH_INI || c.Ue == c.G, "lstur_plan_create(ini needs Ue == G)");
  LSTUR_REQUIRE(c.arch != LSTUR_ARCH_ADD || c.Ue == c.G, "lstur_plan_create(add needs Ue == G)");
  LSTUR_REQUIRE((c.arch != LSTUR_ARCH_INI_CON && c.arch != LSTUR_ARCH_INI_CAT) || c.Ue > c.G, "lstur_plan_create(ini+con needs Ue > G)");
  LSTUR_REQUIRE(c.arch != LSTUR_ARCH_INI_ADD || c.Ue == 2 * c.G, "lstur_plan_create('inagru' needs Ue == 2G)");
  LSTUR_REQUIRE((c.arch != LSTUR_ARCH_ATT_PAIR && c.arch != LSTUR_ARCH_ALPHA) || c.Ue == c.G, "lstur_plan_create('atgru' / 'algru' need Ue == G)");
  LSTUR_REQUIRE(!dot || U == D, "lstur_plan_create('dot' scorer needs user dim == doc dim)");
  if (prec_tc(c) && !lstur_tc_supported(c.L, c.E, c.F, c.KS)) {
    set_error("lstur_plan_create: shape (L=%d,E=%d,F=%d,KS=%d) not supported by the tensor-core conv kernel", c.L, c.E, c.F, c.KS);
    return LSTUR_ERR_UNSUPPORTED;
  }

  LSTUR_REQUIRE(!c.trainable_word_emb || (c.save_for_backward && c.E % 4 == 0 && c.E <= 512),
                "lstur_plan_create(trainable word table: training plan, E % 4 == 0, E <= 512)");
  LSTUR_REQUIRE(!c.save_for_backward || prec_tc(c) || c.F <= 1024,
                "lstur_plan_create(fp32 training plan: F <= 1024, the limit of the attention backward)");
  lstur_plan* p = new lstur_plan();
  p->c = c;
  p->c.Dd = Dd;
  p->Nh = c.B * c.W;
  p->Nc = c.B * c.C;
  p->N = p->Nh + p->Nc;
  p->Lp = c.L + c.KS - 1;
  p->D = D;
  const long long N = p->N, Nh = p->Nh, B = c.B, Lp = p->Lp;
  const int G = c.G, F = c.F, E = c.E;
  const bool bw = c.save_for_backward != 0;
  const int Uc = arch_uc(c);
  const bool con_dense = c.arch == LSTUR_ARCH_CON_DENSE || c.arch == LSTUR_ARCH_INI_CON;
  const bool tcp = prec_tc(c);
  p->tc_prec = tcp;
  // the tensor-core news encoder runs over the compacted list of live titles (lstur_compact_titles): everything inside
  // the encoder (tokens_c, C16, att_a, att_w, keep bits, dPre image, dX rows) is indexed by the compacted title index
  p->compact_titles = tcp;
  // ascending list of the unmasked (user, step) rows: the only rows of the GRU-side GEMMs that matter
  p->live_hist_rows = has_rnn && tcp;
  // batch rows sorted by history length (lstur_first_live_step) once the recurrence kernels' 4-CTA clusters of 32 rows
  // outnumber the SMs: the kernel is a W-step dependency chain per tile, so with every tile resident its time is that of
  // the longest history whatever the order (measured at B = 1024: 3.39 ms with the sort, 3.36 without); in a second wave
  // short tiles pair up
  p->gru_sort = has_gru && B > 1184 && B <= 16384;
  p->tc_gru = has_gru && tcp && lstur_gru_tc_supported(c.B, c.W, G);
  p->cat_head = con_dense || c.arch == LSTUR_ARCH_CON_CAT || c.arch == LSTUR_ARCH_INI_CAT;

  // ---- dense parameter layout
  DenseLayout& t = p->dense;
  add_dense(p, t.conv_w, (long long)c.KS * E * F);
  add_dense(p, t.conv_b, F);
  add_dense(p, t.att_w, F);
  add_dense(p, t.att_b, 1);
  p->dense_head = (p->dense_count + 3) & ~3LL;     // title-encoder bucket: its gradients are the last to become final
  if (c.use_dense) {
    add_dense(p, t.dense_w, (long long)F * Dd);
    add_dense(p, t.dense_b, Dd);
  }
  if (c.dv) add_dense(p, t.vert_emb, (long long)c.n_vert * c.dv);
  if (c.ds) add_dense(p, t.subvert_emb, (long long)c.n_subvert * c.ds);
  if (has_gru) {
    add_dense(p, t.gru_wx, (long long)D * 3 * G);
    add_dense(p, t.gru_wh, (long long)G * 3 * G);
    add_dense(p, t.gru_b, 3 * G);
  }
  if (has_lstm) {
    add_dense(p, t.lstm_wx, (long long)D * 4 * G);
    add_dense(p, t.lstm_wh, (long long)G * 4 * G);
    add_dense(p, t.lstm_b, 4 * G);
  }
  // SimpleAttentionMaskSupport over the history (W steps of width D) or, 'atgru', over the 2G entries of [GRU ; id vector]
  // taken as 2G steps of width 1: keras.backend.expand_dims(x, -1) + concatenate(axis=-2) in task/cook.py:186-188
  const int Da = arch_hist_att(c.arch) ? D : c.arch == LSTUR_ARCH_ATT_PAIR ? 1 : 0;
  const int Wa = arch_hist_att(c.arch) ? c.W : 2 * G;
  if (Da) {
    add_dense(p, t.uatt_w, Da);
    add_dense(p, t.uatt_b, 1);
  }
  if (c.arch == LSTUR_ARCH_ALPHA) add_dense(p, t.alpha, 1);
  if (con_dense) {
    add_dense(p, t.con_w, (long long)(G + Uc) * c.U);
    add_dense(p, t.con_b, c.U);
  }
  if (dnn) {
    add_dense(p, t.sh_w, (long long)(c.U + D) * c.Hs);
    add_dense(p, t.sh_b, c.Hs);
    add_dense(p, t.so_w, c.Hs);
    add_dense(p, t.so_b, 1);
  } else if (ddot) {
    add_dense(p, t.su_w, (long long)c.U * c.Hs);
    add_dense(p, t.su_b, c.Hs);
    add_dense(p, t.sd_w, (long long)D * c.Hs);
    add_dense(p, t.sd_b, c.Hs);
  }
  LSTUR_REQUIRE(c.aux_nv >= 0 && (c.aux_nv == 0 || c.aux_hidden > 0) && c.cls_nv >= 0, "lstur_plan_create(aux_nv / cls_nv)");
  if (c.aux_nv) {   // vertical classifier of ...VertSup (task/paper.py:948-952)
    add_dense(p, t.vs_w1, (long long)D * c.aux_hidden);
    add_dense(p, t.vs_b1, c.aux_hidden);
    add_dense(p, t.vs_w2, (long long)c.aux_hidden * c.aux_nv);
    add_dense(p, t.vs_b2, c.aux_nv);
  }
  if (c.cls_nv) {   // vertical model of ...VertAlt (task/paper.py:1128-1136)
    add_dense(p, t.vcls_w, (long long)D * c.cls_nv);
    add_dense(p, t.vcls_b, c.cls_nv);
  }
  p->dense_count = (p->dense_count + 3) & ~3LL;

  // ---- workspace
  WsLayout& r = p->ws;
  add_ws(p, r.tokens, N * c.L);
  if (!tcp) add_ws(p, r.Xp, N * Lp * E);
  if (!tcp) add_ws(p, r.Cp, N * Lp * F);
  if (tcp) {
    add_ws(p, r.emb_bf16, ((long long)c.V * lstur_tc_padded_e(E) + 1) / 2);
    add_ws(p, r.wimg, (lstur_tc_wimg_elems(E, F) + 1) / 2);
    add_ws(p, r.C16, (N * c.L * F + 1) / 2);
    if (bw && c.dropout > 0.f) add_ws(p, r.xmask, (long long)(lstur_tc_xmask_bytes((int)N, c.L, E) + 3) / 4);
  }
  if (p->compact_titles) {
    add_ws(p, r.title_flags, lstur_compact_titles_scratch_ints((int)N));
    add_ws(p, r.live_idx, N);
    add_ws(p, r.n_live, 1);
    add_ws(p, r.tokens_c, N * c.L);
  }
  add_ws(p, r.att_a, N * c.L);
  add_ws(p, r.att_w, N * c.L);
  add_ws(p, r.pooled, N * F);
  add_ws(p, r.doc_vec, N * D);
  if (c.dv + c.ds) {
    add_ws(p, r.title_vert, N);
    add_ws(p, r.title_subvert, N);
    if (bw) {
      size_t a = c.dv ? lstur_small_table_grad_workspace_bytes(c.n_vert, c.dv) : 0;
      size_t b2 = c.ds ? lstur_small_table_grad_workspace_bytes(c.n_subvert, c.ds) : 0;
      add_ws(p, r.vert_grad_ws, (long long)((a > b2 ? a : b2) / 4) + 4);
    }
  }
  add_ws(p, r.hist_mask, Nh);
  add_ws(p, r.gru_mask, Nh);
  if (has_user) add_ws(p, r.u0, B * c.Ue);
  if (p->live_hist_rows) {
    add_ws(p, r.hist_live_idx, Nh);
    add_ws(p, r.n_hist_live, 1);
    add_ws(p, r.hist_live_scratch, lstur_compact_titles_scratch_ints((int)Nh));
    add_ws(p, r.hist_live_dummy, Nh);
  }
  if (has_rnn) {
    add_ws(p, r.XW, Nh * NG * G);
    add_ws(p, r.hT, B * G);
    if (p->gru_sort) {
      add_ws(p, r.gru_key, B);
      add_ws(p, r.gru_order, B);
      add_ws(p, r.gru_sort_scratch, 3 * B + 2);
    }
    if (bw && has_gru) {
      for (Region* x : {&r.Z, &r.R, &r.HH, &r.HP, &r.RH}) add_ws(p, *x, Nh * G);
    }
    if (bw && has_lstm) {
      for (Region* x : {&r.LI, &r.LF, &r.LG, &r.LO, &r.LCP, &r.LHP, &r.LTC}) add_ws(p, *x, Nh * G);
    }
  }
  if (Da) {
    add_ws(p, r.ua_a, B * Wa);
    add_ws(p, r.ua_w, B * Wa);
    if (bw) add_ws(p, r.ua_partial, B * (Da + 1));
  }
  if (c.arch == LSTUR_ARCH_ATT_PAIR) {
    add_ws(p, r.seq2, B * 2 * G);
    add_ws(p, r.mask2, B * 2 * G);
    if (bw) add_ws(p, r.d_seq2, B * 2 * G);
  }
  if (c.arch == LSTUR_ARCH_ALPHA && bw) {
    add_ws(p, r.d_hT, B * G);
    add_ws(p, r.d_uh, B * c.Ue);
    add_ws(p, r.alpha_partial, B);
  }
  if (p->cat_head) add_ws(p, r.cat, B * (G + Uc));
  add_ws(p, r.user_vec, B * c.U);
  if (dnn) {
    add_ws(p, r.sc_cat, (long long)p->Nc * (c.U + D));
    add_ws(p, r.sc_hid, (long long)p->Nc * c.Hs);
    add_ws(p, r.sc_raw, p->Nc);
    add_ws(p, r.sc_ones, B);
    track_gemm(p, (int)p->Nc, c.Hs, c.U + D);
  } else if (ddot) {
    add_ws(p, r.sc_uh, B * c.Hs);
    add_ws(p, r.sc_dh, (long long)p->Nc * c.Hs);
    track_gemm(p, (int)B, c.Hs, c.U);
    track_gemm(p, (int)p->Nc, c.Hs, D);
  }
  if (c.aux_nv) {
    add_ws(p, r.vs_label, N);
    add_ws(p, r.vs_hid, N * c.aux_hidden);
    add_ws(p, r.vs_logit, N * c.aux_nv);
    add_ws(p, r.vs_probs, N * c.aux_nv);
    add_ws(p, r.vs_loss_rows, N);
    add_ws(p, r.vs_loss, 1);
    track_gemm(p, (int)N, c.aux_hidden, D);
    track_gemm(p, (int)N, c.aux_nv, c.aux_hidden);
    if (bw) {
      add_ws(p, r.vs_dlogit, N * c.aux_nv);
      add_ws(p, r.vs_dhid, N * c.aux_hidden);
      add_ws(p, r.vs_ddoc, N * D);
      track_gemm(p, c.aux_hidden, c.aux_nv, (int)N);
      track_gemm(p, (int)N, c.aux_hidden, c.aux_nv);
      track_gemm(p, D, c.aux_hidden, (int)N);
      track_gemm(p, (int)N, D, c.aux_hidden);
    }
  }
  if (c.cls_nv) {
    add_ws(p, r.vc_label, N);
    add_ws(p, r.vc_logit, N * c.cls_nv);
    add_ws(p, r.vc_probs, N * c.cls_nv);
    add_ws(p, r.vc_loss_rows, N);
    add_ws(p, r.vc_loss, 1);
    track_gemm(p, (int)N, c.cls_nv, D);
    if (bw) {
      add_ws(p, r.vc_dlogit, N * c.cls_nv);
      track_gemm(p, D, c.cls_nv, (int)N);
      track_gemm(p, (int)N, D, c.cls_nv);
    }
  }
  add_ws(p, r.logits, B * c.C);
  add_ws(p, r.probs, B * c.C);
  add_ws(p, r.loss_rows, B);
  add_ws(p, r.loss, 1);
  if (!tcp) track_gemm(p, (int)(N * Lp), F, c.KS * E);
  track_gemm(p, (int)N, Dd, F);
  if (bw) {
    add_ws(p, r.d_user_vec, B * c.U);
    if (bce) add_ws(p, r.d_logits, B * c.C);
    add_ws(p, r.d_doc_vec, N * D);
    add_ws(p, r.d_pooled, N * F);
    if (!tcp) add_ws(p, r.dPre, N * Lp * F);
    if (tcp) {
      add_ws(p, r.dpre_img, (long long)(lstur_tc_dpre_img_bytes((int)N, c.L, F) / 4));
      add_ws(p, r.wgrad_partial, (long long)(lstur_tc_wgrad_partial_bytes((int)N, E, F) / 4));
    }
    if (c.trainable_word_emb) {   // conv input gradient + word-table scatter (task/paper.py:136)
      if (tcp) {
        add_ws(p, r.wimg_d, (lstur_tc_wimg_dgrad_elems(E, F) + 1) / 2);
        add_ws(p, r.dx16, (N * c.L * lstur_tc_padded_e(E) + 1) / 2);
      } else {
        add_ws(p, r.dXp, N * Lp * E);
        track_gemm(p, (int)(N * Lp), E, F);
      }
      add_ws(p, r.wg_ws, (long long)(lstur_word_grad_workspace_bytes(N * c.L, c.V, E) / 4) + 4);
    }
    add_ws(p, r.attn_partials, (long long)lstur_attn_bwd_grid((int)N) * (2 * F + 1));
    if (has_rnn) {
      add_ws(p, r.WhT, (long long)NG * G * G);
      if (has_gru) add_ws(p, r.gru_db_partial, (long long)lstur_gru_tc_db_rows((int)B) * 3 * G);
      add_ws(p, r.dA, Nh * NG * G);
      add_ws(p, r.dh0, B * G);
    }
    if (con_dense) add_ws(p, r.d_cat, B * (G + Uc));
    if (dnn) {
      add_ws(p, r.sc_dhid, (long long)p->Nc * c.Hs);
      add_ws(p, r.sc_whid, (long long)p->Nc * c.Hs);
      add_ws(p, r.sc_dcat, (long long)p->Nc * (c.U + D));
      add_ws(p, r.sc_dlogit, p->Nc);
      add_ws(p, r.sc_scratch, B);
      track_gemm(p, c.U + D, c.Hs, (int)p->Nc);
      track_gemm(p, (int)p->Nc, c.U + D, c.Hs);
    } else if (ddot) {
      add_ws(p, r.sc_duh, B * c.Hs);
      add_ws(p, r.sc_ddh, (long long)p->Nc * c.Hs);
      track_gemm(p, c.U, c.Hs, (int)B);
      track_gemm(p, D, c.Hs, (int)p->Nc);
      track_gemm(p, (int)B, c.U, c.Hs);
      track_gemm(p, (int)p->Nc, D, c.Hs);
    }
    if (has_user) {
      add_ws(p, r.sorted_pos, B);
      add_ws(p, r.user_rows, B);
      add_ws(p, r.seg_start, B + 1);
      add_ws(p, r.inverse, B);
      add_ws(p, r.n_user_rows, 1);
      add_ws(p, r.d_user_rows, B * c.Ue);
      add_ws(p, r.d_u0, B * c.Ue);
    }
    if (!tcp) track_gemm(p, c.KS * E, F, (int)(N * Lp));
    track_gemm(p, F, Dd, (int)N);
    track_gemm(p, (int)N, F, Dd);
    if (has_rnn) {
      track_gemm(p, D, NG * G, (int)Nh);
      track_gemm(p, G, has_lstm ? 4 * G : 2 * G, (int)Nh);
      track_gemm(p, (int)Nh, D, NG * G);
    }
    if (con_dense) track_gemm(p, G + Uc, c.U, (int)B);
  }
  if (has_rnn) track_gemm(p, (int)Nh, NG * G, D);
  if (!bw) {   // lstur_score_impressions: one chunk's users and their scales, rebased candidate offsets and pair -> impression rows
    add_ws(p, r.ev_user, B);
    add_ws(p, r.ev_scale, B);
    add_ws(p, r.ev_scale2, B);
    add_ws(p, r.ev_off, B + 1);
    add_ws(p, r.ev_pair_row, p->Nc);
  }
  add_ws(p, r.gemm_ws, (long long)(p->gemm_ws_bytes / 4) + 4);
  {
    int cols = NG * G > D ? NG * G : D;
    if (c.U > cols) cols = c.U;
    if (c.Hs > cols) cols = c.Hs;
    if (c.aux_hidden > cols) cols = c.aux_hidden;
    if (c.aux_nv > cols) cols = c.aux_nv;
    if (c.cls_nv > cols) cols = c.cls_nv;
    add_ws(p, r.colsum_ws, (long long)1024 * cols);
  }
  p->ws_bytes = (p->ws_bytes + 255) & ~(size_t)255;
  *out = p;
  return LSTUR_OK;
}

extern "C" void lstur_plan_destroy(lstur_plan* plan) { delete plan; }
// The caller wrote the word-embedding table (or moved the workspace): derived copies must be rebuilt on the next forward.
extern "C" int lstur_plan_invalidate_tables(lstur_plan* plan) {
  LSTUR_REQUIRE(plan != nullptr, "lstur_plan_invalidate_tables");
  plan->emb16_src = nullptr;
  plan->emb16_dst = nullptr;
  return LSTUR_OK;
}
extern "C" size_t lstur_plan_workspace_bytes(const lstur_plan* plan) { return plan ? plan->ws_bytes : 0; }
extern "C" long long lstur_plan_dense_count(const lstur_plan* plan) { return plan ? plan->dense_count : 0; }

extern "C" int lstur_plan_dense_offset(const lstur_plan* plan, const char* name, long long* offset, long long* count) {
  LSTUR_REQUIRE(plan && name, "lstur_plan_dense_offset");
  const Region* t = dense_tensor(plan, name);
  if (!t) {
    set_error("lstur_plan_dense_offset: no tensor '%s' in this configuration", name);
    return LSTUR_ERR_ARG;
  }
  if (offset) *offset = (long long)t->off;
  if (count) *count = t->count;
  return LSTUR_OK;
}

extern "C" int lstur_plan_view(const lstur_plan* plan, void* workspace, const char* name, void** ptr, long long* count) {
  LSTUR_REQUIRE(plan && name && ptr, "lstur_plan_view");
  const Region* r = ws_region(plan, name);
  if (!r) {
    set_error("lstur_plan_view: no workspace region '%s'", name);
    return LSTUR_ERR_ARG;
  }
  *ptr = (char*)workspace + r->off;
  if (count) *count = r->count;
  return LSTUR_OK;
}

namespace {

// Tensor-core news encoder forward (k1-k6) over the first n title slots: tokens -> C16, pooled, att_a, att_w.
int encode_titles_tc(lstur_plan* p, const lstur_weights* w, void* ws, int n, int training, unsigned seed, cudaStream_t st) {
  const lstur_config& c = p->c;
  void* emb = p->ws.emb_bf16(ws);
  void* wimg = p->ws.wimg(ws);
  const int fp16 = c.precision == LSTUR_PREC_FP16_TC;
  if (p->emb16_src != (const void*)w->word_emb || p->emb16_dst != emb) {
    RC(lstur_pack_word_emb_16(c.V, c.E, w->word_emb, emb, fp16, st));
    p->emb16_src = w->word_emb;
    p->emb16_dst = emb;
  }
  RC(lstur_pack_conv_w_tc(c.E, c.F, p->dense.conv_w(w->dense), wimg, fp16, st));
  // Live titles only: an all-pad title (left padding of a short history) pools to exactly 0 and back-propagates exactly 0,
  // so the kernels run over the compacted title list; pooled rows of the dead titles are zeroed here.
  int* n_live = p->ws.n_live(ws);
  int* live_idx = p->ws.live_idx(ws);
  int* tok_c = p->ws.tokens_c(ws);
  float* pooled = p->ws.pooled(ws);
  RC(lstur_compact_titles(n, c.L, p->ws.tokens(ws), p->ws.title_flags(ws), live_idx, n_live, tok_c, st));
  cudaMemsetAsync(pooled, 0, (size_t)n * c.F * sizeof(float), st);
  PROBE_BEGIN(p, LSTUR_PROBE_CONV_FWD, st);
  // a training forward leaves the X-dropout keep bits for the weight-gradient kernel (workspace region xmask)
  void* xm = (training && c.dropout > 0.f && n == p->N) ? p->ws.xmask(ws) : nullptr;
  RC(lstur_news_conv_tc_fwd_m(n, c.L, c.E, c.F, c.V, tok_c, emb, wimg, p->dense.conv_b(w->dense), p->dense.att_w(w->dense),
                              p->dense.att_b(w->dense), p->ws.C16(ws), pooled, p->ws.att_a(ws), p->ws.att_w(ws),
                              training ? c.dropout : 0.f, seed, fp16, 0, xm, n_live, live_idx, st));
  PROBE_END(p, LSTUR_PROBE_CONV_FWD, st);
  return LSTUR_OK;
}

// News encoder (k1-k7) over the first n title slots of the workspace: tokens[0..n) -> doc_vec[0..n).
int encode_titles(lstur_plan* p, const lstur_weights* w, void* ws, int n, int training, unsigned seed, cudaStream_t st) {
  const lstur_config& c = p->c;
  const int Lp = p->Lp, D = p->D, L = c.L, E = c.E, F = c.F;
  const float drop = training ? c.dropout : 0.f;
  int* tok = p->ws.tokens(ws);
  float* pooled = p->ws.pooled(ws);
  float* docv = p->ws.doc_vec(ws);
  if (p->tc_prec) {
    RC(encode_titles_tc(p, w, ws, n, training, seed, st));
  } else {
    float* Xp = p->ws.Xp(ws);
    float* Cp = p->ws.Cp(ws);
    PROBE_BEGIN(p, LSTUR_PROBE_GATHER, st);
    RC(lstur_embed_gather_pad(n, L, E, c.V, c.KS, w->word_emb, tok, Xp, drop, seed * 2u + 0u, st));
    PROBE_END(p, LSTUR_PROBE_GATHER, st);
    PROBE_BEGIN(p, LSTUR_PROBE_CONV_FWD, st);
    RC(lstur_gemm_f32(0, 0, n * Lp - (c.KS - 1), F, c.KS * E, Xp, E, p->dense.conv_w(w->dense), F, Cp, F,
                      p->dense.conv_b(w->dense), LSTUR_GEMM_RELU, p->ws.gemm_ws(ws), p->gemm_ws_bytes, st));
    PROBE_END(p, LSTUR_PROBE_CONV_FWD, st);
    RC(lstur_attn_pool_fwd(n, L, F, Cp, (long long)Lp * F, tok, p->dense.att_w(w->dense), p->dense.att_b(w->dense),
                           pooled, F, p->ws.att_a(ws), p->ws.att_w(ws), drop, seed * 2u + 1u, st));
  }
  if (c.use_dense) {
    // with compacted titles, Dense over the live titles only; an all-pad title pools to 0, so its vector is the bias
    RC(gemm_mrows(p, ws, p->compact_titles, p->ws.live_idx(ws), p->ws.n_live(ws), 0, n, c.Dd, F, pooled, F,
                  p->dense.dense_w(w->dense), c.Dd, docv, D, p->dense.dense_b(w->dense), LSTUR_GEMM_PRECISE, st));
    if (p->compact_titles)
      RC(lstur_fill_rows_where(n, c.Dd, p->ws.title_flags(ws), 0, p->dense.dense_b(w->dense), docv, D, st));
  } else {
    cudaMemcpy2DAsync(docv, (size_t)D * 4, pooled, (size_t)F * 4, (size_t)F * 4, n, cudaMemcpyDeviceToDevice, st);
  }
  return LSTUR_OK;
}

// User encoder (k10-k12) on the history rows of doc_vec / gru_mask already in the workspace -> user_vec (B, U).
int user_vector(const lstur_plan* p, const lstur_weights* w, const lstur_batch* b, void* ws, cudaStream_t st) {
  const lstur_config& c = p->c;
  const int Nh = p->Nh, D = p->D, G = c.G, B = c.B;
  const gemm_fn GEMM = pick_gemm(p);
  float* docv = p->ws.doc_vec(ws);
  void* gws = p->ws.gemm_ws(ws);
  const size_t gwsb = p->gemm_ws_bytes;
  float* gmask = p->ws.gru_mask(ws);
  // 4. user embedding (k10)
  float* uvec = p->ws.user_vec(ws);
  float* u0 = p->ws.u0(ws);
  float* cat = p->ws.cat(ws);
  if (arch_has_user(c.arch)) {
    LSTUR_REQUIRE(w->user_emb != nullptr, "lstur_forward");
    const bool two = b->user_scale2 != nullptr && arch_uc(c) != c.Ue;   // independent multipliers for the two tables
    RC(lstur_row_gather(B, c.Ue, c.n_users, w->user_emb, b->user, two ? nullptr : b->user_scale, u0, c.Ue, st));
    if (two) {
      if (b->user_scale) RC(lstur_scale_rows(B, c.G, b->user_scale, u0, c.Ue, st));
      RC(lstur_scale_rows(B, c.Ue - c.G, b->user_scale2, u0 + c.G, c.Ue, st));
    }
  }
  // 5. GRU (k11-k12)
  if (arch_has_gru(c.arch)) {
    float* XW = p->ws.XW(ws);
    int* hl_idx = p->ws.hist_live_idx(ws);
    int* hl_n = p->ws.n_hist_live(ws);
    if (p->live_hist_rows) {   // unmasked (user, step) rows, ascending (the weight gradients of the backward reduce over them too)
      RC(lstur_compact_titles(Nh, 1, reinterpret_cast<const int*>(gmask), p->ws.hist_live_scratch(ws), hl_idx, hl_n,
                              p->ws.hist_live_dummy(ws), st));
    }
    // with the tcgen05 recurrence, the input projection of the unmasked steps only: the recurrence discards what it
    // computes for a masked step (select, not multiply), so the rows of XW behind masked steps are never used
    RC(gemm_mrows(p, ws, p->live_hist_rows && p->tc_gru, hl_idx, hl_n, 0, Nh, 3 * G, D, docv, D,
                  p->dense.gru_wx(w->dense), 3 * G, XW, 3 * G, p->dense.gru_b(w->dense), LSTUR_GEMM_PRECISE, st));
    float* hT = p->ws.hT(ws);
    float* hdst = hT;
    long long ldo = G;
    const bool ini = c.arch == LSTUR_ARCH_INI || c.arch == LSTUR_ARCH_INI_CON || c.arch == LSTUR_ARCH_INI_CAT ||
                     c.arch == LSTUR_ARCH_INI_ADD;
    const bool con_dense = c.arch == LSTUR_ARCH_CON_DENSE || c.arch == LSTUR_ARCH_INI_CON;
    const int Uc = arch_uc(c);
    if (c.arch == LSTUR_ARCH_INI || c.arch == LSTUR_ARCH_NOID || c.arch == LSTUR_ARCH_INI_ADD) hdst = uvec;
    if (p->cat_head) { hdst = cat; ldo = G + Uc; }
    if (c.arch == LSTUR_ARCH_ATT_PAIR) { hdst = p->ws.seq2(ws); ldo = 2 * G; }
    // tiles of 32 batch rows skip the steps at which all their rows are masked: order the rows by their first live step
    int* order = p->ws.gru_order(ws);
    if (p->gru_sort) {
      int* key = p->ws.gru_key(ws);
      int* scr = p->ws.gru_sort_scratch(ws);
      RC(lstur_first_live_step(B, c.W, gmask, key, st));
      RC(lstur_sort_unique_i32(B, key, order, scr, scr + B, scr + 2 * B + 1, scr + 3 * B + 1, st));
    }
    PROBE_BEGIN(p, LSTUR_PROBE_GRU_FWD, st);
    RC((p->tc_gru ? lstur_gru_fwd_tc : lstur_gru_fwd)(B, c.W, G, XW, gmask, ini ? u0 : nullptr, c.Ue,
                                                      p->dense.gru_wh(w->dense), c.rec_act, hdst, ldo, p->ws.Z(ws),
                                                      p->ws.R(ws), p->ws.HH(ws), p->ws.HP(ws), p->ws.RH(ws), order, st));
    PROBE_END(p, LSTUR_PROBE_GRU_FWD, st);
    if (p->cat_head) {
      cudaMemcpy2DAsync(cat + G, (size_t)(G + Uc) * 4, u0 + (c.Ue - Uc), (size_t)c.Ue * 4, (size_t)Uc * 4, B,
                        cudaMemcpyDeviceToDevice, st);
      if (con_dense) {
        RC(GEMM(0, 0, B, c.U, G + Uc, cat, G + Uc, p->dense.con_w(w->dense), c.U, uvec, c.U, p->dense.con_b(w->dense),
                LSTUR_GEMM_PRECISE, gws, gwsb, st));
      } else {
        cudaMemcpyAsync(uvec, cat, (size_t)B * c.U * 4, cudaMemcpyDeviceToDevice, st);
      }
    } else if (c.arch == LSTUR_ARCH_ADD) {
      cudaMemcpyAsync(uvec, hT, (size_t)B * G * 4, cudaMemcpyDeviceToDevice, st);
      RC(lstur_axpby((long long)B * G, 1.f, u0, 1.f, uvec, st));
    } else if (c.arch == LSTUR_ARCH_INI_ADD) {     // 'inagru': GRU(initial_state = table 1) + table 2 (task/cook.py:177-183)
      RC(lstur_add_rows(B, G, 1.f, u0 + G, c.Ue, 1.f, uvec, c.U, st));
    } else if (c.arch == LSTUR_ARCH_ATT_PAIR) {    // 'atgru': attention over the 2G scalar "steps" of [GRU output ; id vector]
      float* seq2 = p->ws.seq2(ws);
      float* mask2 = p->ws.mask2(ws);
      cudaMemcpy2DAsync(seq2 + G, (size_t)2 * G * 4, u0, (size_t)c.Ue * 4, (size_t)G * 4, B, cudaMemcpyDeviceToDevice, st);
      RC(lstur_rows_nonzero((long long)2 * G * B, 1, seq2, 1, mask2, st));       // Masking() on one-feature steps
      RC(lstur_seq_attn_fwd(B, 2 * G, 1, seq2, mask2, p->dense.uatt_w(w->dense), p->dense.uatt_b(w->dense), uvec, c.U,
                            p->ws.ua_a(ws), p->ws.ua_w(ws), st));
    } else if (c.arch == LSTUR_ARCH_ALPHA) {       // 'algru': models.AlphaAdd (models.py:540-554)
      RC(lstur_alpha_add_fwd(B, G, p->dense.alpha(w->dense), hT, G, u0, c.Ue, uvec, c.U, st));
    }
  } else if (arch_has_lstm(c.arch)) {   // 'ilstm': [LSTM(history) ‖ id vector] (task/cook.py:161-163)
    float* XW = p->ws.XW(ws);
    RC(GEMM(0, 0, Nh, 4 * G, D, docv, D, p->dense.lstm_wx(w->dense), 4 * G, XW, 4 * G, p->dense.lstm_b(w->dense),
            LSTUR_GEMM_PRECISE, gws, gwsb, st));
    RC(lstur_lstm_fwd(B, c.W, G, XW, gmask, p->dense.lstm_wh(w->dense), c.rec_act, uvec, c.U, p->ws.LI(ws), p->ws.LF(ws),
                      p->ws.LG(ws), p->ws.LO(ws), p->ws.LCP(ws), p->ws.LHP(ws), p->ws.LTC(ws), st));
    cudaMemcpy2DAsync(uvec + G, (size_t)c.U * 4, u0, (size_t)c.Ue * 4, (size_t)c.Ue * 4, B, cudaMemcpyDeviceToDevice, st);
  } else if (arch_hist_avg(c.arch)) {   // 'niavg' / cook 'iavg': masked mean of the history vectors (models.py:422-441)
    RC(lstur_masked_mean_fwd(B, c.W, D, docv, gmask, uvec, c.U, st));
    if (c.arch == LSTUR_ARCH_AVG_CAT)
      cudaMemcpy2DAsync(uvec + D, (size_t)c.U * 4, u0, (size_t)c.Ue * 4, (size_t)c.Ue * 4, B, cudaMemcpyDeviceToDevice, st);
  } else if (arch_hist_att(c.arch)) {   // 'att' / cook 'iatt': attention pooling of the history (models.py:474-489)
    RC(lstur_seq_attn_fwd(B, c.W, D, docv, gmask, p->dense.uatt_w(w->dense), p->dense.uatt_b(w->dense), uvec, c.U,
                          p->ws.ua_a(ws), p->ws.ua_w(ws), st));
    if (c.arch == LSTUR_ARCH_ATT_CAT)
      cudaMemcpy2DAsync(uvec + D, (size_t)c.U * 4, u0, (size_t)c.Ue * 4, (size_t)c.Ue * 4, B, cudaMemcpyDeviceToDevice, st);
  } else {
    cudaMemcpyAsync(uvec, u0, (size_t)B * c.Ue * 4, cudaMemcpyDeviceToDevice, st);
  }
  return LSTUR_OK;
}

// Operands of the scorer's final dot product, user side u (B rows) and document side d (one row per pair):
struct ScoreOperands {
  const float* u;
  long long ldu;
  const float* d;
  long long ldd;
  int dim;
};
// the scorer up to that product for n_pairs (user, candidate) pairs: user_vec against the candidate rows of doc_vec
// ('dot'), relu Dense on [u ‖ d] then Dense(1), the raw scores against a vector of ones ('dnn', task/paper.py:448-451,
// 222-226), or Dense(Hs) on both sides, tanh in the paper flavour and linear in cook ('ddot', task/paper.py:452-455).
// pair_row gives each pair's user row; NULL = C consecutive pairs per user.
int score_operands(const lstur_plan* p, const lstur_weights* w, void* ws, int n_pairs, const int* pair_row,
                   ScoreOperands* s, cudaStream_t st) {
  const lstur_config& c = p->c;
  const int D = p->D, B = c.B;
  const gemm_fn GEMM = pick_gemm(p);
  void* gws = p->ws.gemm_ws(ws);
  const size_t gwsb = p->gemm_ws_bytes;
  const float* uvec = p->ws.user_vec(ws);
  const float* cand = p->ws.doc_vec(ws) + (size_t)p->Nh * D;
  *s = ScoreOperands{uvec, c.U, cand, D, D};
  if (c.score_model == LSTUR_SCORE_DNN) {
    const int K2 = c.U + D;
    float* sc_cat = p->ws.sc_cat(ws);
    float* hid = p->ws.sc_hid(ws);
    float* raw = p->ws.sc_raw(ws);
    float* ones = p->ws.sc_ones(ws);
    RC(lstur_pair_concat(n_pairs, pair_row ? 1 : c.C, c.U, D, uvec, c.U, cand, D, sc_cat, pair_row, st));
    RC(GEMM(0, 0, n_pairs, c.Hs, K2, sc_cat, K2, p->dense.sh_w(w->dense), c.Hs, hid, c.Hs, p->dense.sh_b(w->dense),
            LSTUR_GEMM_RELU | LSTUR_GEMM_PRECISE, gws, gwsb, st));
    RC(lstur_rowdot_bias(n_pairs, c.Hs, hid, p->dense.so_w(w->dense), p->dense.so_b(w->dense), raw, st));
    RC(lstur_fill(B, 1.f, ones, st));
    *s = ScoreOperands{ones, 1, raw, 1, 1};
  } else if (c.score_model != LSTUR_SCORE_DOT) {
    float* uh = p->ws.sc_uh(ws);
    float* dh = p->ws.sc_dh(ws);
    RC(GEMM(0, 0, B, c.Hs, c.U, uvec, c.U, p->dense.su_w(w->dense), c.Hs, uh, c.Hs, p->dense.su_b(w->dense),
            LSTUR_GEMM_PRECISE, gws, gwsb, st));
    RC(GEMM(0, 0, n_pairs, c.Hs, D, cand, D, p->dense.sd_w(w->dense), c.Hs, dh, c.Hs, p->dense.sd_b(w->dense),
            LSTUR_GEMM_PRECISE, gws, gwsb, st));
    if (c.score_model == LSTUR_SCORE_DDOT) {
      RC(lstur_tanh_fwd((long long)B * c.Hs, uh, st));
      RC(lstur_tanh_fwd((long long)n_pairs * c.Hs, dh, st));
    }
    *s = ScoreOperands{uh, c.Hs, dh, c.Hs, c.Hs};
  }
  return LSTUR_OK;
}

// User encoder + scorer + loss (k10-k14) on doc_vec / gru_mask already in the workspace.
int user_and_score(const lstur_plan* p, const lstur_weights* w, const lstur_batch* b, void* ws, cudaStream_t st) {
  const lstur_config& c = p->c;
  const int B = c.B;
  RC(user_vector(p, w, b, ws, st));
  // 6. score + softmax + loss (k13-k14): the softmax / CE kernel fuses the final dot product, the sigmoid head takes raw
  // scores
  ScoreOperands s;
  RC(score_operands(p, w, ws, p->Nc, nullptr, &s, st));
  float* logits = p->ws.logits(ws);
  float* probs = p->ws.probs(ws);
  float* loss_rows = p->ws.loss_rows(ws);
  float* loss = p->ws.loss(ws);
  if (c.loss_model != LSTUR_LOSS_WEIGHTED_BCE) {
    RC(lstur_score_softmax_ce(B, c.C, s.dim, s.u, s.ldu, s.d, s.ldd, b->label, logits, probs, loss_rows, loss, nullptr, 0,
                              nullptr, 0, 0.f, st));
  } else {
    // sigmoid head + weighted BCE (task/paper.py:222-256, task/seq2vec.py:213-216); without labels (inference) only
    // the probabilities are produced
    RC(lstur_score_sigmoid(p->Nc, c.C, s.dim, s.u, s.ldu, s.d, s.ldd, logits, 0, st));
    if (b->label) RC(lstur_bce_loss(p->Nc, logits, b->label, c.gain, c.bce_neg, probs, loss_rows, loss, nullptr, 0.f, st));
    else RC(lstur_score_sigmoid(p->Nc, c.C, s.dim, s.u, s.ldu, s.d, s.ldd, probs, 1, st));
  }
  return cuda_status("lstur_forward");
}

// lstur_encode_docs / lstur_encode_titles: the n title rows, gathered by document id (doc_ids) or given (tokens), through
// the news encoder into doc_vec_out (n, ldo).
int encode_rows(lstur_plan* p, const lstur_weights* w, void* ws, int n, const int* doc_ids, const int* tokens,
                float* doc_vec_out, long long ldo, cudaStream_t st, const char* entry) {
  if (n == 0) return LSTUR_OK;
  const lstur_config& c = p->c;
  int* tok = p->ws.tokens(ws);
  if (doc_ids) RC(lstur_token_gather(n, c.L, c.n_docs, w->doc_tokens, doc_ids, tok, st));
  else cudaMemcpyAsync(tok, tokens, (size_t)n * c.L * sizeof(int), cudaMemcpyDeviceToDevice, st);
  RC(encode_titles(p, w, ws, n, 0, 0u, st));
  cudaMemcpy2DAsync(doc_vec_out, (size_t)ldo * 4, p->ws.doc_vec(ws), (size_t)p->D * 4, (size_t)p->D * 4, n,
                    cudaMemcpyDeviceToDevice, st);
  return cuda_status(entry);
}

}  // namespace

extern "C" int lstur_forward(lstur_plan* p, const lstur_weights* w, const lstur_batch* b, void* ws, int training,
                             unsigned seed, cudaStream_t st) {
  LSTUR_REQUIRE(p && w && b && ws, "lstur_forward");
  LSTUR_REQUIRE(w->dense && w->word_emb && b->user, "lstur_forward");
  const lstur_config& c = p->c;
  const int N = p->N, Nh = p->Nh, Nc = p->Nc, D = p->D, L = c.L;
  const bool bw = c.save_for_backward != 0;
  LSTUR_REQUIRE(!training || bw, "lstur_forward(training needs a save_for_backward plan)");
  p->last_seed = seed;
  p->last_training = training;
  int* tok = p->ws.tokens(ws);
  float* docv = p->ws.doc_vec(ws);
  // 1. title tokens (k0)
  if (b->hist_tok) {
    LSTUR_REQUIRE(b->cand_tok != nullptr, "lstur_forward");
    cudaMemcpyAsync(tok, b->hist_tok, (size_t)Nh * L * 4, cudaMemcpyDeviceToDevice, st);
    cudaMemcpyAsync(tok + (size_t)Nh * L, b->cand_tok, (size_t)Nc * L * 4, cudaMemcpyDeviceToDevice, st);
  } else {
    LSTUR_REQUIRE(b->hist_doc && b->cand_doc && w->doc_tokens, "lstur_forward");
    RC(lstur_token_gather(Nh, L, c.n_docs, w->doc_tokens, b->hist_doc, tok, st));
    RC(lstur_token_gather(Nc, L, c.n_docs, w->doc_tokens, b->cand_doc, tok + (size_t)Nh * L, st));
  }
  // 2. news encoder (k1-k7)
  RC(encode_titles(p, w, ws, N, training, seed, st));
  if (c.dv + c.ds) {   // [title ‖ Vemb[vert] ‖ Semb[subvert]] (task/cook.py:99-113)
    const float* vemb = p->dense.vert_emb(w->dense);
    const float* semb = p->dense.subvert_emb(w->dense);
    int* tv = p->ws.title_vert(ws);
    int* ts = p->ws.title_subvert(ws);
    if (b->hist_vert || b->hist_subvert || b->cand_vert || b->cand_subvert) {   // ids per title slot (cook .npz protocol)
      LSTUR_REQUIRE((c.dv == 0 || (b->hist_vert && b->cand_vert)) && (c.ds == 0 || (b->hist_subvert && b->cand_subvert)),
                    "lstur_forward(vertical concat: per-slot ids for both history and candidates)");
      RC(lstur_vert_concat(Nh, D, c.Dd, c.dv, c.ds, Nh, c.n_vert, c.n_subvert, nullptr, b->hist_vert, b->hist_subvert,
                           vemb, semb, docv, tv, ts, st));
      RC(lstur_vert_concat(Nc, D, c.Dd, c.dv, c.ds, Nc, c.n_vert, c.n_subvert, nullptr, b->cand_vert, b->cand_subvert,
                           vemb, semb, docv + (size_t)Nh * D, tv + Nh, ts + Nh, st));
    } else {
      LSTUR_REQUIRE(b->hist_doc && b->cand_doc && (c.dv == 0 || w->doc_vert) && (c.ds == 0 || w->doc_subvert),
                    "lstur_forward(vertical concat needs doc ids and the doc_vert / doc_subvert tables, or per-slot ids)");
      RC(lstur_vert_concat(Nh, D, c.Dd, c.dv, c.ds, c.n_docs, c.n_vert, c.n_subvert, b->hist_doc, w->doc_vert, w->doc_subvert,
                           vemb, semb, docv, tv, ts, st));
      RC(lstur_vert_concat(Nc, D, c.Dd, c.dv, c.ds, c.n_docs, c.n_vert, c.n_subvert, b->cand_doc, w->doc_vert, w->doc_subvert,
                           vemb, semb, docv + (size_t)Nh * D, tv + Nh, ts + Nh, st));
    }
  }
  // 3. history mask (k9)
  RC(lstur_hist_mask_apply(Nh, L, D, tok, docv, D, p->ws.hist_mask(ws), p->ws.gru_mask(ws), st));
  RC(user_and_score(p, w, b, ws, st));
  // auxiliary vertical classifier over [history vectors (masked) ; candidate vectors] (task/paper.py:973-990); without
  // labels (test_model, :992-997) the head is not part of the graph
  const bool aux_labels = (b->hist_vert && b->cand_vert) || (b->hist_doc && b->cand_doc && w->doc_vert);
  p->last_aux = 0;
  if (c.aux_nv && aux_labels) {
    const gemm_fn GEMM = pick_gemm(p);
    void* gws = p->ws.gemm_ws(ws);
    const size_t gwsb = p->gemm_ws_bytes;
    int* lab = p->ws.vs_label(ws);
    if (b->hist_vert && b->cand_vert) {
      cudaMemcpyAsync(lab, b->hist_vert, (size_t)Nh * 4, cudaMemcpyDeviceToDevice, st);
      cudaMemcpyAsync(lab + Nh, b->cand_vert, (size_t)Nc * 4, cudaMemcpyDeviceToDevice, st);
    } else {
      RC(lstur_token_gather(Nh, 1, c.n_docs, w->doc_vert, b->hist_doc, lab, st));
      RC(lstur_token_gather(Nc, 1, c.n_docs, w->doc_vert, b->cand_doc, lab + Nh, st));
    }
    float* hid = p->ws.vs_hid(ws);
    float* lg = p->ws.vs_logit(ws);
    RC(GEMM(0, 0, N, c.aux_hidden, D, docv, D, p->dense.vs_w1(w->dense), c.aux_hidden, hid, c.aux_hidden,
            p->dense.vs_b1(w->dense), LSTUR_GEMM_RELU | LSTUR_GEMM_PRECISE, gws, gwsb, st));
    RC(GEMM(0, 0, N, c.aux_nv, c.aux_hidden, hid, c.aux_hidden, p->dense.vs_w2(w->dense), c.aux_nv, lg, c.aux_nv,
            p->dense.vs_b2(w->dense), LSTUR_GEMM_PRECISE, gws, gwsb, st));
    RC(lstur_softmax_ce_labels(N, c.aux_nv, lg, lab, p->ws.vs_probs(ws), p->ws.vs_loss_rows(ws), p->ws.vs_loss(ws),
                               nullptr, 0.f, st));
    p->last_aux = 1;
  }
  return cuda_status("lstur_forward");
}

// ---- decomposed inference (task/test_pipeline.py:37-211): doc vectors once, then users against the cached vectors
// doc_vec_out[i, :] = doc_encoder(title of doc_ids[i]) for n <= B*(W+C) documents (test_doc_vec, :37-75).
extern "C" int lstur_encode_docs(lstur_plan* p, const lstur_weights* w, void* ws, int n, const int* doc_ids,
                                 float* doc_vec_out, long long ldo, cudaStream_t st) {
  LSTUR_REQUIRE(p && w && ws && w->dense && w->word_emb && w->doc_tokens, "lstur_encode_docs");
  LSTUR_REQUIRE(n >= 0 && n <= p->N && doc_ids && doc_vec_out && ldo >= p->D, "lstur_encode_docs");
  return encode_rows(p, w, ws, n, doc_ids, nullptr, doc_vec_out, ldo, st, "lstur_encode_docs");
}

// doc_encoder.predict on explicit token rows (the `doc_encoder` layer of the model, task/paper.py:160; used by
// TestPipeline.get_doc_parser / test_doc_vec on parsed titles): tokens (n, L) on the device, n <= B*(W+C).
extern "C" int lstur_encode_titles(lstur_plan* p, const lstur_weights* w, void* ws, int n, const int* tokens,
                                   float* doc_vec_out, long long ldo, cudaStream_t st) {
  LSTUR_REQUIRE(p && w && ws && w->dense && w->word_emb, "lstur_encode_titles");
  LSTUR_REQUIRE(n >= 0 && n <= p->N && tokens && doc_vec_out && ldo >= p->D, "lstur_encode_titles");
  return encode_rows(p, w, ws, n, nullptr, tokens, doc_vec_out, ldo, st, "lstur_encode_titles");
}

// User encoder + scorer over cached document vectors (test_user_vec / test_user_doc_score, :77-211): history and
// candidate vectors are rows of doc_vec_table (n_rows, ld); a history slot whose vector is all zero (unknown / pad
// document, :104-108) is masked, exactly as keras Masking() does inside the user encoder.
extern "C" int lstur_forward_docvecs(lstur_plan* p, const lstur_weights* w, const lstur_batch* b, void* ws,
                                     const float* doc_vec_table, long long ld, int n_rows, cudaStream_t st) {
  LSTUR_REQUIRE(p && w && b && ws && w->dense && b->user && b->hist_doc && b->cand_doc, "lstur_forward_docvecs");
  LSTUR_REQUIRE(doc_vec_table && ld >= p->D && n_rows > 0, "lstur_forward_docvecs");
  const lstur_config& c = p->c;
  const int Nh = p->Nh, Nc = p->Nc, D = p->D;
  p->last_training = 0;
  float* docv = p->ws.doc_vec(ws);
  // lstur_row_gather reads `ld`-strided rows when table rows are wider than D: gather D columns per row
  LSTUR_REQUIRE(ld == D, "lstur_forward_docvecs(ld must equal the document-vector width)");
  RC(lstur_row_gather(Nh, D, n_rows, doc_vec_table, b->hist_doc, nullptr, docv, D, st));
  RC(lstur_row_gather(Nc, D, n_rows, doc_vec_table, b->cand_doc, nullptr, docv + (size_t)Nh * D, D, st));
  RC(lstur_hist_mask_apply(Nh, c.L, D, nullptr, docv, D, p->ws.hist_mask(ws), p->ws.gru_mask(ws), st));
  return user_and_score(p, w, b, ws, st);
}

// Ranking of whole impressions against cached document vectors (the validation / test pass of Seq2VecPaperSoftmax.callback,
// task/paper.py:497-524): impression i has the user user[i], the history hist_doc[i, :W] and the candidates
// cand_doc[cand_off[i] .. cand_off[i+1]); scores_out[j] = sigmoid(score(user vector of j's impression, doc_vec_table[cand_doc[j]]))
// with the plan's own scorer, the value of the test head.  The user encoder runs once per impression, on chunks of at
// most B impressions and B*C pairs.  cand_off is HOST memory (the chunks are cut on the host; each chunk's offsets are
// copied to the device); every other array is on the device.  A history slot is masked when its document's title is all
// zero tokens (weights->doc_tokens), as in lstur_forward; a candidate keeps its table row whatever its title.
extern "C" int lstur_score_impressions(lstur_plan* p, const lstur_weights* w, void* ws, int n_impr, const int* user,
                                       const float* user_scale, const float* user_scale2, const int* hist_doc,
                                       const int* cand_off, const int* cand_doc, const float* doc_vec_table, int n_rows,
                                       float* scores_out, cudaStream_t st) {
  LSTUR_REQUIRE(p && w && ws && w->dense && w->doc_tokens && n_impr >= 0, "lstur_score_impressions");
  LSTUR_REQUIRE(n_impr == 0 || (user && hist_doc && cand_off && cand_doc && doc_vec_table && n_rows > 0 && scores_out),
                "lstur_score_impressions");
  const lstur_config& c = p->c;
  LSTUR_REQUIRE(c.save_for_backward == 0, "lstur_score_impressions(needs an inference plan: save_for_backward = 0)");
  LSTUR_REQUIRE(c.loss_model == LSTUR_LOSS_SOFTMAX_CE, "lstur_score_impressions(the softmax-family test head)");
  const int Nh = p->Nh, Nc = p->Nc, D = p->D, B = c.B, L = c.L;
  for (int i = 0; i < n_impr; ++i) {
    const int n = cand_off[i + 1] - cand_off[i];
    if (n < 0) {
      set_error("lstur_score_impressions: cand_off decreases at impression %d", i);
      return LSTUR_ERR_ARG;
    }
    if (n > Nc) {
      set_error("lstur_score_impressions: impression %d has %d candidates, more than one chunk of the plan holds "
                "(B*C = %d*%d = %d): build the plan with more rows or candidates", i, n, B, c.C, Nc);
      return LSTUR_ERR_ARG;
    }
  }
  if (n_impr == 0) return LSTUR_OK;
  float* docv = p->ws.doc_vec(ws);
  float* cand = docv + (size_t)Nh * D;
  float* uvec = p->ws.user_vec(ws);
  int* tok = p->ws.tokens(ws);
  int* ev_user = p->ws.ev_user(ws);
  int* ev_off = p->ws.ev_off(ws);
  int* pair_row = p->ws.ev_pair_row(ws);
  lstur_batch b;
  memset(&b, 0, sizeof(b));
  b.user = ev_user;
  float* ev_scale = user_scale ? p->ws.ev_scale(ws) : nullptr;
  float* ev_scale2 = user_scale2 ? p->ws.ev_scale2(ws) : nullptr;
  b.user_scale = ev_scale;
  b.user_scale2 = ev_scale2;
  std::vector<int> off;
  p->last_training = 0;
  for (int i0 = 0; i0 < n_impr;) {
    int i1 = i0;
    while (i1 < n_impr && i1 - i0 < B && cand_off[i1 + 1] - cand_off[i0] <= Nc) ++i1;
    const int m = i1 - i0, p0 = cand_off[i0], np = cand_off[i1] - p0;
    off.assign(cand_off + i0, cand_off + i1 + 1);
    cudaMemcpyAsync(ev_off, off.data(), (size_t)(m + 1) * 4, cudaMemcpyHostToDevice, st);
    RC(lstur_csr_rows(m, ev_off, pair_row, st));
    // users and history rows of the chunk; rows m..B are padding (user 0, all history slots masked)
    cudaMemsetAsync(ev_user, 0, (size_t)B * 4, st);
    cudaMemcpyAsync(ev_user, user + i0, (size_t)m * 4, cudaMemcpyDeviceToDevice, st);
    if (ev_scale) {
      cudaMemsetAsync(ev_scale, 0, (size_t)B * 4, st);
      cudaMemcpyAsync(ev_scale, user_scale + i0, (size_t)m * 4, cudaMemcpyDeviceToDevice, st);
    }
    if (ev_scale2) {
      cudaMemsetAsync(ev_scale2, 0, (size_t)B * 4, st);
      cudaMemcpyAsync(ev_scale2, user_scale2 + i0, (size_t)m * 4, cudaMemcpyDeviceToDevice, st);
    }
    const long long nh = (long long)m * c.W;
    RC(lstur_token_gather((int)nh, L, c.n_docs, w->doc_tokens, hist_doc + (size_t)i0 * c.W, tok, st));
    RC(lstur_row_gather((int)nh, D, n_rows, doc_vec_table, hist_doc + (size_t)i0 * c.W, nullptr, docv, D, st));
    if (nh < Nh) {
      cudaMemsetAsync(tok + nh * L, 0, (size_t)(Nh - nh) * L * 4, st);
      cudaMemsetAsync(docv + nh * D, 0, (size_t)(Nh - nh) * D * 4, st);
    }
    RC(lstur_hist_mask_apply(Nh, L, D, tok, docv, D, p->ws.hist_mask(ws), p->ws.gru_mask(ws), st));
    RC(user_vector(p, w, &b, ws, st));
    float* out = scores_out + p0;
    const int* cd = cand_doc + p0;
    if (c.score_model == LSTUR_SCORE_DOT) {
      RC(lstur_score_sigmoid_ragged(np, D, pair_row, uvec, c.U, cd, doc_vec_table, D, out, st));
    } else {
      RC(lstur_row_gather(np, D, n_rows, doc_vec_table, cd, nullptr, cand, D, st));
      ScoreOperands s;
      RC(score_operands(p, w, ws, np, pair_row, &s, st));
      RC(lstur_score_sigmoid_ragged(np, s.dim, pair_row, s.u, s.ldu, nullptr, s.d, s.ldd, out, st));
    }
    i0 = i1;
  }
  return cuda_status("lstur_score_impressions");
}

namespace {

// News-encoder backward (k1-k7) over the first n title slots: d_doc_vec[0..n) -> dense gradients of the Dense / attention /
// conv tensors and, with a trainable word table, d word_emb.
int encoder_backward(const lstur_plan* p, const lstur_weights* w, void* ws, int n, float* dgrad, float* word_grad,
                     float grad_scale, cudaStream_t st) {
  const lstur_config& c = p->c;
  const int Lp = p->Lp, D = p->D, L = c.L, E = c.E, F = c.F;
  void* gws = p->ws.gemm_ws(ws);
  const size_t gwsb = p->gemm_ws_bytes;
  float* cws = p->ws.colsum_ws(ws);
  const size_t cwsb = p->ws.colsum_ws.bytes();
  float* d_docv = p->ws.d_doc_vec(ws);
  float* d_pooled = p->ws.d_pooled(ws);
  float* pooled = p->ws.pooled(ws);
  const int* n_live = p->ws.n_live(ws);
  const int* live_idx = p->ws.live_idx(ws);
  const float* dpool = d_pooled;
  long long lddp = F;
  if (c.use_dense) {
    // d pooled of the live titles only: the attention backward runs over the compacted list and never reads the other rows
    RC(gemm_mrows(p, ws, p->compact_titles, live_idx, n_live, 1, n, F, c.Dd, d_docv, D, p->dense.dense_w(w->dense), c.Dd,
                  d_pooled, F, nullptr, 0, st));
    // pooled is zero for the all-pad titles: reduce over the live titles of the compacted list
    RC(gemm_tn_rows(p, ws, p->compact_titles, live_idx, n_live, F, c.Dd, n, pooled, F, d_docv, D, p->dense.dense_w(dgrad),
                    c.Dd, st));
    RC(lstur_colsum(n, c.Dd, d_docv, D, p->dense.dense_b(dgrad), 0, cws, cwsb, st));
  } else {
    dpool = d_docv; lddp = D;
  }
  // everything but the title-encoder bucket is final here: a data-parallel caller starts its exchange on another stream
  if (p->ev_tail_ready) cudaEventRecord(p->ev_tail_ready, st);
  // the dropout streams are replayed only if the saved forward was a training forward (an inference forward followed by
  // a backward differentiates the inference graph)
  const float bwd_drop = p->last_training ? c.dropout : 0.f;
  if (p->tc_prec) {
    const int fp16 = c.precision == LSTUR_PREC_FP16_TC;
    void* img = p->ws.dpre_img(ws);
    void* xmask = bwd_drop > 0.f ? p->ws.xmask(ws) : nullptr;
    // power-of-two loss scale of the 16-bit dPre image: the gradients carry grad_scale = 1 / global batch, which would
    // put them in fp16's subnormal range; 16 x the per-impression magnitude leaves 2^12 of headroom
    float img_scale = 1.f;
    if (grad_scale > 0.f && grad_scale < 1.f) {
      int ex = 0;
      frexpf(1.f / grad_scale, &ex);          // 1/grad_scale = m * 2^ex, m in [0.5, 1)
      img_scale = ldexpf(1.f, ex - 1 + 4);
    }
    const int* tok_c = p->ws.tokens_c(ws);
    PROBE_BEGIN(p, LSTUR_PROBE_ATTN_BWD, st);
    RC(lstur_attn_pool_bwd_img(fp16, n, L, F, p->ws.C16(ws), p->ws.att_a(ws), p->ws.att_w(ws), dpool, lddp,
                               p->dense.att_w(w->dense), img, bwd_drop, img_scale, p->dense.att_w(dgrad),
                               p->dense.conv_b(dgrad), p->dense.att_b(dgrad), 0, p->ws.attn_partials(ws),
                               p->ws.attn_partials.bytes(), n_live, live_idx, st));
    PROBE_END(p, LSTUR_PROBE_ATTN_BWD, st);
    PROBE_BEGIN(p, LSTUR_PROBE_CONV_WGRAD, st);
    RC(lstur_conv_wgrad_tc_m(n, L, E, F, c.V, tok_c, p->ws.emb_bf16(ws), img, p->dense.conv_w(dgrad), bwd_drop, p->last_seed,
                             fp16, p->ws.wgrad_partial(ws), p->ws.wgrad_partial.bytes(), xmask, img_scale, n_live, st));
    PROBE_END(p, LSTUR_PROBE_CONV_WGRAD, st);
    if (c.trainable_word_emb) {
      // d X = dPre (*) Wc^T on tcgen05, then d word_emb = segment-sorted sum of the token rows (x the X-dropout mask)
      void* wimg_d = p->ws.wimg_d(ws);
      void* dx16 = p->ws.dx16(ws);
      RC(lstur_pack_conv_w_dgrad_tc(E, F, p->dense.conv_w(w->dense), wimg_d, fp16, st));
      PROBE_BEGIN(p, LSTUR_PROBE_CONV_DGRAD, st);
      RC(lstur_conv_dgrad_tc(n, L, E, F, img, wimg_d, dx16, 1.f, fp16, 0, n_live, st));
      PROBE_END(p, LSTUR_PROBE_CONV_DGRAD, st);
      PROBE_BEGIN(p, LSTUR_PROBE_SCATTER, st);
      RC(lstur_word_grad_scatter_16(n, L, E, c.V, tok_c, dx16, fp16, 1.f / ((1.f - bwd_drop) * img_scale), xmask, word_grad,
                                    p->ws.wg_ws(ws), p->ws.wg_ws.bytes(), n_live, st));
      PROBE_END(p, LSTUR_PROBE_SCATTER, st);
    }
  } else {
    float* dPre = p->ws.dPre(ws);
    RC(lstur_attn_pool_bwd(n, L, Lp, F, p->ws.Cp(ws), (long long)Lp * F, p->ws.att_a(ws), p->ws.att_w(ws), dpool, lddp,
                           p->dense.att_w(w->dense), dPre, (long long)Lp * F, bwd_drop, p->dense.att_w(dgrad),
                           p->dense.conv_b(dgrad), p->dense.att_b(dgrad), 0, p->ws.attn_partials(ws),
                           p->ws.attn_partials.bytes(), st));
    // d_conv_w[(j,e),f] = sum_m Xp[m+j, e] * dPre[m, f]
    PROBE_BEGIN(p, LSTUR_PROBE_CONV_WGRAD, st);
    RC(lstur_gemm_f32(1, 0, c.KS * E, F, n * Lp - (c.KS - 1), p->ws.Xp(ws), E, dPre, F, p->dense.conv_w(dgrad), F, nullptr,
                      0, gws, gwsb, st));
    PROBE_END(p, LSTUR_PROBE_CONV_WGRAD, st);
    if (c.trainable_word_emb) {
      // d Xp[m + j, e] += sum_f dPre[m, f] * Wc[j, e, f]: one accumulating GEMM per tap into the overlapping windows of the
      // zero-haloed title buffer, then the same segment-sorted scatter
      float* dXp = p->ws.dXp(ws);
      cudaMemsetAsync(dXp, 0, (size_t)n * Lp * E * sizeof(float), st);
      PROBE_BEGIN(p, LSTUR_PROBE_CONV_DGRAD, st);
      for (int j = 0; j < c.KS; ++j)
        RC(lstur_gemm_f32(0, 1, n * Lp - (c.KS - 1), E, F, dPre, F, p->dense.conv_w(w->dense) + (size_t)j * E * F, F,
                          dXp + (size_t)j * E, E, nullptr, LSTUR_GEMM_ACCUM, gws, gwsb, st));
      PROBE_END(p, LSTUR_PROBE_CONV_DGRAD, st);
      PROBE_BEGIN(p, LSTUR_PROBE_SCATTER, st);
      RC(lstur_word_grad_scatter_f32(n, L, c.KS, E, c.V, p->ws.tokens(ws), dXp, bwd_drop, p->last_seed * 2u + 0u, 1.f,
                                     word_grad, p->ws.wg_ws(ws), p->ws.wg_ws.bytes(), st));
      PROBE_END(p, LSTUR_PROBE_SCATTER, st);
    }
  }
  return LSTUR_OK;
}

}  // namespace

// ---- vertical model of Seq2VecPaperSoftmaxDaysIdVertAlt (task/paper.py:1128-1136): Dense(cls_nv, softmax)(doc_encoder(title)),
// categorical cross-entropy; trained on (title, vertical) batches in alternation with the click model, which shares the
// doc_encoder weights.  tokens (n, L) and labels (n) on the device, n <= B*(W+C).
extern "C" int lstur_title_cls_forward(lstur_plan* p, const lstur_weights* w, void* ws, int n, const int* tokens,
                                       const int* labels, int training, unsigned seed, cudaStream_t st) {
  LSTUR_REQUIRE(p && w && ws && w->dense && w->word_emb && tokens && labels, "lstur_title_cls_forward");
  const lstur_config& c = p->c;
  LSTUR_REQUIRE(c.cls_nv > 0 && n > 0 && n <= p->N, "lstur_title_cls_forward(plan without cls_nv, or n out of range)");
  LSTUR_REQUIRE(!training || c.save_for_backward, "lstur_title_cls_forward(training needs a save_for_backward plan)");
  p->last_seed = seed; p->last_training = training; p->last_cls_n = n;
  const int D = p->D;
  cudaMemcpyAsync(p->ws.tokens(ws), tokens, (size_t)n * c.L * sizeof(int), cudaMemcpyDeviceToDevice, st);
  cudaMemcpyAsync(p->ws.vc_label(ws), labels, (size_t)n * sizeof(int), cudaMemcpyDeviceToDevice, st);
  RC(encode_titles(p, w, ws, n, training, seed, st));
  float* lg = p->ws.vc_logit(ws);
  RC(pick_gemm(p)(0, 0, n, c.cls_nv, D, p->ws.doc_vec(ws), D, p->dense.vcls_w(w->dense), c.cls_nv, lg, c.cls_nv,
                  p->dense.vcls_b(w->dense), LSTUR_GEMM_PRECISE, p->ws.gemm_ws(ws), p->gemm_ws_bytes, st));
  RC(lstur_softmax_ce_labels(n, c.cls_nv, lg, p->ws.vc_label(ws), p->ws.vc_probs(ws), p->ws.vc_loss_rows(ws),
                             p->ws.vc_loss(ws), nullptr, 0.f, st));
  return cuda_status("lstur_title_cls_forward");
}

// Gradients of the vertical model: dgrad (whole arena; only vcls_* and the title-encoder tensors are non-zero) and, with a
// trainable word table, word_grad.  grad_scale = 1 / (global number of titles).
extern "C" int lstur_title_cls_backward(const lstur_plan* p, const lstur_weights* w, void* ws, float* dgrad,
                                        float* word_grad, float grad_scale, cudaStream_t st) {
  LSTUR_REQUIRE(p && w && ws && dgrad, "lstur_title_cls_backward");
  const lstur_config& c = p->c;
  const int n = p->last_cls_n, D = p->D, nv = c.cls_nv;
  LSTUR_REQUIRE(nv > 0 && c.save_for_backward && n > 0, "lstur_title_cls_backward(needs a lstur_title_cls_forward on a training plan)");
  LSTUR_REQUIRE(!c.trainable_word_emb || word_grad != nullptr, "lstur_title_cls_backward(trainable word table needs word_grad)");
  const gemm_fn GEMM = pick_gemm(p);
  void* gws = p->ws.gemm_ws(ws);
  const size_t gwsb = p->gemm_ws_bytes;
  float* dlg = p->ws.vc_dlogit(ws);
  cudaMemsetAsync(dgrad, 0, (size_t)p->dense_count * 4, st);
  RC(lstur_softmax_ce_labels(n, nv, p->ws.vc_logit(ws), p->ws.vc_label(ws), nullptr, nullptr, nullptr, dlg, grad_scale, st));
  RC(GEMM(1, 0, D, nv, n, p->ws.doc_vec(ws), D, dlg, nv, p->dense.vcls_w(dgrad), nv, nullptr, 0, gws, gwsb, st));
  RC(lstur_colsum(n, nv, dlg, nv, p->dense.vcls_b(dgrad), 0, p->ws.colsum_ws(ws), p->ws.colsum_ws.bytes(), st));
  RC(GEMM(0, 1, n, D, nv, dlg, nv, p->dense.vcls_w(w->dense), nv, p->ws.d_doc_vec(ws), D, nullptr, 0, gws, gwsb, st));
  RC(encoder_backward(p, w, ws, n, dgrad, word_grad, grad_scale, st));
  return cuda_status("lstur_title_cls_backward");
}

extern "C" int lstur_backward(const lstur_plan* p, const lstur_weights* w, const lstur_batch* b, void* ws,
                              float* dgrad, float grad_scale, cudaStream_t st) {
  return lstur_backward_w(p, w, b, ws, dgrad, nullptr, grad_scale, st);
}

extern "C" int lstur_backward_w(const lstur_plan* p, const lstur_weights* w, const lstur_batch* b, void* ws,
                                float* dgrad, float* word_grad, float grad_scale, cudaStream_t st) {
  LSTUR_REQUIRE(p && w && b && ws && dgrad, "lstur_backward");
  const lstur_config& c = p->c;
  LSTUR_REQUIRE(c.save_for_backward != 0, "lstur_backward");
  LSTUR_REQUIRE(!c.trainable_word_emb || word_grad != nullptr, "lstur_backward(trainable word table needs word_grad: lstur_backward_w)");
  const int N = p->N, Nh = p->Nh, D = p->D, G = c.G, B = c.B;
  void* gws = p->ws.gemm_ws(ws);
  const size_t gwsb = p->gemm_ws_bytes;
  const gemm_fn GEMM = pick_gemm(p);
  float* cws = p->ws.colsum_ws(ws);
  const size_t cwsb = p->ws.colsum_ws.bytes();
  float* docv = p->ws.doc_vec(ws);
  float* uvec = p->ws.user_vec(ws);
  float* d_uvec = p->ws.d_user_vec(ws);
  float* d_docv = p->ws.d_doc_vec(ws);
  float* gmask = p->ws.gru_mask(ws);
  cudaMemsetAsync(dgrad, 0, (size_t)p->dense_count * 4, st);
  // 1. loss / score backward
  const float* cand = docv + (size_t)Nh * D;
  float* d_cand = d_docv + (size_t)Nh * D;
  const bool bce = c.loss_model == LSTUR_LOSS_WEIGHTED_BCE;
  float* d_logits = p->ws.d_logits(ws);
  if (bce) {
    LSTUR_REQUIRE(b->label != nullptr, "lstur_backward(weighted BCE needs labels)");
    RC(lstur_bce_loss(p->Nc, p->ws.logits(ws), b->label, c.gain, c.bce_neg, nullptr, nullptr, nullptr, d_logits,
                      grad_scale, st));
  }
  if (c.score_model == LSTUR_SCORE_DOT) {
    if (bce) RC(lstur_dot_score_bwd(B, c.C, D, uvec, c.U, cand, D, d_logits, d_uvec, c.U, d_cand, D, st));
    else RC(lstur_score_softmax_ce(B, c.C, D, uvec, c.U, cand, D, b->label, nullptr, nullptr, nullptr, nullptr,
                                   d_uvec, c.U, d_cand, D, grad_scale, st));
  } else if (c.score_model == LSTUR_SCORE_DNN) {
    const int K2 = c.U + D, Hs = c.Hs;
    const long long Nc = p->Nc;
    float* hid = p->ws.sc_hid(ws);
    float* dhid = p->ws.sc_dhid(ws);
    float* whid = p->ws.sc_whid(ws);
    float* dcat = p->ws.sc_dcat(ws);
    float* dl = bce ? d_logits : p->ws.sc_dlogit(ws);
    if (!bce) RC(lstur_score_softmax_ce(B, c.C, 1, p->ws.sc_ones(ws), 1, p->ws.sc_raw(ws), 1, b->label, nullptr, nullptr,
                                        nullptr, nullptr, p->ws.sc_scratch(ws), 1, dl, 1, grad_scale, st));
    RC(lstur_dnn_out_bwd(Nc, Hs, hid, p->dense.so_w(w->dense), dl, dhid, whid, st));
    RC(lstur_colsum(Nc, Hs, whid, Hs, p->dense.so_w(dgrad), 0, cws, cwsb, st));
    RC(lstur_colsum(Nc, 1, dl, 1, p->dense.so_b(dgrad), 0, cws, cwsb, st));
    RC(lstur_colsum(Nc, Hs, dhid, Hs, p->dense.sh_b(dgrad), 0, cws, cwsb, st));
    RC(GEMM(1, 0, K2, Hs, (int)Nc, p->ws.sc_cat(ws), K2, dhid, Hs, p->dense.sh_w(dgrad), Hs, nullptr, 0, gws, gwsb, st));
    RC(GEMM(0, 1, (int)Nc, K2, Hs, dhid, Hs, p->dense.sh_w(w->dense), Hs, dcat, K2, nullptr, 0, gws, gwsb, st));
    RC(lstur_pair_split(B, c.C, c.U, D, dcat, d_uvec, c.U, d_cand, D, st));
  } else {
    const int Hs = c.Hs;
    const long long Nc = p->Nc;
    float* uh = p->ws.sc_uh(ws);
    float* dh = p->ws.sc_dh(ws);
    float* duh = p->ws.sc_duh(ws);
    float* ddh = p->ws.sc_ddh(ws);
    if (bce) RC(lstur_dot_score_bwd(B, c.C, Hs, uh, Hs, dh, Hs, d_logits, duh, Hs, ddh, Hs, st));
    else RC(lstur_score_softmax_ce(B, c.C, Hs, uh, Hs, dh, Hs, b->label, nullptr, nullptr, nullptr, nullptr, duh, Hs, ddh,
                                   Hs, grad_scale, st));
    if (c.score_model == LSTUR_SCORE_DDOT) {
      RC(lstur_tanh_bwd((long long)B * Hs, uh, duh, st));
      RC(lstur_tanh_bwd(Nc * Hs, dh, ddh, st));
    }
    RC(lstur_colsum(B, Hs, duh, Hs, p->dense.su_b(dgrad), 0, cws, cwsb, st));
    RC(lstur_colsum(Nc, Hs, ddh, Hs, p->dense.sd_b(dgrad), 0, cws, cwsb, st));
    RC(GEMM(1, 0, c.U, Hs, B, uvec, c.U, duh, Hs, p->dense.su_w(dgrad), Hs, nullptr, 0, gws, gwsb, st));
    RC(GEMM(1, 0, D, Hs, (int)Nc, cand, D, ddh, Hs, p->dense.sd_w(dgrad), Hs, nullptr, 0, gws, gwsb, st));
    RC(GEMM(0, 1, B, c.U, Hs, duh, Hs, p->dense.su_w(w->dense), Hs, d_uvec, c.U, nullptr, 0, gws, gwsb, st));
    RC(GEMM(0, 1, (int)Nc, D, Hs, ddh, Hs, p->dense.sd_w(w->dense), Hs, d_cand, D, nullptr, 0, gws, gwsb, st));
  }
  // 2. user-encoder head backward
  const float* dhT = d_uvec;
  long long lddh = c.U;
  const float* du0 = nullptr;
  long long lddu0 = 0;
  const int Uc = arch_uc(c);
  if (c.arch == LSTUR_ARCH_CON_DENSE || c.arch == LSTUR_ARCH_INI_CON) {
    float* d_cat = p->ws.d_cat(ws);
    const int K2 = G + Uc;
    RC(GEMM(0, 1, B, K2, c.U, d_uvec, c.U, p->dense.con_w(w->dense), c.U, d_cat, K2, nullptr, 0, gws, gwsb, st));
    RC(GEMM(1, 0, K2, c.U, B, p->ws.cat(ws), K2, d_uvec, c.U, p->dense.con_w(dgrad), c.U, nullptr, 0, gws, gwsb, st));
    RC(lstur_colsum(B, c.U, d_uvec, c.U, p->dense.con_b(dgrad), 0, cws, cwsb, st));
    dhT = d_cat; lddh = K2; du0 = d_cat + G; lddu0 = K2;
  } else if (c.arch == LSTUR_ARCH_CON_CAT || c.arch == LSTUR_ARCH_INI_CAT) {
    du0 = d_uvec + G; lddu0 = c.U;
  } else if (c.arch == LSTUR_ARCH_ADD || c.arch == LSTUR_ARCH_VO || c.arch == LSTUR_ARCH_INI_ADD) {
    du0 = d_uvec; lddu0 = c.U;
  } else if (c.arch == LSTUR_ARCH_LSTM_CAT) {
    du0 = d_uvec + G; lddu0 = c.U;
  } else if (c.arch == LSTUR_ARCH_AVG_CAT || c.arch == LSTUR_ARCH_ATT_CAT) {
    du0 = d_uvec + D; lddu0 = c.U;
  } else if (c.arch == LSTUR_ARCH_ATT_PAIR) {
    float* d_seq2 = p->ws.d_seq2(ws);
    float* part = p->ws.ua_partial(ws);
    RC(lstur_seq_attn_bwd(B, 2 * G, 1, p->ws.seq2(ws), p->dense.uatt_w(w->dense), p->ws.ua_a(ws), p->ws.ua_w(ws), d_uvec,
                          c.U, nullptr, d_seq2, part, st));
    RC(lstur_colsum(B, 1, part, 2, p->dense.uatt_w(dgrad), 0, cws, cwsb, st));
    RC(lstur_colsum(B, 1, part + 1, 2, p->dense.uatt_b(dgrad), 0, cws, cwsb, st));
    dhT = d_seq2; lddh = 2 * G; du0 = d_seq2 + G; lddu0 = 2 * G;
  } else if (c.arch == LSTUR_ARCH_ALPHA) {
    float* d_hT = p->ws.d_hT(ws);
    float* d_uh = p->ws.d_uh(ws);
    float* part = p->ws.alpha_partial(ws);
    RC(lstur_alpha_add_bwd(B, G, p->dense.alpha(w->dense), p->ws.hT(ws), G, p->ws.u0(ws), c.Ue, d_uvec, c.U, d_hT, G, d_uh,
                           c.Ue, part, st));
    RC(lstur_colsum(B, 1, part, 1, p->dense.alpha(dgrad), 0, cws, cwsb, st));
    dhT = d_hT; lddh = G; du0 = d_uh; lddu0 = c.Ue;
  }
  // 3. GRU backward
  if (arch_has_gru(c.arch)) {
    float* dA = p->ws.dA(ws);
    float* dh0 = p->ws.dh0(ws);
    float* HP = p->ws.HP(ws);
    // row order of the last forward (the mask has not changed since)
    const int* order = p->ws.gru_order(ws);
    PROBE_BEGIN(p, LSTUR_PROBE_GRU_BWD, st);
    if (p->tc_gru) {
      // the kernel also leaves per-(tile, row group) column sums of dA: the bias gradient needs no second pass over dA
      float* dbp = p->ws.gru_db_partial(ws);
      RC(lstur_gru_bwd_tc(B, c.W, G, gmask, p->ws.Z(ws), p->ws.R(ws), p->ws.HH(ws), HP, p->dense.gru_wh(w->dense), c.rec_act,
                          dhT, lddh, dA, dh0, G, order, dbp, st));
      RC(lstur_colsum(lstur_gru_tc_db_rows(B), 3 * G, dbp, 3 * G, p->dense.gru_b(dgrad), 0, cws, cwsb, st));
    } else {
      float* WhT = p->ws.WhT(ws);
      RC(lstur_transpose(G, 3 * G, p->dense.gru_wh(w->dense), WhT, st));
      RC(lstur_gru_bwd(B, c.W, G, gmask, p->ws.Z(ws), p->ws.R(ws), p->ws.HH(ws), HP, WhT, c.rec_act, dhT, lddh, dA, dh0, G,
                       order, st));
      RC(lstur_colsum(Nh, 3 * G, dA, 3 * G, p->dense.gru_b(dgrad), 0, cws, cwsb, st));
    }
    PROBE_END(p, LSTUR_PROBE_GRU_BWD, st);
    // with the row list of the forward: dA is zero on masked steps, so the weight gradients reduce over the unmasked
    // (user, step) rows only (half of them with the left-padded histories of short click logs)
    const bool rows = p->live_hist_rows;
    const int* hl_idx = p->ws.hist_live_idx(ws);
    const int* hl_n = p->ws.n_hist_live(ws);
    float* dwh = p->dense.gru_wh(dgrad);
    RC(gemm_tn_rows(p, ws, rows, hl_idx, hl_n, D, 3 * G, Nh, docv, D, dA, 3 * G, p->dense.gru_wx(dgrad), 3 * G, st));
    RC(gemm_tn_rows(p, ws, rows, hl_idx, hl_n, G, 2 * G, Nh, HP, G, dA, 3 * G, dwh, 3 * G, st));
    RC(gemm_tn_rows(p, ws, rows, hl_idx, hl_n, G, G, Nh, p->ws.RH(ws), G, dA + 2 * G, 3 * G, dwh + 2 * G, 3 * G, st));
    // dH = dA . Wx^T  (rows of masked steps are zero because dA is zero there; the row-listed GEMM leaves them to the memset)
    if (rows) cudaMemsetAsync(d_docv, 0, (size_t)Nh * D * sizeof(float), st);
    RC(gemm_mrows(p, ws, rows, hl_idx, hl_n, 1, Nh, D, 3 * G, dA, 3 * G, p->dense.gru_wx(w->dense), 3 * G, d_docv, D,
                  nullptr, 0, st));
    if (c.arch == LSTUR_ARCH_INI) { du0 = dh0; lddu0 = G; }
    if (c.arch == LSTUR_ARCH_INI_CON || c.arch == LSTUR_ARCH_INI_CAT || c.arch == LSTUR_ARCH_INI_ADD) {   // d row = [d h0 ‖ d of the concat / add part]
      float* d_u0 = p->ws.d_u0(ws);
      cudaMemcpy2DAsync(d_u0, (size_t)c.Ue * 4, dh0, (size_t)G * 4, (size_t)G * 4, B, cudaMemcpyDeviceToDevice, st);
      cudaMemcpy2DAsync(d_u0 + G, (size_t)c.Ue * 4, du0, (size_t)lddu0 * 4, (size_t)Uc * 4, B, cudaMemcpyDeviceToDevice, st);
      du0 = nullptr;
    }
  } else if (arch_has_lstm(c.arch)) {
    float* WhT = p->ws.WhT(ws);
    float* dA = p->ws.dA(ws);
    RC(lstur_transpose(G, 4 * G, p->dense.lstm_wh(w->dense), WhT, st));
    RC(lstur_lstm_bwd(B, c.W, G, gmask, p->ws.LI(ws), p->ws.LF(ws), p->ws.LG(ws), p->ws.LO(ws), p->ws.LCP(ws), p->ws.LTC(ws),
                      WhT, c.rec_act, dhT, lddh, dA, st));
    RC(lstur_colsum(Nh, 4 * G, dA, 4 * G, p->dense.lstm_b(dgrad), 0, cws, cwsb, st));
    RC(GEMM(1, 0, D, 4 * G, Nh, docv, D, dA, 4 * G, p->dense.lstm_wx(dgrad), 4 * G, nullptr, 0, gws, gwsb, st));
    RC(GEMM(1, 0, G, 4 * G, Nh, p->ws.LHP(ws), G, dA, 4 * G, p->dense.lstm_wh(dgrad), 4 * G, nullptr, 0, gws, gwsb, st));
    RC(GEMM(0, 1, Nh, D, 4 * G, dA, 4 * G, p->dense.lstm_wx(w->dense), 4 * G, d_docv, D, nullptr, 0, gws, gwsb, st));
  } else if (arch_hist_avg(c.arch)) {
    RC(lstur_masked_mean_bwd(B, c.W, D, d_uvec, c.U, gmask, p->ws.hist_mask(ws), d_docv, st));
  } else if (arch_hist_att(c.arch)) {
    float* part = p->ws.ua_partial(ws);
    RC(lstur_seq_attn_bwd(B, c.W, D, docv, p->dense.uatt_w(w->dense), p->ws.ua_a(ws), p->ws.ua_w(ws), d_uvec, c.U,
                          p->ws.hist_mask(ws), d_docv, part, st));
    RC(lstur_colsum(B, D, part, D + 1, p->dense.uatt_w(dgrad), 0, cws, cwsb, st));
    RC(lstur_colsum(B, 1, part + D, D + 1, p->dense.uatt_b(dgrad), 0, cws, cwsb, st));
  } else {
    cudaMemsetAsync(d_docv, 0, (size_t)Nh * D * 4, st);
  }
  // 4. user-embedding gradient: dedup + segment-sorted sum (k10 backward)
  if (arch_has_user(c.arch)) {
    RC(lstur_sort_unique_i32(B, b->user, p->ws.sorted_pos(ws), p->ws.user_rows(ws), p->ws.seg_start(ws), p->ws.inverse(ws),
                             p->ws.n_user_rows(ws), st));
    // contiguous per-sample copy (also what the data-parallel sparse exchange sends); the user-vector multiplier
    // (dgru / id_keep) scales the gradient of its embedding row
    float* d_u0 = p->ws.d_u0(ws);
    if (du0) cudaMemcpy2DAsync(d_u0, (size_t)c.Ue * 4, du0, (size_t)lddu0 * 4, (size_t)c.Ue * 4, B, cudaMemcpyDeviceToDevice, st);
    if (b->user_scale2 != nullptr && arch_uc(c) != c.Ue) {
      if (b->user_scale) RC(lstur_scale_rows(B, G, b->user_scale, d_u0, c.Ue, st));
      RC(lstur_scale_rows(B, c.Ue - G, b->user_scale2, d_u0 + G, c.Ue, st));
    } else if (b->user_scale) RC(lstur_scale_rows(B, c.Ue, b->user_scale, d_u0, c.Ue, st));
    RC(lstur_segment_sum_rows(B, c.Ue, p->ws.n_user_rows(ws), p->ws.seg_start(ws), p->ws.sorted_pos(ws), d_u0, c.Ue,
                              p->ws.d_user_rows(ws), st));
  }
  // 5a. vertical / subvertical Embedding backward (task/cook.py:99-103): the extra columns of d doc_vec
  if (c.dv + c.ds) {
    float* vws = p->ws.vert_grad_ws(ws);
    const size_t vwsb = p->ws.vert_grad_ws.bytes();
    if (c.dv) RC(lstur_small_table_grad(N, D, c.Dd, c.dv, c.n_vert, p->ws.title_vert(ws), d_docv, p->dense.vert_emb(dgrad),
                                        vws, vwsb, st));
    if (c.ds) RC(lstur_small_table_grad(N, D, c.Dd + c.dv, c.ds, c.n_subvert, p->ws.title_subvert(ws), d_docv,
                                        p->dense.subvert_emb(dgrad), vws, vwsb, st));
  }
  // 5b. auxiliary vertical classifier backward (task/paper.py:973-990): loss += aux_gain * mean over the B*(W+C) positions
  if (c.aux_nv && p->last_aux) {
    const int Hd = c.aux_hidden, nv = c.aux_nv;
    float* hid = p->ws.vs_hid(ws);
    float* dlg = p->ws.vs_dlogit(ws);
    float* dhid = p->ws.vs_dhid(ws);
    float* ddoc = p->ws.vs_ddoc(ws);
    RC(lstur_softmax_ce_labels(N, nv, p->ws.vs_logit(ws), p->ws.vs_label(ws), nullptr, nullptr, nullptr, dlg,
                               c.aux_gain * grad_scale / (float)(c.W + c.C), st));
    RC(GEMM(1, 0, Hd, nv, N, hid, Hd, dlg, nv, p->dense.vs_w2(dgrad), nv, nullptr, 0, gws, gwsb, st));
    RC(lstur_colsum(N, nv, dlg, nv, p->dense.vs_b2(dgrad), 0, cws, cwsb, st));
    RC(GEMM(0, 1, N, Hd, nv, dlg, nv, p->dense.vs_w2(w->dense), nv, dhid, Hd, nullptr, 0, gws, gwsb, st));
    RC(lstur_relu_bwd((long long)N * Hd, hid, dhid, st));
    RC(GEMM(1, 0, D, Hd, N, docv, D, dhid, Hd, p->dense.vs_w1(dgrad), Hd, nullptr, 0, gws, gwsb, st));
    RC(lstur_colsum(N, Hd, dhid, Hd, p->dense.vs_b1(dgrad), 0, cws, cwsb, st));
    RC(GEMM(0, 1, N, D, Hd, dhid, Hd, p->dense.vs_w1(w->dense), Hd, ddoc, D, nullptr, 0, gws, gwsb, st));
    RC(lstur_scale_rows(Nh, D, p->ws.hist_mask(ws), ddoc, D, st));     // the classifier saw doc_vec * history mask
    RC(lstur_axpby((long long)N * D, 1.f, ddoc, 1.f, d_docv, st));
  }
  // 5. news-encoder backward over all N titles
  RC(encoder_backward(p, w, ws, N, dgrad, word_grad, grad_scale, st));
  return cuda_status("lstur_backward");
}
