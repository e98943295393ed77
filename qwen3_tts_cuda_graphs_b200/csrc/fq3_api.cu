// fq3_api.cu — host side of libfq3.so: engine construction, phase-program builders, C ABI (include/fq3.h).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <array>
#include <vector>

#include "../../include/fq3.h"
#include "fq3_kernel.cuh"

using namespace fq3;

namespace {

thread_local std::string g_err;
int fail(int code, const std::string& msg) {
  g_err = msg;
  return -code;
}
#define CK(call)                                                                                     \
  do {                                                                                               \
    cudaError_t _e = (call);                                                                         \
    if (_e != cudaSuccess)                                                                           \
      return fail(FQ3_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(_e) + " @" + __FILE__ + ":" + \
                                  std::to_string(__LINE__));                                         \
  } while (0)

inline size_t round_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct StackHost {
  fq3_stack_desc d;
  std::vector<uint64_t> offs;
  int qdim() const { return d.n_q_heads * d.head_dim; }
  int kvdim() const { return d.n_kv_heads * d.head_dim; }
  int qkvdim() const { return qdim() + 2 * kvdim(); }
  int kmax() const { return std::max(std::max(d.hidden, d.inter), qdim()); }
};

}  // namespace

struct fq3_engine {
  int dev = 0, G = 0;
  size_t smem_max = 0;
  fq3_model_desc desc{};
  StackHost tk, pr;
  std::vector<uint64_t> lm_head_offs, pred_embed_offs;
  int max_rows = 8;
  int ncb = 15;
  void* bufs[kNumBufs] = {};
  int ld[kNumBufs] = {};
  size_t buf_bytes[kNumBufs] = {};
  StackRt rt[2]{};
  StreamState* d_st = nullptr;
  StreamPolicy* d_spol = nullptr;  // [max_streams] per-stream sampling policies (fq3_set_stream_policy), zeroed = none
  std::vector<uint8_t> spol_on;    // host mirror of the records' `on` flags, in call order: a launch none of whose streams has a
                                   // record gets no record pointer, so its samplers issue no extra load on the critical path
  std::vector<StreamState> h_st;
  std::vector<int> text_rows;      // per stream: text rows given by the host (n_trailing; only host calls change it)
  std::vector<uint8_t> text_open;  // per stream: fq3_open_text was called and the text has not been closed since
  LLWord* attn_part = nullptr;
  size_t attn_part_bytes = 0;
  int* err_host = nullptr;
  int* err_dev = nullptr;
  float* pred_logits_all = nullptr;
  int frames_rows = 0;  // streams of the last persistent launch if it ran the reference-shaped frame program, else 0
  uint8_t* seen_scratch = nullptr;
  Phase *d_frames = nullptr, *d_pred = nullptr, *d_talker = nullptr, *d_prefill = nullptr, *d_linear = nullptr, *d_wide = nullptr;
  std::vector<Phase> h_frames, h_pred, h_talker, h_prefill, h_wide;  // host copies (shared-memory sizing)
  int n_frames_ph = 0, n_pred_ph = 0, n_talker_ph = 0, n_prefill_ph = 0, n_wide_ph = 0;
  int ref_stages = 0;     // ring stages of a single-stream launch of the frame program (the wide program copies its k-splits)
  int wide_rows = 0;      // streams per lock-step group of the wide frame program (0: not available for this model)
  std::vector<uint8_t> in_wpin;  // per stream: the predictor's pass-0 input rows live in BUF_WPIN (1) or in the pair layout (0)
  uint8_t* tiled = nullptr;               // fragment images of every GEMV matrix (fq3_tile_weights_kernel); Phase::w_off indexes it
  size_t tiled_bytes = 0;
  std::vector<std::pair<uint64_t, uint64_t>> tiled_map;  // arena byte offset -> image byte offset
  uint8_t* lin_img = nullptr;             // scratch image of fq3_linear's matrix
  size_t lin_img_bytes = 0;
  size_t tiled_used = 0;
  int64_t launches = 0;
  long long* prof = nullptr;
  std::vector<Plan> plans;                 // GEMV partitions, one per distinct (N, K, SwiGLU)
  int n_sms = 0;                           // SMs of the device (G <= n_sms: the rest stays free for the codec)
  std::vector<std::array<int, 3>> plan_keys;
  long ring_cap = 0;      // optional cap on the weight ring (FQ3_RING_KB), 0 = all remaining shared memory
  int prof_cta = -1;
  uint32_t epoch = 1;     // LL epoch counter (monotonic across launches)
  int lin_words = 0;      // capacity (words per row) of the fq3_linear staging buffers
  unsigned long long watchdog_ns = 4000000000ull;
  std::vector<void*> owned;
};

namespace {

template <class T>
int dalloc(fq3_engine* e, T** p, size_t n, bool zero = true) {
  void* q = nullptr;
  CK(cudaMalloc(&q, std::max<size_t>(n * sizeof(T), 16)));
  if (zero) CK(cudaMemset(q, 0, std::max<size_t>(n * sizeof(T), 16)));
  e->owned.push_back(q);
  *p = reinterpret_cast<T*>(q);
  return 0;
}

uint32_t off16(uint64_t byte_off) { return (uint32_t)(byte_off >> 4); }

// Partition of one GEMV shape over the grid (fq3_common.cuh: Plan): 8-row groups per CTA, the twelve consumer warps of a
// CTA split between groups and k-parts.
bool make_plan(int G, int N, int K, bool swiglu, Plan* out) {
  if (N < 2 || (N & 1) || K < 64 || (K % 64)) return false;
  if (swiglu && (N & 3)) return false;
  Plan pl{};
  pl.ro_shift = swiglu ? 2 : 1;
  const int n_groups = (N + kGroupRows - 1) / kGroupRows;
  pl.g_base = n_groups / G;
  pl.g_rem = n_groups - pl.g_base * G;
  const int g_max = pl.g_base + (pl.g_rem ? 1 : 0);
  pl.nch = K / kChunkK;
  pl.wpg = g_max >= kConsumerWarps ? 1 : std::max(1, std::min(kConsumerWarps / std::max(1, g_max), pl.nch));
  pl.gpr = kConsumerWarps / pl.wpg;
  pl.spg = (K * 16 + kStageBytes - 1) / kStageBytes;
  pl.inv_k = 1.0f / (float)K;
  *out = pl;
  return true;
}
int plan_for(fq3_engine* e, int N, int K, bool swiglu) {
  const std::array<int, 3> key{N, K, swiglu ? 1 : 0};
  for (size_t i = 0; i < e->plan_keys.size(); ++i)
    if (e->plan_keys[i] == key) return (int)i;
  Plan pl{};
  if (!make_plan(e->G, N, K, swiglu, &pl) || (int)e->plans.size() >= kMaxPlans - 1) return -1;
  e->plans.push_back(pl);
  e->plan_keys.push_back(key);
  return (int)e->plans.size() - 1;
}
static bool g_plan_fail = false;
uint8_t plan_id(fq3_engine* e, int N, int K, bool swiglu) {
  const int id = plan_for(e, N, K, swiglu);
  if (id < 0) { g_plan_fail = true; return 0; }
  return (uint8_t)id;
}

// One decoder layer = 5 phases (DESIGN.md §3.2).
void push_layer(fq3_engine* e, std::vector<Phase>& v, const StackHost& s, uint8_t stack, int layer, bool rows2, uint8_t aux,
                bool keep) {
  const uint64_t* o = &s.offs[(size_t)layer * 8];
  const uint16_t r2 = rows2 ? F_ROWS2 : 0, kp = keep ? F_L2_KEEP : 0;
  const uint8_t X = stack == ST_TALKER ? BUF_TX : BUF_PX, Q = stack == ST_TALKER ? BUF_TQKV : BUF_PQKV,
                A = stack == ST_TALKER ? BUF_TATT : BUF_PATT, C = stack == ST_TALKER ? BUF_TACT : BUF_PACT;
  Phase p{};
  p.stack = stack; p.layer = (uint8_t)layer; p.aux = aux;
  // 1. RMSNorm + fused QKV projection
  p.type = PH_GEMV; p.flags = F_PRENORM | r2 | kp; p.in_buf = X; p.out_buf = Q; p.res_buf = 0;
  p.w_off = off16(o[1]); p.g_off = off16(o[0]); p.b_off = 0; p.N = s.qkvdim(); p.K = s.d.hidden;
  p.plan = plan_id(e, p.N, p.K, false);
  v.push_back(p);
  // 2. q/k norm + RoPE + KV append + attention
  p.type = PH_ATTN; p.flags = r2; p.in_buf = Q; p.out_buf = A; p.w_off = 0; p.g_off = off16(o[2]); p.b_off = off16(o[3]);
  p.N = 0; p.K = 0; p.plan = 0;
  v.push_back(p);
  // 3. o_proj + residual
  p.type = PH_GEMV; p.flags = F_RESID | r2 | kp; p.in_buf = A; p.out_buf = X; p.res_buf = X;
  p.w_off = off16(o[4]); p.g_off = 0; p.b_off = 0; p.N = s.d.hidden; p.K = s.qdim();
  p.plan = plan_id(e, p.N, p.K, false);
  v.push_back(p);
  // 4. RMSNorm + gate/up + SiLU*mul
  p.flags = F_PRENORM | F_SWIGLU | r2 | kp; p.in_buf = X; p.out_buf = C; p.res_buf = 0;
  p.w_off = off16(o[6]); p.g_off = off16(o[5]); p.N = 2 * s.d.inter; p.K = s.d.hidden;
  p.plan = plan_id(e, p.N, p.K, true);
  v.push_back(p);
  // 5. down_proj + residual
  p.flags = F_RESID | r2 | kp; p.in_buf = C; p.out_buf = X; p.res_buf = X;
  p.w_off = off16(o[7]); p.g_off = 0; p.N = s.d.hidden; p.K = s.d.inter;
  p.plan = plan_id(e, p.N, p.K, false);
  v.push_back(p);
}

void push_predictor(std::vector<Phase>& v, fq3_engine* e, bool only) {
  for (int i = 0; i < e->ncb; ++i) {
    const bool r2 = (i == 0);
    if (e->desc.has_s2m) {
      Phase p{};
      p.type = PH_GEMV; p.stack = ST_PRED; p.aux = (uint8_t)i; p.flags = F_BIAS | F_L2_KEEP | (r2 ? F_ROWS2 : 0);
      p.in_buf = BUF_PIN; p.out_buf = BUF_PX; p.w_off = off16(e->desc.s2m_w_off); p.b_off = off16(e->desc.s2m_b_off);
      p.N = e->pr.d.hidden; p.K = e->tk.d.hidden;
      p.plan = plan_id(e, p.N, p.K, false);
      v.push_back(p);
    }
    for (int l = 0; l < e->pr.d.n_layers; ++l) push_layer(e, v, e->pr, ST_PRED, l, r2, (uint8_t)i, true);
    Phase h{};
    h.type = PH_GEMV; h.stack = ST_PRED; h.aux = (uint8_t)i;
    h.flags = F_PRENORM | F_OUT_F32 | F_L2_KEEP | (r2 ? F_ROWS2 : 0);
    h.in_buf = BUF_PX; h.out_buf = BUF_LOGITS; h.w_off = off16(e->lm_head_offs[i]);
    h.g_off = off16(e->pr.d.final_norm_off); h.N = e->pr.d.vocab; h.K = e->pr.d.hidden;
    h.plan = plan_id(e, h.N, h.K, false);
    v.push_back(h);
    Phase s{};
    s.type = PH_SAMPLE; s.stack = ST_PRED; s.aux = (uint8_t)i; s.skind = only ? SMP_PRED_ONLY : SMP_PRED;
    s.flags = r2 ? F_ROWS2 : 0;
    v.push_back(s);
  }
}

// Predictor of the wide frame program (more than four lock-step streams).  Pass 0 of the reference feeds two rows per stream,
// [past_hidden ; codec_embed(token)] (predictor_graph.py:125-139); here it runs as two single-row passes — 0a: past_hidden at
// position 0 (it only has to leave its K/V rows behind: no head, no sampler, and the last layer stops after attention), 0b:
// codec_embed(token) at position 1 — so every GEMV phase stages one row per stream.  Causal attention makes that the same
// arithmetic.  Input rows come from BUF_WPIN (by stream slot).
void push_predictor_wide(std::vector<Phase>& v, fq3_engine* e) {
  const int L = e->pr.d.n_layers;
  for (int half = 0; half < 2; ++half) {
    const uint16_t fb = half ? F_WPIN_B : 0;
    const size_t first = v.size();
    if (e->desc.has_s2m) {
      Phase p{};
      p.type = PH_GEMV; p.stack = ST_PRED; p.aux = 0; p.flags = F_BIAS | F_L2_KEEP | F_IN_PREV | fb;
      p.in_buf = BUF_WPIN; p.out_buf = BUF_PX; p.w_off = off16(e->desc.s2m_w_off); p.b_off = off16(e->desc.s2m_b_off);
      p.N = e->pr.d.hidden; p.K = e->tk.d.hidden;
      p.plan = plan_id(e, p.N, p.K, false);
      v.push_back(p);
    }
    for (int l = 0; l < L; ++l) {
      const size_t at = v.size();
      push_layer(e, v, e->pr, ST_PRED, l, false, 0, true);
      if (l == 0 && !e->desc.has_s2m) {  // layer 0 reads its input and residual rows straight from BUF_WPIN
        v[at].in_buf = BUF_WPIN; v[at].flags |= F_IN_PREV | fb;
        v[at + 2].res_buf = BUF_WPIN; v[at + 2].flags |= fb;
      }
      if (half == 0) v[at + 1].flags |= F_PASS0A;
      if (half == 0 && l == L - 1) v.resize(at + 2);
    }
    (void)first;
  }
  for (int i = 0; i < e->ncb; ++i) {
    if (i > 0) {
      if (e->desc.has_s2m) {
        Phase p{};
        p.type = PH_GEMV; p.stack = ST_PRED; p.aux = (uint8_t)i; p.flags = F_BIAS | F_L2_KEEP;
        p.in_buf = BUF_PIN; p.out_buf = BUF_PX; p.w_off = off16(e->desc.s2m_w_off); p.b_off = off16(e->desc.s2m_b_off);
        p.N = e->pr.d.hidden; p.K = e->tk.d.hidden;
        p.plan = plan_id(e, p.N, p.K, false);
        v.push_back(p);
      }
      for (int l = 0; l < L; ++l) push_layer(e, v, e->pr, ST_PRED, l, false, (uint8_t)i, true);
    }
    Phase h{};
    h.type = PH_GEMV; h.stack = ST_PRED; h.aux = (uint8_t)i;
    h.flags = F_PRENORM | F_OUT_F32 | F_L2_KEEP;
    h.in_buf = BUF_PX; h.out_buf = BUF_LOGITS; h.w_off = off16(e->lm_head_offs[i]);
    h.g_off = off16(e->pr.d.final_norm_off); h.N = e->pr.d.vocab; h.K = e->pr.d.hidden;
    h.plan = plan_id(e, h.N, h.K, false);
    v.push_back(h);
    Phase sm{};
    sm.type = PH_SAMPLE; sm.stack = ST_PRED; sm.aux = (uint8_t)i; sm.skind = SMP_PRED;
    v.push_back(sm);
  }
}

void push_talker(std::vector<Phase>& v, fq3_engine* e, bool last_row_head) {
  for (int l = 0; l < e->tk.d.n_layers; ++l) push_layer(e, v, e->tk, ST_TALKER, l, false, 0, false);
  Phase h{};
  h.type = PH_GEMV; h.stack = ST_TALKER;
  h.flags = F_PRENORM | F_OUT_F32 | F_WRITE_NORMED | (last_row_head ? F_LAST_ROW : 0);
  h.in_buf = BUF_TX; h.out_buf = BUF_LOGITS; h.w_off = off16(e->desc.codec_head_off);
  h.g_off = off16(e->tk.d.final_norm_off); h.N = e->tk.d.vocab; h.K = e->tk.d.hidden;
  h.plan = plan_id(e, h.N, h.K, false);
  v.push_back(h);
}

// Point every GEMV phase of a program at the fragment image of its matrix (built on first use), then upload the program.
int upload(fq3_engine* e, std::vector<Phase>& v, Phase** d) {
  const uint8_t* arena = reinterpret_cast<const uint8_t*>(e->desc.arena);
  // kinds: phases that agree in everything but their weights (the consumers' view), numbered in order of appearance
  std::vector<std::array<uint32_t, 8>> kinds;
  for (Phase& ph : v) {
    if (ph.type != PH_GEMV) continue;
    const std::array<uint32_t, 8> key{ph.flags, ph.in_buf, ph.out_buf, ph.res_buf, ph.N, ph.K, ph.plan, ph.b_off};
    size_t k = 0;
    while (k < kinds.size() && kinds[k] != key) ++k;
    if (k == kinds.size()) kinds.push_back(key);
    if (k >= (size_t)kMaxKinds) return -1;
    ph.kind = (uint8_t)k;
  }
  for (Phase& ph : v) {
    if (ph.type != PH_GEMV) continue;
    if (ph.N % 8) return -1;  // model matrices: whole 8-row groups (the image has the size of the matrix)
    const uint64_t aoff = (uint64_t)ph.w_off * 16;
    uint64_t ioff = ~0ull;
    for (auto& m : e->tiled_map)
      if (m.first == aoff) ioff = m.second;
    if (ioff == ~0ull) {
      size_t used = 0;
      if (!e->tiled_map.empty()) used = e->tiled_used;
      ioff = used;
      const size_t bytes = (size_t)ph.N * ph.K * 2;
      if (ioff + bytes > e->tiled_bytes) return -1;
      fq3_tile_weights_kernel<<<256, 256>>>(reinterpret_cast<const bf16*>(arena + aoff), reinterpret_cast<uint4*>(e->tiled + ioff), (int)ph.N,
                                            (int)ph.K);
      if (cudaGetLastError() != cudaSuccess) return -1;
      e->tiled_map.push_back({aoff, ioff});
      e->tiled_used = (ioff + bytes + 1023) / 1024 * 1024;
    }
    ph.w_off = off16(ioff);
  }
  if (dalloc(e, d, v.size(), false)) return -1;
  if (cudaMemcpy(*d, v.data(), v.size() * sizeof(Phase), cudaMemcpyHostToDevice) != cudaSuccess) return -1;
  return 0;
}

void fill_common(fq3_engine* e, LaunchParams& p) {
  p.arena = reinterpret_cast<const uint8_t*>(e->desc.arena);
  p.tiled = e->tiled;
  for (int i = 0; i < kNumBufs; ++i) { p.bufs[i] = e->bufs[i]; p.ld[i] = e->ld[i]; }
  p.stacks[0] = e->rt[0];
  p.stacks[1] = e->rt[1];
  p.st = e->d_st;
  p.attn_part = e->attn_part;
  for (size_t i = 0; i < e->plans.size(); ++i) p.plans[i] = e->plans[i];
  p.err = e->err_dev;
  p.n_code_groups = e->desc.n_code_groups;
  p.eos_id = e->desc.eos_id;
  p.has_s2m = e->desc.has_s2m;
  p.max_frames = e->desc.max_frames;
  p.codec_embed = reinterpret_cast<const bf16*>(p.arena + e->desc.codec_embed_off);
  for (int i = 0; i < e->ncb; ++i) p.pred_embeds[i] = reinterpret_cast<const bf16*>(p.arena + e->pred_embed_offs[i]);
  p.pred_logits_all = nullptr;
  p.pos_override = -1;
  p.watchdog_ns = e->watchdog_ns;
  p.debug = (16 << 16) | 32;  // poll back-off: sleep 32 ns after 16 immediate retries (FQ3_DEBUG = tries << 16 | ns)
  p.prof = e->prof;
  p.prof_cta = e->prof_cta;
  if (const char* d = getenv("FQ3_DEBUG")) p.debug = atoi(d);
  p.n_iters = 1;
  p.stream0 = 0;
  p.wide = 0;
  p.max_streams = e->desc.max_streams;
}

int check_device_fault(fq3_engine* e) {
  if (e->err_host && e->err_host[0] != 0) {
    char b[256];
    snprintf(b, sizeof b, "device watchdog fault: code=%d cta=%d phase=%d detail=%d (1=grid barrier 2=ring full-wait "
                          "3=ring empty-wait 4=frame handshake 5=bad phase)",
             e->err_host[0], e->err_host[1], e->err_host[2], e->err_host[3]);
    return fail(FQ3_E_DEVICE_FAULT, b);
  }
  return 0;
}

// rows of the B operand a GEMV phase stages (kernel: phase_m / b_rows)
int phase_rows_host(const Phase& ph, int n_rows) {
  if (ph.flags & F_LAST_ROW) return 1;
  return (ph.flags & F_ROWS2) ? 2 * n_rows : n_rows;
}

// Every API entry that launches the persistent kernel reserves its LL epochs first — before it stages any input.  Phase i
// of iteration `it` of a launch carries epoch_base + it * n_phases + i + 1; the 32-bit counter wraps after ~4e9 phases
// (hours of serving).  On a wrap the epoch halves of all LL words are reset to 0 ("written before the launch") and the
// payloads are kept, so the state that crosses launches (predictor input rows, frame control records) survives.
int reserve_epochs(fq3_engine* e, uint64_t span, cudaStream_t s) {
  if (int r = check_device_fault(e)) return r;
  if ((uint64_t)e->epoch + span >= 0xFFFFFF00ull) {
    for (int i = 0; i < kNumBufs; ++i)
      if (e->buf_bytes[i]) fq3_ll_clear_epochs_kernel<<<64, 256, 0, s>>>(reinterpret_cast<LLWord*>(e->bufs[i]), e->buf_bytes[i] / sizeof(LLWord));
    fq3_ll_clear_epochs_kernel<<<64, 256, 0, s>>>(e->attn_part, e->attn_part_bytes / sizeof(LLWord));
    fq3_ctl_clear_epochs_kernel<<<1, 64, 0, s>>>(e->d_st, e->desc.max_streams);
    e->launches += 2;
    CK(cudaGetLastError());
    e->epoch = 1;
  }
  return 0;
}

// Launch the persistent kernel: one CTA per SM, cooperative (all CTAs must be co-resident: they poll each other's words).
// smem: header | scratch | program | norm-weight slots | activation rows | weight ring (16 KB stages, everything that is left).
// shared-memory carve-up of a launch: fills p.xbuf_bytes / prog_bytes / gam_bytes / n_stages; returns the fixed bytes or < 0
long carve(fq3_engine* e, LaunchParams& p, const Phase* prog_host) {
  size_t xbytes = 0, gamma_elems = 0;
  for (int i = 0; i < p.n_phases; ++i) {
    const Phase& ph = prog_host[i];
    if (ph.type != PH_GEMV) continue;
    const int M = phase_rows_host(ph, p.n_rows);
    if (M > (p.wide ? kMaxWide : kMaxRows)) return fail(FQ3_E_UNSUPPORTED, "more activation rows than the GEMV stage takes");
    // single-stream rows alternate between two buffers; the rows of a multi-row phase are padded (kernel: xrow_stride)
    xbytes = std::max(xbytes, (M == 1 && !p.wide) ? (size_t)4 * ph.K : (size_t)M * ((size_t)ph.K * 2 + 64));
    if (ph.flags & F_PRENORM) gamma_elems = std::max(gamma_elems, (size_t)ph.K);
  }
  p.xbuf_bytes = (int)round_up(xbytes, 2048);
  p.prog_bytes = (int)round_up((size_t)kKindBytes + kUnitBytes + (size_t)p.n_phases * sizeof(Phase), 1024);
  p.gam_bytes = (int)round_up(gamma_elems * 2, 1024);
  // Shared memory and L1 share 256 KB per SM: staying at or below the 196 KB carve-out leaves 60 KB of L1 for the table
  // reads of the attention and sampling phases.
  const long fixed = kHeaderBytes + kScratchBytes + (long)p.xbuf_bytes + (long)p.prog_bytes + (long)kGammaSlots * p.gam_bytes;
  const long budget = e->ring_cap > 0 ? (long)e->smem_max : std::min<long>((long)e->smem_max, 196L * 1024);
  long avail = budget - fixed;
  if (avail < 6L * kStageBytes) avail = (long)e->smem_max - fixed;
  if (e->ring_cap > 0) avail = std::min(avail, e->ring_cap);
  p.n_stages = (int)std::min<long>(kMaxStages, avail / kStageBytes);
  if (p.n_stages < 2) return fail(FQ3_E_INVALID, "not enough shared memory for the weight ring");
  return fixed;
}

int launch(fq3_engine* e, LaunchParams& p, const Phase* prog_host, cudaStream_t s) {
  const int grid = e->G;
  const long fixed = carve(e, p, prog_host);
  if (fixed < 0) return (int)fixed;
  // one representative phase per GEMV kind (the kernel resolves the kinds at start)
  p.n_kinds = 0;
  for (int i = 0; i < p.n_phases; ++i) {
    const Phase& ph = prog_host[i];
    if (ph.type != PH_GEMV) continue;
    if (ph.kind >= kMaxKinds) return fail(FQ3_E_INVALID, "phase kind out of range");
    if (ph.kind >= p.n_kinds) {
      p.n_kinds = ph.kind + 1;
      p.kind_phase[ph.kind] = (uint16_t)i;
    }
  }
  const size_t smem = (size_t)fixed + (size_t)p.n_stages * kStageBytes;
  // A round of a GEMV phase (gpr groups x spg stages) must fit in the ring (kernel: gemv_phase_consume).  Shapes that do not
  // (1.7B gate/up: 12 groups x 2 stages per CTA) take fewer groups per round and more warps per group.
  for (int i = 0; i < p.n_phases; ++i) {
    const Phase& ph = prog_host[i];
    if (ph.type != PH_GEMV) continue;
    Plan& pl = p.plans[ph.plan];
    if (pl.spg > p.n_stages) return fail(FQ3_E_UNSUPPORTED, "K too large for the weight ring");
    const int g_max = pl.g_base + (pl.g_rem ? 1 : 0);
    const bool follow_ref = p.mode == MODE_FRAMES && (p.wide || p.n_rows > 1) && e->ref_stages > 0;
    if (follow_ref && std::min(pl.gpr, g_max) * pl.spg > e->ref_stages) {
      // the k-split (warps per group) a single-stream launch of the frame program uses for this shape: a batched launch must
      // add a row's products in the same order, whatever its own (smaller) ring allows
      pl.gpr = e->ref_stages / pl.spg;
      pl.wpg = std::max(1, std::min(kConsumerWarps / pl.gpr, pl.nch));
    }
    if (std::min(pl.gpr, g_max) * pl.spg > p.n_stages) {
      pl.gpr = p.n_stages / pl.spg;
      if (!follow_ref) pl.wpg = std::max(1, std::min(kConsumerWarps / pl.gpr, pl.nch));  // batched frame loops: same k-split, more rounds
    }
  }

  const uint64_t span = (uint64_t)p.n_iters * (uint64_t)p.n_phases + 2;
  if ((uint64_t)e->epoch + span >= 0xFFFFFFF0ull) return fail(FQ3_E_INVALID, "LL epochs were not reserved for this launch");
  p.epoch_base = e->epoch;
  e->epoch += (uint32_t)span;
  void* args[] = {&p};
  void* fn = p.wide ? (void*)fq3_stream_kernel<false, true> : (p.prof ? (void*)fq3_stream_kernel<true, false> : (void*)fq3_stream_kernel<false, false>);
  CK(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(kThreads), args, smem, s));
  e->launches += 1;
  e->frames_rows = (p.mode == MODE_FRAMES && !p.wide) ? p.n_rows : 0;
  return 0;
}

// ---- plain <-> LL conversions at the ABI boundary ----
int pack_ll(fq3_engine* e, int buf, int row0, const void* src, int ld_src, int rows, int cols, cudaStream_t s) {
  LLWord* dst = reinterpret_cast<LLWord*>(e->bufs[buf]) + (size_t)row0 * e->ld[buf];
  const int n = rows * cols;
  fq3_pack_ll_kernel<<<std::max(1, std::min(64, (n + 255) / 256)), 256, 0, s>>>(dst, e->ld[buf], reinterpret_cast<const bf16*>(src),
                                                                          ld_src, rows, cols);
  e->launches += 1;
  CK(cudaGetLastError());
  return 0;
}
int unpack_f32(fq3_engine* e, void* dst, int ld_dst, int buf, int row0, int rows, int cols, cudaStream_t s) {
  const LLWord* src = reinterpret_cast<const LLWord*>(e->bufs[buf]) + (size_t)row0 * e->ld[buf];
  const int n = rows * cols;
  fq3_unpack_ll_f32_kernel<<<std::max(1, std::min(64, (n + 255) / 256)), 256, 0, s>>>(reinterpret_cast<float*>(dst), ld_dst, src,
                                                                                e->ld[buf], rows, cols);
  e->launches += 1;
  CK(cudaGetLastError());
  return 0;
}
int unpack_bf16(fq3_engine* e, void* dst, int ld_dst, int buf, int row0, int rows, int cols, cudaStream_t s) {
  const LLWord* src = reinterpret_cast<const LLWord*>(e->bufs[buf]) + (size_t)row0 * e->ld[buf];
  const int n = rows * cols;
  fq3_unpack_ll_bf16_kernel<<<std::max(1, std::min(64, (n + 255) / 256)), 256, 0, s>>>(reinterpret_cast<bf16*>(dst), ld_dst, src,
                                                                                 e->ld[buf], rows, cols);
  e->launches += 1;
  CK(cudaGetLastError());
  return 0;
}

Policy to_policy(const fq3_policy* q) {
  Policy p{};
  p.do_sample = q->do_sample; p.top_k = q->top_k; p.top_p = q->top_p; p.temperature = q->temperature;
  p.rep_pen = q->repetition_penalty; p.min_new_tokens = q->min_new_tokens; p.suppress_tail = q->suppress_tail;
  p.seed = q->seed;
  return p;
}
SubPolicy to_sub(const fq3_subpolicy* q) {
  SubPolicy p{};
  p.do_sample = q->do_sample; p.top_k = q->top_k; p.top_p = q->top_p; p.temperature = q->temperature;
  return p;
}

// The rows that cross launches — [past_hidden ; codec_embed(token)] of every stream — live in the pair layout (rows 2s, 2s+1 of
// BUF_PIN / BUF_PX: prefill, set_loop_state and the frame program of up to four streams) or in BUF_WPIN (the wide program).
// Bring streams [s0, s0 + n) into the layout the next launch reads.
int sync_pin_layout(fq3_engine* e, int s0, int n, bool to_wpin, cudaStream_t s) {
  const int pb = e->desc.has_s2m ? BUF_PIN : BUF_PX;
  for (int i = s0; i < s0 + n; ++i) {
    if ((e->in_wpin[i] != 0) == to_wpin) continue;
    fq3_wpin_from_pairs_kernel<<<1, 256, 0, s>>>(reinterpret_cast<LLWord*>(e->bufs[BUF_WPIN]), e->ld[BUF_WPIN], reinterpret_cast<LLWord*>(e->bufs[pb]),
                                                 e->ld[pb], i, e->desc.max_streams, to_wpin ? 0 : 1);
    e->launches += 1;
    CK(cudaGetLastError());
    e->in_wpin[i] = to_wpin ? 1 : 0;
  }
  return 0;
}

int check_stack(const fq3_stack_desc& d, const char* name) {
  if (d.head_dim != kHeadDim) return fail(FQ3_E_UNSUPPORTED, std::string(name) + ": head_dim must be 128");
  if (d.hidden % 64 || d.inter % 64) return fail(FQ3_E_UNSUPPORTED, std::string(name) + ": dims must be multiples of 64");
  if (d.n_q_heads % d.n_kv_heads) return fail(FQ3_E_UNSUPPORTED, std::string(name) + ": nq % nkv != 0");
  if (d.n_q_heads / d.n_kv_heads > kGq) return fail(FQ3_E_UNSUPPORTED, std::string(name) + ": more than 2 q heads per kv head");
  if (d.vocab > kMaxVocab) return fail(FQ3_E_UNSUPPORTED, std::string(name) + ": vocab exceeds sampling scratch");
  if (d.vocab % 4) return fail(FQ3_E_UNSUPPORTED, std::string(name) + ": vocab must be a multiple of 4");
  return 0;
}

}  // namespace

extern "C" {

int fq3_abi_version(void) { return FQ3_ABI_VERSION; }
const char* fq3_last_error(void) { return g_err.c_str(); }

static int create_impl(const fq3_model_desc* desc, fq3_engine* e);

int fq3_create(const fq3_model_desc* desc, fq3_engine** out) {
  if (!desc || !out) return fail(FQ3_E_INVALID, "null argument");
  *out = nullptr;
  fq3_engine* e = new fq3_engine();
  const int r = create_impl(desc, e);
  if (r) {  // every early return of create_impl lands here: nothing leaks
    const std::string msg = g_err;
    fq3_destroy(e);
    g_err = msg;
    return r;
  }
  *out = e;
  return 0;
}

static int create_impl(const fq3_model_desc* desc, fq3_engine* e) {
  if (desc->abi_version != FQ3_ABI_VERSION) return fail(FQ3_E_INVALID, "ABI version mismatch");
  if (int r = check_stack(desc->talker, "talker")) return r;
  if (int r = check_stack(desc->predictor, "predictor")) return r;
  if (desc->n_code_groups < 2 || desc->n_code_groups > FQ3_MAX_CODE_GROUPS) return fail(FQ3_E_INVALID, "n_code_groups");
  if (desc->max_streams < 1) return fail(FQ3_E_INVALID, "max_streams");
  if (!desc->has_s2m && desc->talker.hidden != desc->predictor.hidden)
    return fail(FQ3_E_INVALID, "talker/predictor widths differ but no small_to_mtp projection given");
  e->desc = *desc;
  CK(cudaGetDevice(&e->dev));
  int sms = 0, smem_optin = 0, coop = 0;
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, e->dev));
  CK(cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, e->dev));
  CK(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, e->dev));
  if (!coop) return fail(FQ3_E_UNSUPPORTED, "device lacks cooperative launch");
  // 128 CTAs: the partitions of every model shape come out even (whole 8-row groups per CTA, the K-splits fill the 128
  // rows of an MMA tile), the exchange has fewer parties, and the remaining SMs stay free for the codec decode of the
  // previous streaming chunk (DESIGN.md §3.4).  FQ3_GRID overrides.
  e->n_sms = sms;
  e->G = std::min(sms, 128);
  if (const char* g = getenv("FQ3_GRID")) e->G = std::max(1, std::min(sms, atoi(g)));
  if (const char* rk = getenv("FQ3_RING_KB")) e->ring_cap = std::max(16L, atol(rk)) * 1024L;
  if (const char* pc = getenv("FQ3_PROF")) {
    e->prof_cta = atoi(pc);
    if (dalloc(e, &e->prof, 512 * 160 * 2)) return -FQ3_E_CUDA;
  }
  if (const char* w = getenv("FQ3_WATCHDOG_MS")) e->watchdog_ns = (unsigned long long)atoll(w) * 1000000ull;
  e->smem_max = (size_t)smem_optin;
  CK(cudaFuncSetAttribute(fq3_stream_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_optin));
  CK(cudaFuncSetAttribute(fq3_stream_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_optin));
  CK(cudaFuncSetAttribute(fq3_stream_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_optin));
  int occ = 0;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fq3_stream_kernel<false, false>, kThreads, smem_optin));
  if (occ < 1) return fail(FQ3_E_UNSUPPORTED, "stream kernel does not fit on an SM");

  e->ncb = desc->n_code_groups - 1;
  e->tk.d = desc->talker;
  e->pr.d = desc->predictor;
  e->tk.offs.assign(desc->talker.layer_offs, desc->talker.layer_offs + (size_t)desc->talker.n_layers * 8);
  e->pr.offs.assign(desc->predictor.layer_offs, desc->predictor.layer_offs + (size_t)desc->predictor.n_layers * 8);
  e->lm_head_offs.assign(desc->lm_head_offs, desc->lm_head_offs + e->ncb);
  e->pred_embed_offs.assign(desc->pred_embed_offs, desc->pred_embed_offs + e->ncb);
  e->tk.d.layer_offs = nullptr;
  e->pr.d.layer_offs = nullptr;

  const int B = desc->max_streams;
  const int R = std::max(2 * B, 2 * kMaxRows);
  e->max_rows = R;
  const uint8_t* arena = reinterpret_cast<const uint8_t*>(desc->arena);
  // --- static KV caches (StaticCache of talker_graph.py:43 / predictor_graph.py:61) ---
  for (int s = 0; s < 2; ++s) {
    const StackHost& sh = s == 0 ? e->tk : e->pr;
    StackRt& r = e->rt[s];
    r.hidden = sh.d.hidden; r.inter = sh.d.inter; r.n_layers = sh.d.n_layers; r.nq = sh.d.n_q_heads;
    r.nkv = sh.d.n_kv_heads; r.vocab = sh.d.vocab; r.eps = sh.d.rms_eps; r.max_pos = sh.d.max_pos;
    r.rope_len = sh.d.rope_len; r.n_slots = B;
    const size_t n = (size_t)sh.d.n_layers * B * sh.d.n_kv_heads * sh.d.max_pos * kHeadDim;
    if (dalloc(e, &r.kcache, n)) return -FQ3_E_CUDA;
    if (dalloc(e, &r.vcache, n)) return -FQ3_E_CUDA;
    r.rope_cos = reinterpret_cast<const bf16*>(arena + sh.d.rope_cos_off);
    r.rope_sin = reinterpret_cast<const bf16*>(arena + sh.d.rope_sin_off);
  }
  // --- activation buffers ---
  auto mk = [&](int id, int width, size_t elt, int rows) -> int {
    void* q = nullptr;
    if (dalloc(e, reinterpret_cast<uint8_t**>(&q), (size_t)rows * width * elt)) return -1;
    e->bufs[id] = q;
    e->ld[id] = width;
    e->buf_bytes[id] = (size_t)rows * width * elt;
    return 0;
  };
  const int Ht = e->tk.d.hidden, Hp = e->pr.d.hidden;
  const size_t LL = sizeof(LLWord);  // LL buffers: width in packed words (two bf16 per word)
  if (mk(BUF_TX, Ht / 2, LL, R) || mk(BUF_TQKV, e->tk.qkvdim() / 2, LL, R) || mk(BUF_TATT, e->tk.qdim() / 2, LL, R) ||
      mk(BUF_TACT, e->tk.d.inter / 2, LL, R) || mk(BUF_PX, Hp / 2, LL, R) || mk(BUF_PQKV, e->pr.qkvdim() / 2, LL, R) ||
      mk(BUF_PATT, e->pr.qdim() / 2, LL, R) || mk(BUF_PACT, e->pr.d.inter / 2, LL, R) ||
      mk(BUF_LOGITS, std::max(e->tk.d.vocab, e->pr.d.vocab) / 2, LL, R) || mk(BUF_HID, Ht, 2, R))
    return -FQ3_E_CUDA;
  e->buf_bytes[BUF_HID] = 0;  // plain bf16, not an LL buffer
  if (desc->has_s2m) {
    if (mk(BUF_PIN, Ht / 2, LL, R)) return -FQ3_E_CUDA;
  } else {
    e->bufs[BUF_PIN] = e->bufs[BUF_PX];
    e->ld[BUF_PIN] = e->ld[BUF_PX];
  }
  if (mk(BUF_WPIN, Ht / 2, LL, 2 * B)) return -FQ3_E_CUDA;
  e->lin_words = 32768;
  if (mk(BUF_LIN_IN, e->lin_words, LL, kMaxRows) || mk(BUF_LIN_OUT, e->lin_words, LL, kMaxRows) ||
      mk(BUF_LIN_RES, e->lin_words, LL, kMaxRows))
    return -FQ3_E_CUDA;
  const int nqmax = std::max(e->tk.d.n_q_heads, e->pr.d.n_q_heads);
  e->attn_part_bytes = (size_t)R * nqmax * kMaxSplits * kPartStride * sizeof(LLWord);
  if (dalloc(e, &e->attn_part, (size_t)R * nqmax * kMaxSplits * kPartStride)) return -FQ3_E_CUDA;
  if (dalloc(e, &e->pred_logits_all, (size_t)e->ncb * e->pr.d.vocab)) return -FQ3_E_CUDA;
  if (dalloc(e, &e->seen_scratch, (size_t)kMaxVocab * 4)) return -FQ3_E_CUDA;
  CK(cudaHostAlloc(reinterpret_cast<void**>(&e->err_host), 64, cudaHostAllocMapped));
  memset(e->err_host, 0, 64);
  CK(cudaHostGetDevicePointer(reinterpret_cast<void**>(&e->err_dev), e->err_host, 0));
  // --- per-stream state ---
  e->h_st.resize(B);
  e->in_wpin.assign(B, 0);
  e->spol_on.assign(B, 0);
  e->text_rows.assign(B, 0);
  e->text_open.assign(B, 0);
  if (dalloc(e, &e->d_st, B)) return -FQ3_E_CUDA;
  if (dalloc(e, &e->d_spol, B)) return -FQ3_E_CUDA;
  for (int b = 0; b < B; ++b) {
    StreamState& s = e->h_st[b];
    memset(&s, 0, sizeof s);
    bf16 *tr = nullptr, *pe = nullptr;
    if (dalloc(e, &tr, (size_t)e->tk.d.max_pos * Ht)) return -FQ3_E_CUDA;
    if (dalloc(e, &pe, (size_t)Ht)) return -FQ3_E_CUDA;
    if (dalloc(e, &s.held, (size_t)Ht)) return -FQ3_E_CUDA;
    if (dalloc(e, &s.codes, (size_t)desc->max_frames * desc->n_code_groups)) return -FQ3_E_CUDA;
    if (dalloc(e, &s.seen, (size_t)round_up(e->tk.d.vocab, 16))) return -FQ3_E_CUDA;
    s.trailing = tr;
    s.pad_embed = pe;
  }
  CK(cudaMemcpy(e->d_st, e->h_st.data(), sizeof(StreamState) * B, cudaMemcpyHostToDevice));
  // --- programs + tiled weight images ---
  auto gemv_bytes = [&](const StackHost& sh) {
    return (size_t)sh.d.n_layers * ((size_t)sh.qkvdim() * sh.d.hidden + (size_t)sh.d.hidden * sh.qdim() + 3ull * sh.d.hidden * sh.d.inter) * 2;
  };
  e->tiled_bytes = gemv_bytes(e->tk) + gemv_bytes(e->pr) + (size_t)e->tk.d.vocab * e->tk.d.hidden * 2 +
                   (size_t)e->ncb * e->pr.d.vocab * e->pr.d.hidden * 2 + (desc->has_s2m ? (size_t)e->pr.d.hidden * e->tk.d.hidden * 2 : 0) +
                   1024 * (size_t)(8 * (e->tk.d.n_layers + e->pr.d.n_layers) + e->ncb + 8);
  if (dalloc(e, &e->tiled, e->tiled_bytes, false)) return -FQ3_E_CUDA;
  std::vector<Phase>& v = e->h_frames;
  push_predictor(v, e, false);
  push_talker(v, e, false);
  {
    Phase s{};
    s.type = PH_SAMPLE; s.stack = ST_TALKER; s.skind = SMP_TALKER;
    v.push_back(s);
  }
  push_predictor(e->h_pred, e, true);
  push_talker(e->h_talker, e, false);
  push_talker(e->h_prefill, e, true);
  {
    Phase s{};
    s.type = PH_SAMPLE; s.stack = ST_TALKER; s.skind = SMP_PREFILL;
    e->h_prefill.push_back(s);
  }
  push_predictor_wide(e->h_wide, e);
  push_talker(e->h_wide, e, false);
  {
    Phase s{};
    s.type = PH_SAMPLE; s.stack = ST_TALKER; s.skind = SMP_TALKER;
    e->h_wide.push_back(s);
  }
  if (g_plan_fail) { g_plan_fail = false; return fail(FQ3_E_UNSUPPORTED, "a GEMV shape of this model cannot be partitioned (odd N or K % 64)"); }
  e->n_frames_ph = (int)e->h_frames.size();
  e->n_pred_ph = (int)e->h_pred.size();
  e->n_talker_ph = (int)e->h_talker.size();
  e->n_prefill_ph = (int)e->h_prefill.size();
  e->n_wide_ph = (int)e->h_wide.size();
  if (upload(e, e->h_wide, &e->d_wide)) return fail(FQ3_E_CUDA, "wide program upload");
  {
    // streams per lock-step group of the wide program: the padded activation rows of the longest K next to a ring that holds
    // one group of that K plus one more stage (at least four stages)
    const int kmax = std::max(e->tk.kmax(), e->pr.kmax());
    const long fixed = kHeaderBytes + kScratchBytes + (long)round_up((size_t)kKindBytes + kUnitBytes + (size_t)e->n_wide_ph * sizeof(Phase), 1024) +
                       (long)kGammaSlots * (long)round_up((size_t)std::max(e->tk.d.hidden, e->pr.d.hidden) * 2, 1024);
    const long spg_max = ((long)kmax * 16 + kStageBytes - 1) / kStageBytes;
    const long avail = (long)e->smem_max - fixed - std::max(4L, spg_max + 1) * kStageBytes - 2048;
    e->wide_rows = (int)std::max<long>(0, std::min<long>(avail / ((long)kmax * 2 + 64), kMaxWide));
  }
  {
    LaunchParams q{};
    q.n_phases = e->n_frames_ph; q.n_rows = 1;
    if (carve(e, q, e->h_frames.data()) < 0) return -FQ3_E_INVALID;
    e->ref_stages = q.n_stages;
  }
  if (upload(e, e->h_frames, &e->d_frames) || upload(e, e->h_pred, &e->d_pred) || upload(e, e->h_talker, &e->d_talker) ||
      upload(e, e->h_prefill, &e->d_prefill))
    return fail(FQ3_E_CUDA, "program upload / weight tiling (matrix rows must be a multiple of 8)");
  if (dalloc(e, &e->d_linear, 1)) return -FQ3_E_CUDA;
  CK(cudaDeviceSynchronize());
  return 0;
}

int fq3_destroy(fq3_engine* e) {
  if (!e) return 0;
  cudaDeviceSynchronize();
  for (void* p : e->owned) if (p) cudaFree(p);
  if (e->err_host) cudaFreeHost(e->err_host);
  delete e;
  return 0;
}

int fq3_num_sms(const fq3_engine* e) { return e ? e->G : 0; }  /* CTAs of the engine's grid */
int64_t fq3_launch_count(const fq3_engine* e) { return e ? e->launches : 0; }

static int check_stream(fq3_engine* e, int idx) {
  if (!e) return fail(FQ3_E_INVALID, "null engine");
  if (idx < 0 || idx >= e->desc.max_streams) return fail(FQ3_E_INVALID, "stream index out of range");
  return 0;
}

// LaunchParams::spol of a launch over streams [s0, s0 + n): the records when one of them has one, else null
static const StreamPolicy* spol_for(const fq3_engine* e, int s0, int n) {
  for (int i = s0; i < s0 + n; ++i)
    if (e->spol_on[i]) return e->d_spol;
  return nullptr;
}

int fq3_reset_stream(fq3_engine* e, int idx, void* stream) {
  if (int r = check_stream(e, idx)) return r;
  fq3_reset_stream_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(e->d_st + idx, e->tk.d.vocab, e->d_spol + idx);
  e->spol_on[idx] = 0;
  e->launches += 1;
  CK(cudaGetLastError());
  return 0;
}

int fq3_retire_stream(fq3_engine* e, int idx, void* stream) {
  if (int r = check_stream(e, idx)) return r;
  fq3_set_state_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(e->d_st + idx, 0, 0, 0, 32, 0, 0, 0);
  e->launches += 1;
  CK(cudaGetLastError());
  return 0;
}

int fq3_set_stream_policy(fq3_engine* e, int idx, const fq3_policy* policy, void* stream) {
  if (int r = check_stream(e, idx)) return r;
  Policy pol{};
  if (policy) {
    if (policy->top_k < 0) return fail(FQ3_E_INVALID, "top_k < 0");
    if (!(policy->top_p > 0.0f && policy->top_p <= 1.0f)) return fail(FQ3_E_INVALID, "top_p outside (0, 1]");
    if (policy->do_sample && !(policy->temperature > 0.0f)) return fail(FQ3_E_INVALID, "temperature <= 0 with do_sample");
    if (!(policy->repetition_penalty > 0.0f)) return fail(FQ3_E_INVALID, "repetition_penalty <= 0");
    if (policy->suppress_tail < 0 || policy->suppress_tail > e->tk.d.vocab) return fail(FQ3_E_INVALID, "suppress_tail outside [0, V]");
    pol = to_policy(policy);
  }
  fq3_set_stream_policy_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(e->d_spol + idx, policy ? 1 : 0, pol);
  e->spol_on[idx] = policy ? 1 : 0;
  e->launches += 1;
  CK(cudaGetLastError());
  return 0;
}

int fq3_set_generation_state(fq3_engine* e, int idx, int n_left_pad, int rope_delta, void* stream) {
  if (int r = check_stream(e, idx)) return r;
  fq3_set_state_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(e->d_st + idx, 0, 0, 0, 2, n_left_pad, rope_delta, 0);
  e->launches += 1;
  CK(cudaGetLastError());
  return 0;
}

int fq3_set_text_conditioning(fq3_engine* e, int idx, const void* trailing, int n_trailing, const void* pad_embed,
                              void* stream) {
  if (int r = check_stream(e, idx)) return r;
  const int Ht = e->tk.d.hidden;
  if (n_trailing < 0 || n_trailing > e->tk.d.max_pos) return fail(FQ3_E_TOO_LONG, "trailing text longer than max_seq_len");
  cudaStream_t s = (cudaStream_t)stream;
  if (n_trailing > 0)
    CK(cudaMemcpyAsync(const_cast<bf16*>(e->h_st[idx].trailing), trailing, (size_t)n_trailing * Ht * 2,
                       cudaMemcpyDeviceToDevice, s));
  CK(cudaMemcpyAsync(const_cast<bf16*>(e->h_st[idx].pad_embed), pad_embed, (size_t)Ht * 2, cudaMemcpyDeviceToDevice, s));
  fq3_set_state_kernel<<<1, 32, 0, s>>>(e->d_st + idx, 0, 0, 0, 4, 0, 0, n_trailing);  // closed text
  e->text_rows[idx] = n_trailing;
  e->text_open[idx] = 0;
  e->launches += 1;
  CK(cudaGetLastError());
  return 0;
}

int fq3_open_text(fq3_engine* e, int idx, const void* pad_embed, void* stream) {
  if (int r = check_stream(e, idx)) return r;
  if (!pad_embed) return fail(FQ3_E_INVALID, "null pad_embed");
  cudaStream_t s = (cudaStream_t)stream;
  CK(cudaMemcpyAsync(const_cast<bf16*>(e->h_st[idx].pad_embed), pad_embed, (size_t)e->tk.d.hidden * 2, cudaMemcpyDeviceToDevice, s));
  fq3_set_state_kernel<<<1, 32, 0, s>>>(e->d_st + idx, 0, 0, 0, 4 | 64, 0, 0, 0);
  e->text_rows[idx] = 0;
  e->text_open[idx] = 1;
  e->launches += 1;
  CK(cudaGetLastError());
  return 0;
}

int fq3_append_text(fq3_engine* e, int idx, const void* rows, int n, int close, void* stream) {
  if (int r = check_stream(e, idx)) return r;
  if (!e->text_open[idx]) return fail(FQ3_E_INVALID, "the stream's text is not open (fq3_open_text)");
  if (n < 0 || (n > 0 && !rows)) return fail(FQ3_E_INVALID, "bad text rows");
  const int total = e->text_rows[idx] + n;
  if (total > e->tk.d.max_pos) return fail(FQ3_E_TOO_LONG, "trailing text longer than max_seq_len");
  cudaStream_t s = (cudaStream_t)stream;
  const int Ht = e->tk.d.hidden;
  if (n > 0)
    CK(cudaMemcpyAsync(const_cast<bf16*>(e->h_st[idx].trailing) + (size_t)e->text_rows[idx] * Ht, rows, (size_t)n * Ht * 2,
                       cudaMemcpyDeviceToDevice, s));
  fq3_set_state_kernel<<<1, 32, 0, s>>>(e->d_st + idx, 0, 0, 0, close ? 4 : 4 | 64, 0, 0, total);
  e->text_rows[idx] = total;
  e->text_open[idx] = close ? 0 : 1;
  e->launches += 1;
  CK(cudaGetLastError());
  return 0;
}

int fq3_import_kv(fq3_engine* e, int idx, int layer, const void* k, const void* v, int T, void* stream) {
  if (int r = check_stream(e, idx)) return r;
  const StackRt& S = e->rt[0];
  if (layer < 0 || layer >= S.n_layers) return fail(FQ3_E_INVALID, "layer out of range");
  if (T > S.max_pos) {
    char b[200];
    snprintf(b, sizeof b, "Input is too long: prefill has %d tokens but max_seq_len=%d. Use shorter text or shorter "
                          "reference audio.", T, S.max_pos);
    return fail(FQ3_E_TOO_LONG, b);
  }
  if (T <= 0) return 0;
  const size_t base = ((size_t)layer * S.n_slots + idx) * S.nkv * (size_t)S.max_pos * kHeadDim;
  fq3_import_kv_kernel<<<64, 256, 0, (cudaStream_t)stream>>>(S.kcache + base, S.vcache + base,
                                                             reinterpret_cast<const bf16*>(k),
                                                             reinterpret_cast<const bf16*>(v), S.nkv, T, S.max_pos);
  e->launches += 1;
  CK(cudaGetLastError());
  return 0;
}

int fq3_set_loop_state(fq3_engine* e, int idx, int token, const void* past_hidden, int position, int gen_step,
                       void* stream) {
  if (int r = check_stream(e, idx)) return r;
  if (token < 0 || token >= e->tk.d.vocab) return fail(FQ3_E_INVALID, "token out of range");
  cudaStream_t s = (cudaStream_t)stream;
  const int Ht = e->tk.d.hidden;
  fq3_set_state_kernel<<<1, 32, 0, s>>>(e->d_st + idx, token, position, gen_step, 1 | 8 | 16, 0, 0, 0);
  e->launches += 1;
  CK(cudaGetLastError());
  bf16* hid = reinterpret_cast<bf16*>(e->bufs[BUF_HID]) + (size_t)idx * e->ld[BUF_HID];
  const bf16* emb = reinterpret_cast<const bf16*>(reinterpret_cast<const uint8_t*>(e->desc.arena) + e->desc.codec_embed_off) +
                    (size_t)token * Ht;
  CK(cudaMemcpyAsync(hid, past_hidden, (size_t)Ht * 2, cudaMemcpyDeviceToDevice, s));
  e->in_wpin[idx] = 0;
  if (int r = pack_ll(e, BUF_PIN, 2 * idx, past_hidden, Ht, 1, Ht, s)) return r;
  if (int r = pack_ll(e, BUF_PIN, 2 * idx + 1, emb, Ht, 1, Ht, s)) return r;
  return 0;
}

// rows of a prompt one launch of the prefill program takes: bounded by the activation staging buffer next to a ring of at
// least six stages
static int prefill_rows(const fq3_engine* e) {
  const long fixed = kHeaderBytes + kScratchBytes + (long)round_up((size_t)kKindBytes + kUnitBytes + (size_t)e->n_prefill_ph * sizeof(Phase), 1024) +
                     (long)kGammaSlots * (long)round_up((size_t)e->tk.d.hidden * 2, 1024);
  const long spg_max = ((long)e->tk.kmax() * 16 + kStageBytes - 1) / kStageBytes;
  const long avail = (long)e->smem_max - fixed - std::max(6L, spg_max + 1) * kStageBytes;
  return (int)std::max<long>(1, std::min<long>(avail / ((long)e->tk.kmax() * 2 + 64), kMaxRows));
}

// rows [start, T) of the prompt go through the persistent kernel; the K/V rows of [0, start) must already be in the cache
static int prefill_impl(fq3_engine* e, int idx, const void* embeds_from_start, int T, int start, int n_left_pad, const fq3_policy* policy,
                        void* out_logits, void* stream) {
  if (int r = check_stream(e, idx)) return r;
  if (!embeds_from_start || !policy || T <= 0 || start < 0 || start >= T) return fail(FQ3_E_INVALID, "bad prefill arguments");
  if (T > e->tk.d.max_pos) {
    char b[200];
    snprintf(b, sizeof b, "Input is too long: prefill has %d tokens but max_seq_len=%d. Use shorter text or shorter "
                          "reference audio.", T, e->tk.d.max_pos);
    return fail(FQ3_E_TOO_LONG, b);
  }
  cudaStream_t s = (cudaStream_t)stream;
  const int Ht = e->tk.d.hidden;
  const int Mmax = prefill_rows(e);
  if (int r = reserve_epochs(e, (uint64_t)((T - start + Mmax - 1) / Mmax) * (uint64_t)(e->n_prefill_ph + 2), s)) return r;
  fq3_reset_stream_kernel<<<1, 256, 0, s>>>(e->d_st + idx, e->tk.d.vocab, nullptr);  // the policy record survives
  fq3_set_state_kernel<<<1, 32, 0, s>>>(e->d_st + idx, 0, 0, 0, 2, n_left_pad, -n_left_pad, 0);
  e->launches += 2;
  for (int c0 = start; c0 < T; c0 += Mmax) {
    const int rows = std::min(Mmax, T - c0);
    const bool final = (c0 + rows == T);
    if (int r = pack_ll(e, BUF_TX, 0, reinterpret_cast<const bf16*>(embeds_from_start) + (size_t)(c0 - start) * Ht, Ht, rows, Ht, s)) return r;
    LaunchParams p{};
    fill_common(e, p);
    p.prog = e->d_prefill;
    p.n_phases = final ? e->n_prefill_ph : e->n_prefill_ph - 2;  // drop head + sample on non-final chunks
    p.mode = MODE_PREFILL;
    p.n_rows = rows;
    p.stream0 = idx;
    p.pf_pos0 = c0; p.pf_n_pad = n_left_pad; p.pf_rope_delta = -n_left_pad; p.pf_final = final;
    p.pol = to_policy(policy);
    p.spol = spol_for(e, idx, 1);
    if (int r = launch(e, p, e->h_prefill.data(), s)) return r;
  }
  fq3_set_state_kernel<<<1, 32, 0, s>>>(e->d_st + idx, 0, T, 0, 8, 0, 0, 0);
  e->in_wpin[idx] = 0;  // SMP_PREFILL published the stream's predictor rows in the pair layout
  e->launches += 1;
  CK(cudaGetLastError());
  if (out_logits)
    if (int r = unpack_f32(e, out_logits, e->tk.d.vocab, BUF_LOGITS, 0, 1, e->tk.d.vocab, s)) return r;
  return 0;
}

int fq3_prefill(fq3_engine* e, int idx, const void* embeds, int T, int n_left_pad, const fq3_policy* policy,
                void* out_logits, void* stream) {
  return prefill_impl(e, idx, embeds, T, 0, n_left_pad, policy, out_logits, stream);
}

int fq3_prefill_tail(fq3_engine* e, int idx, const void* embeds_tail, int T, int n_tail, const fq3_policy* policy, void* out_logits,
                     void* stream) {
  if (n_tail < 1 || n_tail > T) return fail(FQ3_E_INVALID, "bad prefill tail");
  return prefill_impl(e, idx, embeds_tail, T, T - n_tail, 0, policy, out_logits, stream);
}

int fq3_prefill_head(fq3_engine* e, int idx, const void* last_hidden, int T, const fq3_policy* policy, void* out_logits, void* stream) {
  if (int r = check_stream(e, idx)) return r;
  if (!last_hidden || !policy || T <= 0) return fail(FQ3_E_INVALID, "bad prefill_head arguments");
  if (T > e->tk.d.max_pos) {
    char b[200];
    snprintf(b, sizeof b, "Input is too long: prefill has %d tokens but max_seq_len=%d. Use shorter text or shorter "
                          "reference audio.", T, e->tk.d.max_pos);
    return fail(FQ3_E_TOO_LONG, b);
  }
  cudaStream_t s = (cudaStream_t)stream;
  const int Ht = e->tk.d.hidden;
  if (int r = reserve_epochs(e, 4, s)) return r;
  fq3_reset_stream_kernel<<<1, 256, 0, s>>>(e->d_st + idx, e->tk.d.vocab, nullptr);  // the policy record survives
  fq3_set_state_kernel<<<1, 32, 0, s>>>(e->d_st + idx, 0, 0, 0, 2, 0, 0, 0);
  e->launches += 2;
  if (int r = pack_ll(e, BUF_TX, 0, last_hidden, Ht, 1, Ht, s)) return r;
  LaunchParams p{};
  fill_common(e, p);
  // the last two phases of the prefill program: final norm + codec_head on the row, then the first-token sampler
  p.prog = e->d_prefill + (e->n_prefill_ph - 2);
  p.n_phases = 2;
  p.mode = MODE_PREFILL;
  p.n_rows = 1;
  p.stream0 = idx;
  p.pf_pos0 = T - 1; p.pf_n_pad = 0; p.pf_rope_delta = 0; p.pf_final = 1;
  p.pol = to_policy(policy);
  p.spol = spol_for(e, idx, 1);
  if (int r = launch(e, p, e->h_prefill.data() + (e->n_prefill_ph - 2), s)) return r;
  fq3_set_state_kernel<<<1, 32, 0, s>>>(e->d_st + idx, 0, T, 0, 8, 0, 0, 0);
  e->in_wpin[idx] = 0;
  e->launches += 1;
  CK(cudaGetLastError());
  if (out_logits)
    if (int r = unpack_f32(e, out_logits, e->tk.d.vocab, BUF_LOGITS, 0, 1, e->tk.d.vocab, s)) return r;
  return 0;
}

void* fq3_kv_cache_ptr(fq3_engine* e, int idx, int layer, int which) {
  if (!e || idx < 0 || idx >= e->desc.max_streams || layer < 0 || layer >= e->rt[0].n_layers) return nullptr;
  const StackRt& S = e->rt[0];
  const size_t base = ((size_t)layer * S.n_slots + idx) * S.nkv * (size_t)S.max_pos * kHeadDim;
  return (which ? S.vcache : S.kcache) + base;
}

int fq3_talker_step(fq3_engine* e, int idx, const void* embeds, int position, void* out_hidden, void* out_logits,
                    void* stream) {
  if (int r = check_stream(e, idx)) return r;
  if (position < 0 || position >= e->tk.d.max_pos) return fail(FQ3_E_TOO_LONG, "position outside the static KV cache");
  cudaStream_t s = (cudaStream_t)stream;
  const int Ht = e->tk.d.hidden;
  if (int r = reserve_epochs(e, (uint64_t)e->n_talker_ph + 2, s)) return r;
  if (int r = pack_ll(e, BUF_TX, 0, embeds, Ht, 1, Ht, s)) return r;
  LaunchParams p{};
  fill_common(e, p);
  p.prog = e->d_talker;
  p.n_phases = e->n_talker_ph;
  p.mode = MODE_TALKER_STEP;
  p.n_rows = 1;
  p.stream0 = idx;
  p.pos_override = position;
  if (int r = launch(e, p, e->h_talker.data(), s)) return r;
  if (out_hidden) CK(cudaMemcpyAsync(out_hidden, e->bufs[BUF_HID], (size_t)Ht * 2, cudaMemcpyDeviceToDevice, s));
  if (out_logits)
    if (int r = unpack_f32(e, out_logits, e->tk.d.vocab, BUF_LOGITS, 0, 1, e->tk.d.vocab, s)) return r;
  return 0;
}

int fq3_predictor_run(fq3_engine* e, int idx, const void* pred_input, const fq3_subpolicy* sub, uint64_t seed,
                      void* out_codes_i64, void* out_logits, void* stream) {
  if (int r = check_stream(e, idx)) return r;
  if (!pred_input || !sub || !out_codes_i64) return fail(FQ3_E_INVALID, "bad predictor arguments");
  cudaStream_t s = (cudaStream_t)stream;
  const int Ht = e->tk.d.hidden;
  if (int r = reserve_epochs(e, (uint64_t)e->n_pred_ph + 2, s)) return r;
  if (int r = pack_ll(e, BUF_PIN, 0, pred_input, Ht, 2, Ht, s)) return r;
  LaunchParams p{};
  fill_common(e, p);
  p.prog = e->d_pred;
  p.n_phases = e->n_pred_ph;
  p.mode = MODE_PREDICTOR;
  p.n_rows = 1;
  p.stream0 = idx;
  p.sub = to_sub(sub);
  p.pol.seed = seed;
  p.pred_logits_all = out_logits ? e->pred_logits_all : nullptr;
  if (int r = launch(e, p, e->h_pred.data(), s)) return r;
  fq3_codes_to_i64_kernel<<<1, 32, 0, s>>>(reinterpret_cast<const int*>(reinterpret_cast<const uint8_t*>(e->d_st + idx) +
                                                                         offsetof(StreamState, cur_codes)),
                                           e->ncb, reinterpret_cast<long long*>(out_codes_i64));
  e->launches += 1;
  CK(cudaGetLastError());
  if (out_logits)
    CK(cudaMemcpyAsync(out_logits, e->pred_logits_all, (size_t)e->ncb * e->pr.d.vocab * 4, cudaMemcpyDeviceToDevice, s));
  return 0;
}

int fq3_sample(fq3_engine* e, const void* logits_f32, int V, const void* history_i64, int n_history,
               const fq3_policy* policy, int eos_id, int suppress_eos, int flags, uint64_t draw_index,
               void* out_token_i64, void* stream) {
  if (!e || !logits_f32 || !policy || !out_token_i64) return fail(FQ3_E_INVALID, "bad sample arguments");
  if (V <= 0 || V > kMaxVocab) return fail(FQ3_E_UNSUPPORTED, "vocab exceeds sampling scratch");
  SampleArgs a{};
  a.V = V; a.do_sample = policy->do_sample; a.top_k = policy->top_k; a.top_p = policy->top_p;
  a.temperature = policy->temperature; a.rep_pen = policy->repetition_penalty; a.seen = nullptr;
  a.suppress_start = policy->suppress_tail > 0 ? std::max(0, V - policy->suppress_tail) : V;
  a.eos = eos_id; a.suppress_eos = suppress_eos; a.round_bf16 = flags & 1; a.seed = policy->seed; a.draw = draw_index;
  a.next_emb = nullptr; a.emb_row_bytes = 0;
  fq3_sample_kernel<<<1, kConsumerThreads, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const float*>(logits_f32), a, reinterpret_cast<const long long*>(history_i64), n_history,
      e->seen_scratch, reinterpret_cast<long long*>(out_token_i64));
  e->launches += 1;
  CK(cudaGetLastError());
  return 0;
}

int fq3_apply_repetition_penalty(fq3_engine* e, void* logits_f32, int V, const void* history_i64, int n_history,
                                 float penalty, int flags, void* stream) {
  if (!e || !logits_f32) return fail(FQ3_E_INVALID, "bad arguments");
  if (V <= 0 || V > kMaxVocab * 4) return fail(FQ3_E_UNSUPPORTED, "vocab exceeds scratch");
  if (penalty == 1.0f || n_history <= 0 || !history_i64) return 0;  // sampling.py:22-23
  fq3_rep_penalty_kernel<<<1, kConsumerThreads, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<float*>(logits_f32), V, reinterpret_cast<const long long*>(history_i64), n_history, penalty,
      flags & 1, e->seen_scratch);
  e->launches += 1;
  CK(cudaGetLastError());
  return 0;
}

int fq3_decode_frames(fq3_engine* e, int n_streams, int n_frames, const fq3_policy* policy, const fq3_subpolicy* sub,
                      void* stream) {
  if (!e || !policy || !sub) return fail(FQ3_E_INVALID, "bad decode arguments");
  if (n_streams < 1 || n_streams > e->desc.max_streams) return fail(FQ3_E_INVALID, "n_streams out of range");
  if (n_frames <= 0) return 0;
  // The wide program takes over from three streams on where the model has one (measured at 0.6B dims, ms per frame-step,
  // reference-shaped / wide: 2 streams 2.18 / 2.17, 3: 2.39 / 2.25, 4: 2.77 / 2.35; one stream 1.55 / 2.01).  FQ3_WIDE_FROM overrides.
  int wide_from = 3;
  if (const char* wf = getenv("FQ3_WIDE_FROM")) wide_from = std::max(1, atoi(wf));
  if ((n_streams >= wide_from && e->wide_rows > kMaxRows / 2) || 2 * n_streams > kMaxRows) {
    // more than four streams: the wide frame program, in lock-step groups of up to wide_rows streams, one launch per group
    // (a group streams the weights once for all its streams; groups follow each other on the stream)
    // (1.7B dims: a 6144-column row is 12 KB and the ring must hold a six-stage group: three rows fit — not worth it next to the
    // four streams of the reference-shaped program; the host then runs groups of four through that one)
    if (e->wide_rows <= kMaxRows / 2)
      return fail(FQ3_E_UNSUPPORTED, "more than four lock-step streams do not fit this model's staging buffer: decode in groups of fq3_lockstep_group()");
    const int n_groups = (n_streams + e->wide_rows - 1) / e->wide_rows;
    const int per = (n_streams + n_groups - 1) / n_groups;  // even groups
    // all streams first: a group's working rows overwrite pair-layout rows of other groups' streams
    if (int r = sync_pin_layout(e, 0, n_streams, true, (cudaStream_t)stream)) return r;
    for (int s0 = 0; s0 < n_streams; s0 += per) {
      const int n = std::min(per, n_streams - s0);
      if (int r = reserve_epochs(e, (uint64_t)n_frames * (uint64_t)e->n_wide_ph + 2, (cudaStream_t)stream)) return r;
      LaunchParams p{};
      fill_common(e, p);
      p.prog = e->d_wide;
      p.n_phases = e->n_wide_ph;
      p.mode = MODE_FRAMES;
      p.wide = 1;
      p.n_rows = n;
      p.stream0 = s0;
      p.n_iters = n_frames;
      p.pol = to_policy(policy);
      p.spol = spol_for(e, s0, n);
      p.sub = to_sub(sub);
      if (int r = launch(e, p, e->h_wide.data(), (cudaStream_t)stream)) return r;
    }
    return 0;
  }
  if (int r = reserve_epochs(e, (uint64_t)n_frames * (uint64_t)e->n_frames_ph + 2, (cudaStream_t)stream)) return r;
  if (int r = sync_pin_layout(e, 0, n_streams, false, (cudaStream_t)stream)) return r;
  LaunchParams p{};
  fill_common(e, p);
  p.prog = e->d_frames;
  p.n_phases = e->n_frames_ph;
  p.mode = MODE_FRAMES;
  p.n_rows = n_streams;
  p.n_iters = n_frames;
  p.pol = to_policy(policy);
  p.spol = spol_for(e, 0, n_streams);
  p.sub = to_sub(sub);
  return launch(e, p, e->h_frames.data(), (cudaStream_t)stream);
}

// The engine runs every launch on one grid of G <= n_sms CTAs.  When G < n_sms the rest of the device is free for other
// work next to the frame loop (the codec decode of the previous streaming chunk): that is what "reduced grid" reports.
int fq3_set_decode_grid(fq3_engine* e, int n_ctas) {
  if (!e) return fail(FQ3_E_INVALID, "null engine");
  if (n_ctas <= 0 || n_ctas == e->G || n_ctas == e->n_sms) return 0;
  return fail(FQ3_E_UNSUPPORTED, "the decode grid is fixed at engine creation (FQ3_GRID)");
}
int fq3_assemble_prompt(fq3_engine* e, const void* tp_rows, const void* desc_i32x4, int n_rows, const void* spk_rows,
                        const void* ref_codes_i32, void* out_bf16, void* stream) {
  if (!e || !desc_i32x4 || !out_bf16 || n_rows < 0) return fail(FQ3_E_INVALID, "bad assemble_prompt arguments");
  if (n_rows == 0) return 0;
  PromptTables tb{};
  const uint8_t* arena = reinterpret_cast<const uint8_t*>(e->desc.arena);
  tb.codec_embed = reinterpret_cast<const bf16*>(arena + e->desc.codec_embed_off);
  for (int i = 0; i < e->ncb; ++i) tb.pred_embeds[i] = reinterpret_cast<const bf16*>(arena + e->pred_embed_offs[i]);
  tb.ncb = e->ncb;
  fq3_assemble_prompt_kernel<<<n_rows, 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const bf16*>(tp_rows), reinterpret_cast<const int4*>(desc_i32x4), e->tk.d.hidden, tb,
      reinterpret_cast<const bf16*>(spk_rows), reinterpret_cast<const int*>(ref_codes_i32), e->desc.n_code_groups,
      reinterpret_cast<bf16*>(out_bf16));
  e->launches += 1;
  CK(cudaGetLastError());
  return 0;
}

int fq3_lockstep_group(const fq3_engine* e) { return e ? std::max(e->wide_rows, kMaxRows / 2) : 0; }  /* 4 = no wide program */
int fq3_reduced_grid(const fq3_engine* e) { return (e && e->G < e->n_sms) ? e->G : 0; }

int fq3_clear_fault(fq3_engine* e, void* stream) {
  if (!e) return fail(FQ3_E_INVALID, "null engine");
  cudaStreamSynchronize((cudaStream_t)stream);
  if (cudaGetLastError() != cudaSuccess) return fail(FQ3_E_CUDA, "the CUDA context is in an error state: rebuild the engine");
  if (e->err_host) memset(e->err_host, 0, 64);
  // a faulted launch may have left half-written phases behind: forget every epoch
  for (int i = 0; i < kNumBufs; ++i)
    if (e->buf_bytes[i]) CK(cudaMemsetAsync(e->bufs[i], 0, e->buf_bytes[i], (cudaStream_t)stream));
  CK(cudaMemsetAsync(e->attn_part, 0, e->attn_part_bytes, (cudaStream_t)stream));
  e->epoch = 1;
  return 0;
}

int fq3_debug_set_epoch(fq3_engine* e, uint32_t epoch) {
  if (!e || epoch == 0) return fail(FQ3_E_INVALID, "bad arguments");
  e->epoch = epoch;
  return 0;
}

// The frame program ends with the talker's head and sampler: until the next launch, stream b's BUF_LOGITS row holds the
// logits its last talker sampling phase consumed (the predictor's heads write that row earlier in the frame).
int fq3_debug_read_talker_logits(fq3_engine* e, int idx, void* out_f32, void* stream) {
  if (int r = check_stream(e, idx)) return r;
  if (!out_f32) return fail(FQ3_E_INVALID, "null output");
  if (idx >= e->frames_rows)
    return fail(FQ3_E_INVALID, "the last launch was not a reference-shaped fq3_decode_frames launch that ran this stream");
  return unpack_f32(e, out_f32, e->tk.d.vocab, BUF_LOGITS, idx, 1, e->tk.d.vocab, (cudaStream_t)stream);
}

int fq3_get_status(fq3_engine* e, int idx, fq3_status* out, void* stream) {
  if (int r = check_stream(e, idx)) return r;
  cudaError_t se = cudaStreamSynchronize((cudaStream_t)stream);
  if (int r = check_device_fault(e)) return r;
  if (se != cudaSuccess) return fail(FQ3_E_CUDA, std::string("stream sync: ") + cudaGetErrorString(se));
  StreamState s;
  CK(cudaMemcpy(&s, e->d_st + idx, sizeof s, cudaMemcpyDeviceToHost));
  out->n_frames = s.n_frames; out->done = s.done; out->position = s.position; out->gen_step = s.gen_step;
  out->token = s.token; out->error = e->err_host[0];
  return 0;
}

int fq3_read_codes(fq3_engine* e, int idx, int first, int n, int32_t* codes_out, void* stream) {
  if (int r = check_stream(e, idx)) return r;
  if (first < 0 || n < 0 || first + n > e->desc.max_frames) return fail(FQ3_E_INVALID, "frame range");
  if (n == 0) return 0;
  const int g = e->desc.n_code_groups;
  CK(cudaMemcpyAsync(codes_out, e->h_st[idx].codes + (size_t)first * g, (size_t)n * g * 4, cudaMemcpyDeviceToHost,
                     (cudaStream_t)stream));
  CK(cudaStreamSynchronize((cudaStream_t)stream));
  return 0;
}

/* debug: copy the per-phase clock marks of the profiled CTA (FQ3_PROF=<cta>) */
int fq3_debug_read_prof(fq3_engine* e, long long* out, int n_words) {
  if (!e || !e->prof) return fail(FQ3_E_INVALID, "profiling not enabled (FQ3_PROF)");
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(out, e->prof, sizeof(long long) * std::min(n_words, 512 * 160 * 2), cudaMemcpyDeviceToHost));
  CK(cudaMemset(e->prof, 0, sizeof(long long) * 512 * 160 * 2));
  return 0;
}

int fq3_last_hidden(fq3_engine* e, int row, void* out_bf16, void* stream) {
  if (!e || !out_bf16 || row < 0 || row >= e->max_rows) return fail(FQ3_E_INVALID, "bad arguments");
  const int Ht = e->tk.d.hidden;
  CK(cudaMemcpyAsync(out_bf16, reinterpret_cast<const bf16*>(e->bufs[BUF_HID]) + (size_t)row * e->ld[BUF_HID], (size_t)Ht * 2,
                     cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return 0;
}

void* fq3_codes_device_ptr(fq3_engine* e, int idx) {
  if (!e || idx < 0 || idx >= e->desc.max_streams) return nullptr;
  return e->h_st[idx].codes;
}

int fq3_linear(fq3_engine* e, const void* W, const void* x, void* y, int M, int N, int K, int flags, const void* gamma,
               float eps, const void* bias, const void* residual, void* stream) {
  if (!e || !W || !x || !y) return fail(FQ3_E_INVALID, "null argument");
  if (M < 1 || M > kMaxRows) return fail(FQ3_E_UNSUPPORTED, "M must be in [1, 8]");
  if (K % 64 || N < 2 || (N & 1) || K / 2 > e->lin_words || N / 2 > e->lin_words)
    return fail(FQ3_E_UNSUPPORTED, "K must be a multiple of 64 and N even");
  if ((flags & 8) && (N % 4)) return fail(FQ3_E_INVALID, "SwiGLU needs N to be a multiple of 4");
  Plan lin_plan{};
  if (!make_plan(e->G, N, K, (flags & 8) != 0, &lin_plan)) return fail(FQ3_E_UNSUPPORTED, "shape cannot be partitioned");
  cudaStream_t s = (cudaStream_t)stream;
  if (int r = reserve_epochs(e, 3, s)) return r;
  // tiled image of this matrix (the model's own matrices are tiled once at fq3_create)
  const size_t img_bytes = (size_t)((N + 7) / 8 * 8) * K * 2;
  if (img_bytes > e->lin_img_bytes) {
    CK(cudaStreamSynchronize(s));
    if (e->lin_img) {
      cudaFree(e->lin_img);
      for (void*& q : e->owned) if (q == e->lin_img) q = nullptr;
      e->lin_img = nullptr;
    }
    e->lin_img_bytes = 0;
    if (dalloc(e, &e->lin_img, img_bytes, false)) return -FQ3_E_CUDA;
    e->lin_img_bytes = img_bytes;
  }
  fq3_tile_weights_kernel<<<256, 256, 0, s>>>(reinterpret_cast<const bf16*>(W), reinterpret_cast<uint4*>(e->lin_img), N, K);
  e->launches += 1;
  CK(cudaGetLastError());
  Phase ph{};
  ph.type = PH_GEMV;
  ph.flags = F_ABSPTR | ((flags & 1) ? F_PRENORM : 0) | ((flags & 2) ? F_BIAS : 0) | ((flags & 4) ? F_RESID : 0) |
             ((flags & 8) ? F_SWIGLU : 0) | ((flags & 16) ? F_OUT_F32 : 0) | ((flags & 32) ? F_SILU : 0);
  ph.in_buf = BUF_LIN_IN; ph.out_buf = BUF_LIN_OUT; ph.res_buf = BUF_LIN_RES;
  ph.N = (uint32_t)N; ph.K = (uint32_t)K;
  ph.plan = (uint8_t)(kMaxPlans - 1);
  CK(cudaMemcpyAsync(e->d_linear, &ph, sizeof ph, cudaMemcpyHostToDevice, s));
  LaunchParams p{};
  fill_common(e, p);
  p.prog = e->d_linear;
  p.n_phases = 1;
  p.mode = MODE_LINEAR;
  p.n_rows = M;
  const int No = (flags & 8) ? N / 2 : N;
  if (int r = pack_ll(e, BUF_LIN_IN, 0, x, K, M, K, s)) return r;
  if (flags & 4) {
    if (!residual) return fail(FQ3_E_INVALID, "residual flag without a residual pointer");
    if (int r = pack_ll(e, BUF_LIN_RES, 0, residual, No, M, No, s)) return r;
  }
  p.lin_W = e->lin_img; p.lin_gamma = gamma; p.lin_bias = bias; p.lin_eps = eps;
  p.plans[kMaxPlans - 1] = lin_plan;
  if (int r = launch(e, p, &ph, s)) return r;
  if (flags & 16) return unpack_f32(e, y, No, BUF_LIN_OUT, 0, M, No, s);
  return unpack_bf16(e, y, No, BUF_LIN_OUT, 0, M, No, s);
}

}  // extern "C"
