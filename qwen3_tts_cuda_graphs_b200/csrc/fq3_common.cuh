// fq3_common.cuh — shared device/host definitions for the persistent weight-streaming decode kernel.
//
// The kernel is a small "phase machine": a program is a flat list of 32-byte phase descriptors (GEMV /
// attention / sampling).  One CTA per SM runs the whole program.  Every GEMV weight matrix is kept in HBM as a
// *fragment image*: groups of 8 consecutive rows, each group a run of 512-byte blocks (8 rows x 32 columns) laid out
// so that one 16-byte shared-memory load per lane yields the mma.m16n8k16 B fragments of two k-steps.  A producer
// warp streams a CTA's groups through a shared-memory ring of 16 KB stages with cp.async.bulk (TMA bulk copy, SASS
// UBLKCP) — one contiguous copy per stage — and runs ahead of the consumers across phases and frames, so HBM stays
// busy while the CTAs wait for each other.  The activations are the A operand (one stream per A row), so after the
// k loop every lane holds the dot products of one (stream, output word).  See DESIGN.md §3.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace fq3 {

typedef __nv_bfloat16 bf16;

// ---- geometry ---------------------------------------------------------------------------------
constexpr int kConsumerWarps = 12;  // three warpgroups of consumers
constexpr int kConsumerThreads = kConsumerWarps * 32;  // 384
constexpr int kThreads = kConsumerThreads + 128;       // + the producer's warpgroup (warp 12 streams the weights, warps 13-15 only hand their
                                                       // registers over: setmaxnreg moves 72 registers per thread of this warpgroup to the
                                                       // consumers, 128 -> 152 per consumer thread)
constexpr int kProducerRegs = 56;
constexpr int kConsumerRegs = 152;
constexpr int kPollWarps = 8;              // consumer warps 0-7 poll, normalise and stage a single-stream activation row; the
constexpr int kPollThreads = kPollWarps * 32;  // group leaders sit on the other warps where they can (resolve_unit)
constexpr int kMaxStages = 16;             // mbarrier pairs: ring stages in flight per SM
constexpr int kGroupRows = 8;              // weight rows per group = the n dimension of mma.m16n8k16
constexpr int kChunkK = 32;                // columns per fragment block (two k-steps of 16)
constexpr int kBlockBytes = kGroupRows * kChunkK * 2;  // 512: one warp-wide 16-byte load
constexpr int kStageBytes = 16 * 1024;     // ring stage: up to 32 blocks (1024 columns) of ONE group
constexpr int kStageChunks = kStageBytes / kBlockBytes;  // 32
constexpr int kHeadDim = 128;              // talker and predictor heads (asserted on the host)
constexpr int kMaxRows = 8;                // activation rows (tokens) per launch, GEMV register tile
constexpr int kMaxWide = 16;               // streams of one lock-step group of the wide frame program: the 16 A rows of mma.m16n8k16
constexpr int kMaxSplits = 16;             // split-KV partitions per (sequence, kv head)
constexpr int kSplitLen = 4 * kConsumerWarps;              // positions one CTA sweeps per (row, kv head) before the context is split over CTAs
constexpr int kPartStride = 132;           // floats per attention partial: m, l, pad, pad, o[128]
constexpr int kNumBufs = 16;
constexpr int kMaxVocab = 5120;            // sampling scratch holds V fp32 logits in 20 KB
// scratch: GEMV partial sums of the k-parts [12 warps][32 lanes][4] fp32 = 6 KB;
//          attention q rows fp32 [2][128] | fresh K/V rows bf16 [8][2][128] | warp partials [12][2][132] = 17.4 KB;
//          sampling 20 KB logits + histogram + reductions = 21.5 KB
constexpr int kScratchBytes = 24 * 1024;
// smem header: full[16] | empty[16] | ctl: go flag, [8..23] frame positions, [24..39] frame done flags | red[16][8] | gfull[4] | gempty[4] |
// stream consts
constexpr int kEmptyOffset = 128;
constexpr int kCtlOffset = 256;
constexpr int kFramePosIdx = 8;          // ints from the start of ctl
constexpr int kFrameDoneIdx = 8 + kMaxWide;
constexpr int kRedOffset = 512;          // float [kMaxWide][8]: RMSNorm partial sums per (row, eighth of the row)
constexpr int kGFullOffset = 1024;
constexpr int kGEmptyOffset = 1056;
constexpr int kStreamConstOffset = 1088;  // int [16] n_pad | [16] rope_delta of the streams of this launch
constexpr int kHeaderBytes = 2048;
constexpr int kGammaSlots = 4;             // norm-weight vectors in flight (streamed by the producer like the weights)
constexpr int kMaxPlans = 24;

// ---- LL (low-latency) activation words ---------------------------------------------------------
// Every activation that crosses CTAs travels in 8-byte words {payload, epoch}.  payload = two bf16 values
// (elements 2w, 2w+1 of the vector: every exchanged activation is bf16-rounded at that point in the
// reference as well), one fp32 (split-attention partials) or one int (frame control record).  A single
// 8-byte store is atomic, so a reader that sees the expected epoch also sees the payload: consumers poll
// the data itself and no grid-wide barrier, fence or atomic sits between two phases (DESIGN.md §3.3).
typedef uint2 LLWord;

// ---- phase descriptors ------------------------------------------------------------------------
enum PhaseType : uint8_t { PH_END = 0, PH_GEMV = 1, PH_ATTN = 2, PH_SAMPLE = 3 };
enum StackId : uint8_t { ST_TALKER = 0, ST_PRED = 1 };
enum SampleKind : uint8_t { SMP_PRED = 0, SMP_TALKER = 1, SMP_PREFILL = 2, SMP_PRED_ONLY = 3 };

enum PhaseFlags : uint16_t {
  F_PRENORM = 1,        // x <- RMSNorm(x) * gamma before the product
  F_BIAS = 2,           // + bias
  F_RESID = 4,          // out = res + y
  F_SWIGLU = 8,         // rows are (gate_j, up_j) pairs; out[j] = silu(gate) * up
  F_OUT_F32 = 16,       // store bf16-rounded value as fp32 (logits)
  F_ROWS2 = 32,         // predictor pass 0: two rows per stream
  F_LAST_ROW = 64,      // only the last input row is used (prefill head)
  F_WRITE_NORMED = 128, // CTA 0 also stores the normalised input rows (past_hidden)
  F_L2_KEEP = 256,      // weights are re-read soon (predictor): L2 evict_last hint
  F_ABSPTR = 512,       // fq3_linear: absolute pointers taken from LaunchParams
  F_SILU = 1024,        // out = silu(out) after bias (text_projection fc1, model.py:395-403)
  // wide frame program (more than four lock-step streams): predictor pass 0 runs as two single-row passes (0a: past_hidden at
  // position 0, 0b: codec_embed(token) at position 1) whose input rows live in BUF_WPIN, addressed by stream slot
  F_PASS0A = 2048,      // ATTN: position 0
  F_WPIN_B = 4096,      // GEMV: BUF_WPIN rows [max_streams + slot] (0b) instead of [slot] (0a)
  F_IN_PREV = 8192      // GEMV: the input was published by the last phase of the previous iteration (or before the launch)
};

struct __align__(16) Phase {
  uint8_t type;
  uint8_t stack;
  uint8_t layer;
  uint8_t aux;  // predictor pass index / sample kind payload
  uint16_t flags;
  uint8_t in_buf, out_buf;
  uint32_t w_off;  // weight offset in 16-byte units from the arena base (ATTN: unused)
  uint32_t g_off;  // GEMV: gamma;  ATTN: q_norm gamma
  uint32_t b_off;  // GEMV: bias;   ATTN: k_norm gamma
  uint32_t N;
  uint32_t K;
  uint8_t res_buf;
  uint8_t skind; // SAMPLE: SampleKind
  uint8_t plan;  // GEMV: index into LaunchParams::plans
  uint8_t kind;  // GEMV: index into the launch's table of resolved phase kinds (KindDesc)
};
static_assert(sizeof(Phase) == 32, "Phase must stay 32 bytes");

enum BufId : uint8_t {
  BUF_TX = 0, BUF_TQKV, BUF_TATT, BUF_TACT, BUF_PX, BUF_PQKV, BUF_PATT, BUF_PACT, BUF_PIN,
  BUF_LOGITS, BUF_HID, BUF_LIN_IN, BUF_LIN_OUT, BUF_LIN_RES, BUF_WPIN, BUF_COUNT
};

// Host-computed partition of one GEMV shape (N, K, SwiGLU) over the grid, in groups of 8 consecutive weight rows.
// Inside a CTA a group is shared by `wpg` warps, each taking a contiguous part of the K / 32 fragment blocks
// ("k-part"); gpr = 12 / wpg groups are in flight at once and a CTA with more groups goes round again.  A group's
// image (8 * K * 2 bytes, contiguous) travels through spg = ceil(K / 1024) ring stages.
struct Plan {
  int g_base, g_rem;  // 8-row groups per CTA: the first g_rem CTAs take g_base + 1
  int wpg;            // warps per group (k-parts)
  int gpr;            // groups per round
  int spg;            // ring stages per group
  int nch;            // fragment blocks per group = K / 32
  int ro_shift;       // log2 of the weight rows behind one packed output word: 1 (plain) or 2 (SwiGLU: two (gate, up) pairs)
  float inv_k;        // 1 / K
};
// A GEMV phase "kind": everything a consumer needs that does not change from layer to layer (buffers, shape, this CTA's
// share, the warps' units).  The kernel resolves each kind of a launch once, at start, into shared memory; a phase then
// costs a few 16-byte loads instead of a page of address arithmetic on the critical path between two exchanges.
constexpr int kMaxKinds = 32;
struct __align__(16) KindDesc {
  const LLWord* in;            // first input row (F_LAST_ROW applied)
  int Kq, flags;               // 16-byte word pairs per row; Phase::flags
  LLWord* out;
  const LLWord* res;
  const uint32_t* bias;
  int ldout, ldres;
  int g, grp0, wpg, gpr;       // this CTA's 8-row groups, first group; warps per group, groups per round
  int spg, nch, ro_shift, n_stages;  // stages per group, blocks per group, log2 rows per word, stages of the phase on this CTA
  float eps, inv_k;
  int n_rounds, wpgrp;         // rounds; words per group
  int M, n_words, K, fast;     // activation rows, packed output words of the matrix, columns, M == 1 && K <= 3072 (three quads per polling thread)
  int ldin, norm, pad0, pad1;
};
static_assert(sizeof(KindDesc) == 128, "KindDesc is eight 16-byte lines");
struct __align__(16) UnitDesc {  // one consumer warp's unit of a kind
  int wgrp, kp;    // group inside a round, k-part (wgrp >= gpr: the warp has no unit)
  int ch0, ch1;    // blocks [ch0, ch1) of the group
};
constexpr int kKindBytes = kMaxKinds * (int)sizeof(KindDesc);                    // 4 KB
constexpr int kUnitBytes = kMaxKinds * kConsumerWarps * (int)sizeof(UnitDesc);   // 6 KB

// ---- run-time structures ----------------------------------------------------------------------
struct StackRt {
  int hidden, inter, n_layers, nq, nkv, vocab;
  float eps;
  int max_pos;    // KV capacity per slot
  int rope_len;
  int n_slots;
  bf16* kcache;   // [layer][slot][kv_head][max_pos][128]
  bf16* vcache;
  const bf16* rope_cos;  // [rope_len][128]
  const bf16* rope_sin;
};

struct StreamState {  // one per stream, device memory
  int token;
  int position;
  int gen_step;
  int n_frames;
  int done;
  int n_pad;
  int rope_delta;
  int n_trailing;
  int text_open;          // fq3_open_text: rows past n_trailing may still arrive; a frame that needs one waits (done = 4)
  unsigned long long draws;
  const bf16* trailing;   // [n_trailing, H_t]
  const bf16* pad_embed;  // [H_t]
  bf16* held;             // [H_t] past_hidden of a waiting stream (done = 4): its BUF_HID row is overwritten while it idles
  int* codes;             // [max_frames, 16]
  uint8_t* seen;          // [V_t] first-codebook history bitmap (repetition penalty)
  int cur_codes[32];
  LLWord ctl[4];          // per-frame control record published by the talker sampler: done, position, gen_step, n_frames
};

struct Policy {
  int do_sample, top_k;
  float top_p, temperature, rep_pen;
  int min_new_tokens, suppress_tail;
  unsigned long long seed;
};
struct SubPolicy {
  int do_sample, top_k;
  float top_p, temperature;
};
// A stream's own sampling policy (fq3_set_stream_policy), one per stream in device memory.  on != 0: the stream's talker /
// prefill sampler takes pol instead of LaunchParams::pol and its predictor sampler takes pol.seed; the Philox key is then
// pol.seed ^ K * 1 whatever the slot, so the draws depend on the stream's seed and draw counter alone.
struct StreamPolicy {
  int on;
  Policy pol;
};

enum Mode : int { MODE_FRAMES = 0, MODE_TALKER_STEP = 1, MODE_PREDICTOR = 2, MODE_PREFILL = 3, MODE_LINEAR = 4 };

struct LaunchParams {
  const Phase* prog;
  int n_phases;
  int n_kinds;                       // GEMV phase kinds of this launch
  uint16_t kind_phase[kMaxKinds];    // a phase index of every kind (its representative)
  int n_iters;
  int mode;
  int n_rows;    // base row count M (streams for decode, chunk rows for prefill, M for linear)
  int wide;      // wide frame program: up to kMaxWide streams, pass 0 split, BUF_WPIN
  int max_streams;
  int stream0;   // first stream index (single-stream entry points)
  int pos_override;  // >=0: talker position for MODE_TALKER_STEP
  int pf_pos0, pf_n_pad, pf_rope_delta, pf_final;
  const uint8_t* arena;
  const uint8_t* tiled;  // fragment images of the GEMV matrices (Phase::w_off indexes this buffer)
  void* bufs[kNumBufs];
  int ld[kNumBufs];
  StackRt stacks[2];
  StreamState* st;
  Policy pol;
  SubPolicy sub;
  const StreamPolicy* spol;  // [max_streams] per-stream policies; null when no stream of the launch has one, or the launch takes its policy explicitly
  LLWord* attn_part;  // split-attention partials as fp32 LL words [row][q head][split][kPartStride]
  int* err;  // mapped host memory: [0]=code [1]=cta [2]=phase [3]=detail
  // model constants used by the sampling phases
  int n_code_groups, eos_id, has_s2m, max_frames;
  const bf16* codec_embed;            // [V_t, H_t]
  const bf16* pred_embeds[32];        // [V_p, H_t] each
  float* pred_logits_all;             // optional [15, V_p] dump (MODE_PREDICTOR)
  // fq3_linear
  const void* lin_W;  // tiled image of the matrix
  const void* lin_gamma;
  const void* lin_bias;
  float lin_eps;
  // smem carve-up
  int n_stages, xbuf_bytes, prog_bytes, gam_bytes;  // ring stages of 16 KB; bytes of the activation staging buffer / of the kind tables + program copy / of ONE norm-weight slot (1 KB multiples)
  Plan plans[kMaxPlans];
  unsigned epoch_base;  // LL epoch of the phase before this launch's first phase
  unsigned long long watchdog_ns;
  long long* prof;  // optional per-phase clock64 marks [n_phases][8] of CTA prof_cta (FQ3_PROF)
  int prof_cta;
  int debug;  // timing ablations (FQ3_DEBUG): 1 no LL wait, 2 no GEMV math, 4 no attention
};

enum DevErr : int { DE_NONE = 0, DE_LL_WAIT = 1, DE_FULL_WAIT = 2, DE_EMPTY_WAIT = 3, DE_HANDSHAKE = 4, DE_BAD_PHASE = 5, DE_CTL_WAIT = 6, DE_ASSERT = 7 };

}  // namespace fq3
