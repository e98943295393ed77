// fq3_kernel.cuh — the persistent weight-streaming decode kernel (sm_100a), v9.
//
// Replaces the CUDA-graph replays of talker_graph.py:97-107,198-214 and predictor_graph.py:115-167 and
// the eager per-frame glue of generate.py:149-199 (reference paths under /root/reference/faster_qwen3_tts).
//
// Structure of one CTA (one per SM, all co-resident):
//   warp 12      producer: walks the phase program and streams this CTA's row groups of every GEMV phase's weight
//                image through a shared-memory ring of 16 KB stages with cp.async.bulk (TMA bulk copy), one
//                contiguous copy per stage.  Weight addresses never depend on activations or sampled ids, so it
//                runs ahead of the consumers across phases and frames.
//   warps 0..11  consumers: per phase, poll-read the input activations (LL words), normalise and stage them; then a
//                warp multiplies one group of 8 weight rows over its part of K with mma.sync.m16n8k16 (weights = B
//                operand as they arrived, activations = A operand, one stream per row), the parts of a group meet in
//                shared memory and the group's first warp applies the epilogue and publishes.
// There is no grid barrier: phases are chained by the data itself (payload + epoch in one 8-byte word).
#pragma once
#include "fq3_common.cuh"

namespace fq3 {

// =================================================================================================
// PTX helpers
// =================================================================================================
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }

// TMA bulk copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP).
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint64_t* bar, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(dst),
      "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s_a(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(dst),
      "l"(src), "r"(bytes), "r"(bar), "l"(policy)
      : "memory");
}
__device__ __forceinline__ uint64_t policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
// a fixed 40 % of the lines stay (evict_last), the rest is streamed: weights that are re-read every pass but exceed L2
__device__ __forceinline__ uint64_t policy_keep_fraction() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.L2::evict_first.b64 %0, 0.4;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}

__device__ __forceinline__ void cbar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(kConsumerThreads) : "memory"); }

__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ int ld_volatile_shared_i32(const int* p) {
  int v;
  asm volatile("ld.volatile.shared.s32 %0, [%1];" : "=r"(v) : "r"(smem_u32(p)) : "memory");
  return v;
}
__device__ __forceinline__ void st_volatile_shared_i32(int* p, int v) {
  asm volatile("st.volatile.shared.s32 [%0], %1;" ::"r"(smem_u32(p)), "r"(v) : "memory");
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}

// LL words: relaxed gpu-scope 8-byte accesses served by L2 (the coherence point).
__device__ __forceinline__ LLWord ll_ld(const LLWord* p) {
  LLWord w;
  asm volatile("ld.relaxed.gpu.global.v2.u32 {%0, %1}, [%2];" : "=r"(w.x), "=r"(w.y) : "l"(p) : "memory");
  return w;
}
// two adjacent words with one 16-byte request (each word is validated by its own epoch, so tearing is harmless)
__device__ __forceinline__ void ll_ld2(const LLWord* p, LLWord& a, LLWord& b) {
  asm volatile("ld.relaxed.gpu.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(a.x), "=r"(a.y), "=r"(b.x), "=r"(b.y) : "l"(p) : "memory");
}
// Publishing store.  A plain st.relaxed.gpu may linger in the SM's write path for about a microsecond before L2 (and the
// pollers) see it; a reduction is sent to L2 at once and needs no reply.  Epochs only grow, so with the epoch in the high
// half max.u64 installs exactly {payload, epoch} (measured: 17 % off the step time against st.relaxed.gpu).
__device__ __forceinline__ void ll_st(LLWord* p, uint32_t payload, uint32_t ep) {
  const unsigned long long val = ((unsigned long long)ep << 32) | payload;
  asm volatile("red.relaxed.gpu.global.max.u64 [%0], %1;" ::"l"(p), "l"(val) : "memory");
}
__device__ __forceinline__ void ll_st2(LLWord* p, uint32_t pay0, uint32_t pay1, uint32_t ep) {
  ll_st(p, pay0, ep);
  ll_st(p + 1, pay1, ep);
}
__device__ __forceinline__ void ll_stf(LLWord* p, float v, uint32_t ep) { ll_st(p, __float_as_uint(v), ep); }

__device__ __forceinline__ float bf16r(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }
__device__ __forceinline__ float bf_lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf_hi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// =================================================================================================
// Shared-memory layout
// =================================================================================================
struct Smem {
  uint64_t* full;    // [kMaxStages]
  uint64_t* empty;   // [kMaxStages]
  int* ctl;          // [0] producer go flag, [kFramePosIdx ..] frame positions, [kFrameDoneIdx ..] frame done flags
  float* red;        // [kMaxWide][8] RMSNorm partial sums
  unsigned char* scratch;
  KindDesc* kinds;   // [kMaxKinds] resolved GEMV phase kinds
  UnitDesc* units;   // [kMaxKinds][kConsumerWarps]
  Phase* prog;       // copy of the phase program (a global read per phase would sit on the critical path)
  unsigned char* gam;  // [kGammaSlots][gam_bytes] norm weights, streamed by the producer
  unsigned char* xbuf;  // activation rows of the current GEMV phase, in A-fragment order
  unsigned char* ring;
};

__device__ __forceinline__ Smem carve_smem(unsigned char* base, const LaunchParams& p) {
  Smem s;
  s.full = reinterpret_cast<uint64_t*>(base);
  s.empty = reinterpret_cast<uint64_t*>(base + kEmptyOffset);
  s.ctl = reinterpret_cast<int*>(base + kCtlOffset);
  s.red = reinterpret_cast<float*>(base + kRedOffset);
  s.scratch = base + kHeaderBytes;
  s.kinds = reinterpret_cast<KindDesc*>(s.scratch + kScratchBytes);
  s.units = reinterpret_cast<UnitDesc*>(s.scratch + kScratchBytes + kKindBytes);
  s.prog = reinterpret_cast<Phase*>(s.scratch + kScratchBytes + kKindBytes + kUnitBytes);
  s.gam = s.scratch + kScratchBytes + p.prog_bytes;
  s.xbuf = s.gam + kGammaSlots * p.gam_bytes;
  s.ring = s.xbuf + p.xbuf_bytes;  // header, scratch, program, norm-weight slots and xbuf are 1 KB multiples
  return s;
}

// =================================================================================================
// Watchdog: a protocol bug must surface as an error, never as a hung GPU.
// =================================================================================================
__device__ __noinline__ void device_fault(const LaunchParams& p, int code, int phase, int detail) {
  volatile int* e = p.err;
  if (e[0] == 0) {
    e[1] = blockIdx.x;
    e[2] = phase;
    e[3] = detail;
    e[0] = code;
  }
  __threadfence_system();
  asm volatile("trap;");
}

struct Spin {
  unsigned long long t0;
  unsigned n;
  __device__ __forceinline__ Spin() : t0(0), n(0) {}
  __device__ __forceinline__ void tick(const LaunchParams& p, int code, int phase, int detail) {
    if ((++n & 0x3ff) == 0) {
      unsigned long long t = globaltimer_ns();
      if (t0 == 0) t0 = t;
      else if (t - t0 > p.watchdog_ns) device_fault(p, code, phase, detail);
    }
  }
};

__device__ __noinline__ void mbar_wait_slow(uint64_t* bar, uint32_t parity, const LaunchParams& p, int code, int phase) {
  Spin s;
  while (!mbar_try_wait(bar, parity)) s.tick(p, code, phase, (int)parity);
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, const LaunchParams& p, int code, int phase) {
  if (mbar_try_wait(bar, parity)) return;
  mbar_wait_slow(bar, parity, p, code, phase);
}

// Slow path of an LL read: poll until the word carries `ep`.  The first retries are immediate (the common case is
// a word that lands within one more L2 round trip); after that back off a little.
__device__ __noinline__ LLWord ll_spin(const LLWord* ptr, uint32_t ep, const LaunchParams& p, int phase) {
  Spin s;
  LLWord w;
  unsigned tries = 0;
  do {
    if (++tries > 4) __nanosleep(40);
    s.tick(p, DE_LL_WAIT, phase, (int)ep);
    w = ll_ld(ptr);
  } while (w.y != ep);
  return w;
}
// Validate a word that was loaded earlier (loads are issued in batches so their L2 round trips overlap);
// ep == 0 accepts whatever is there — inputs written before the launch.  Returns the 32-bit payload.
__device__ __forceinline__ uint32_t ll_check(LLWord w, const LLWord* ptr, uint32_t ep, const LaunchParams& p, int phase) {
  if (ep != 0 && w.y != ep) w = ll_spin(ptr, ep, p, phase);
  return w.x;
}
__device__ __forceinline__ uint32_t ll_wait(const LLWord* ptr, uint32_t ep, const LaunchParams& p, int phase) {
  return ll_check(ll_ld(ptr), ptr, ep, p, phase);
}

// Device-side bounds checks (compute-sanitizer is not available on the GPU pool): a violated invariant surfaces as
// FQ3_E_DEVICE_FAULT with code DE_ASSERT, the phase index and a site-specific detail.
#ifndef FQ3_CHECKS
#define FQ3_CHECKS 0
#endif
#if FQ3_CHECKS
#define FQ3_ASSERT(cond, pidx, detail) do { if (!(cond)) device_fault(p, DE_ASSERT, (pidx), (detail)); } while (0)
#else
#define FQ3_ASSERT(cond, pidx, detail) do { } while (0)
#endif

// FQ3_PROF=-2: every CTA records the global-timer time of its phase start (k = 0) and of its first output store (k = 1)
__device__ __forceinline__ void prof_cta_time(const LaunchParams& p, int pidx, int k) {
  if (p.prof && p.prof_cta == -2 && threadIdx.x == 0 && pidx >= 0 && pidx < 512)
    p.prof[((size_t)pidx * 160 + blockIdx.x) * 2 + k] = (long long)globaltimer_ns();
}
// FQ3_PROF=-3: every warp of CTA 0 records clock64 at two points of a phase (k = 0, 1)
__device__ __forceinline__ void prof_warp_time(const LaunchParams& p, int pidx, int k) {
  if (p.prof && p.prof_cta == -3 && blockIdx.x == 0 && (threadIdx.x & 31) == 0 && pidx >= 0 && pidx < 512)
    p.prof[((size_t)pidx * 160 + 16 * (k >> 1) + (threadIdx.x >> 5)) * 2 + (k & 1)] = clock64();
}
__device__ __forceinline__ void prof_mark(const LaunchParams& p, int pidx, int slot, int thread = 0) {
  if (p.prof && (int)threadIdx.x == thread && (int)blockIdx.x == p.prof_cta && pidx >= 0 && pidx < 512) p.prof[(size_t)pidx * 16 + slot] = clock64();
}
// FQ3_PROF=<cta> with the wide program: thread 0 of that CTA adds cycles per category (scripts/wide_prof.py)
#ifndef FQ3_WIDE_PROF
#define FQ3_WIDE_PROF 0  // build with -DFQ3_WIDE_PROF=1 for scripts/wide_prof.py (the marks cost ~700 cycles each and a few per cent when idle)
#endif
__device__ __forceinline__ void prof_acc(const LaunchParams& p, int cat, long long& t, int thread = 0) {
  if (FQ3_WIDE_PROF && p.prof && (int)threadIdx.x == thread && (int)blockIdx.x == p.prof_cta) {
    const long long now = clock64();
    p.prof[cat] += now - t;
    t = now;
  }
}
constexpr int kProfLeader = (kConsumerWarps - 1) * 32;  // lane 0 of warp 11: the leader of group 0 (resolve_unit)

// SiLU in fp32; the result is rounded to bf16 right away, so the fast exp / divide (a few ulp of fp32) do not show
__device__ __forceinline__ float silu_f(float x) { return __fdividef(x, 1.f + __expf(-x)); }

__device__ __forceinline__ int phase_rows(const Phase& ph, const LaunchParams& p) {
  return (ph.flags & F_ROWS2) ? 2 * p.n_rows : p.n_rows;
}

__device__ __forceinline__ uint2 ldg_keep_u2(const void* ptr, uint64_t pol) {
  uint2 v;
  asm volatile("ld.global.nc.L2::cache_hint.v2.u32 {%0, %1}, [%2], %3;" : "=r"(v.x), "=r"(v.y) : "l"(ptr), "l"(pol));
  return v;
}

__device__ __forceinline__ Phase load_phase(const Phase* prog_smem, int i) {
  // uniform shared-memory address: two broadcast 16-byte reads
  union { Phase ph; uint4 q[2]; } u;
  const uint32_t a = smem_u32(prog_smem + i);
  u.q[0] = lds128(a);
  u.q[1] = lds128(a + 16u);
  return u.ph;
}

// =================================================================================================
// GEMV phase
//
// A lone warp issues a dependent instruction only every ~5 cycles, so what bounds a phase is the number of instructions
// between "the input words are visible" and "the output words are stored".  The multiply is arranged so that nothing
// has to be re-shuffled afterwards: a warp takes one group of 8 weight rows and a contiguous part of K; the weights are
// the B operand of mma.m16n8k16 (n = row inside the group) exactly as they arrive from HBM — the image is stored in
// fragment order, one 16-byte load per lane feeds two k-steps — and the activations are the A operand, one stream per A
// row.  After the k loop lane (g, t) holds the dot products of stream g with rows 2t and 2t+1 of the group: one packed
// output word.  Where a group is shared by several warps (k-parts) the partial words go through shared memory once and
// the first warp of the group adds them in part order.  Everything that does not depend on the input (partition,
// addresses, gamma / residual / bias fetches, the wait for the weight stage) happens between issuing the first poll loads
// and looking at their result — that window (an L2 round trip) is otherwise idle.
//
// (A tcgen05 version of this phase — weights as a pre-swizzled A operand, K-splits on the M dimension, accumulator in
// tensor memory — was built and measured first: an SS-mode tcgen05.mma streams its A rows from shared memory at one row
// per cycle, 128 cycles per k-step whatever N is, which is slower than shared-memory loads + mma.sync for a GEMV:
// profiles/r02a_tcgen05_gemv_phase_profile_rejected.log.)
// =================================================================================================
struct Ctx {  // per-thread constants (shared-memory addresses as 32-bit shared-window offsets)
  uint32_t full, empty, red, scratch, xs, ring, gfull, gempty, gam;
  int n_stages, gam_bytes;
  uint32_t kinds, units, xhalf;
  const Phase* prog;
};
__device__ __forceinline__ Ctx make_ctx(unsigned char* smem_base, const LaunchParams& p) {
  const Smem sm = carve_smem(smem_base, p);
  Ctx c;
  c.full = smem_u32(sm.full);
  c.empty = smem_u32(sm.empty);
  c.red = smem_u32(sm.red);
  c.scratch = smem_u32(sm.scratch);
  c.xs = smem_u32(sm.xbuf);
  c.ring = smem_u32(sm.ring);
  c.n_stages = p.n_stages;
  c.gfull = smem_u32(smem_base + kGFullOffset);
  c.gempty = smem_u32(smem_base + kGEmptyOffset);
  c.gam = smem_u32(sm.gam);
  c.gam_bytes = p.gam_bytes;
  c.xhalf = (uint32_t)p.xbuf_bytes / 2u;
  c.kinds = smem_u32(sm.kinds);
  c.units = smem_u32(sm.units);
  c.prog = sm.prog;
  return c;
}
__device__ __forceinline__ bool mbar_try_wait_a(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_arrive_a(uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }
__device__ __forceinline__ float lds_f32(uint32_t a) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ float2 lds_f32x2(uint32_t a) {
  float2 v;
  asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(a));
  return v;
}
__device__ __forceinline__ float4 lds_f32x4(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts_f32(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
__device__ __forceinline__ void sts_f32x2(uint32_t a, float v0, float v1) { asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(a), "f"(v0), "f"(v1) : "memory"); }
__device__ __forceinline__ void sts_u32(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ uint2 lds_u32x2(uint32_t a) {
  uint2 v;
  asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
  return v;
}
// named barrier of the warps that share a weight group (ids 2 .. 13; 0 = __syncthreads, 1 = all consumers)
__device__ __forceinline__ void group_bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

// D(16x8, fp32) += A(16x16, bf16, row) * B(16x8, bf16, col)
__device__ __forceinline__ void mma_bf16(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// Ring cursor: slot and lap parity of the next stage of this CTA (same sequence on the producer and on every consumer).
struct RingCur {
  int slot;
  uint32_t lap;
  __device__ __forceinline__ void advance(int n, int n_stages) {
    slot += n;
    while (slot >= n_stages) { slot -= n_stages; lap ^= 1u; }
  }
};

// exact a / b for 0 <= a < 2^20, 1 <= b < 2^12 (the +0.5 keeps the float quotient away from integer boundaries)
__device__ __forceinline__ int small_div(int a, int b) { return (int)__fdividef((float)a + 0.5f, (float)b); }

// This CTA's share of a GEMV phase (producer and consumers must agree).
struct Slab {
  int g, grp0;  // 8-row groups of this CTA and the index of its first group
  int n_stages; // ring stages the phase takes on this CTA = g * spg
};
__device__ __forceinline__ Slab get_slab(const Phase& ph, const LaunchParams& p) {
  const Plan& pl = p.plans[ph.plan];
  const int cta = blockIdx.x;
  Slab s;
  s.g = pl.g_base + (cta < pl.g_rem ? 1 : 0);
  s.grp0 = cta * pl.g_base + min(cta, pl.g_rem);
  s.n_stages = s.g * pl.spg;
  return s;
}

// Kernel start: resolve the GEMV phase kinds of this launch (thread k < n_kinds) and the warps' units (fq3_common.cuh: KindDesc).
__device__ __forceinline__ void resolve_kind(const LaunchParams& p, const Phase& ph, KindDesc& kd) {
  const Plan& pl = p.plans[ph.plan];
  const Slab sb = get_slab(ph, p);
  const uint32_t flags = ph.flags;
  int M = (flags & F_ROWS2) ? 2 * p.n_rows : p.n_rows, row_off = 0;
  if (flags & F_LAST_ROW) { row_off = M - 1; M = 1; }
  const int K = (int)ph.K;
  // rows of BUF_WPIN are addressed by stream slot (they cross launches): [slot] = past_hidden, [max_streams + slot] = codec_embed(token)
  const int wpin_row = p.stream0 + ((flags & F_WPIN_B) ? p.max_streams : 0);
  if (ph.in_buf == BUF_WPIN) row_off += wpin_row;
  kd.ldin = p.ld[ph.in_buf];
  kd.in = reinterpret_cast<const LLWord*>(p.bufs[ph.in_buf]) + (size_t)row_off * kd.ldin;
  kd.Kq = K >> 2;
  kd.flags = (int)flags;
  kd.out = reinterpret_cast<LLWord*>(p.bufs[ph.out_buf]);
  kd.ldout = p.ld[ph.out_buf];
  kd.ldres = (flags & F_RESID) ? p.ld[ph.res_buf] : 0;
  kd.res = (flags & F_RESID) ? reinterpret_cast<const LLWord*>(p.bufs[ph.res_buf]) + (size_t)(ph.res_buf == BUF_WPIN ? wpin_row : 0) * kd.ldres : nullptr;
  kd.bias = nullptr;
  if (flags & F_BIAS)
    kd.bias = reinterpret_cast<const uint32_t*>((flags & F_ABSPTR) ? p.lin_bias : static_cast<const void*>(p.arena + (size_t)ph.b_off * 16));
  kd.g = sb.g; kd.grp0 = sb.grp0; kd.wpg = pl.wpg; kd.gpr = pl.gpr;
  kd.spg = pl.spg; kd.nch = pl.nch; kd.ro_shift = pl.ro_shift; kd.n_stages = sb.n_stages;
  kd.eps = (flags & F_ABSPTR) ? p.lin_eps : p.stacks[ph.stack].eps;
  kd.inv_k = pl.inv_k;
  kd.n_rounds = sb.g ? (sb.g + pl.gpr - 1) / pl.gpr : 0;
  kd.wpgrp = 8 >> pl.ro_shift;
  kd.M = M; kd.n_words = (int)ph.N >> pl.ro_shift; kd.K = K;
  kd.fast = (M == 1) && (kd.Kq <= 3 * kPollThreads);
  kd.norm = (flags & F_PRENORM) ? 1 : 0;
  kd.pad0 = 0; kd.pad1 = 0;
}
// Which unit a warp takes.  The first warp of a group ("leader", k-part 0) adds the parts, applies the epilogue and publishes:
// it is the last warp of its CTA to leave a phase.  Leaders therefore sit on the highest warps — warps 8-11 do not poll the
// next phase's input (kPollWarps), so a leader's way from its store to the next phase overlaps the pollers' wait, norm and
// staging instead of delaying them.  The other k-parts fill the warps from 0 up.
__device__ __forceinline__ void resolve_unit(const KindDesc& kd, int warp, UnitDesc& u) {
  const int wpg = kd.wpg, gpr = kd.gpr;
  if (warp >= kConsumerWarps - gpr) {
    u.wgrp = kConsumerWarps - 1 - warp;
    u.kp = 0;
  } else if (wpg > 1 && warp < gpr * (wpg - 1)) {
    u.wgrp = warp / (wpg - 1);
    u.kp = 1 + warp - u.wgrp * (wpg - 1);
  } else {
    u.wgrp = gpr;  // no unit
    u.kp = 0;
  }
  u.ch0 = (u.kp * kd.nch) / wpg;
  u.ch1 = ((u.kp + 1) * kd.nch) / wpg;
}
__device__ __forceinline__ void poll_bar_sync() { asm volatile("bar.sync 14, %0;" ::"n"(kPollThreads) : "memory"); }

// Values computed before the poll must not be sunk behind it by the compiler: an empty asm pins them in a register.
__device__ __forceinline__ void pin(uint32_t& v) { asm volatile("" : "+r"(v)); }
__device__ __forceinline__ void pin(int& v) { asm volatile("" : "+r"(v)); }
__device__ __forceinline__ void pin(float& v) { asm volatile("" : "+f"(v)); }
template <class T>
__device__ __forceinline__ void pin(T*& v) { asm volatile("" : "+l"(v)); }

// Two neighbouring LL words in one 16-byte request.  ld.relaxed.gpu was the fastest of the flavours tried (volatile, .cv, .cg,
// relaxed.sys, acquire.gpu: profiles/r01b_ll_store_flavours.log).
__device__ __forceinline__ uint4 ll_ld_pair(const LLWord* p) {
  uint4 v;
  asm volatile("ld.relaxed.gpu.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
  return v;
}
// bf16(bf16(x * rs) * g) for two packed elements: fp32 product + one packed round, then a packed bf16 multiply (the bf16 x bf16
// product is exact in fp32, so rounding it once to bf16 is what the fp32 route does as well)
__device__ __forceinline__ uint32_t norm_pair(uint32_t x, float rs, uint32_t g) {
  const __nv_bfloat162 xr = __floats2bfloat162_rn(bf_lo(x) * rs, bf_hi(x) * rs);
  const __nv_bfloat162 y = __hmul2(xr, *reinterpret_cast<const __nv_bfloat162*>(&g));
  return *reinterpret_cast<const uint32_t*>(&y);
}

// Shared-memory copy of an activation row, in the order the A fragments want it: a 32-column block is 64 bytes, lane t's
// 16 bytes hold columns {2t, 2t+1 | 8+2t, 9+2t | 16+2t, 17+2t | 24+2t, 25+2t} (= a0, a2 of k-step 0, a0, a2 of k-step 1).
// A quad q (columns 4q .. 4q+3, the two LL words a thread polls with one request) lands in two 4-byte slots 16 bytes apart.
// (Every shared-memory load instruction costs a pass per quarter-warp whether its lanes are predicated off or read the same
// address, so one 16-byte load per block is the cheapest way to fetch a stream's fragments; storing the row in both k-step
// orders to save the register moves below was measured and is slower: profiles/r02b_gemv_variants.log.)
constexpr uint32_t kXBlock = 64;
__device__ __forceinline__ uint32_t xrow_bytes(int K) { return (uint32_t)K * 2u; }
__device__ __forceinline__ uint32_t xquad_off(int q) {
  const int qq = q & 7;  // quad inside the block
  return (uint32_t)(q >> 3) * kXBlock + (uint32_t)(qq & 1) * 32u + (uint32_t)((qq >> 2) * 2 + ((qq >> 1) & 1)) * 4u;
}
__device__ __forceinline__ void xquad_store(uint32_t addr, uint32_t lo, uint32_t hi) {
  sts_u32(addr, lo);
  sts_u32(addr + 16u, hi);
}

// Shared-memory stride of the activation rows of a multi-row phase: 64 bytes of padding put rows g and g + 1 in different
// banks, so the 16-byte A-fragment loads of a quarter-warp (two rows x four lanes) do not collide.
__device__ __forceinline__ uint32_t xrow_stride(int K) { return (uint32_t)K * 2u + 64u; }

// Multi-row activation load (several rows, or rows too long for the register path): raw payloads go through shared memory,
// each thread re-reads exactly what it wrote.  HF rounding points (Qwen3RMSNorm): fp32 mean-square, x*rsqrt -> bf16,
// * weight -> bf16.  The sum of squares of a row is built exactly as the single-stream register path builds it — eight
// "virtual warps" per row, lane l of virtual warp v owns quads 32v + l + 256j and adds them in j order, a shuffle tree per
// virtual warp, the eight sums in a fixed tree — so a stream's arithmetic does not depend on how many streams (or prompt rows)
// share the launch.  A unit = (row, virtual warp); a warp keeps UNITS units (up to UNITS * kMaxJ 16-byte requests per lane) in flight.
constexpr int kMaxJ = 6;  // quads per lane of a unit: K <= 6144
template <int UNITS, int JC, bool ENTRY_BARRIER = false>
__device__ __forceinline__ void load_x_rows_impl(const LaunchParams& p, uint32_t flags, const LLWord* in, int ld, uint32_t gam, float eps,
                                         int K, int M, uint32_t ep_in, int pidx, uint32_t xs, uint32_t red, long long* tprof = nullptr) {
  const int Kq = K >> 2;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool norm = (flags & F_PRENORM) != 0;
  const int n_units = M * 8;
  const uint32_t rstride = xrow_stride(K);
  const float inv_k = __frcp_rn((float)K);  // = the host's 1.0f / K (Plan::inv_k)
  // (every CTA reads the same rows in the same order.  Starting each CTA at a different unit — so that they do not all ask L2 for
  // the same lines at once — was measured and is 9 % slower at 16 streams, and so are twelve requests per lane instead of six:
  // L2 serves the common lines well, the staging is bound by the bytes, M * K * 8 per CTA and phase.)
  auto unit_of = [&](int u) { return u; };
  FQ3_ASSERT(Kq <= 256 * kMaxJ && M <= kMaxWide, pidx, 310000 + M);
  if (ENTRY_BARRIER && warp >= n_units) cbar_sync();  // a warp without a unit still meets the others (below: behind the first requests)
#pragma unroll 1
  for (int u0 = warp; u0 < n_units; u0 += UNITS * kConsumerWarps) {
    float ss[UNITS];
#pragma unroll
    for (int h = 0; h < UNITS; ++h) ss[h] = 0.f;
#pragma unroll 1
    for (int j0 = 0; j0 * 256 < Kq; j0 += JC) {  // JC quads per lane and unit at a time
      uint4 w[UNITS][JC];
#pragma unroll
      for (int h = 0; h < UNITS; ++h) {
        const bool uok = u0 + h * kConsumerWarps < n_units;
        const int u = unit_of(u0 + h * kConsumerWarps);
        const LLWord* src = in + (size_t)(u >> 3) * ld;
        const int qb = (u & 7) * 32 + lane + 256 * j0;
#pragma unroll
        for (int j = 0; j < JC; ++j) {
          w[h][j] = make_uint4(0u, ep_in, 0u, ep_in);  // absent quads: payload 0, never waited for
          if (uok && qb + 256 * j < Kq) w[h][j] = ll_ld_pair(src + 2 * (qb + 256 * j));
        }
      }
      // the block barrier that lets go of the previous phase's rows and partial words waits in the shadow of the first requests
      if (ENTRY_BARRIER && u0 == warp && j0 == 0) cbar_sync();
      if (ep_in != 0) {
        Spin spin;
        unsigned tries = 0;
        while (true) {
          bool bad = false;
#pragma unroll
          for (int h = 0; h < UNITS; ++h) {
#pragma unroll
            for (int j = 0; j < JC; ++j) bad |= (w[h][j].y != ep_in) | (w[h][j].w != ep_in);
          }
          if (!bad) break;
          if (++tries > 4) __nanosleep(40);
          spin.tick(p, DE_LL_WAIT, pidx, (int)ep_in);
#pragma unroll
          for (int h = 0; h < UNITS; ++h) {  // only the quads that are still missing are requested again
            const int u = unit_of(u0 + h * kConsumerWarps);
            const LLWord* src = in + (size_t)(u >> 3) * ld;
            const int qb = (u & 7) * 32 + lane + 256 * j0;
#pragma unroll
            for (int j = 0; j < JC; ++j)
              if ((w[h][j].y != ep_in) | (w[h][j].w != ep_in)) w[h][j] = ll_ld_pair(src + 2 * (qb + 256 * j));
          }
        }
      }
#pragma unroll
      for (int h = 0; h < UNITS; ++h) {
        const bool uok = u0 + h * kConsumerWarps < n_units;
        const int u = unit_of(u0 + h * kConsumerWarps);
        const int qb = (u & 7) * 32 + lane + 256 * j0;
        const uint32_t xrow = xs + (uint32_t)(u >> 3) * rstride;
#pragma unroll
        for (int j = 0; j < JC; ++j) {
          const int q = qb + 256 * j;
          if (uok && q < Kq) xquad_store(xrow + xquad_off(q), w[h][j].x, w[h][j].z);
          const float x0 = bf_lo(w[h][j].x), x1 = bf_hi(w[h][j].x), x2 = bf_lo(w[h][j].z), x3 = bf_hi(w[h][j].z);
          ss[h] += fmaf(x0, x0, x1 * x1) + fmaf(x2, x2, x3 * x3);  // first quad: 0 + sq = sq exactly; absent quads add 0
        }
      }
    }
    if (norm) {
#pragma unroll
      for (int h = 0; h < UNITS; ++h) {
        const bool uok = u0 + h * kConsumerWarps < n_units;
        const int u = unit_of(u0 + h * kConsumerWarps);
        const float t = warp_sum(ss[h]);
        if (uok && lane == 0) sts_f32(red + (uint32_t)u * 4u, t);
      }
    }
  }
  cbar_sync();
  if (tprof) prof_acc(p, 1, *tprof);
  if (!norm) return;
  // rescale: UNITS units of a warp side by side (independent chains); the norm phases have K <= 2048, two quads per lane
#pragma unroll 1
  for (int u0 = warp; u0 < n_units; u0 += UNITS * kConsumerWarps) {
#pragma unroll
    for (int h = 0; h < UNITS; ++h) {
      if (u0 + h * kConsumerWarps < n_units) {
        const int u = unit_of(u0 + h * kConsumerWarps);
        const int m = u >> 3, qb = (u & 7) * 32 + lane;
        const float4 r0 = lds_f32x4(red + (uint32_t)m * 32u), r1 = lds_f32x4(red + (uint32_t)m * 32u + 16u);
        const float tot = ((r0.x + r0.y) + (r0.z + r0.w)) + ((r1.x + r1.y) + (r1.z + r1.w));
        const float rs = rsqrtf(fmaf(tot, inv_k, eps));
        const bool wr = (flags & F_WRITE_NORMED) && (int)blockIdx.x == (m % (int)gridDim.x);
        const uint32_t xrow = xs + (uint32_t)m * rstride;
#pragma unroll 2
        for (int q = qb; q < Kq; q += 256) {
          const uint2 gg = lds_u32x2(gam + (uint32_t)q * 8u);
          const uint32_t a = xrow + xquad_off(q);
          const uint32_t y0 = norm_pair(lds_u32(a), rs, gg.x), y1 = norm_pair(lds_u32(a + 16u), rs, gg.y);
          xquad_store(a, y0, y1);
          if (wr) reinterpret_cast<uint2*>(reinterpret_cast<bf16*>(p.bufs[BUF_HID]) + (size_t)m * p.ld[BUF_HID])[q] = make_uint2(y0, y1);
        }
      }
    }
  }
  cbar_sync();
  if (tprof) prof_acc(p, 2, *tprof);
}

// out of line for the tuned single-stream kernel (a cold path there: predictor pass 0, prefill chunks); the wide kernel inlines it
template <int UNITS, int JC>
__device__ __noinline__ void load_x_rows(const LaunchParams& p, uint32_t flags, const LLWord* in, int ld, uint32_t gam, float eps,
                                         int K, int M, uint32_t ep_in, int pidx, uint32_t xs, uint32_t red) {
  load_x_rows_impl<UNITS, JC, false>(p, flags, in, ld, gam, eps, K, M, ep_in, pidx, xs, red, nullptr);
}

// Sum of the k-parts of one (stream, output word) in the order the single-stream path adds them (its shuffle tree): part g is
// paired with part g + 8, the eight pairs are added as ((0+1)+(2+3))+((4+5)+(6+7)).  pa = this lane's word of part 0; parts
// lie `stride` bytes apart; y0 / y1 enter as the lane's own part-0 sums.
__device__ __forceinline__ float2 tree_parts(float y0, float y1, uint32_t pa, uint32_t stride, int wpg) {
  float P0[8], P1[8];
#pragma unroll
  for (int g = 0; g < 8; ++g) {
    float s0 = 0.f, s1 = 0.f;
    if (g != 0 && g < wpg) { const float2 v = lds_f32x2(pa + (uint32_t)g * stride); s0 = v.x; s1 = v.y; }
    if (g + 8 < wpg) { const float2 v = lds_f32x2(pa + (uint32_t)(g + 8) * stride); s0 += v.x; s1 += v.y; }
    if (g == 0) { s0 += y0; s1 += y1; }
    P0[g] = s0; P1[g] = s1;
  }
  return make_float2(((P0[0] + P0[1]) + (P0[2] + P0[3])) + ((P0[4] + P0[5]) + (P0[6] + P0[7])),
                     ((P1[0] + P1[1]) + (P1[2] + P1[3])) + ((P1[4] + P1[5]) + (P1[6] + P1[7])));
}

template <bool PROF>
__device__ __forceinline__ void gemv_phase_consume(const Ctx& c, const Phase& ph, const LaunchParams& p, RingCur& cur, RingCur& gcur, uint32_t& gst,
                                                   int pidx, uint32_t ep) {
  // the phase's kind and this warp's unit, resolved at kernel start (resolve_kind / resolve_unit): eight + one 16-byte loads
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  RingCur cur0 = cur, gcur0 = gcur;  // by value: the cursors stay in registers
  const uint32_t kda = c.kinds + (uint32_t)ph.kind * (uint32_t)sizeof(KindDesc);
  const uint4 k0 = lds128(kda);  // in | Kq | flags
  const uint4 k3 = lds128(kda + 48u);  // g | grp0 | wpg | gpr
  const uint4 ud = lds128(c.units + (uint32_t)(ph.kind * kConsumerWarps + warp) * (uint32_t)sizeof(UnitDesc));
  if (k3.x == 0u) return;  // more CTAs than row groups: nothing to do here (the producer skips the phase as well)
  const uint32_t flags = k0.w;
  const int Kq = (int)k0.z;  // 16-byte word pairs ("quads": columns 4q .. 4q+3) per row; thread tid owns quads tid and tid + 384
  const LLWord* in = reinterpret_cast<const LLWord*>(((unsigned long long)k0.y << 32) | k0.x);
  const uint32_t ep_in = (pidx == 0 && ep == p.epoch_base + 1) ? 0u : ep - 1;
  const bool norm = (flags & F_PRENORM) != 0;
  if (PROF) prof_mark(p, pidx, 0);
  if (PROF) prof_cta_time(p, pidx, 0);
  if (PROF) prof_warp_time(p, pidx, 0);

  // ---- issue the first poll of this thread's input words (single-stream rows: warps 0-7, quads tid, tid + 256, tid + 512)
  const uint4 k6 = lds128(kda + 96u);  // M | n_words | K | fast
  const bool fast = k6.w != 0u;
  const bool poller = tid < kPollThreads;
  const bool have0 = poller && tid < Kq, have1 = poller && tid + kPollThreads < Kq, have2 = poller && tid + 2 * kPollThreads < Kq;
  const LLWord* src = in + 2 * tid;
  uint4 w0 = make_uint4(0u, ep_in, 0u, ep_in), w1 = w0, w2 = w0;
  if (fast) {
    if (have0) w0 = ll_ld_pair(src);
    if (have1) w1 = ll_ld_pair(src + 2 * kPollThreads);
    if (have2) w2 = ll_ld_pair(src + 4 * kPollThreads);
  }

  // ---- everything that does not depend on the input: overlaps the round trip of the poll
  const uint4 k1 = lds128(kda + 16u);  // out | res
  const uint4 k2 = lds128(kda + 32u);  // bias | ldout | ldres
  const uint4 k4 = lds128(kda + 64u);  // spg | nch | ro_shift | n_stages
  const uint4 k5 = lds128(kda + 80u);  // eps | inv_k | n_rounds | wpgrp
  const int M = (int)k6.x, n_words = (int)k6.y, K = (int)k6.z;
  FQ3_ASSERT(M >= 1 && M <= kMaxRows && (K & 63) == 0 && (M == 1 ? 2 * K * 2 : M * (int)xrow_stride(K)) <= p.xbuf_bytes, pidx, 300000 + M);
  struct { int g, grp0, n_stages; } sb = {(int)k3.x, (int)k3.y, (int)k4.w};
  const int wpg = (int)k3.z, gpr = (int)k3.w, spg = (int)k4.x, ro_shift = (int)k4.z;
  const int g8 = lane >> 2, t = lane & 3;
  // this warp's unit: group (round * gpr + wgrp), k-part kp = blocks [ch0, ch1)
  const int wgrp = (int)ud.x, kp = (int)ud.y;
  const bool w_act = wgrp < gpr;
  int ch0 = (int)ud.z, ch1 = (int)ud.w;
  // norm weights arrive through the producer's stream (slot gcur of the small gamma ring)
  uint32_t gsrc = c.gam + (uint32_t)gcur0.slot * (uint32_t)c.gam_bytes + (uint32_t)tid * 8u;
  uint32_t gfullb = c.gfull + (uint32_t)gcur0.slot * 8u, gemptyb = c.gempty + (uint32_t)gcur0.slot * 8u;
  const uint32_t glap = gcur0.lap;
  if (norm) gcur0.advance(1, kGammaSlots);
  float eps = __uint_as_float(k5.x);
  float inv_k = __uint_as_float(k5.y);
  // Single-stream rows and the partial words alternate between two buffers from one GEMV phase to the next: a warp that is
  // already staging phase i + 1 cannot disturb a warp that still multiplies phase i, and no barrier has to open the phase.
  const uint32_t par = gst & 1u;
  const uint32_t xs = c.xs + (fast ? par * c.xhalf : 0u);
  uint32_t xdst0 = xs + xquad_off(tid), xdst1 = xs + xquad_off(tid + kPollThreads), xdst2 = xs + xquad_off(tid + 2 * kPollThreads);
  // A rows: stream min(g8, M - 1) (rows beyond M repeat the last stream; their results are not read)
  uint32_t xrow = xs + (uint32_t)min(g8, M - 1) * xrow_stride(K) + (uint32_t)t * 16u;
  const uint32_t lane_w = (uint32_t)lane * 16u;
  const uint32_t pbase = c.scratch + par * (uint32_t)(kConsumerWarps * 32 * 8);
  uint32_t pdst = pbase + (uint32_t)((wgrp * wpg + kp) * 32 + lane) * 8u;  // this lane's partial word (two fp32), by unit
  LLWord* out = reinterpret_cast<LLWord*>(((unsigned long long)k1.y << 32) | k1.x);
  const LLWord* resp = reinterpret_cast<const LLWord*>(((unsigned long long)k1.w << 32) | k1.z);
  const uint32_t* biasp = reinterpret_cast<const uint32_t*>(((unsigned long long)k2.y << 32) | k2.x);
  const int ldout = (int)k2.z, ldres = (int)k2.w;
  // finishing lane: stream g8, rows 2t, 2t+1 of the group -> plain: word 4 * group + t; SwiGLU: element 4 * group + t, the even lane
  // of a pair publishes word 2 * group + t / 2
  const bool f_lane = w_act && kp == 0 && g8 < M && (ro_shift == 1 || (t & 1) == 0);
  const int f_sub = (ro_shift == 1) ? t : (t >> 1);
  const int wpgrp = (int)k5.w;  // words per group
  int gi = wgrp;                     // group of round 0
  int f_word = (sb.grp0 + gi) * wpgrp + f_sub;
  uint32_t res0 = 0u, bias0 = 0u;
  const bool g_ok0 = w_act && gi < sb.g;
  if (f_lane && g_ok0 && f_word < n_words) {
    if (flags & F_RESID) res0 = ll_ld(resp + (size_t)g8 * ldres + f_word).x;
    if (flags & F_BIAS) bias0 = __ldg(biasp + f_word);
  }
  // the first stage this warp reads: wait for it now (it landed long ago; a wait after the poll would sit on the critical path)
  RingCur my = cur0;
  const bool pre_ok = g_ok0;  // a round never takes more stages than the ring has slots (fq3_api.cu: launch), so the stage's
                              // slot was handed back by an earlier phase and its copy needs nothing from this one
  if (g_ok0) my.advance(gi * spg + (ch0 >> 5), c.n_stages);
  if (pre_ok) {
    if (!mbar_try_wait_a(c.full + (uint32_t)my.slot * 8u, my.lap)) {
      Spin spin;
      while (!mbar_try_wait_a(c.full + (uint32_t)my.slot * 8u, my.lap)) spin.tick(p, DE_FULL_WAIT, pidx, my.slot);
    }
  }
  int n_rounds = (int)k5.z;  // 1 for every shape of the 0.6B model
  uint32_t wa0 = c.ring + lane_w + (uint32_t)my.slot * kStageBytes + (uint32_t)(ch0 & (kStageChunks - 1)) * kBlockBytes;
  uint32_t xa0 = xrow + (uint32_t)ch0 * kXBlock;
  // Experiment (FQ3_PRE > 0, off): the stage is in shared memory long before the activations are, so the first FQ3_PRE weight
  // blocks of this warp's unit could wait in registers and leave only the activation loads between "input visible" and
  // "output stored".  Measured slower at 4 and 8 blocks even with 152 registers per thread (profiles/r02b_gemv_variants.log):
  // the fragments are spilled around the poll loop.
#ifndef FQ3_PRE
#define FQ3_PRE 0
#endif
  constexpr int kPre = FQ3_PRE > 0 ? FQ3_PRE : 1;
  uint4 wreg[kPre];
  int npre = 0;
  if (pre_ok && FQ3_PRE > 0) {
    npre = min(min(ch1, (ch0 | (kStageChunks - 1)) + 1) - ch0, kPre);
#pragma unroll
    for (int i = 0; i < kPre; ++i)
      if (i < npre) wreg[i] = lds128(wa0 + (uint32_t)i * kBlockBytes);
  }
  // the norm weights were queued by the producer long ago as well
  uint2 g0 = make_uint2(0u, 0u), g1 = g0, g2 = g0;
  if (fast && norm) {
    if (poller) {
      if (!mbar_try_wait_a(gfullb, glap)) {
        Spin spin;
        while (!mbar_try_wait_a(gfullb, glap)) spin.tick(p, DE_FULL_WAIT, pidx, 100);
      }
      if (have0) g0 = lds_u32x2(gsrc);
      if (have1) g1 = lds_u32x2(gsrc + kPollThreads * 8);
      if (have2) g2 = lds_u32x2(gsrc + 2 * kPollThreads * 8);
    } else if (lane == 0) {
      mbar_arrive_a(gemptyb);  // the other warps do not read the norm weights
    }
  }
  pin(gemptyb); pin(eps); pin(inv_k); pin(xdst0); pin(xdst1); pin(xdst2); pin(pdst); pin(f_word); pin(ch0); pin(ch1); pin(wa0); pin(xa0); pin(n_rounds);
  pin(g0.x); pin(g0.y); pin(g1.x); pin(g1.y); pin(g2.x); pin(g2.y);
  // No barrier closes a GEMV phase, so a warp may arrive here while others still multiply the previous phase's activations or
  // read its partial words.  Single-stream phases are protected by the alternating buffers (above); multi-row phases use one
  // buffer and meet here, in the shadow of the poll — and so does a single-stream phase that follows a multi-row one.
  if (!fast || (gst & 2u)) cbar_sync();

  // ---- wait for the input, normalise, stage it in shared memory
  if (fast) {
    if (poller) {
      if (ep_in != 0) {
        unsigned tries = 0;
        while ((w0.y != ep_in) | (w0.w != ep_in) | (w1.y != ep_in) | (w1.w != ep_in) | (w2.y != ep_in) | (w2.w != ep_in)) {
          if (++tries > (unsigned)(p.debug >> 16)) __nanosleep((unsigned)(p.debug & 0xffff));
          if (tries > (unsigned)(p.watchdog_ns >> 8)) device_fault(p, DE_LL_WAIT, pidx, (int)ep_in);
          if (have0 && ((w0.y != ep_in) | (w0.w != ep_in))) w0 = ll_ld_pair(src);
          if (have1 && ((w1.y != ep_in) | (w1.w != ep_in))) w1 = ll_ld_pair(src + 2 * kPollThreads);
          if (have2 && ((w2.y != ep_in) | (w2.w != ep_in))) w2 = ll_ld_pair(src + 4 * kPollThreads);
        }
      }
      if (PROF) prof_mark(p, pidx, 7);
      if (PROF) prof_warp_time(p, pidx, 5);
      if (!norm) {
        if (have0) xquad_store(xdst0, w0.x, w0.z);
        if (have1) xquad_store(xdst1, w1.x, w1.z);
        if (have2) xquad_store(xdst2, w2.x, w2.z);
      } else {
        float ss;
        {  // absent pairs carry payload 0
          const float a0 = bf_lo(w0.x), a1 = bf_hi(w0.x), a2 = bf_lo(w0.z), a3 = bf_hi(w0.z);
          const float b0 = bf_lo(w1.x), b1 = bf_hi(w1.x), b2 = bf_lo(w1.z), b3 = bf_hi(w1.z);
          const float c0 = bf_lo(w2.x), c1 = bf_hi(w2.x), c2 = bf_lo(w2.z), c3 = bf_hi(w2.z);
          ss = (fmaf(a0, a0, a1 * a1) + fmaf(a2, a2, a3 * a3)) + (fmaf(b0, b0, b1 * b1) + fmaf(b2, b2, b3 * b3)) +
               (fmaf(c0, c0, c1 * c1) + fmaf(c2, c2, c3 * c3));
        }
        ss = warp_sum(ss);
        if (lane == 0) sts_f32(c.red + (uint32_t)warp * 4u, ss);
        if (PROF) prof_mark(p, pidx, 15);
        poll_bar_sync();  // the eight polling warps
        if (PROF) prof_mark(p, pidx, 14);
        float tot;
        {
          const float4 r0 = lds_f32x4(c.red), r1 = lds_f32x4(c.red + 16u);
          static_assert(kPollWarps == 8, "the RMSNorm reduction reads eight per-warp sums");
          tot = ((r0.x + r0.y) + (r0.z + r0.w)) + ((r1.x + r1.y) + (r1.z + r1.w));
        }
        const float rs = rsqrtf(fmaf(tot, inv_k, eps));
        const bool wr = (flags & F_WRITE_NORMED) && blockIdx.x == 0;
        if (have0) {
          const uint32_t y0 = norm_pair(w0.x, rs, g0.x), y1 = norm_pair(w0.z, rs, g0.y);
          xquad_store(xdst0, y0, y1);
          if (wr) reinterpret_cast<uint2*>(p.bufs[BUF_HID])[tid] = make_uint2(y0, y1);
        }
        if (have1) {
          const uint32_t y0 = norm_pair(w1.x, rs, g1.x), y1 = norm_pair(w1.z, rs, g1.y);
          xquad_store(xdst1, y0, y1);
          if (wr) reinterpret_cast<uint2*>(p.bufs[BUF_HID])[tid + kPollThreads] = make_uint2(y0, y1);
        }
        if (have2) {
          const uint32_t y0 = norm_pair(w2.x, rs, g2.x), y1 = norm_pair(w2.z, rs, g2.y);
          xquad_store(xdst2, y0, y1);
          if (wr) reinterpret_cast<uint2*>(p.bufs[BUF_HID])[tid + 2 * kPollThreads] = make_uint2(y0, y1);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive_a(gemptyb);
      }
    }
    if (PROF) prof_warp_time(p, pidx, 6);
    cbar_sync();  // all twelve warps: the activation row is staged (red[] is safe as well: the next norm phase lies behind this barrier)
    if (PROF) prof_warp_time(p, pidx, 1);
  } else {
    if (norm && !mbar_try_wait_a(gfullb, glap)) {
      Spin spin;
      while (!mbar_try_wait_a(gfullb, glap)) spin.tick(p, DE_FULL_WAIT, pidx, 100);
    }
    load_x_rows<1, 3>(p, flags, in, (int)lds_u32(kda + 112u), gsrc - (uint32_t)tid * 8u, eps, K, M, ep_in, pidx, c.xs, c.red);
    if (norm) {  // load_x_rows ends with a barrier after the last read of the norm weights
      if (lane == 0) mbar_arrive_a(gemptyb);
    }
  }
  if (PROF) prof_mark(p, pidx, 1);

  // ---- multiply, reduce the k-parts, publish, hand the group's stages back
#pragma unroll 1
  for (int r = 0; r < n_rounds; ++r) {
    // A round re-uses the ring slots of the round before.  mbarrier phases only tell adjacent uses of a slot apart, so
    // nobody may wait for a slot's next use before all readers of the current one are through: rounds are separated by a
    // block barrier (it also protects the partial words).
    if (r != 0) cbar_sync();
    gi = r * gpr + wgrp;
    if (!(w_act && gi < sb.g)) continue;  // (all warps of a group skip together)
    if (r != 0) {
      my = cur0;
      my.advance(gi * spg + (ch0 >> 5), c.n_stages);
      const uint32_t fb = c.full + (uint32_t)my.slot * 8u;
      Spin spin;
      while (!mbar_try_wait_a(fb, my.lap)) spin.tick(p, DE_FULL_WAIT, pidx, my.slot);
      wa0 = c.ring + lane_w + (uint32_t)my.slot * kStageBytes + (uint32_t)(ch0 & (kStageChunks - 1)) * kBlockBytes;
    }
    float acc[4] = {0.f, 0.f, 0.f, 0.f}, acc2[4] = {0.f, 0.f, 0.f, 0.f};  // two accumulator chains (k-step 0 / 1 of a block)
    int ch = ch0;
    uint32_t wa = wa0, xa = xa0;
    if (PROF && r == 0) prof_mark(p, pidx, 8);
    if (PROF && r == 0) prof_warp_time(p, pidx, 2);
    if (r == 0 && npre > 0) {
      // blocks whose weights wait in registers: only the activation loads remain, one ahead of the MMAs
      uint4 xv = lds128(xa);
#pragma unroll
      for (int i = 0; i < kPre; ++i) {
        if (i < npre) {
          uint4 xn = xv;
          if (ch0 + i + 1 < ch1) xn = lds128(xa + (uint32_t)(i + 1) * kXBlock);
          mma_bf16(acc, xv.x, xv.x, xv.y, xv.y, wreg[i].x, wreg[i].y);
          mma_bf16(acc2, xv.z, xv.z, xv.w, xv.w, wreg[i].z, wreg[i].w);
          xv = xn;
        }
      }
      ch += npre;
      wa += (uint32_t)npre * kBlockBytes;
      xa += (uint32_t)npre * kXBlock;
    }
#pragma unroll 1
    while (ch < ch1) {
      if (ch != ch0 && (ch & (kStageChunks - 1)) == 0) {  // the unit goes on in the next stage of the group
        my.advance(1, c.n_stages);
        const uint32_t fb = c.full + (uint32_t)my.slot * 8u;
        if (!mbar_try_wait_a(fb, my.lap)) {
          Spin spin;
          while (!mbar_try_wait_a(fb, my.lap)) spin.tick(p, DE_FULL_WAIT, pidx, my.slot);
        }
        wa = c.ring + lane_w + (uint32_t)my.slot * kStageBytes;
      }
      const int ce = min(ch1, (ch | (kStageChunks - 1)) + 1);  // end of this stage's blocks
      // software-pipelined: the loads of block i + 1 are in flight while block i is multiplied
      uint4 wv = lds128(wa), xv = lds128(xa);
#pragma unroll 2
      for (int n = ce - ch - 1; n > 0; --n) {
        wa += kBlockBytes;
        xa += kXBlock;
        const uint4 wn = lds128(wa), xn = lds128(xa);
        mma_bf16(acc, xv.x, xv.x, xv.y, xv.y, wv.x, wv.y);
        mma_bf16(acc2, xv.z, xv.z, xv.w, xv.w, wv.z, wv.w);
        wv = wn; xv = xn;
      }
      mma_bf16(acc, xv.x, xv.x, xv.y, xv.y, wv.x, wv.y);
      mma_bf16(acc2, xv.z, xv.z, xv.w, xv.w, wv.z, wv.w);
      wa += kBlockBytes;
      xa += kXBlock;
      ch = ce;
    }
    if (PROF && r == 0) prof_mark(p, pidx, 9);
    if (PROF && r == 0) prof_warp_time(p, pidx, 3);
    // ---- finish the unit: stream g8, rows 2t, 2t+1 of group gi -> partial words -> epilogue -> publish
    float y0 = acc[0] + acc2[0], y1 = acc[1] + acc2[1];
    if (wpg > 1) {
      if (kp != 0) sts_f32x2(pdst, y0, y1);
      group_bar_sync(2 + wgrp, wpg * 32);
      if (kp == 1) {
        // every warp of the group has finished reading the group's stages (its k loop lies in front of the group barrier):
        // the second warp hands them back, one arrival per stage — the first one is busy with the output
        if (lane == 0) {
          int rs = cur0.slot + gi * spg;
          while (rs >= c.n_stages) rs -= c.n_stages;
          for (int s2 = 0; s2 < spg; ++s2) {
            mbar_arrive_a(c.empty + (uint32_t)rs * 8u);
            if (++rs == c.n_stages) rs = 0;
          }
        }
      } else if (kp == 0) {
        if (wpg <= 4) {
          // few parts: every lane adds the partial words of its own (stream, word) in part order
#pragma unroll
          for (int k2 = 1; k2 < 4; ++k2) {
            if (k2 < wpg) {
              const float2 v = lds_f32x2(pdst + (uint32_t)k2 * 256u);
              y0 += v.x; y1 += v.y;
            }
          }
        } else if (M == 1) {
          // many parts, one stream: lane (g8, t) adds the parts g8, g8 + 8 of word t, three shuffles add the eight slices in
          // a fixed order (the A rows of a single stream are copies: every lane's own accumulator equals lane t's)
          float s0 = 0.f, s1 = 0.f;
          const uint32_t q0 = pbase + (uint32_t)(wgrp * wpg * 32 + t) * 8u;
          if (g8 != 0 && g8 < wpg) { const float2 v = lds_f32x2(q0 + (uint32_t)g8 * 256u); s0 = v.x; s1 = v.y; }
          if (g8 + 8 < wpg) { const float2 v = lds_f32x2(q0 + (uint32_t)(g8 + 8) * 256u); s0 += v.x; s1 += v.y; }
          if (g8 == 0) { s0 += y0; s1 += y1; }
#pragma unroll
          for (int o = 4; o <= 16; o <<= 1) {
            s0 += __shfl_xor_sync(0xffffffffu, s0, o);
            s1 += __shfl_xor_sync(0xffffffffu, s1, o);
          }
          y0 = s0; y1 = s1;
        } else {
          // many parts, several streams: the single-stream tree once per stream (stream m's own sums sit in lanes (m, t));
          // lane (m, t) keeps the result
          float r0 = y0, r1 = y1;
#pragma unroll 1
          for (int m = 0; m < M; ++m) {
            float s0 = 0.f, s1 = 0.f;
            const uint32_t q0 = pbase + (uint32_t)(wgrp * wpg * 32 + m * 4 + t) * 8u;
            if (g8 != 0 && g8 < wpg) { const float2 v = lds_f32x2(q0 + (uint32_t)g8 * 256u); s0 = v.x; s1 = v.y; }
            if (g8 + 8 < wpg) { const float2 v = lds_f32x2(q0 + (uint32_t)(g8 + 8) * 256u); s0 += v.x; s1 += v.y; }
            const float o0 = __shfl_sync(0xffffffffu, y0, m * 4 + t), o1 = __shfl_sync(0xffffffffu, y1, m * 4 + t);
            if (g8 == 0) { s0 += o0; s1 += o1; }
#pragma unroll
            for (int o = 4; o <= 16; o <<= 1) {
              s0 += __shfl_xor_sync(0xffffffffu, s0, o);
              s1 += __shfl_xor_sync(0xffffffffu, s1, o);
            }
            if (g8 == m) { r0 = s0; r1 = s1; }
          }
          y0 = r0; y1 = r1;
        }
      }
    }
    if (PROF && r == 0) prof_mark(p, pidx, 10, kProfLeader);
    if (kp == 0) {
      if (r != 0) {
        f_word = (sb.grp0 + gi) * wpgrp + f_sub;
        if (f_lane && f_word < n_words) {
          if (flags & F_RESID) res0 = ll_ld(resp + (size_t)g8 * ldres + f_word).x;
          if (flags & F_BIAS) bias0 = __ldg(biasp + f_word);
        }
      }
      float lo, hi;
      if (flags & F_SWIGLU) {
        // (y0, y1) = (gate, up) of element 4 * group + t; the odd lane of a pair hands its element to the even one
        const float e = bf16r(bf16r(silu_f(bf16r(y0))) * bf16r(y1));
        lo = e;
        hi = __shfl_down_sync(0xffffffffu, e, 1);
      } else {
        lo = y0; hi = y1;
        if (flags & F_BIAS) { lo += bf_lo(bias0); hi += bf_hi(bias0); }
        lo = bf16r(lo); hi = bf16r(hi);
        if (flags & F_SILU) { lo = bf16r(silu_f(lo)); hi = bf16r(silu_f(hi)); }
      }
      if (flags & F_RESID) { lo = bf16r(bf_lo(res0) + lo); hi = bf16r(bf_hi(res0) + hi); }
      if (PROF) prof_cta_time(p, pidx, 1);
      if (f_lane && f_word < n_words) ll_st(out + (size_t)g8 * ldout + f_word, pack_bf16x2(lo, hi), ep);
      if (PROF && r == 0) prof_mark(p, pidx, 11, kProfLeader);
      if (PROF && r == 0) prof_warp_time(p, pidx, 7);
      if (wpg == 1) {  // a group of one warp hands its own stages back
        __syncwarp();
        if (lane == 0) {
          int rs = cur0.slot + gi * spg;
          while (rs >= c.n_stages) rs -= c.n_stages;
          for (int s2 = 0; s2 < spg; ++s2) {
            mbar_arrive_a(c.empty + (uint32_t)rs * 8u);
            if (++rs == c.n_stages) rs = 0;
          }
        }
      }
    }
  }
  cur0.advance(sb.n_stages, c.n_stages);
  cur = cur0;
  gcur = gcur0;
  gst = ((gst & 1u) ^ 1u) | (fast ? 0u : 2u);
  if (PROF) prof_mark(p, pidx, 3, kProfLeader);
  if (PROF) prof_warp_time(p, pidx, 4);
}


// GEMV phase of the wide frame program: up to kMaxWide = 16 lock-step streams, all 16 A rows of the MMA in use (rows g8 and
// g8 + 8 of a lane's fragments are different streams; a lane ends up with two output words).  Same arithmetic per stream as the
// single-stream path (load_x_rows, tree_parts, the same accumulator chains), so a stream's tokens do not depend on its
// neighbours.  What grows with the batch is the staging: every CTA polls M * K / 2 LL words per phase.
// (Inlined into the wide kernel: as a separate function its cursors lived in local memory, and with 227 KB of shared memory the
// 28 KB of L1 that are left do not hold 384 threads' stack frames — every access to them was an L2 round trip, 14 % of the
// samples of an ncu capture.  The kind / unit descriptors are read from shared memory field by field for the same reason.)
struct KindRegs {  // the fields of a KindDesc, loaded with eight 16-byte shared-memory reads
  const LLWord* in; int Kq, flags; LLWord* out; const LLWord* res; const uint32_t* bias; int ldout, ldres;
  int g, grp0, wpg, gpr, spg, nch, ro_shift, n_stages; float eps, inv_k; int n_rounds, wpgrp, M, n_words, K, fast, ldin, norm;
};
__device__ __forceinline__ KindRegs load_kind(uint32_t kda) {
  const uint4 k0 = lds128(kda), k1 = lds128(kda + 16u), k2 = lds128(kda + 32u), k3 = lds128(kda + 48u), k4 = lds128(kda + 64u),
              k5 = lds128(kda + 80u), k6 = lds128(kda + 96u), k7 = lds128(kda + 112u);
  KindRegs r;
  r.in = reinterpret_cast<const LLWord*>(((unsigned long long)k0.y << 32) | k0.x); r.Kq = (int)k0.z; r.flags = (int)k0.w;
  r.out = reinterpret_cast<LLWord*>(((unsigned long long)k1.y << 32) | k1.x);
  r.res = reinterpret_cast<const LLWord*>(((unsigned long long)k1.w << 32) | k1.z);
  r.bias = reinterpret_cast<const uint32_t*>(((unsigned long long)k2.y << 32) | k2.x); r.ldout = (int)k2.z; r.ldres = (int)k2.w;
  r.g = (int)k3.x; r.grp0 = (int)k3.y; r.wpg = (int)k3.z; r.gpr = (int)k3.w;
  r.spg = (int)k4.x; r.nch = (int)k4.y; r.ro_shift = (int)k4.z; r.n_stages = (int)k4.w;
  r.eps = __uint_as_float(k5.x); r.inv_k = __uint_as_float(k5.y); r.n_rounds = (int)k5.z; r.wpgrp = (int)k5.w;
  r.M = (int)k6.x; r.n_words = (int)k6.y; r.K = (int)k6.z; r.fast = (int)k6.w;
  r.ldin = (int)k7.x; r.norm = (int)k7.y;
  return r;
}
__device__ __forceinline__ void gemv_phase_consume_wide(const Ctx& c, const Phase& ph, const LaunchParams& p, RingCur& cur, RingCur& gcur, uint32_t& gst,
                                                        int pidx, uint32_t ep) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const KindRegs kd = load_kind(c.kinds + (uint32_t)ph.kind * (uint32_t)sizeof(KindDesc));
  struct { int wgrp, kp, ch0, ch1; } ud;
  {
    const uint4 u4 = lds128(c.units + (uint32_t)(ph.kind * kConsumerWarps + warp) * (uint32_t)sizeof(UnitDesc));
    ud.wgrp = (int)u4.x; ud.kp = (int)u4.y; ud.ch0 = (int)u4.z; ud.ch1 = (int)u4.w;
  }
  if (kd.g == 0) return;
  const uint32_t flags = (uint32_t)kd.flags;
  const int M = kd.M, K = kd.K, n_words = kd.n_words;
  const bool norm = (flags & F_PRENORM) != 0;
  uint32_t ep_in = (pidx == 0 && ep == p.epoch_base + 1) ? 0u : ep - 1;
  if (flags & F_IN_PREV) {  // rows published by the talker sampler of the previous iteration (epoch = this iteration's base)
    const uint32_t ep0 = ep - (uint32_t)pidx - 1u;
    ep_in = (ep0 == p.epoch_base) ? 0u : ep0;
  }
  FQ3_ASSERT(M >= 1 && M <= kMaxWide && (K & 63) == 0 && M * (int)xrow_stride(K) <= p.xbuf_bytes, pidx, 320000 + M);
  if ((flags & (F_IN_PREV | F_WPIN_B)) == (F_IN_PREV | F_WPIN_B) && pidx > 0) {
    // First phase of pass 0b.  Its input (BUF_WPIN) is older than the iteration, so unlike every other phase it does not depend
    // on the phase before it — pass 0a's last attention — and a CTA without an attention item there (fewer than 16 streams) is
    // already here while others still poll that attention's q / k / v words in the buffer THIS phase publishes into: a word of
    // this phase landing first makes their exact-epoch poll spin for good (seen once as a watchdog fault, with the codec of a
    // serving loop running beside the kernel).  An attention item reads all its inputs before it computes any output, so one
    // output word per (stream, kv head) with the previous phase's epoch proves the buffer is free; the block barrier inside
    // load_x_rows keeps every warp's publish behind this wait.
    const StackRt& Sp = p.stacks[ST_PRED];
    const int n_items = M * Sp.nkv;
    const int words_per_item = (Sp.nq / Sp.nkv) * (kHeadDim / 2);
    for (int it = tid; it < n_items; it += kConsumerWarps * 32) {
      const int g = it / Sp.nkv, kvh = it - g * Sp.nkv;
      (void)ll_wait(reinterpret_cast<const LLWord*>(p.bufs[BUF_PATT]) + (size_t)g * p.ld[BUF_PATT] + (size_t)kvh * words_per_item, ep - 1u, p, pidx);
    }
  }
  const uint32_t gsrc = c.gam + (uint32_t)gcur.slot * (uint32_t)c.gam_bytes;
  const uint32_t gfullb = c.gfull + (uint32_t)gcur.slot * 8u, gemptyb = c.gempty + (uint32_t)gcur.slot * 8u;
  const uint32_t glap = gcur.lap;
  if (norm) gcur.advance(1, kGammaSlots);
  long long tp = (FQ3_WIDE_PROF && p.prof) ? clock64() : 0ll;
  // (the block barrier behind which the previous phase's activation rows and partial words may be overwritten sits inside
  // load_x_rows, behind the first poll requests: ENTRY_BARRIER)
  if (norm && !mbar_try_wait_a(gfullb, glap)) {
    Spin spin;
    while (!mbar_try_wait_a(gfullb, glap)) spin.tick(p, DE_FULL_WAIT, pidx, 100);
  }
  // the output lanes' residual / bias words are older than this phase's input: request them now, under the poll
  const int g8 = lane >> 2, t = lane & 3;
  const int f_sub = (kd.ro_shift == 1) ? t : (t >> 1);
  const bool t_ok = (kd.ro_shift == 1) || ((t & 1) == 0);
  uint32_t res_pre[2] = {0u, 0u}, bias_pre = 0u;
  {
    const int f_word = (kd.grp0 + ud.wgrp) * kd.wpgrp + f_sub;
    if (ud.wgrp < kd.gpr && ud.kp == 0 && ud.wgrp < kd.g && t_ok && f_word < n_words) {
      if (flags & F_RESID) {
        if (g8 < M) res_pre[0] = ll_ld(kd.res + (size_t)g8 * kd.ldres + f_word).x;
        if (g8 + 8 < M) res_pre[1] = ll_ld(kd.res + (size_t)(g8 + 8) * kd.ldres + f_word).x;
      }
      if (flags & F_BIAS) bias_pre = __ldg(kd.bias + f_word);
    }
  }
  {
    long long* tpp = (FQ3_WIDE_PROF && p.prof) ? &tp : nullptr;
    // six 16-byte requests per lane in flight (twelve was measured: slower — every CTA asks L2 for the same lines)
    if (K <= 1024) load_x_rows_impl<6, 1, true>(p, flags, kd.in, kd.ldin, gsrc, kd.eps, K, M, ep_in, pidx, c.xs, c.red, tpp);
    else if (K <= 2048) load_x_rows_impl<3, 2, true>(p, flags, kd.in, kd.ldin, gsrc, kd.eps, K, M, ep_in, pidx, c.xs, c.red, tpp);
    else load_x_rows_impl<2, 3, true>(p, flags, kd.in, kd.ldin, gsrc, kd.eps, K, M, ep_in, pidx, c.xs, c.red, tpp);
  }
  if (norm && lane == 0) mbar_arrive_a(gemptyb);

  const int wgrp = ud.wgrp, kp = ud.kp, ch0 = ud.ch0, ch1 = ud.ch1;
  const int wpg = kd.wpg, gpr = kd.gpr, spg = kd.spg, wpgrp = kd.wpgrp;
  const bool w_act = wgrp < gpr;
  const uint32_t rstride = xrow_stride(K);
  const uint32_t xlo = c.xs + (uint32_t)min(g8, M - 1) * rstride + (uint32_t)t * 16u;
  const uint32_t xhi = c.xs + (uint32_t)min(g8 + 8, M - 1) * rstride + (uint32_t)t * 16u;
  const uint32_t lane_w = (uint32_t)lane * 16u;
  // partial words: [unit][half: streams g8 / g8 + 8][lane] two fp32
  const uint32_t pdst = c.scratch + (uint32_t)((wgrp * wpg + kp) * 64 + lane) * 8u;
#pragma unroll 1
  for (int r = 0; r < kd.n_rounds; ++r) {
    if (r != 0) cbar_sync();  // rounds re-use ring slots and partial words (gemv_phase_consume)
    const int gi = r * gpr + wgrp;
    if (!(w_act && gi < kd.g)) continue;
    RingCur my = cur;
    my.advance(gi * spg + (ch0 >> 5), c.n_stages);
    {
      const uint32_t fb = c.full + (uint32_t)my.slot * 8u;
      Spin spin;
      while (!mbar_try_wait_a(fb, my.lap)) spin.tick(p, DE_FULL_WAIT, pidx, my.slot);
    }
    uint32_t wa = c.ring + lane_w + (uint32_t)my.slot * kStageBytes + (uint32_t)(ch0 & (kStageChunks - 1)) * kBlockBytes;
    float acc[4] = {0.f, 0.f, 0.f, 0.f}, acc2[4] = {0.f, 0.f, 0.f, 0.f};
    int ch = ch0;
    long long tq = (FQ3_WIDE_PROF && p.prof) ? clock64() : 0ll;
    if (FQ3_WIDE_PROF && p.prof) { tq = tp; prof_acc(p, 8, tq, kProfLeader); }  // 8: from the staging barrier to the weights being there
#pragma unroll 1
    while (ch < ch1) {
      if (ch != ch0 && (ch & (kStageChunks - 1)) == 0) {
        my.advance(1, c.n_stages);
        const uint32_t fb = c.full + (uint32_t)my.slot * 8u;
        Spin spin;
        while (!mbar_try_wait_a(fb, my.lap)) spin.tick(p, DE_FULL_WAIT, pidx, my.slot);
        wa = c.ring + lane_w + (uint32_t)my.slot * kStageBytes;
      }
      const int ce = min(ch1, (ch | (kStageChunks - 1)) + 1);
      uint32_t xa = (uint32_t)ch * kXBlock;
      uint4 wv = lds128(wa), xl = lds128(xlo + xa), xh = lds128(xhi + xa);
#pragma unroll 2
      for (int n = ce - ch - 1; n > 0; --n) {
        wa += kBlockBytes;
        xa += kXBlock;
        const uint4 wn = lds128(wa), xln = lds128(xlo + xa), xhn = lds128(xhi + xa);
        mma_bf16(acc, xl.x, xh.x, xl.y, xh.y, wv.x, wv.y);
        mma_bf16(acc2, xl.z, xh.z, xl.w, xh.w, wv.z, wv.w);
        wv = wn; xl = xln; xh = xhn;
      }
      mma_bf16(acc, xl.x, xh.x, xl.y, xh.y, wv.x, wv.y);
      mma_bf16(acc2, xl.z, xh.z, xl.w, xh.w, wv.z, wv.w);
      wa += kBlockBytes;
      ch = ce;
    }
    // lane (g8, t): streams g8 (y[0], y[1]) and g8 + 8 (y[2], y[3]), rows 2t, 2t+1 of group gi
    float y[4] = {acc[0] + acc2[0], acc[1] + acc2[1], acc[2] + acc2[2], acc[3] + acc2[3]};
    prof_acc(p, 9, tq, kProfLeader);  // 9: k loop
    if (wpg > 1) {
      if (kp != 0) {
        sts_f32x2(pdst, y[0], y[1]);
        sts_f32x2(pdst + 256u, y[2], y[3]);
      }
      group_bar_sync(2 + wgrp, wpg * 32);
      if (kp == 1) {
        if (lane == 0) {  // every warp of the group is through with the group's stages: hand them back
          int rs = cur.slot + gi * spg;
          while (rs >= c.n_stages) rs -= c.n_stages;
          for (int s2 = 0; s2 < spg; ++s2) {
            mbar_arrive_a(c.empty + (uint32_t)rs * 8u);
            if (++rs == c.n_stages) rs = 0;
          }
        }
      } else if (kp == 0) {
        if (wpg <= 4) {
#pragma unroll
          for (int k2 = 1; k2 < 4; ++k2) {
            if (k2 < wpg) {
              const float2 v0 = lds_f32x2(pdst + (uint32_t)k2 * 512u), v1 = lds_f32x2(pdst + (uint32_t)k2 * 512u + 256u);
              y[0] += v0.x; y[1] += v0.y; y[2] += v1.x; y[3] += v1.y;
            }
          }
        } else {
          const float2 v0 = tree_parts(y[0], y[1], pdst, 512u, wpg), v1 = tree_parts(y[2], y[3], pdst + 256u, 512u, wpg);
          y[0] = v0.x; y[1] = v0.y; y[2] = v1.x; y[3] = v1.y;
        }
      }
    }
    prof_acc(p, 10, tq, kProfLeader);  // 10: k-parts through shared memory
    if (kp == 0) {
      const int f_word = (kd.grp0 + gi) * wpgrp + f_sub;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int row = g8 + 8 * h;
        const bool f_lane = row < M && t_ok && f_word < n_words;
        const float y0 = y[2 * h], y1 = y[2 * h + 1];
        uint32_t res0 = res_pre[h], bias0 = bias_pre;
        if (f_lane && r != 0) {
          if (flags & F_RESID) res0 = ll_ld(kd.res + (size_t)row * kd.ldres + f_word).x;
          if (flags & F_BIAS) bias0 = __ldg(kd.bias + f_word);
        }
        float lo, hi;
        if (flags & F_SWIGLU) {
          const float e = bf16r(bf16r(silu_f(bf16r(y0))) * bf16r(y1));
          lo = e;
          hi = __shfl_down_sync(0xffffffffu, e, 1);
        } else {
          lo = y0; hi = y1;
          if (flags & F_BIAS) { lo += bf_lo(bias0); hi += bf_hi(bias0); }
          lo = bf16r(lo); hi = bf16r(hi);
          if (flags & F_SILU) { lo = bf16r(silu_f(lo)); hi = bf16r(silu_f(hi)); }
        }
        if (flags & F_RESID) { lo = bf16r(bf_lo(res0) + lo); hi = bf16r(bf_hi(res0) + hi); }
        if (f_lane) ll_st(kd.out + (size_t)row * kd.ldout + f_word, pack_bf16x2(lo, hi), ep);
      }
      prof_acc(p, 11, tq, kProfLeader);  // 11: epilogue + publish
      if (wpg == 1) {
        __syncwarp();
        if (lane == 0) {
          int rs = cur.slot + gi * spg;
          while (rs >= c.n_stages) rs -= c.n_stages;
          for (int s2 = 0; s2 < spg; ++s2) {
            mbar_arrive_a(c.empty + (uint32_t)rs * 8u);
            if (++rs == c.n_stages) rs = 0;
          }
        }
      }
    }
  }
  cur.advance(kd.n_stages, c.n_stages);
  gst = ((gst & 1u) ^ 1u) | 2u;
  prof_acc(p, 3, tp);
  if (FQ3_WIDE_PROF && p.prof && tid == 0 && (int)blockIdx.x == p.prof_cta) p.prof[6] += 1;
}

// Producer side of one GEMV phase: stream this CTA's groups through the ring, one contiguous bulk copy per stage (up to
// 16 KB = 1024 columns of one group's image).  The phase's norm weights travel in the same stream.  Returns false when the
// consumers asked to stop (frame loop finished early).
template <bool PROF>
__device__ __forceinline__ bool gemv_phase_produce(const Ctx& c, const Phase& ph, const LaunchParams& p, int* ctl, RingCur& cur, RingCur& gcur, uint32_t& issued,
                                                   uint32_t& gissued, int pidx, uint64_t pol_stream, uint64_t pol_keep, uint64_t pol_gamma) {
  const Slab sb = get_slab(ph, p);
  if (sb.g == 0) return true;
  const int K = (int)ph.K;
  const uint32_t gbytes = (uint32_t)K * 16u;  // one group: 8 rows
  const unsigned char* W = ((ph.flags & F_ABSPTR) ? reinterpret_cast<const unsigned char*>(p.lin_W) : p.tiled + (size_t)ph.w_off * 16) +
                           (size_t)sb.grp0 * gbytes;
  const uint64_t pol = (ph.flags & F_L2_KEEP) ? pol_keep : pol_stream;
  if (PROF && (int)blockIdx.x == p.prof_cta && pidx < 512) p.prof[(size_t)pidx * 16 + 4] = clock64();
  if (ph.flags & F_PRENORM) {
    const unsigned char* gp = (ph.flags & F_ABSPTR) ? reinterpret_cast<const unsigned char*>(p.lin_gamma) : p.arena + (size_t)ph.g_off * 16;
    const uint32_t gfullb = c.gfull + (uint32_t)gcur.slot * 8u, gemptyb = c.gempty + (uint32_t)gcur.slot * 8u;
    Spin spin;
    while (!mbar_try_wait_a(gemptyb, gcur.lap ^ 1u)) {
      if (ld_volatile_shared_i32(ctl) < 0) return false;
      __nanosleep(100);
      spin.tick(p, DE_EMPTY_WAIT, pidx, 100 + gcur.slot);
    }
    if (ld_volatile_shared_i32(ctl) < 0) return false;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(gfullb), "r"((uint32_t)K * 2u) : "memory");
    bulk_g2s_a(c.gam + (uint32_t)gcur.slot * (uint32_t)c.gam_bytes, gp, (uint32_t)K * 2u, gfullb, pol_gamma);
    gcur.advance(1, kGammaSlots);
    ++gissued;
  }
#pragma unroll 1
  for (int gi = 0; gi < sb.g; ++gi) {
#pragma unroll 1
    for (uint32_t off = 0; off < gbytes; off += kStageBytes) {
      const uint32_t bytes = min((uint32_t)kStageBytes, gbytes - off);
      const uint32_t fullb = c.full + (uint32_t)cur.slot * 8u, emptyb = c.empty + (uint32_t)cur.slot * 8u;
      Spin spin;
      while (!mbar_try_wait_a(emptyb, cur.lap ^ 1u)) {
        if (ld_volatile_shared_i32(ctl) < 0) return false;
        __nanosleep(100);  // the ring is full most of the time
        spin.tick(p, DE_EMPTY_WAIT, pidx, cur.slot);
      }
      if (ld_volatile_shared_i32(ctl) < 0) return false;
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(fullb), "r"(bytes) : "memory");
      bulk_g2s_a(c.ring + (uint32_t)cur.slot * kStageBytes, W + (size_t)gi * gbytes + off, bytes, fullb, pol);
      cur.advance(1, c.n_stages);
      ++issued;
    }
  }
  if (PROF && (int)blockIdx.x == p.prof_cta && pidx < 512) p.prof[(size_t)pidx * 16 + 5] = clock64();
  return true;
}

// =================================================================================================
// Attention phase: q/k RMSNorm + RoPE + KV append + GQA decode attention (+ split-KV combine).
// One work item = (group, query row, kv head, split): one query row and its (<= 2) q heads.  A decode step has one
// row per stream; a prefill chunk spreads its rows over CTAs — every item re-derives the chunk's K/V rows up to its own
// (identical bytes from every writer, so the redundant stores are benign) and needs no cross-CTA ordering.
// =================================================================================================
struct Group {
  int first_row, nrows, slot, pos0, n_pad, rope_delta;
};
__device__ __forceinline__ int num_groups(const LaunchParams& p) { return p.mode == MODE_PREFILL ? 1 : p.n_rows; }
__device__ __forceinline__ Group get_group(const Phase& ph, const LaunchParams& p, int g, const int* frame_pos) {
  Group r;
  if (p.mode == MODE_PREFILL) {
    r.first_row = 0; r.nrows = p.n_rows; r.slot = p.stream0; r.pos0 = p.pf_pos0; r.n_pad = p.pf_n_pad;
    r.rope_delta = p.pf_rope_delta;
    return r;
  }
  r.nrows = (ph.flags & F_ROWS2) ? 2 : 1;
  r.first_row = g * r.nrows;
  r.slot = p.stream0 + g;
  if (ph.stack == ST_TALKER) {
    // a stream whose prompt filled the whole cache (T == max_seq_len) still runs the talker phases of its last frame; their
    // result is discarded (done = 2), so any in-range row will do (generate.py:174-177 returns one frame and breaks)
    r.pos0 = min((p.pos_override >= 0) ? p.pos_override : frame_pos[g], p.stacks[ST_TALKER].max_pos - 1);
    // launch constants of the stream, parked in shared memory by the frame loop (two L2 round trips per attention phase otherwise)
    const int* sconst = frame_pos + (kStreamConstOffset - kCtlOffset) / 4 - kFramePosIdx;
    r.n_pad = sconst[g];
    r.rope_delta = sconst[kMaxWide + g];
  } else {
    r.pos0 = (ph.flags & (F_ROWS2 | F_PASS0A)) ? 0 : (int)ph.aux + 1;
    r.n_pad = 0;
    r.rope_delta = 0;
  }
  return r;
}
// one CTA sweeps up to kSplitLen positions of one (row, kv head); longer contexts are split over CTAs
__device__ __forceinline__ int num_splits(int L, int cap) {
  const int want = (L + kSplitLen - 1) / kSplitLen;
  return max(1, min(want, cap));
}

// RMSNorm over the 128-wide head + rotary embedding; lane owns elements [4*lane, 4*lane+4).
struct RopeRegs {
  uint2 g2, c2, s2;
};
// issued before the q/k words are polled, so the table reads overlap the wait
__device__ __forceinline__ RopeRegs rope_load(const bf16* gamma, const bf16* cosp, const bf16* sinp, int lane) {
  RopeRegs r;
  const uint64_t keep = policy_evict_last();
  r.g2 = ldg_keep_u2(gamma + lane * 4, keep);
  r.c2 = ldg_keep_u2(cosp + lane * 4, keep);
  r.s2 = ldg_keep_u2(sinp + lane * 4, keep);
  return r;
}
__device__ __forceinline__ void head_norm_rope(float (&x)[4], const RopeRegs& rr, float eps, int lane) {
  const uint2 g2 = rr.g2, c2 = rr.c2, s2 = rr.s2;
  float ss = x[0] * x[0] + x[1] * x[1] + x[2] * x[2] + x[3] * x[3];
  ss = warp_sum(ss);
  const float rs = rsqrtf(ss * (1.f / kHeadDim) + eps);
  const float g[4] = {bf_lo(g2.x), bf_hi(g2.x), bf_lo(g2.y), bf_hi(g2.y)};
  const float c[4] = {bf_lo(c2.x), bf_hi(c2.x), bf_lo(c2.y), bf_hi(c2.y)};
  const float sn[4] = {bf_lo(s2.x), bf_hi(s2.x), bf_lo(s2.y), bf_hi(s2.y)};
  float y[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) y[i] = bf16r(bf16r(x[i] * rs) * g[i]);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float partner = __shfl_xor_sync(0xffffffffu, y[i], 16);
    const float rot = (lane < 16) ? -partner : partner;
    x[i] = bf16r(bf16r(y[i] * c[i]) + bf16r(rot * sn[i]));
  }
}

// a warp reads one 128-wide head (64 LL words, two per lane) of the qkv row
__device__ __forceinline__ void ll_head_wait(const LLWord* src, uint32_t ep, LLWord& a, LLWord& b, const LaunchParams& p, int phase) {
  ll_ld2(src, a, b);
  if (ep == 0) return;
  Spin spin;
  unsigned tries = 0;
  while (__any_sync(0xffffffffu, a.y != ep || b.y != ep)) {
    if (++tries > 4) __nanosleep(40);
    spin.tick(p, DE_LL_WAIT, phase, (int)ep);
    ll_ld2(src, a, b);
  }
}

constexpr int kGq = 2;  // q heads per kv head handled by one item (talker and predictor: 16 / 8)
constexpr int kAttnPre = 2;  // cached positions per half-warp whose K/V rows are requested before the q/k/v poll
constexpr int kAttnShort = 2 * kAttnPre * kConsumerWarps;  // 48 positions: at most kAttnPre per half-warp

// Scratch layout: qs fp32 [kGq][128] (1 KB) | fresh K,V rows bf16 [kMaxRows][2][128] (4 KB) | warp partials fp32 [16][kGq][kPartStride]
// Positions are dealt to half-warps (position a + 2*warp + half, stride 2 * kConsumerWarps); a lane owns 8 of the 128 dims (one 16-byte
// piece of the K row and of the V row).  Every half-warp keeps its own online softmax; the 32 partial states are merged in
// a fixed order, so the result is deterministic.
template <bool PROF>
__device__ __forceinline__ void attn_row(const Phase& ph, const LaunchParams& p, unsigned char* smem_base, const Group& gr, int r, int kvh, int sp,
                                      int nsplit, uint32_t ep, int pidx) {
  const Smem sm = carve_smem(smem_base, p);
  const StackRt& S = p.stacks[ph.stack];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int gq = S.nq / S.nkv;
  const int qb = ph.stack == ST_TALKER ? BUF_TQKV : BUF_PQKV, ab = ph.stack == ST_TALKER ? BUF_TATT : BUF_PATT;
  const LLWord* qkv = reinterpret_cast<const LLWord*>(p.bufs[qb]) + (size_t)gr.first_row * p.ld[qb];
  const int ldq = p.ld[qb];
  constexpr int HW = kHeadDim / 2;  // words per head
  const size_t head_base = (((size_t)ph.layer * S.n_slots + gr.slot) * S.nkv + kvh) * (size_t)S.max_pos * kHeadDim;
  bf16* Kc = S.kcache + head_base;
  bf16* Vc = S.vcache + head_base;
  const int pos = gr.pos0 + r;         // position of this query row; it attends to [n_pad, pos]
  // rows in front of n_pad are the left padding of a batched prompt: they attend to nothing (L <= 0) and publish zeros
  FQ3_ASSERT(pos >= 0 && pos < S.max_pos && gr.n_pad >= 0 && gq <= kGq, pidx, 200000 + pos);
  const int L = pos + 1 - gr.n_pad;
  FQ3_ASSERT(r >= 0 && r < kMaxRows && sp >= 0 && sp < nsplit && nsplit <= kMaxSplits, pidx, 210000 + sp);
  const int per = (L + nsplit - 1) / nsplit;
  const int a = gr.n_pad + sp * per;
  const int b = min(a + per, pos + 1);
  float* qs = reinterpret_cast<float*>(sm.scratch);
  uint4* fresh = reinterpret_cast<uint4*>(sm.scratch + 1024);  // [row][K|V][16 pieces of 16 bytes]
  float* wp = reinterpret_cast<float*>(sm.scratch + 1024 + 4096);
  const uint32_t ep_in = ep - 1;
  const int hw = lane >> 4, dl = lane & 15;
  if (PROF) prof_mark(p, pidx, 0);

  // -- step 0: request the first cached K/V rows of this half-warp before waiting for q (their addresses are known)
  uint4 kpre[kAttnPre], vpre[kAttnPre];
#pragma unroll
  for (int u = 0; u < kAttnPre; ++u) {
    const int i = a + warp * 2 + hw + u * 2 * kConsumerWarps;
    kpre[u] = make_uint4(0u, 0u, 0u, 0u);
    vpre[u] = kpre[u];
    if (i < b && i < gr.pos0) {
      kpre[u] = __ldcg(reinterpret_cast<const uint4*>(Kc + (size_t)i * kHeadDim) + dl);
      vpre[u] = __ldcg(reinterpret_cast<const uint4*>(Vc + (size_t)i * kHeadDim) + dl);
    }
  }
  cbar_sync();  // the scratch may still be read by the previous phase's finishing threads
  if (threadIdx.x < kGq * kAttnShort) wp[threadIdx.x] = -INFINITY;  // score slots of the short-range path

  // -- step 1: one warp per item: q heads (norm + rope, pre-scaled) to smem; K/V rows pos0..pos of this chunk that fall
  //    into [a, b) to the cache and to smem (norm + rope on K).
  for (int it = warp; it < gq + 2 * (r + 1); it += kConsumerWarps) {  // q heads, then (K row, V row) of every chunk row
    if (it < gq) {
      const int rp = min(max(pos + gr.rope_delta, 0), S.rope_len - 1);
      const LLWord* src = qkv + (size_t)r * ldq + (kvh * gq + it) * HW + lane * 2;
      const RopeRegs rr = rope_load(reinterpret_cast<const bf16*>(p.arena + (size_t)ph.g_off * 16), S.rope_cos + (size_t)rp * kHeadDim,
                                    S.rope_sin + (size_t)rp * kHeadDim, lane);
      LLWord w0, w1;
      ll_head_wait(src, ep_in, w0, w1, p, pidx);
      float x[4] = {bf_lo(w0.x), bf_hi(w0.x), bf_lo(w1.x), bf_hi(w1.x)};
      head_norm_rope(x, rr, S.eps, lane);
      const float scale = rsqrtf((float)kHeadDim);
      *reinterpret_cast<float4*>(qs + it * kHeadDim + lane * 4) = make_float4(x[0] * scale, x[1] * scale, x[2] * scale, x[3] * scale);
    } else {
      const int r2 = (it - gq) >> 1;
      const bool is_v = ((it - gq) & 1) != 0;
      const int kp = gr.pos0 + r2;
      if (kp >= a && kp < b) {
        const LLWord* row = qkv + (size_t)r2 * ldq;
        uint2* f = reinterpret_cast<uint2*>(fresh + (size_t)r2 * 32);
        if (is_v) {
          const LLWord* vsrc = row + (S.nq + S.nkv + kvh) * HW + lane * 2;
          LLWord v0, v1;
          ll_head_wait(vsrc, ep_in, v0, v1, p, pidx);
          const uint2 vv = make_uint2(v0.x, v1.x);
          *reinterpret_cast<uint2*>(Vc + (size_t)kp * kHeadDim + lane * 4) = vv;
          f[32 + lane] = vv;
        } else {
          const int rp = min(max(kp + gr.rope_delta, 0), S.rope_len - 1);
          const LLWord* ksrc = row + (S.nq + kvh) * HW + lane * 2;
          const RopeRegs rr = rope_load(reinterpret_cast<const bf16*>(p.arena + (size_t)ph.b_off * 16), S.rope_cos + (size_t)rp * kHeadDim,
                                        S.rope_sin + (size_t)rp * kHeadDim, lane);
          LLWord k0, k1;
          ll_head_wait(ksrc, ep_in, k0, k1, p, pidx);
          float x[4] = {bf_lo(k0.x), bf_hi(k0.x), bf_lo(k1.x), bf_hi(k1.x)};
          head_norm_rope(x, rr, S.eps, lane);
          const uint2 kk = make_uint2(pack_bf16x2(x[0], x[1]), pack_bf16x2(x[2], x[3]));
          *reinterpret_cast<uint2*>(Kc + (size_t)kp * kHeadDim + lane * 4) = kk;
          f[lane] = kk;
        }
      }
    }
  }
  cbar_sync();
  if (PROF) prof_mark(p, pidx, 1);

  float qr[kGq][8];
#pragma unroll
  for (int j = 0; j < kGq; ++j) {
    const float4 q0 = *reinterpret_cast<const float4*>(qs + j * kHeadDim + dl * 8);
    const float4 q1 = *reinterpret_cast<const float4*>(qs + j * kHeadDim + dl * 8 + 4);
    qr[j][0] = q0.x; qr[j][1] = q0.y; qr[j][2] = q0.z; qr[j][3] = q0.w;
    qr[j][4] = q1.x; qr[j][5] = q1.y; qr[j][6] = q1.z; qr[j][7] = q1.w;
  }
  // -- step 2 (short range, <= two positions per half-warp: every decode item, since a split never exceeds kSplitLen): two
  //    passes instead of an online softmax.  Every half-warp scores its positions and parks the V rows in shared memory;
  //    after ONE barrier the 128 output threads run max / exp / weighted sum over the <= 48 scores in position order.
  if (b - a <= kAttnShort) {
    float* sc = wp;                                                  // [kGq][kAttnShort]
    uint4* vst = reinterpret_cast<uint4*>(wp + kGq * kAttnShort);    // [kAttnShort][16 pieces]
    float sv[2][kGq];
    uint4 vv[2];
    int idx[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int i = a + warp * 2 + hw + u * 2 * kConsumerWarps;
      idx[u] = (i < b) ? i - a : -1;
      uint4 kk = make_uint4(0u, 0u, 0u, 0u);
      vv[u] = kk;
      if (i < b) {
        if (i >= gr.pos0) {
          const uint4* f = fresh + (size_t)(i - gr.pos0) * 32;
          kk = f[dl];
          vv[u] = f[16 + dl];
        } else {
          kk = kpre[u];
          vv[u] = vpre[u];
        }
      }
      const float k[8] = {bf_lo(kk.x), bf_hi(kk.x), bf_lo(kk.y), bf_hi(kk.y), bf_lo(kk.z), bf_hi(kk.z), bf_lo(kk.w), bf_hi(kk.w)};
#pragma unroll
      for (int j = 0; j < kGq; ++j) {
        float t = 0.f;
#pragma unroll
        for (int d = 0; d < 8; ++d) t = fmaf(qr[j][d], k[d], t);
        sv[u][j] = t;
      }
    }
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) {
#pragma unroll
      for (int u = 0; u < 2; ++u) {
#pragma unroll
        for (int j = 0; j < kGq; ++j) sv[u][j] += __shfl_xor_sync(0xffffffffu, sv[u][j], o);
      }
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      // every slot of the V staging area is written (zeros beyond the range): the output loop below reads whole groups of four
      vst[(warp * 2 + hw + u * 2 * kConsumerWarps) * 16 + dl] = vv[u];
      if (idx[u] >= 0 && dl < kGq) sc[dl * kAttnShort + idx[u]] = (dl == 0) ? sv[u][0] : sv[u][1];
    }
    if (PROF) prof_mark(p, pidx, 2);
    cbar_sync();
    // probabilities once per (head, position) — not once per output word: thread (j, i) finds the head's maximum and stores
    // exp(s_i - max); the scores beyond n are -inf (cleared at the top of the phase) and give 0
    float* pr = reinterpret_cast<float*>(vst + kAttnShort * 16);  // [kGq][kAttnShort] | maxima [kGq]
    const int n = b - a;
    const int n4 = (n + 3) >> 2;
    if (threadIdx.x < kGq * kAttnShort) {
      const int j = threadIdx.x / kAttnShort, i = threadIdx.x - j * kAttnShort;
      const float4* s4 = reinterpret_cast<const float4*>(sc + j * kAttnShort);
      float Mx = -INFINITY;
      for (int g4 = 0; g4 < n4; ++g4) {
        const float4 v = s4[g4];
        Mx = fmaxf(Mx, fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w)));
      }
      pr[threadIdx.x] = expf(sc[threadIdx.x] - Mx);
      if (i == 0) pr[kGq * kAttnShort + j] = Mx;
    }
    cbar_sync();
    if (threadIdx.x < gq * HW) {  // a thread owns one packed output word
      const int j = threadIdx.x / HW, wd = threadIdx.x - j * HW;
      const int qh = kvh * gq + j;
      const int row = gr.first_row + r;
      const float4* p4 = reinterpret_cast<const float4*>(pr + j * kAttnShort);
      const float Mx = pr[kGq * kAttnShort + j];
      const uint32_t* vw = reinterpret_cast<const uint32_t*>(vst) + wd;
      float Lsum = 0.f, O0 = 0.f, O1 = 0.f;
      // four positions per step, loads first (the slots beyond n hold probability 0 and a zero V row: they add nothing)
#pragma unroll 3
      for (int g4 = 0; g4 < n4; ++g4) {
        const float4 v = p4[g4];
        const uint32_t w0 = vw[(4 * g4) * HW], w1 = vw[(4 * g4 + 1) * HW], w2 = vw[(4 * g4 + 2) * HW], w3 = vw[(4 * g4 + 3) * HW];
        Lsum += v.x; O0 = fmaf(v.x, bf_lo(w0), O0); O1 = fmaf(v.x, bf_hi(w0), O1);
        Lsum += v.y; O0 = fmaf(v.y, bf_lo(w1), O0); O1 = fmaf(v.y, bf_hi(w1), O1);
        Lsum += v.z; O0 = fmaf(v.z, bf_lo(w2), O0); O1 = fmaf(v.z, bf_hi(w2), O1);
        Lsum += v.w; O0 = fmaf(v.w, bf_lo(w3), O0); O1 = fmaf(v.w, bf_hi(w3), O1);
      }
      if (nsplit == 1) {
        const float y0 = bf16r(Lsum > 0.f ? O0 / Lsum : 0.f), y1 = bf16r(Lsum > 0.f ? O1 / Lsum : 0.f);
        ll_st(reinterpret_cast<LLWord*>(p.bufs[ab]) + (size_t)row * p.ld[ab] + qh * HW + wd, pack_bf16x2(y0, y1), ep);
      } else {
        LLWord* dst = p.attn_part + (((size_t)row * S.nq + qh) * kMaxSplits + sp) * kPartStride;
        if (wd == 0) ll_st2(dst, __float_as_uint(Mx), __float_as_uint(Lsum), ep);
        ll_st2(dst + 4 + 2 * wd, __float_as_uint(O0), __float_as_uint(O1), ep);
      }
    }
    if (PROF) prof_mark(p, pidx, 3);
    return;
  }
  // -- step 2 (long range): online softmax per half-warp
  float m_run[kGq], l_run[kGq], acc[kGq][8];
#pragma unroll
  for (int j = 0; j < kGq; ++j) {
    m_run[j] = -INFINITY; l_run[j] = 0.f;
#pragma unroll
    for (int d = 0; d < 8; ++d) acc[j][d] = 0.f;
  }
  auto step = [&](const uint4& kk, const uint4& vv, bool valid) {
    const float k[8] = {bf_lo(kk.x), bf_hi(kk.x), bf_lo(kk.y), bf_hi(kk.y), bf_lo(kk.z), bf_hi(kk.z), bf_lo(kk.w), bf_hi(kk.w)};
    const float v[8] = {bf_lo(vv.x), bf_hi(vv.x), bf_lo(vv.y), bf_hi(vv.y), bf_lo(vv.z), bf_hi(vv.z), bf_lo(vv.w), bf_hi(vv.w)};
    float s[kGq];
#pragma unroll
    for (int j = 0; j < kGq; ++j) {
      float t = 0.f;
#pragma unroll
      for (int d = 0; d < 8; ++d) t = fmaf(qr[j][d], k[d], t);
      s[j] = t;
    }
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) {
#pragma unroll
      for (int j = 0; j < kGq; ++j) s[j] += __shfl_xor_sync(0xffffffffu, s[j], o);
    }
    if (valid) {
#pragma unroll
      for (int j = 0; j < kGq; ++j) {
        const float m_new = fmaxf(m_run[j], s[j]);
        const float corr = expf(m_run[j] - m_new);  // exp(-inf) = 0 on the first position
        const float pj = expf(s[j] - m_new);
        l_run[j] = l_run[j] * corr + pj;
#pragma unroll
        for (int d = 0; d < 8; ++d) acc[j][d] = fmaf(pj, v[d], acc[j][d] * corr);
        m_run[j] = m_new;
      }
    }
  };
  {
    // both halves of a warp run the same trip count (the shuffles name all 32 lanes); a half past the end skips the update
    int u = 0;
#pragma unroll 1
    for (int i0 = a + warp * 2; i0 < b; i0 += 2 * kConsumerWarps, ++u) {
      const int i = i0 + hw;
      const bool valid = i < b;
      uint4 kk = make_uint4(0u, 0u, 0u, 0u), vv = kk;
      if (valid) {
        if (i >= gr.pos0) {
          const uint4* f = fresh + (size_t)(i - gr.pos0) * 32;
          kk = f[dl];
          vv = f[16 + dl];
        } else if (u < kAttnPre) {
          kk = (u == 0) ? kpre[0] : kpre[1];
          vv = (u == 0) ? vpre[0] : vpre[1];
        } else {
          kk = __ldcg(reinterpret_cast<const uint4*>(Kc + (size_t)i * kHeadDim) + dl);
          vv = __ldcg(reinterpret_cast<const uint4*>(Vc + (size_t)i * kHeadDim) + dl);
        }
      }
      step(kk, vv, valid);
    }
  }
  // merge the two halves of a warp (fixed order: half 0, then half 1), then one state per warp and head to shared memory
#pragma unroll
  for (int j = 0; j < kGq; ++j) {
    const float m_o = __shfl_xor_sync(0xffffffffu, m_run[j], 16);
    const float l_o = __shfl_xor_sync(0xffffffffu, l_run[j], 16);
    const float m_new = fmaxf(m_run[j], m_o);
    const float c_s = (m_run[j] == -INFINITY) ? 0.f : expf(m_run[j] - m_new);
    const float c_o = (m_o == -INFINITY) ? 0.f : expf(m_o - m_new);
    float o8[8];
#pragma unroll
    for (int d = 0; d < 8; ++d) {
      const float a_o = __shfl_xor_sync(0xffffffffu, acc[j][d], 16);
      o8[d] = acc[j][d] * c_s + a_o * c_o;
    }
    const float l_new = l_run[j] * c_s + l_o * c_o;
    if (hw == 0) {
      float* w = wp + ((size_t)warp * kGq + j) * kPartStride;
      if (dl == 0) { w[0] = m_new; w[1] = l_new; }
      *reinterpret_cast<float4*>(w + 4 + dl * 8) = make_float4(o8[0], o8[1], o8[2], o8[3]);
      *reinterpret_cast<float4*>(w + 8 + dl * 8) = make_float4(o8[4], o8[5], o8[6], o8[7]);
    }
  }
  if (PROF) prof_mark(p, pidx, 2);
  cbar_sync();
  if (threadIdx.x < gq * HW) {  // a thread owns one packed output word
    const int j = threadIdx.x / HW, wd = threadIdx.x - j * HW;
    const int qh = kvh * gq + j;
    const int row = gr.first_row + r;
    const int nw = min(kConsumerWarps, (b - a + 1) >> 1);  // warps that saw at least one position
    float Mx = -INFINITY;
    for (int w = 0; w < nw; ++w) Mx = fmaxf(Mx, wp[((size_t)w * kGq + j) * kPartStride]);
    float Lsum = 0.f, O0 = 0.f, O1 = 0.f;
    for (int w = 0; w < nw; ++w) {
      const float* q = wp + ((size_t)w * kGq + j) * kPartStride;
      const float f = (q[0] == -INFINITY) ? 0.f : expf(q[0] - Mx);
      Lsum += q[1] * f;
      const float2 o2 = *reinterpret_cast<const float2*>(q + 4 + 2 * wd);
      O0 += o2.x * f; O1 += o2.y * f;
    }
    if (nsplit == 1) {
      const float y0 = bf16r(Lsum > 0.f ? O0 / Lsum : 0.f), y1 = bf16r(Lsum > 0.f ? O1 / Lsum : 0.f);
      ll_st(reinterpret_cast<LLWord*>(p.bufs[ab]) + (size_t)row * p.ld[ab] + qh * HW + wd, pack_bf16x2(y0, y1), ep);
    } else {
      LLWord* dst = p.attn_part + (((size_t)row * S.nq + qh) * kMaxSplits + sp) * kPartStride;
      if (wd == 0) ll_st2(dst, __float_as_uint(Mx), __float_as_uint(Lsum), ep);
      ll_st2(dst + 4 + 2 * wd, __float_as_uint(O0), __float_as_uint(O1), ep);
    }
  }
  if (PROF) prof_mark(p, pidx, 3);
}

// One step of the split-KV merge: fold the partial state (ms, ls, a0, a1) of the next split into the running one.  Shared by the
// cross-CTA combine and by the single-CTA multi-split item of the wide program, so both add in the same order with the same
// expressions (the batch must not change a stream's arithmetic).
__device__ __forceinline__ void combine_step(float& Mx, float& Lsum, float& O0, float& O1, float ms, float ls, float a0, float a1) {
  if (ms != -INFINITY) {
    const float m_new = fmaxf(Mx, ms);
    const float c_old = (Mx == -INFINITY) ? 0.f : expf(Mx - m_new);
    const float c_new = expf(ms - m_new);
    Lsum = Lsum * c_old + ls * c_new;
    O0 = O0 * c_old + a0 * c_new;
    O1 = O1 * c_old + a1 * c_new;
    Mx = m_new;
  }
}

// Split-KV combine (contexts beyond kSplitLen): the CTA of split 0 polls the partials of all splits (its own included)
// and merges them in split order.
__device__ __forceinline__ void attn_combine(const Phase& ph, const LaunchParams& p, const Group& gr, int r, int kvh, int nsplit, uint32_t ep,
                                          int pidx) {
  const StackRt& S = p.stacks[ph.stack];
  const int gq = S.nq / S.nkv;
  const int ab = ph.stack == ST_TALKER ? BUF_TATT : BUF_PATT;
  constexpr int HW = kHeadDim / 2;
  if (threadIdx.x < gq * HW) {
    const int j = threadIdx.x / HW, wd = threadIdx.x - j * HW;
    const int qh = kvh * gq + j;
    const int row = gr.first_row + r;
    const LLWord* src = p.attn_part + (((size_t)row * S.nq + qh) * kMaxSplits) * kPartStride;
    // four splits at a time: issue the loads first (the round trips overlap), then validate / re-poll and fold them into
    // the running state in split order
    float Mx = -INFINITY, Lsum = 0.f, O0 = 0.f, O1 = 0.f;
#pragma unroll 1
    for (int s0 = 0; s0 < nsplit; s0 += 4) {
      LLWord wm[4], wl[4], wa[4], wb[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (s0 + u < nsplit) {
          const LLWord* q = src + (size_t)(s0 + u) * kPartStride;
          ll_ld2(q, wm[u], wl[u]);
          ll_ld2(q + 4 + 2 * wd, wa[u], wb[u]);
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (s0 + u < nsplit) {
          const LLWord* q = src + (size_t)(s0 + u) * kPartStride;
          const float ms = __uint_as_float(ll_check(wm[u], q, ep, p, pidx));
          const float ls = __uint_as_float(ll_check(wl[u], q + 1, ep, p, pidx));
          const float a0 = __uint_as_float(ll_check(wa[u], q + 4 + 2 * wd, ep, p, pidx));
          const float a1 = __uint_as_float(ll_check(wb[u], q + 5 + 2 * wd, ep, p, pidx));
          combine_step(Mx, Lsum, O0, O1, ms, ls, a0, a1);
        }
      }
    }
    const float y0 = bf16r(Lsum > 0.f ? O0 / Lsum : 0.f), y1 = bf16r(Lsum > 0.f ? O1 / Lsum : 0.f);
    ll_st(reinterpret_cast<LLWord*>(p.bufs[ab]) + (size_t)row * p.ld[ab] + qh * HW + wd, pack_bf16x2(y0, y1), ep);
  }
}

// Wide program, contexts beyond one split: ONE CTA takes all splits of a (stream, kv head) in turn — same split boundaries, same
// per-split two-pass softmax, same merge order as the cross-CTA scheme (attn_row + attn_combine), so the result is bit-identical
// to the single-stream run; but q is normalised once, nothing travels through global memory between the splits, and the K/V rows
// of split s + 1 are requested while split s is being reduced.  Decode rows only (one row per stream), splits of <= kAttnShort.
__device__ __forceinline__ void attn_item_multi(const Phase& ph, const LaunchParams& p, unsigned char* smem_base, const Group& gr, int kvh, int nsplit,
                                                uint32_t ep, int pidx) {
  const Smem sm = carve_smem(smem_base, p);
  const StackRt& S = p.stacks[ph.stack];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int gq = S.nq / S.nkv;
  const int qb = ph.stack == ST_TALKER ? BUF_TQKV : BUF_PQKV, ab = ph.stack == ST_TALKER ? BUF_TATT : BUF_PATT;
  const LLWord* qkv = reinterpret_cast<const LLWord*>(p.bufs[qb]) + (size_t)gr.first_row * p.ld[qb];
  constexpr int HW = kHeadDim / 2;
  const size_t head_base = (((size_t)ph.layer * S.n_slots + gr.slot) * S.nkv + kvh) * (size_t)S.max_pos * kHeadDim;
  bf16* Kc = S.kcache + head_base;
  bf16* Vc = S.vcache + head_base;
  const int pos = gr.pos0;
  const int L = pos + 1 - gr.n_pad;
  const int per = (L + nsplit - 1) / nsplit;
  FQ3_ASSERT(pos >= 0 && pos < S.max_pos && per <= kAttnShort && nsplit <= kMaxSplits, pidx, 220000 + pos);
  float* qs = reinterpret_cast<float*>(sm.scratch);
  uint4* fresh = reinterpret_cast<uint4*>(sm.scratch + 1024);
  float* wp = reinterpret_cast<float*>(sm.scratch + 1024 + 4096);
  float* sc = wp;                                                  // [kGq][kAttnShort]
  uint4* vst = reinterpret_cast<uint4*>(wp + kGq * kAttnShort);    // [kAttnShort][16 pieces]
  float* pr = reinterpret_cast<float*>(vst + kAttnShort * 16);     // [kGq][kAttnShort] | maxima [kGq]
  const uint32_t ep_in = ep - 1;
  const int hw = lane >> 4, dl = lane & 15;
  uint4 kpre[kAttnPre], vpre[kAttnPre];
  auto request = [&](int sp) {  // the cached K/V rows of split sp that this half-warp scores
    const int a = gr.n_pad + sp * per, b = min(a + per, pos + 1);
#pragma unroll
    for (int u = 0; u < kAttnPre; ++u) {
      const int i = a + warp * 2 + hw + u * 2 * kConsumerWarps;
      kpre[u] = make_uint4(0u, 0u, 0u, 0u);
      vpre[u] = kpre[u];
      if (i < b && i < pos) {
        kpre[u] = __ldcg(reinterpret_cast<const uint4*>(Kc + (size_t)i * kHeadDim) + dl);
        vpre[u] = __ldcg(reinterpret_cast<const uint4*>(Vc + (size_t)i * kHeadDim) + dl);
      }
    }
  };
  long long tq = (FQ3_WIDE_PROF && p.prof) ? clock64() : 0ll;
  request(0);
  cbar_sync();  // the scratch may still be read by the previous phase's finishing threads
  prof_acc(p, 12, tq);
  // q heads (norm + rope, pre-scaled) and the fresh K / V row of this position: same code as attn_row, one warp each
  for (int it = warp; it < gq + 2; it += kConsumerWarps) {
    if (it < gq) {
      const int rp = min(max(pos + gr.rope_delta, 0), S.rope_len - 1);
      const LLWord* src = qkv + (kvh * gq + it) * HW + lane * 2;
      const RopeRegs rr = rope_load(reinterpret_cast<const bf16*>(p.arena + (size_t)ph.g_off * 16), S.rope_cos + (size_t)rp * kHeadDim,
                                    S.rope_sin + (size_t)rp * kHeadDim, lane);
      LLWord w0, w1;
      ll_head_wait(src, ep_in, w0, w1, p, pidx);
      float x[4] = {bf_lo(w0.x), bf_hi(w0.x), bf_lo(w1.x), bf_hi(w1.x)};
      head_norm_rope(x, rr, S.eps, lane);
      const float scale = rsqrtf((float)kHeadDim);
      *reinterpret_cast<float4*>(qs + it * kHeadDim + lane * 4) = make_float4(x[0] * scale, x[1] * scale, x[2] * scale, x[3] * scale);
    } else {
      const bool is_v = (it - gq) != 0;
      uint2* f = reinterpret_cast<uint2*>(fresh);
      if (is_v) {
        const LLWord* vsrc = qkv + (S.nq + S.nkv + kvh) * HW + lane * 2;
        LLWord v0, v1;
        ll_head_wait(vsrc, ep_in, v0, v1, p, pidx);
        const uint2 vv = make_uint2(v0.x, v1.x);
        *reinterpret_cast<uint2*>(Vc + (size_t)pos * kHeadDim + lane * 4) = vv;
        f[32 + lane] = vv;
      } else {
        const int rp = min(max(pos + gr.rope_delta, 0), S.rope_len - 1);
        const LLWord* ksrc = qkv + (S.nq + kvh) * HW + lane * 2;
        const RopeRegs rr = rope_load(reinterpret_cast<const bf16*>(p.arena + (size_t)ph.b_off * 16), S.rope_cos + (size_t)rp * kHeadDim,
                                      S.rope_sin + (size_t)rp * kHeadDim, lane);
        LLWord k0, k1;
        ll_head_wait(ksrc, ep_in, k0, k1, p, pidx);
        float x[4] = {bf_lo(k0.x), bf_hi(k0.x), bf_lo(k1.x), bf_hi(k1.x)};
        head_norm_rope(x, rr, S.eps, lane);
        const uint2 kk = make_uint2(pack_bf16x2(x[0], x[1]), pack_bf16x2(x[2], x[3]));
        *reinterpret_cast<uint2*>(Kc + (size_t)pos * kHeadDim + lane * 4) = kk;
        f[lane] = kk;
      }
    }
  }
  cbar_sync();
  float qr[kGq][8];
#pragma unroll
  for (int j = 0; j < kGq; ++j) {
    const float4 q0 = *reinterpret_cast<const float4*>(qs + j * kHeadDim + dl * 8);
    const float4 q1 = *reinterpret_cast<const float4*>(qs + j * kHeadDim + dl * 8 + 4);
    qr[j][0] = q0.x; qr[j][1] = q0.y; qr[j][2] = q0.z; qr[j][3] = q0.w;
    qr[j][4] = q1.x; qr[j][5] = q1.y; qr[j][6] = q1.z; qr[j][7] = q1.w;
  }
  float Mx = -INFINITY, Lsum = 0.f, O0 = 0.f, O1 = 0.f;  // running state of an output thread (one packed output word)
  const int oj = threadIdx.x / HW, owd = threadIdx.x - oj * HW;
  prof_acc(p, 13, tq);
#pragma unroll 1
  for (int sp = 0; sp < nsplit; ++sp) {
    const int a = gr.n_pad + sp * per, b = min(a + per, pos + 1);
    const int n = b - a, n4 = (n + 3) >> 2;
    // every half-warp scores its (<= 2) positions of this split and parks their V rows; slots beyond n get -inf
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int idx = warp * 2 + hw + u * 2 * kConsumerWarps;
      const int i = a + idx;
      uint4 kk = make_uint4(0u, 0u, 0u, 0u), vv = kk;
      if (i < b) {
        if (i >= pos) { kk = fresh[dl]; vv = fresh[16 + dl]; }
        else { kk = kpre[u]; vv = vpre[u]; }
      }
      const float k[8] = {bf_lo(kk.x), bf_hi(kk.x), bf_lo(kk.y), bf_hi(kk.y), bf_lo(kk.z), bf_hi(kk.z), bf_lo(kk.w), bf_hi(kk.w)};
      float sv[kGq];
#pragma unroll
      for (int j = 0; j < kGq; ++j) {
        float t = 0.f;
#pragma unroll
        for (int d = 0; d < 8; ++d) t = fmaf(qr[j][d], k[d], t);
        sv[j] = t;
      }
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) {
#pragma unroll
        for (int j = 0; j < kGq; ++j) sv[j] += __shfl_xor_sync(0xffffffffu, sv[j], o);
      }
      vst[idx * 16 + dl] = vv;  // zeros beyond the range
      if (dl < kGq) sc[dl * kAttnShort + idx] = (i < b) ? ((dl == 0) ? sv[0] : sv[1]) : -INFINITY;
    }
    if (sp + 1 < nsplit) request(sp + 1);
    prof_acc(p, 14, tq);
    cbar_sync();
    prof_acc(p, 15, tq);
    if (threadIdx.x < kGq * kAttnShort) {
      const int j = threadIdx.x / kAttnShort, i = threadIdx.x - j * kAttnShort;
      const float4* s4 = reinterpret_cast<const float4*>(sc + j * kAttnShort);
      float m = -INFINITY;
      for (int g4 = 0; g4 < n4; ++g4) {
        const float4 v = s4[g4];
        m = fmaxf(m, fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w)));
      }
      pr[threadIdx.x] = expf(sc[threadIdx.x] - m);
      if (i == 0) pr[kGq * kAttnShort + j] = m;
    }
    prof_acc(p, 18, tq);
    cbar_sync();
    prof_acc(p, 19, tq);
    if (threadIdx.x < gq * HW) {
      const float4* p4 = reinterpret_cast<const float4*>(pr + oj * kAttnShort);
      const float ms = pr[kGq * kAttnShort + oj];
      const uint32_t* vw = reinterpret_cast<const uint32_t*>(vst) + owd;
      float ls = 0.f, a0 = 0.f, a1 = 0.f;
#pragma unroll 3
      for (int g4 = 0; g4 < n4; ++g4) {
        const float4 v = p4[g4];
        const uint32_t w0 = vw[(4 * g4) * HW], w1 = vw[(4 * g4 + 1) * HW], w2 = vw[(4 * g4 + 2) * HW], w3 = vw[(4 * g4 + 3) * HW];
        ls += v.x; a0 = fmaf(v.x, bf_lo(w0), a0); a1 = fmaf(v.x, bf_hi(w0), a1);
        ls += v.y; a0 = fmaf(v.y, bf_lo(w1), a0); a1 = fmaf(v.y, bf_hi(w1), a1);
        ls += v.z; a0 = fmaf(v.z, bf_lo(w2), a0); a1 = fmaf(v.z, bf_hi(w2), a1);
        ls += v.w; a0 = fmaf(v.w, bf_lo(w3), a0); a1 = fmaf(v.w, bf_hi(w3), a1);
      }
      combine_step(Mx, Lsum, O0, O1, ms, ls, a0, a1);
    }
    prof_acc(p, 16, tq);
    cbar_sync();  // the next split overwrites the scores, the parked V rows and the probabilities
    prof_acc(p, 17, tq);
  }
  if (threadIdx.x < gq * HW) {
    const int qh = kvh * gq + oj;
    const float y0 = bf16r(Lsum > 0.f ? O0 / Lsum : 0.f), y1 = bf16r(Lsum > 0.f ? O1 / Lsum : 0.f);
    ll_st(reinterpret_cast<LLWord*>(p.bufs[ab]) + (size_t)gr.first_row * p.ld[ab] + qh * HW + owd, pack_bf16x2(y0, y1), ep);
  }
}


template <bool PROF, bool WIDE>
__device__ __forceinline__ void attn_phase(const Phase& ph, const LaunchParams& p, unsigned char* smem_base, uint32_t ep, int pidx,
                                           const int* frame_pos) {
  const StackRt& S = p.stacks[ph.stack];
  const int G = gridDim.x, cta = blockIdx.x;
  const int ng = num_groups(p);
  if (ng == 1 && p.mode != MODE_PREFILL && !(ph.flags & F_ROWS2)) {
    // one stream, one row (every decode phase except predictor pass 0): items = kv heads x splits, spread over the grid
    const Group gr = get_group(ph, p, 0, frame_pos);
    const int cap = max(1, min(small_div(G, S.nkv), kMaxSplits));
    const int nsplit = num_splits(gr.pos0 + 1 - gr.n_pad, cap);
    const int total = S.nkv * nsplit;
    const int stride = max(1, small_div(G, total));
    const int q = small_div(cta, stride);
    if (cta == q * stride && q < total) {
      const int kvh = small_div(q, nsplit), sp = q - kvh * nsplit;
      attn_row<PROF>(ph, p, smem_base, gr, 0, kvh, sp, nsplit, ep, pidx);
      if (nsplit > 1 && sp == 0) attn_combine(ph, p, gr, 0, kvh, nsplit, ep, pidx);
    }
    return;
  }
  // The split structure of a row depends on its context length alone (the same cap as the single-stream case above), so a
  // stream's attention arithmetic does not change with the number of streams in the launch; with more items than CTAs a
  // CTA takes several, and every CTA publishes all its partials before it waits for anybody else's (two passes).
  const int cap = max(1, min(small_div(G, S.nkv), kMaxSplits));
  if constexpr (WIDE) {
    if (p.mode != MODE_PREFILL && !(ph.flags & F_ROWS2)) {
      // decode rows of the wide program: exactly one item per (stream, kv head) as long as every context fits the two-pass path
      // (nsplit = ceil(L / 48) <= cap) — item -> (stream, kv head) is a division, not a walk over the streams
      int Lmax = 0;
      for (int g = 0; g < ng; ++g) {
        const Group gr = get_group(ph, p, g, frame_pos);
        Lmax = max(Lmax, gr.pos0 + 1 - gr.n_pad);
      }
      if (Lmax <= kAttnShort * cap) {
        const int total = ng * S.nkv;
        const int stride = (total <= G) ? small_div(G, total) : 1;
        int first = cta, step = G;
        if (stride > 1) {
          const int q = small_div(cta, stride);
          first = (cta - q * stride == 0 && q < total) ? q : total;
          step = total;
        }
#pragma unroll 1
        for (int item = first; item < total; item += step) {
          const int g = small_div(item, S.nkv), kvh = item - g * S.nkv;
          const Group gr = get_group(ph, p, g, frame_pos);
          const int nsplit = num_splits(gr.pos0 + 1 - gr.n_pad, cap);
          if (nsplit == 1) attn_row<PROF>(ph, p, smem_base, gr, 0, kvh, 0, 1, ep, pidx);
          else attn_item_multi(ph, p, smem_base, gr, kvh, nsplit, ep, pidx);
        }
        return;
      }
    }
  }
  // wide program: a row whose splits fit the two-pass path is ONE item per kv head (attn_item_multi walks its splits)
  auto row_items = [&](const Group& gr, int r, int& nsplit, bool& multi) {
    const int L = gr.pos0 + r + 1 - gr.n_pad;
    nsplit = num_splits(L, cap);
    multi = WIDE && p.mode != MODE_PREFILL && nsplit > 1 && (L + nsplit - 1) / nsplit <= kAttnShort;
    return S.nkv * (multi ? 1 : nsplit);
  };
  int total = 0;
  for (int g = 0; g < ng; ++g) {
    const Group gr = get_group(ph, p, g, frame_pos);
    for (int r = 0; r < gr.nrows; ++r) {
      int ns; bool mu;
      total += row_items(gr, r, ns, mu);
    }
  }
  // item -> CTA: spread the items over the whole grid (stride) so concurrent items sit on distant SMs
  const int stride = (total <= G) ? small_div(G, total) : 1;
  int first, step;
  if (stride > 1) {
    const int q = small_div(cta, stride);
    first = (cta - q * stride == 0 && q < total) ? q : total;
    step = total;
  } else {
    first = cta;
    step = G;
  }
#pragma unroll 1
  for (int pass = 0; pass < 2; ++pass) {
#pragma unroll 1
    for (int item = first; item < total; item += step) {
      int base = 0;
      bool found = false;
      for (int g = 0; g < ng && !found; ++g) {
        const Group gr = get_group(ph, p, g, frame_pos);
        for (int r = 0; r < gr.nrows; ++r) {
          int nsplit; bool multi;
          const int nitems = row_items(gr, r, nsplit, multi);
          if (item < base + nitems) {
            const int it = item - base;
            if (multi) {
              if constexpr (WIDE) {
                if (pass == 0) attn_item_multi(ph, p, smem_base, gr, it, nsplit, ep, pidx);
              }
            } else {
              const int kvh = small_div(it, nsplit), sp = it - kvh * nsplit;
              if (pass == 0) attn_row<PROF>(ph, p, smem_base, gr, r, kvh, sp, nsplit, ep, pidx);
              else if (nsplit > 1 && sp == 0) attn_combine(ph, p, gr, r, kvh, nsplit, ep, pidx);
            }
            found = true;
            break;
          }
          base += nitems;
        }
      }
    }
  }
}

// =================================================================================================
// Sampling (sampling.py:10-66) — block-wide, 512 consumer threads, one stream per CTA
// =================================================================================================
__device__ __forceinline__ uint32_t f2key(float f) {
  uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key2f(uint32_t k) {
  uint32_t u = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
  return __uint_as_float(u);
}
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
  return c;
}

struct SampleScratch {
  float* sl;       // [V] working logits
  unsigned* hist;  // [256]
  float* redf;     // [32]
  int* redi;       // [32]
};
__device__ __forceinline__ SampleScratch sample_scratch(unsigned char* scratch) {
  SampleScratch s;
  s.sl = reinterpret_cast<float*>(scratch);
  s.hist = reinterpret_cast<unsigned*>(scratch + 20 * 1024);
  s.redf = reinterpret_cast<float*>(scratch + 21 * 1024);
  s.redi = reinterpret_cast<int*>(scratch + 21 * 1024 + 256);
  return s;
}

__device__ __noinline__ float block_sum(float v, float* red) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  v = warp_sum(v);
  cbar_sync();
  if (lane == 0) red[warp] = v;
  cbar_sync();
  float t = 0.f;
#pragma unroll
  for (int w = 0; w < kConsumerWarps; ++w) t += red[w];
  return t;
}
__device__ __noinline__ float block_max(float v, float* red) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  v = warp_max(v);
  cbar_sync();
  if (lane == 0) red[warp] = v;
  cbar_sync();
  float t = -INFINITY;
#pragma unroll
  for (int w = 0; w < kConsumerWarps; ++w) t = fmaxf(t, red[w]);
  return t;
}
// argmax with lowest-index tie-break (torch.argmax on a 1-row tensor)
__device__ __noinline__ int block_argmax(const float* sl, int V, float* redf, int* redi, float* out_val) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float bv = -INFINITY;
  int bi = 0x7fffffff;
  for (int i = threadIdx.x; i < V; i += kConsumerThreads) {
    const float x = sl[i];
    if (x > bv || (x == bv && i < bi)) { bv = x; bi = i; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
  }
  cbar_sync();
  if (lane == 0) { redf[warp] = bv; redi[warp] = bi; }
  cbar_sync();
  bv = redf[0]; bi = redi[0];
#pragma unroll
  for (int w = 1; w < kConsumerWarps; ++w) {
    const float ov = redf[w]; const int oi = redi[w];
    if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
  }
  if (out_val) *out_val = bv;
  return bi == 0x7fffffff ? 0 : bi;
}

// k-th largest value (counting multiplicity) by 4-pass radix select on order-preserving keys.
__device__ __noinline__ float kth_largest(const float* sl, int V, int k, unsigned* hist, int* redi) {
  uint32_t prefix = 0;
  int krem = k;
  const int lane = threadIdx.x & 31;
  for (int pass = 0; pass < 4; ++pass) {
    const int shift = 24 - 8 * pass;
    cbar_sync();
    if (threadIdx.x < 256) hist[threadIdx.x] = 0;
    cbar_sync();
    for (int i = threadIdx.x; i < V; i += kConsumerThreads) {
      const uint32_t key = f2key(sl[i]);
      const bool match = (pass == 0) || ((key >> (shift + 8)) == (prefix >> (shift + 8)));
      if (match) atomicAdd(&hist[(key >> shift) & 0xffu], 1u);
    }
    cbar_sync();
    if (threadIdx.x < 32) {
      // lane l covers bins [255-8l-7, 255-8l], scanned from the top
      unsigned s = 0;
#pragma unroll
      for (int t = 0; t < 8; ++t) s += hist[255 - 8 * lane - t];
      unsigned incl = s;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned n = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += n;
      }
      const unsigned ballot = __ballot_sync(0xffffffffu, incl >= (unsigned)krem);
      const int sel = __ffs(ballot) - 1;
      if (lane == sel) {
        unsigned above = incl - s;
        int digit = 255 - 8 * lane;
        for (int t = 0; t < 8; ++t) {
          const unsigned c = hist[255 - 8 * lane - t];
          if (above + c >= (unsigned)krem) { digit = 255 - 8 * lane - t; break; }
          above += c;
        }
        redi[0] = digit;
        redi[1] = krem - (int)above;
      }
    }
    cbar_sync();
    prefix |= ((uint32_t)redi[0]) << shift;
    krem = redi[1];
  }
  cbar_sync();
  return key2f(prefix);
}

struct SampleArgs {
  int V;
  int do_sample, top_k;
  float top_p, temperature, rep_pen;
  const uint8_t* seen;  // may be null
  int suppress_start;   // ids >= this (except eos) are masked; V => none
  int eos;
  int suppress_eos;
  int round_bf16;       // logits came from a bf16 tensor: round every intermediate like the reference's bf16 ops
  unsigned long long seed, draw;
  const bf16* next_emb;  // optional: embedding table whose row [token] is read right after the draw (L2 prefetch of the candidates)
  int emb_row_bytes;
};

// logits arrive either as LL words (ll != null, epoch ep) or as a plain fp32 array.
__device__ __noinline__ int sample_row(const float* logits_g, const LLWord* ll, uint32_t ep, const LaunchParams* lp, int pidx,
                          const SampleArgs& a, const SampleScratch& sc) {
  float* sl = sc.sl;
  const int V = a.V;
  // 1. load + repetition penalty (sampling.py:22-29, before suppression) + suppression + temperature
  auto prep = [&](int i, float x) {
    if (a.seen && a.rep_pen != 1.0f && __ldcg(a.seen + i)) {
      x = (x > 0.f) ? x / a.rep_pen : x * a.rep_pen;
      if (a.round_bf16) x = bf16r(x);
    }
    if (i >= a.suppress_start && i != a.eos) x = -INFINITY;
    if (a.suppress_eos && i == a.eos) x = -INFINITY;
    if (a.do_sample) {
      x = x / a.temperature;
      if (a.round_bf16) x = bf16r(x);
    }
    sl[i] = x + 0.0f;  // -0 -> +0: the top-p step orders by key, and torch's sort puts both zeros in one tie group
  };
  if (ll) {
    // packed words: word w carries logits 2w, 2w+1 (bf16-rounded by the head phase, like the reference's bf16 Linear)
    constexpr int kLw = (kMaxVocab / 2 + kConsumerThreads - 1) / kConsumerThreads;  // 6
    const int Vw = V >> 1;
    LLWord lw[kLw];
    Spin spin;
    unsigned tries = 0;
    bool bad;
    do {
      bad = false;
#pragma unroll
      for (int j = 0; j < kLw; ++j) {
        const int wi = threadIdx.x + j * kConsumerThreads;
        if (wi < Vw) {
          lw[j] = ll_ld(ll + wi);
          bad |= (lw[j].y != ep);
        }
      }
      if (ep == 0) break;
      if (bad) {
        if (++tries > 4) __nanosleep(40);
        spin.tick(*lp, DE_LL_WAIT, pidx, (int)ep);
      }
    } while (bad);
#pragma unroll
    for (int j = 0; j < kLw; ++j) {
      const int wi = threadIdx.x + j * kConsumerThreads;
      if (wi < Vw) {
        prep(2 * wi, bf_lo(lw[j].x));
        prep(2 * wi + 1, bf_hi(lw[j].x));
      }
    }
  } else {
    for (int i = threadIdx.x; i < V; i += kConsumerThreads) prep(i, __ldcg(logits_g + i));
  }
  cbar_sync();
  float vmax;
  const int imax = block_argmax(sl, V, sc.redf, sc.redi, &vmax);
  if (!a.do_sample) return imax;
  // 2. top-k: keep x >= k-th largest (ties survive, sampling.py:54-56)
  if (a.top_k > 0 && a.top_k < V) {
    const float thr = kth_largest(sl, V, a.top_k, sc.hist, sc.redi);
    for (int i = threadIdx.x; i < V; i += kConsumerThreads)
      if (sl[i] < thr) sl[i] = -INFINITY;
    cbar_sync();
  }
  // 3. top-p on the sorted distribution (sampling.py:57-65): rank j is dropped iff cum_j > top_p and j > 0
  if (a.top_p < 1.0f) {
    float loc = 0.f;
    for (int i = threadIdx.x; i < V; i += kConsumerThreads) loc += expf(sl[i] - vmax);
    const float total = block_sum(loc, sc.redf);
    // fp32: unnormalised masses against top_p * total.  bf16 (the reference's softmax and cumsum of a bf16 tensor, compared
    // with bf16(top_p)): every probability rounded to bf16, and the prefix kept while it would round to at most bf16(top_p),
    // i.e. up to the midpoint P between bf16(top_p) and the next bf16 value.  A prefix exactly on P rounds to the even one of
    // the two, so it is kept iff bf16(top_p) is even (`strict` otherwise).  Both masses grow with the key.
    const bool bf = a.round_bf16;
    auto mass = [&](float x) {
      const float e = expf(x - vmax);
      return bf ? bf16r(e / total) : e;
    };
    float P = a.top_p * total;
    bool strict = false;
    if (bf) {
      const uint32_t b = __float_as_uint(bf16r(a.top_p));
      P = 0.5f * (__uint_as_float(b) + __uint_as_float(b + 0x10000u));
      strict = (b & 0x10000u) != 0;
    }
    uint32_t lo = 0u, hi = 0xffffffffu;  // smallest key t with mass(key >= t) <= P (< P when strict)
    for (int it = 0; it < 32; ++it) {
      const uint32_t mid = lo + ((hi - lo) >> 1);
      float msum = 0.f;
      for (int i = threadIdx.x; i < V; i += kConsumerThreads) {
        const float x = sl[i];
        if (f2key(x) >= mid) msum += mass(x);
      }
      msum = block_sum(msum, sc.redf);
      if (msum < P || (!strict && msum == P)) hi = mid; else lo = mid + 1;
    }
    const uint32_t tkey = hi;
    // boundary value v* = largest key below tkey; its first j ties (index order) may still fit under P
    uint32_t bk = 0;
    for (int i = threadIdx.x; i < V; i += kConsumerThreads) {
      const uint32_t k = f2key(sl[i]);
      if (k < tkey && k > bk) bk = k;
    }
    const float bval = block_max(key2f(bk), sc.redf);
    float above = 0.f;
    for (int i = threadIdx.x; i < V; i += kConsumerThreads)
      if (f2key(sl[i]) >= tkey) above += mass(sl[i]);
    above = block_sum(above, sc.redf);
    int keep_ties = 0;
    if (bval > -INFINITY) {
      const float pe = mass(bval);
      keep_ties = (int)floorf((P - above) / pe);
      if (strict && above + (float)keep_ties * pe >= P) --keep_ties;  // bf16 masses: these sums are exact
      if (keep_ties < 0) keep_ties = 0;
    }
    const int seg = (V + kConsumerThreads - 1) / kConsumerThreads;
    const int i0 = threadIdx.x * seg, i1 = min(V, i0 + seg);
    int cnt = 0;
    for (int i = i0; i < i1; ++i) cnt += (sl[i] == bval) ? 1 : 0;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int n = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += n;
    }
    cbar_sync();
    if (lane == 31) sc.redi[warp] = incl;
    cbar_sync();
    int base = 0;
    for (int w = 0; w < warp; ++w) base += sc.redi[w];
    int rank = base + incl - cnt;
    for (int i = i0; i < i1; ++i) {
      const float x = sl[i];
      if (f2key(x) >= tkey) continue;
      if (x == bval && bval > -INFINITY) {
        if (rank < keep_ties) { ++rank; continue; }
        ++rank;
      }
      if (i != imax) sl[i] = -INFINITY;
    }
    cbar_sync();
  }
  // 4. multinomial(softmax) by inverse CDF on one Philox uniform
  const int seg = (V + kConsumerThreads - 1) / kConsumerThreads;
  const int i0 = threadIdx.x * seg, i1 = min(V, i0 + seg);
  float loc = 0.f;
  for (int i = i0; i < i1; ++i) loc += expf(sl[i] - vmax);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float incl = loc;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float n = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += n;
  }
  cbar_sync();
  if (lane == 31) sc.redf[warp] = incl;
  if (threadIdx.x == 0) sc.redi[16] = 0x7fffffff;
  cbar_sync();
  float base = 0.f, total = 0.f;
  for (int w = 0; w < kConsumerWarps; ++w) {
    if (w < warp) base += sc.redf[w];
    total += sc.redf[w];
  }
  const uint4 rnd = philox4x32_10(make_uint4((uint32_t)a.draw, (uint32_t)(a.draw >> 32), 0u, 0u),
                                  make_uint2((uint32_t)a.seed, (uint32_t)(a.seed >> 32)));
  const float u = (float)(rnd.x >> 8) * (1.0f / 16777216.0f);
  const float target = u * total;
  const float excl = base + incl - loc;
  if (loc > 0.f && target >= excl && target < excl + loc) {
    float c = excl;
    int pick = -1;
    for (int i = i0; i < i1; ++i) {
      const float e = expf(sl[i] - vmax);
      if (e > 0.f) { pick = i; c += e; if (target < c) break; }
    }
    if (pick >= 0) atomicMin(&sc.redi[16], pick);
  }
  cbar_sync();
  int tok = sc.redi[16];
  if (tok == 0x7fffffff) tok = imax;  // rounding fell off the end of the CDF
  return tok;
}

// In-kernel sampler for logits that arrive as packed bf16 LL words (V <= 8 * 384 = 3072), top_p >= 1.
// Thread t owns logits [8t, 8t+8) in registers (four words, two 16-byte loads).  Every intermediate of the reference is a
// bf16 tensor here (round_bf16), so the order-preserving keys have 16 bits and the k-th largest value needs two 8-bit
// radix passes.  Eight barriers in total (the generic sampler behind fq3_sample needs about twenty-five).
// Same semantics as sample_row: penalty -> suppression -> temperature -> keep x >= k-th largest (ties survive) ->
// multinomial by inverse CDF in index order on one Philox uniform; greedy = lowest index of the maximum.
__device__ __forceinline__ uint32_t bf16_key(float x) {  // x is bf16-representable (or -inf)
  const uint32_t b = __float_as_uint(x) >> 16;
  return (b & 0x8000u) ? (~b & 0xffffu) : (b | 0x8000u);
}
__device__ __forceinline__ float bf16_key_value(uint32_t k) {
  const uint32_t b = (k & 0x8000u) ? (k & 0x7fffu) : (~k & 0xffffu);
  return __uint_as_float(b << 16);
}
__device__ __noinline__ int sample_fast(const LLWord* ll, uint32_t ep, const LaunchParams* lp, int pidx, const SampleArgs& a, unsigned char* scratch) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int V = a.V, nw = V >> 1;
  unsigned* hist = reinterpret_cast<unsigned*>(scratch);         // [2][256]
  float* redf = reinterpret_cast<float*>(scratch + 2048);         // [0..15] per-warp maxima, [16..31] per-warp sums
  int* redi = reinterpret_cast<int*>(scratch + 2048 + 128);       // [0..15] argmax indices, [16..19] select state, [20] result
  // ---- poll this thread's four words
  const int w0i = 4 * tid;
  const bool h0 = w0i < nw, h1 = w0i + 2 < nw;
  uint4 wa = make_uint4(0u, ep, 0u, ep), wb = wa;
  if (h0) wa = ll_ld_pair(ll + w0i);
  if (h1) wb = ll_ld_pair(ll + w0i + 2);
  if (tid < 256) { hist[tid] = 0u; hist[256 + tid] = 0u; }
  cbar_sync();  // (0) histograms cleared before anybody adds to them (overlaps the poll round trip)
  if (ep != 0) {
    unsigned tries = 0;
    while ((wa.y != ep) | (wa.w != ep) | (wb.y != ep) | (wb.w != ep)) {
      if (++tries > 4) __nanosleep(32);
      if (tries > (unsigned)(lp->watchdog_ns >> 8)) device_fault(*lp, DE_LL_WAIT, pidx, (int)ep);
      if (h0 && ((wa.y != ep) | (wa.w != ep))) wa = ll_ld_pair(ll + w0i);
      if (h1 && ((wb.y != ep) | (wb.w != ep))) wb = ll_ld_pair(ll + w0i + 2);
    }
  }
  prof_mark(*lp, pidx, 1);
  prof_warp_time(*lp, pidx, 0);
  float x[8] = {bf_lo(wa.x), bf_hi(wa.x), bf_lo(wa.z), bf_hi(wa.z), bf_lo(wb.x), bf_hi(wb.x), bf_lo(wb.z), bf_hi(wb.z)};
  // ---- penalty, suppression, temperature (each result rounded to bf16 like the reference's bf16 tensor ops)
  unsigned long long seen8 = 0ull;
  if (a.seen && a.rep_pen != 1.0f && 8 * tid < V) seen8 = __ldcg(reinterpret_cast<const unsigned long long*>(a.seen + 8 * tid));
  {
    // copies of the policy in registers (the argument block lives in local memory), and a fast path for the common
    // thread whose eight logits need neither penalty nor suppression
    const int V_ = a.V, sup0 = a.suppress_start, eos = a.eos, sup_eos = a.suppress_eos, smp = a.do_sample;
    const float temp = a.temperature, pen = a.rep_pen;
    const int i0 = 8 * tid;
    const bool plain = (seen8 == 0ull) && (i0 + 8 <= V_) && (i0 + 8 <= sup0) && !(sup_eos && eos >= i0 && eos < i0 + 8);
    // x / T, correctly rounded for the finite, normal values that occur here: reciprocal + one fused residual correction
    const float rcp = __frcp_rn(temp);
    auto div_t = [&](float v) {
      const float q = v * rcp;
      return fmaf(fmaf(-q, temp, v), rcp, q);
    };
    if (i0 >= V_) {
#pragma unroll
      for (int j = 0; j < 8; ++j) x[j] = -INFINITY;
    } else if (plain) {
      if (smp) {
#pragma unroll
        for (int j = 0; j < 8; ++j) x[j] = bf16r(div_t(x[j]));
      }
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int i = i0 + j;
        float v = x[j];
        if ((seen8 >> (8 * j)) & 0xffull) v = bf16r((v > 0.f) ? v / pen : v * pen);
        if (i >= sup0 && i != eos) v = -INFINITY;
        if (sup_eos && i == eos) v = -INFINITY;
        if (smp && v > -INFINITY) v = bf16r(div_t(v));
        if (i >= V_) v = -INFINITY;
        x[j] = v;
      }
    }
  }
  // ---- maximum and its lowest index; the first radix pass (high byte of the 16-bit keys) shares its barrier
  const bool want_k = a.do_sample && a.top_k > 0 && a.top_k < V;
  uint32_t key[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) key[j] = bf16_key(x[j]);
  if (want_k && 8 * tid < V) {
    // logits sit in a handful of binades: a thread's eight keys mostly share their high byte, so count those once
    const uint32_t d0 = key[0] >> 8;
    unsigned same = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const bool in = 8 * tid + j < V;
      if (in && (key[j] >> 8) == d0) ++same;
      else if (in) atomicAdd(&hist[key[j] >> 8], 1u);
    }
    if (same) atomicAdd(&hist[d0], same);
  }
  float bv = x[0];
  int bi = 8 * tid;
#pragma unroll
  for (int j = 1; j < 8; ++j)
    if (x[j] > bv) { bv = x[j]; bi = 8 * tid + j; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
  }
  if (lane == 0) { redf[warp] = bv; redi[warp] = bi; }
  prof_warp_time(*lp, pidx, 1);
  cbar_sync();  // (1)
  auto select = [&](unsigned* h, int krem, int slot) {  // warp 0: highest digit whose cumulative count (from the top) reaches krem
    if (warp == 0) {
      unsigned s = 0;
#pragma unroll
      for (int t = 0; t < 8; ++t) s += h[255 - 8 * lane - t];
      unsigned incl = s;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned n = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += n;
      }
      const unsigned ballot = __ballot_sync(0xffffffffu, incl >= (unsigned)krem);
      const int sel = __ffs(ballot) - 1;
      if (lane == sel) {
        unsigned above = incl - s;
        int digit = 255 - 8 * lane;
        for (int t = 0; t < 8; ++t) {
          const unsigned c = h[255 - 8 * lane - t];
          if (above + c >= (unsigned)krem) { digit = 255 - 8 * lane - t; break; }
          above += c;
        }
        redi[16 + 2 * slot] = digit;
        redi[17 + 2 * slot] = krem - (int)above;
      }
    }
  };
  if (want_k) select(hist, a.top_k, 0);
  float vmax = redf[0];
  int imax = redi[0];
#pragma unroll
  for (int w = 1; w < kConsumerWarps; ++w) {
    const float ov = redf[w];
    const int oi = redi[w];
    if (ov > vmax || (ov == vmax && oi < imax)) { vmax = ov; imax = oi; }
  }
  prof_mark(*lp, pidx, 2);
  if (!a.do_sample) return imax;
  // ---- k-th largest value (counting multiplicity): second radix pass over the low byte
  float thr = -INFINITY;
  if (want_k) {
    cbar_sync();  // (2)
    const uint32_t d1 = (uint32_t)redi[16];
    const int krem = redi[17];
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (8 * tid + j < V && (key[j] >> 8) == d1) atomicAdd(&hist[256 + (key[j] & 0xffu)], 1u);
    cbar_sync();  // (3)
    select(hist + 256, krem, 1);
    cbar_sync();  // (4)
    thr = bf16_key_value((d1 << 8) | (uint32_t)redi[18]);
  }
  // the row of the drawn token is read from HBM right after the draw: pull the rows of all surviving candidates into L2 now
  if (a.next_emb && (a.top_k > 0 && a.top_k <= 64)) {
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (x[j] >= thr && x[j] > -INFINITY)
        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(reinterpret_cast<const unsigned char*>(a.next_emb) +
                                                                       (size_t)(8 * tid + j) * a.emb_row_bytes),
                     "r"(a.emb_row_bytes)
                     : "memory");
  }
  prof_mark(*lp, pidx, 4);
  // ---- multinomial(softmax) by inverse CDF in index order
  float e[8], loc = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    e[j] = (x[j] >= thr) ? expf(x[j] - vmax) : 0.f;  // exp(-inf) = 0
    loc += e[j];
  }
  float incl = loc;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float n = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += n;
  }
  if (lane == 31) redf[16 + warp] = incl;
  if (tid == 0) redi[20] = 0x7fffffff;
  cbar_sync();  // (6)
  float base = 0.f, total = 0.f;
#pragma unroll
  for (int w = 0; w < kConsumerWarps; ++w) {
    const float s = redf[16 + w];
    if (w < warp) base += s;
    total += s;
  }
  const uint4 rnd = philox4x32_10(make_uint4((uint32_t)a.draw, (uint32_t)(a.draw >> 32), 0u, 0u),
                                  make_uint2((uint32_t)a.seed, (uint32_t)(a.seed >> 32)));
  const float u = (float)(rnd.x >> 8) * (1.0f / 16777216.0f);
  const float target = u * total;
  const float excl = base + incl - loc;
  if (loc > 0.f && target >= excl && target < excl + loc) {
    float c = excl;
    int pick = -1;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (e[j] > 0.f && (pick < 0 || target >= c)) { pick = 8 * tid + j; }
      c += e[j];
    }
    // pick = last index whose cumulative start is <= target among kept entries == first index with target < cumulative end
    if (pick >= 0) atomicMin(&redi[20], pick);
  }
  cbar_sync();  // (7)
  int tok = redi[20];
  if (tok == 0x7fffffff) tok = imax;  // rounding fell off the end of the CDF
  prof_mark(*lp, pidx, 5);
  return tok;
}

// logits as LL words: the register sampler whenever it applies (top-p needs the sorted distribution: generic path)
__device__ __forceinline__ int sample_ll(const LLWord* ll, uint32_t ep, const LaunchParams& p, int pidx, const SampleArgs& a, unsigned char* scratch) {
  if (a.top_p >= 1.0f && a.V <= 8 * kConsumerThreads && (a.V & 3) == 0) return sample_fast(ll, ep, &p, pidx, a, scratch);
  return sample_row(nullptr, ll, ep, &p, pidx, a, sample_scratch(scratch));
}

// Publish one bf16 row (n elements) as LL words with all consumer threads.
__device__ __forceinline__ void publish_row(LLWord* dst, const bf16* src, int n, uint32_t ep) {
  for (int c = threadIdx.x; c < (n >> 1); c += kConsumerThreads) ll_st(dst + c, __ldg(reinterpret_cast<const uint32_t*>(src) + c), ep);
}
// The same for a waiting stream's held row, which this kernel wrote: read through L2, not the read-only path.
__device__ __noinline__ void publish_held_row(LLWord* dst, const bf16* src, int n, uint32_t ep) {
  for (int c = threadIdx.x; c < (n >> 1); c += kConsumerThreads) ll_st(dst + c, __ldcg(reinterpret_cast<const uint32_t*>(src) + c), ep);
}
// Keep a stream's past_hidden row when it starts waiting for text: each thread copies the words it publishes from held later.
__device__ __noinline__ void hold_row(bf16* dst, const bf16* src, int n) {
  for (int c = threadIdx.x; c < (n >> 1); c += kConsumerThreads)
    __stcg(reinterpret_cast<uint32_t*>(dst) + c, __ldg(reinterpret_cast<const uint32_t*>(src) + c));
}

template <bool WIDE>
__device__ __forceinline__ void sample_phase(const Phase& ph, const LaunchParams& p, unsigned char* smem_base, uint32_t ep, int pidx,
                             const int* frame_done) {
  const Smem sm = carve_smem(smem_base, p);
  const SampleScratch sc = sample_scratch(sm.scratch);
  const int Ht = p.stacks[ST_TALKER].hidden;
  const int ncb = p.n_code_groups - 1;
  const uint32_t ep_in = ep - 1;
  // CTAs without a stream idle through sampling phases: the once-per-step fence that makes this step's KV
  // rows visible to whichever CTA reads them in a later step goes here, off the critical path.
  if ((int)blockIdx.x >= (p.mode == MODE_PREFILL ? 1 : p.n_rows) && threadIdx.x == 0 && ph.skind != SMP_PRED && ph.skind != SMP_PRED_ONLY)
    __threadfence();  // cumulative: covers the K/V rows its CTA mates stored (ordered before by the consumer barriers)
  for (int b = blockIdx.x; b < (p.mode == MODE_PREFILL ? 1 : p.n_rows); b += gridDim.x) {
    prof_mark(p, pidx, 0);
    cbar_sync();  // the scratch may still be read by the previous GEMV phase's finishing threads
    const int slot = p.stream0 + b;
    StreamState* st = p.st + slot;
    const int done = (p.mode == MODE_FRAMES) ? frame_done[b] : 0;
    LLWord* pin = reinterpret_cast<LLWord*>(p.bufs[p.has_s2m ? BUF_PIN : BUF_PX]);
    const int ldpin = p.ld[p.has_s2m ? BUF_PIN : BUF_PX];
    const LLWord* lgbuf = reinterpret_cast<const LLWord*>(p.bufs[BUF_LOGITS]);
    if (ph.skind == SMP_PRED || ph.skind == SMP_PRED_ONLY) {
      const int i = ph.aux;  // codebook step 0..ncb-1
      const int Vp = p.stacks[ST_PRED].vocab;
      const int lrow = (ph.flags & F_ROWS2) ? 2 * b + 1 : b;
      const LLWord* lg = lgbuf + (size_t)lrow * p.ld[BUF_LOGITS];
      if (p.pred_logits_all) {
        for (int v = threadIdx.x; v < (Vp >> 1); v += kConsumerThreads) {
          const uint32_t pay = ll_wait(lg + v, ep_in, p, pidx);
          p.pred_logits_all[(size_t)i * Vp + 2 * v] = bf_lo(pay);
          p.pred_logits_all[(size_t)i * Vp + 2 * v + 1] = bf_hi(pay);
        }
      }
      // codebooks 1..15 keep the launch's SubPolicy; a stream with its own policy keys the draws with its own seed (fq3_common.cuh)
      const bool own = p.spol != nullptr && __ldcg(&p.spol[slot].on) != 0;
      const unsigned long long seed = own ? __ldcg(&p.spol[slot].pol.seed) : p.pol.seed;
      SampleArgs a;
      a.V = Vp; a.do_sample = p.sub.do_sample; a.top_k = p.sub.top_k; a.top_p = p.sub.top_p;
      a.temperature = p.sub.temperature; a.rep_pen = 1.0f; a.seen = nullptr; a.suppress_start = Vp; a.eos = -1;
      a.suppress_eos = 0; a.round_bf16 = 1; a.seed = seed ^ (0x9E3779B97F4A7C15ull * (unsigned long long)(own ? 1 : slot + 1));
      a.draw = __ldcg(&st->draws) + (unsigned long long)(i + 1);
      a.next_emb = p.pred_embeds[i]; a.emb_row_bytes = Ht * 2;
      const int tok = sample_ll(lg, ep_in, p, pidx, a, sm.scratch);
      FQ3_ASSERT(tok >= 0 && tok < Vp, pidx, 100000 + tok);
      if (threadIdx.x == 0) st->cur_codes[i + 1] = tok;
      if (i + 1 < ncb) {
        // next predictor input row: codec_embeds[i](tok)  (predictor_graph.py:144)
        publish_row(pin + (size_t)b * ldpin, p.pred_embeds[i] + (size_t)tok * Ht, Ht, ep);
      } else if (ph.skind == SMP_PRED) {
        // frame complete: append [c0..c15], then build the next talker input (generate.py:159-171)
        const int nfr = __ldcg(&st->n_frames);
        const int c0 = __ldcg(&st->token);
        if (!done) {
          if (threadIdx.x < p.n_code_groups && nfr < p.max_frames) {
            const int code = (threadIdx.x == 0) ? c0 : (threadIdx.x == ncb ? tok : __ldcg(&st->cur_codes[threadIdx.x]));
            st->codes[(size_t)nfr * p.n_code_groups + threadIdx.x] = code;
          }
          if (threadIdx.x == 0) {
            st->n_frames = nfr + 1;
            st->seen[c0] = 1;
            st->draws = __ldcg(&st->draws) + 32ull;
          }
        }
        cbar_sync();
        const int gs = __ldcg(&st->gen_step);
        const int ntr = __ldcg(&st->n_trailing);
        const bf16* text = (gs < ntr) ? st->trailing + (size_t)gs * Ht : st->pad_embed;
        LLWord* tx = reinterpret_cast<LLWord*>(p.bufs[BUF_TX]) + (size_t)b * p.ld[BUF_TX];
        const uint32_t* ce = reinterpret_cast<const uint32_t*>(p.codec_embed + (size_t)c0 * Ht);
        const uint32_t* tx32 = reinterpret_cast<const uint32_t*>(text);
        for (int c = threadIdx.x; c < (Ht >> 1); c += kConsumerThreads) {
          uint32_t v = __ldg(ce + c);
          float s0 = bf_lo(v), s1 = bf_hi(v);
          for (int g = 0; g < ncb; ++g) {
            const int code = (g == ncb - 1) ? tok : __ldcg(&st->cur_codes[g + 1]);
            v = __ldg(reinterpret_cast<const uint32_t*>(p.pred_embeds[g] + (size_t)code * Ht) + c);
            s0 += bf_lo(v); s1 += bf_hi(v);
          }
          const uint32_t t = __ldg(tx32 + c);
          ll_st(tx + c, pack_bf16x2(bf16r(bf16r(s0) + bf_lo(t)), bf16r(bf16r(s1) + bf_hi(t))), ep);
        }
        // static-cache bound (generate.py:174-177): the frame stays, decoding stops after this step
        if (threadIdx.x == 0 && !done) {
          const int pos = __ldcg(&st->position);
          if (pos >= p.stacks[ST_TALKER].max_pos - 1) st->done = 2;
        }
      }
    } else {
      // SMP_TALKER / SMP_PREFILL: first-codebook sampler (generate.py:124-134, :182-197)
      const int Vt = p.stacks[ST_TALKER].vocab;
      const LLWord* lg = lgbuf + (size_t)b * p.ld[BUF_LOGITS];
      const int nfr = __ldcg(&st->n_frames);
      const int done_now = (ph.skind == SMP_PREFILL) ? 0 : __ldcg(&st->done);  // includes this frame's cache-bound stop
      // the stream's own policy when it has one (fq3_set_stream_policy), else the launch's; read once into registers
      const bool own = p.spol != nullptr && __ldcg(&p.spol[slot].on) != 0;
      Policy pol;
      if (own) {
        const Policy* sp = &p.spol[slot].pol;
        pol.do_sample = __ldcg(&sp->do_sample); pol.top_k = __ldcg(&sp->top_k); pol.top_p = __ldcg(&sp->top_p);
        pol.temperature = __ldcg(&sp->temperature); pol.rep_pen = __ldcg(&sp->rep_pen);
        pol.min_new_tokens = __ldcg(&sp->min_new_tokens); pol.suppress_tail = __ldcg(&sp->suppress_tail); pol.seed = __ldcg(&sp->seed);
      } else {
        pol = p.pol;
      }
      SampleArgs a;
      a.V = Vt; a.do_sample = pol.do_sample; a.top_k = pol.top_k; a.top_p = pol.top_p;
      a.temperature = pol.temperature; a.rep_pen = pol.rep_pen;
      a.seen = (ph.skind == SMP_TALKER && nfr > 0) ? st->seen : nullptr;
      a.suppress_start = max(0, Vt - pol.suppress_tail); a.eos = p.eos_id;
      a.suppress_eos = (ph.skind == SMP_PREFILL) ? (pol.min_new_tokens > 0) : (nfr < pol.min_new_tokens);
      a.round_bf16 = 1;
      a.seed = pol.seed ^ (0x9E3779B97F4A7C15ull * (unsigned long long)(own ? 1 : slot + 1));
      a.draw = __ldcg(&st->draws);
      a.next_emb = p.codec_embed; a.emb_row_bytes = Ht * 2;
      int tok = sample_ll(lg, ep_in, p, pidx, a, sm.scratch);
      const bool live = !done_now;
      int new_done = done_now, new_pos = __ldcg(&st->position), new_gs = __ldcg(&st->gen_step);
      if (live) {
        if (ph.skind == SMP_TALKER) { new_pos += 1; new_gs += 1; }
        if (tok == p.eos_id) new_done = 1;  // generate.py:150 — checked before the next frame is built
        // open text (fq3_open_text): the next frame adds text row new_gs; until it has arrived the stream waits, state unchanged
        else if (__ldcg(&st->text_open) && new_gs >= __ldcg(&st->n_trailing)) new_done = 4;
      } else {
        tok = __ldcg(&st->token);
      }
      cbar_sync();  // everyone has read the old state
      if (threadIdx.x == 0) {
        if (live) { st->token = tok; st->draws = a.draw + 1ull; st->position = new_pos; st->gen_step = new_gs; st->done = new_done; }
        // control record every CTA reads at the top of the next frame
        ll_st(&st->ctl[0], (uint32_t)new_done, ep);
        ll_st(&st->ctl[1], (uint32_t)new_pos, ep);
      }
      // predictor pass-0 input rows [past_hidden ; codec_embed(token)] (generate.py:154-155), addressed by
      // stream slot; always re-published so every reader sees this phase's epoch.  A waiting stream's BUF_HID row is the
      // result of an idle talker pass: its past_hidden comes from the row it held when it started waiting.
      const bf16* hid = reinterpret_cast<const bf16*>(p.bufs[BUF_HID]) + (size_t)b * p.ld[BUF_HID];
      LLWord* const hid_dst = WIDE ? reinterpret_cast<LLWord*>(p.bufs[BUF_WPIN]) + (size_t)slot * p.ld[BUF_WPIN]
                                   : pin + (size_t)(2 * slot) * ldpin;
      if (done_now == 4) {
        publish_held_row(hid_dst, st->held, Ht, ep);
      } else {
        if (new_done == 4) hold_row(st->held, hid, Ht);
        publish_row(hid_dst, hid, Ht, ep);
      }
      if constexpr (WIDE) {  // the wide program keeps them in BUF_WPIN (the host converts between the two layouts: fq3_api.cu, sync_pin_layout)
        publish_row(reinterpret_cast<LLWord*>(p.bufs[BUF_WPIN]) + (size_t)(p.max_streams + slot) * p.ld[BUF_WPIN],
                    p.codec_embed + (size_t)tok * Ht, Ht, ep);
      } else {
        publish_row(pin + (size_t)(2 * slot + 1) * ldpin, p.codec_embed + (size_t)tok * Ht, Ht, ep);
      }
      if (threadIdx.x == 0) __threadfence();  // once per step: K/V rows stored by this CTA (see above)
    }
    prof_mark(p, pidx, 6);
    cbar_sync();
    prof_mark(p, pidx, 3);
  }
}

// =================================================================================================
// Kernel
// =================================================================================================
template <bool PROF, bool WIDE>
__global__ void __launch_bounds__(kThreads, 1) fq3_stream_kernel(const __grid_constant__ LaunchParams p) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  const Smem sm = carve_smem(smem_raw, p);
  const Ctx c = make_ctx(smem_raw, p);
  const int tid = threadIdx.x;

  if (tid == 0) {
    for (int s = 0; s < kMaxStages; ++s) {
      mbar_init(&sm.full[s], 1);
      mbar_init(&sm.empty[s], 1);  // the first warp of the stage's group, behind the group barrier
    }
    for (int s = 0; s < kGammaSlots; ++s) {
      mbar_init(reinterpret_cast<uint64_t*>(smem_raw + kGFullOffset) + s, 1);
      mbar_init(reinterpret_cast<uint64_t*>(smem_raw + kGEmptyOffset) + s, kConsumerWarps);
    }
    sm.ctl[0] = 0;
    fence_barrier_init();
  }
  {
    const uint4* src = reinterpret_cast<const uint4*>(p.prog);
    uint4* dst = reinterpret_cast<uint4*>(sm.prog);
    for (int i = tid; i < p.n_phases * 2; i += kThreads) dst[i] = __ldg(src + i);
  }
  __syncthreads();
  // resolve the GEMV phase kinds of this launch, then every warp's unit of every kind
  if (tid < p.n_kinds) resolve_kind(p, sm.prog[p.kind_phase[tid]], sm.kinds[tid]);
  __syncthreads();
  for (int i = tid; i < p.n_kinds * kConsumerWarps; i += kThreads) resolve_unit(sm.kinds[i / kConsumerWarps], i % kConsumerWarps, sm.units[i]);
  __syncthreads();

  // Register budget: the launch gives every thread 128 (64 K / 512); the producer's warpgroup keeps 56 and the three consumer
  // warpgroups grow to 152 — room for the weight blocks a consumer prefetches into registers (gemv_phase_consume) without
  // spilling.
#ifndef FQ3_SETMAXNREG
#define FQ3_SETMAXNREG 1
#endif
#if FQ3_SETMAXNREG
  if (tid >= kConsumerThreads) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kProducerRegs));
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kConsumerRegs));
  }
#endif
  if (tid >= kConsumerThreads) {
    // ------------------------------ producer warp (one thread) ------------------------------
    if (tid == kConsumerThreads) {
      const uint64_t pol_stream = policy_evict_first(), pol_keep = policy_keep_fraction();
      const uint64_t pol_gamma = policy_evict_last();
      RingCur cur{0, 0u}, gcur{0, 0u};
      uint32_t issued = 0, gissued = 0;
      bool ok = true;
      for (int iter = 0; iter < p.n_iters && ok; ++iter) {
        for (int i = 0; i < p.n_phases && ok; ++i) {
          const Phase ph = load_phase(sm.prog, i);
          if (ph.type == PH_GEMV) ok = gemv_phase_produce<PROF>(c, ph, p, sm.ctl, cur, gcur, issued, gissued, i, pol_stream, pol_keep, pol_gamma);
        }
      }
      // drain: shared memory must not be released with bulk copies in flight (the frame loop may stop early)
      const int n = (int)min(issued, (uint32_t)p.n_stages);
      RingCur d = cur;
      for (int k = 0; k < n; ++k) {
        if (d.slot == 0) { d.slot = p.n_stages - 1; d.lap ^= 1u; } else { --d.slot; }
        mbar_wait(&sm.full[d.slot], d.lap, p, DE_FULL_WAIT, -3);
      }
      const int gn = (int)min(gissued, (uint32_t)kGammaSlots);
      d = gcur;
      for (int k = 0; k < gn; ++k) {
        if (d.slot == 0) { d.slot = kGammaSlots - 1; d.lap ^= 1u; } else { --d.slot; }
        mbar_wait(reinterpret_cast<uint64_t*>(smem_raw + kGFullOffset) + d.slot, d.lap, p, DE_FULL_WAIT, -4);
      }
    }
    return;
  }

  // -------------------------------- consumer warps --------------------------------
  RingCur cur{0, 0u}, gcur{0, 0u};
  uint32_t gst = 0u;              // GEMV phase state: bit 0 = activation / partial-word buffer, bit 1 = the last phase was multi-row
  int* frame_pos = sm.ctl + kFramePosIdx;    // [kMaxWide] talker positions of this iteration
  int* frame_done = sm.ctl + kFrameDoneIdx;  // [kMaxWide]
  for (int iter = 0; iter < p.n_iters; ++iter) {
    const uint32_t ep0 = p.epoch_base + (uint32_t)iter * (uint32_t)p.n_phases;
    if (p.mode == MODE_FRAMES || p.mode == MODE_TALKER_STEP) {
      // per-stream frame state: from the stream state at launch, afterwards from the sampler's control record
      if (tid < p.n_rows) {
        const StreamState* st = p.st + p.stream0 + tid;
        int done, pos;
        if (iter == 0) {
          done = __ldcg(&st->done);
          pos = __ldcg(&st->position);
          int* sconst = reinterpret_cast<int*>(smem_raw + kStreamConstOffset);
          sconst[tid] = __ldcg(&st->n_pad);
          sconst[kMaxWide + tid] = __ldcg(&st->rope_delta);
        } else {
          done = (int)ll_wait(&st->ctl[0], ep0, p, -2);
          pos = (int)ll_wait(&st->ctl[1], ep0, p, -2);
        }
        frame_pos[tid] = pos;
        frame_done[tid] = done;
      }
      cbar_sync();
      if (p.mode == MODE_FRAMES && iter > 0) {
        int all_done = 1;
        for (int b = 0; b < p.n_rows; ++b) all_done &= (frame_done[b] != 0);
        if (all_done) {
          if (tid == 0) st_volatile_shared_i32(&sm.ctl[0], -1);  // tells the producer (which prefetches across frames) to stop
          break;
        }
      }
    }
    for (int i = 0; i < p.n_phases; ++i) {
      const Phase ph = load_phase(sm.prog, i);
      const uint32_t ep = ep0 + (uint32_t)i + 1u;
      switch (ph.type) {
        case PH_GEMV:
          if constexpr (WIDE) gemv_phase_consume_wide(c, ph, p, cur, gcur, gst, i, ep);
          else gemv_phase_consume<PROF>(c, ph, p, cur, gcur, gst, i, ep);
          break;
        case PH_ATTN:
          if constexpr (WIDE) {
            long long tp = (FQ3_WIDE_PROF && p.prof) ? clock64() : 0ll;
            attn_phase<PROF, true>(ph, p, smem_raw, ep, i, frame_pos);
            prof_acc(p, 4, tp);
          } else {
            attn_phase<PROF, false>(ph, p, smem_raw, ep, i, frame_pos);
          }
          break;
        case PH_SAMPLE:
          if constexpr (WIDE) {
            long long tp = (FQ3_WIDE_PROF && p.prof) ? clock64() : 0ll;
            sample_phase<WIDE>(ph, p, smem_raw, ep, i, frame_done);
            prof_acc(p, 5, tp);
          } else {
            sample_phase<WIDE>(ph, p, smem_raw, ep, i, frame_done);
          }
          break;
        default: if (tid == 0) device_fault(p, DE_BAD_PHASE, i, ph.type); break;
      }
    }
  }
}

// Fragment image of one GEMV matrix (fq3_common.cuh: Plan).  W is row-major [N][K]; the image keeps groups of 8 rows
// contiguous (8 * K * 2 bytes each, in row order), a group being K / 32 blocks of 512 bytes: lane (r8, t) of a warp reads
// bytes [(4 * r8 + t) * 16, +16) of a block = columns {2t, 2t+1 | 8+2t, 9+2t | 16+2t, 17+2t | 24+2t, 25+2t} of row r8 —
// the B fragments (b0, b1) of two consecutive mma.m16n8k16 k-steps.  Rows beyond N are zeros.
__global__ void fq3_tile_weights_kernel(const bf16* __restrict__ W, uint4* __restrict__ out, int N, int K) {
  const long pieces = (long)((N + 7) / 8) * K;  // 16-byte pieces: K per group
  for (long idx = blockIdx.x * (long)blockDim.x + threadIdx.x; idx < pieces; idx += (long)gridDim.x * blockDim.x) {
    const long grp = idx / K;
    const int pc = (int)(idx - grp * K);
    const int ch = pc >> 5, ln = pc & 31, r8 = ln >> 2, t = ln & 3;
    const long row = grp * 8 + r8;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (row < N) {
      const uint32_t* src = reinterpret_cast<const uint32_t*>(W + (size_t)row * K + ch * kChunkK) + t;
      v = make_uint4(__ldg(src), __ldg(src + 4), __ldg(src + 8), __ldg(src + 12));
    }
    out[idx] = v;
  }
}

// Small kernels -----------------------------------------------------------------------------------
// Stand-alone sampler behind fq3_sample (sampling.py parity tests and the operator-at-a-time host loop).
__global__ void __launch_bounds__(kConsumerThreads, 1)
fq3_sample_kernel(const float* logits, SampleArgs a, const long long* history, int n_history, uint8_t* seen_scratch,
                  long long* out) {
  __shared__ __align__(16) unsigned char scratch[24 * 1024];
  const SampleScratch sc = sample_scratch(scratch);
  if (history && n_history > 0 && a.rep_pen != 1.0f) {
    for (int i = threadIdx.x; i < a.V; i += kConsumerThreads) seen_scratch[i] = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < n_history; i += kConsumerThreads) {
      const long long t = history[i];
      if (t >= 0 && t < a.V) seen_scratch[t] = 1;
    }
    __syncthreads();
    a.seen = seen_scratch;
  } else {
    a.seen = nullptr;
  }
  const int tok = sample_row(logits, nullptr, 0u, nullptr, 0, a, sc);
  if (threadIdx.x == 0) out[0] = tok;
}

// apply_repetition_penalty (sampling.py:10-29) in place on fp32 logits; history marks a bitmap first.
__global__ void __launch_bounds__(kConsumerThreads, 1)
fq3_rep_penalty_kernel(float* logits, int V, const long long* history, int n_history, float penalty, int round_bf16,
                       uint8_t* seen) {
  for (int i = threadIdx.x; i < V; i += kConsumerThreads) seen[i] = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < n_history; i += kConsumerThreads) {
    const long long t = history[i];
    if (t >= 0 && t < V) seen[t] = 1;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < V; i += kConsumerThreads) {
    if (__ldcg(seen + i)) {
      float x = logits[i];
      x = (x > 0.f) ? x / penalty : x * penalty;
      logits[i] = round_bf16 ? bf16r(x) : x;
    }
  }
}

// Wide frame program entry: rows [2 * slot], [2 * slot + 1] of the pair layout -> BUF_WPIN rows [slot], [max_streams + slot]
// (epoch 0: "written before the launch"), or back.  One block, one stream.
__global__ void fq3_wpin_from_pairs_kernel(LLWord* wpin, int ldw, LLWord* pairs, int ldp, int slot, int max_streams, int reverse) {
  for (int c = threadIdx.x; c < ldw; c += blockDim.x) {
    LLWord* a0 = wpin + (size_t)slot * ldw + c;
    LLWord* a1 = wpin + (size_t)(max_streams + slot) * ldw + c;
    LLWord* b0 = pairs + (size_t)(2 * slot) * ldp + c;
    LLWord* b1 = pairs + (size_t)(2 * slot + 1) * ldp + c;
    if (reverse) { *b0 = make_uint2(a0->x, 0u); *b1 = make_uint2(a1->x, 0u); }
    else { *a0 = make_uint2(b0->x, 0u); *a1 = make_uint2(b1->x, 0u); }
  }
}

// Prompt assembly (model.py:331-553, SURVEY.md Appendix A5): one block per prompt row.  A row is text part + codec part:
//   desc.x  index into the projected text rows tp [n_tp, H] (text_projection(text_embedding(id))), -1 = none
//   desc.y  codec part: 0 none | 1 talker codec embedding row desc.z | 2 speaker row desc.z | 3 the 16-codebook embedding sum of
//           reference frame desc.z (generate_icl_prompt: CE(c0), then + emb_g(c_g) one codebook at a time, each add rounded to
//           bf16 like the reference's bf16 tensor adds)
// and the two parts meet in one more bf16 add.  Rows with neither part are the left padding: zeros.
struct PromptTables {
  const bf16* codec_embed;
  const bf16* pred_embeds[32];
  int ncb;
};
__global__ void fq3_assemble_prompt_kernel(const bf16* __restrict__ tp, const int4* __restrict__ desc, int H, PromptTables tb,
                                           const bf16* __restrict__ spk, const int* __restrict__ ref_codes, int n_groups, bf16* __restrict__ out) {
  const int r = blockIdx.x;
  const int4 d = desc[r];
  const int Hw = H >> 1;
  uint32_t* o = reinterpret_cast<uint32_t*>(out + (size_t)r * H);
  const uint32_t* t = d.x >= 0 ? reinterpret_cast<const uint32_t*>(tp + (size_t)d.x * H) : nullptr;
  for (int c = threadIdx.x; c < Hw; c += blockDim.x) {
    float c0 = 0.f, c1 = 0.f;
    bool have_c = d.y != 0;
    if (d.y == 1) {
      const uint32_t v = __ldg(reinterpret_cast<const uint32_t*>(tb.codec_embed + (size_t)d.z * H) + c);
      c0 = bf_lo(v); c1 = bf_hi(v);
    } else if (d.y == 2) {
      const uint32_t v = __ldg(reinterpret_cast<const uint32_t*>(spk + (size_t)d.z * H) + c);
      c0 = bf_lo(v); c1 = bf_hi(v);
    } else if (d.y == 3) {
      const int* codes = ref_codes + (size_t)d.z * n_groups;
      uint32_t v = __ldg(reinterpret_cast<const uint32_t*>(tb.codec_embed + (size_t)codes[0] * H) + c);
      c0 = bf_lo(v); c1 = bf_hi(v);
      for (int g = 0; g < tb.ncb; ++g) {
        v = __ldg(reinterpret_cast<const uint32_t*>(tb.pred_embeds[g] + (size_t)codes[g + 1] * H) + c);
        c0 = bf16r(c0 + bf_lo(v)); c1 = bf16r(c1 + bf_hi(v));
      }
    }
    uint32_t res = 0u;
    if (t) {
      const uint32_t v = __ldg(t + c);
      res = have_c ? pack_bf16x2(bf_lo(v) + c0, bf_hi(v) + c1) : v;
    } else if (have_c) {
      res = pack_bf16x2(c0, c1);
    }
    o[c] = res;
  }
}

// LL-epoch wrap (fq3_api.cu: reserve_epochs): keep the payloads, mark every word "written before the launch"
__global__ void fq3_ll_clear_epochs_kernel(LLWord* w, size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) w[i].y = 0u;
}
__global__ void fq3_ctl_clear_epochs_kernel(StreamState* st, int n) {
  for (int i = threadIdx.x; i < n * 4; i += blockDim.x) st[i >> 2].ctl[i & 3].y = 0u;
}

// spol: the stream's policy record to clear as well (fq3_reset_stream), null where it survives (the reset inside a prefill)
__global__ void fq3_reset_stream_kernel(StreamState* st, int V, StreamPolicy* spol) {
  for (int i = threadIdx.x; i < V; i += blockDim.x) st->seen[i] = 0;
  if (threadIdx.x == 0) {
    st->token = 0; st->position = 0; st->gen_step = 0; st->n_frames = 0; st->done = 0; st->n_pad = 0;
    st->rope_delta = 0; st->draws = 0ull;  // text conditioning (n_trailing) is set separately and survives a reset
    for (int i = 0; i < 32; ++i) st->cur_codes[i] = 0;
    if (spol) spol->on = 0;
  }
}

// fq3_set_stream_policy: the policy travels by value, so no host buffer has to outlive the (stream-ordered) call
__global__ void fq3_set_stream_policy_kernel(StreamPolicy* spol, int on, Policy pol) {
  if (threadIdx.x == 0) {
    spol->pol = pol;
    spol->on = on;
  }
}

__global__ void fq3_set_state_kernel(StreamState* st, int token, int position, int gen_step, int set_mask, int n_pad,
                                     int rope_delta, int n_trailing) {
  if (threadIdx.x == 0) {
    if (set_mask & 1) st->token = token;
    if (set_mask & 2) { st->n_pad = n_pad; st->rope_delta = rope_delta; }
    if (set_mask & 4) {  // text conditioning: n_trailing rows, still open (64) or closed
      st->n_trailing = n_trailing;
      st->text_open = (set_mask & 64) ? 1 : 0;
      // a stream waiting for text runs again once its next row has arrived or its text has ended
      if (st->done == 4 && (!(set_mask & 64) || st->gen_step < n_trailing)) st->done = 0;
    }
    if (set_mask & 8) { st->position = position; st->gen_step = gen_step; }
    if (set_mask & 16) st->done = 0;
    if (set_mask & 32) st->done = 3;  // retired by the host (fq3_retire_stream): idles in lock-step launches until reset
  }
}

// K/V import: src [nkv, T, 128] -> cache [nkv, max_pos, 128] of one (layer, slot)
__global__ void fq3_import_kv_kernel(bf16* kdst, bf16* vdst, const bf16* k, const bf16* v, int nkv, int T, int max_pos) {
  const size_t n = (size_t)nkv * T * (kHeadDim / 8);
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % (kHeadDim / 8));
    const size_t t = (i / (kHeadDim / 8)) % T;
    const size_t h = i / ((size_t)(kHeadDim / 8) * T);
    const size_t d = (h * max_pos + t) * (kHeadDim / 8) + c;
    reinterpret_cast<uint4*>(kdst)[d] = reinterpret_cast<const uint4*>(k)[i];
    reinterpret_cast<uint4*>(vdst)[d] = reinterpret_cast<const uint4*>(v)[i];
  }
}

__global__ void fq3_codes_to_i64_kernel(const int* cur_codes, int n, long long* out) {
  if (threadIdx.x < n) out[threadIdx.x] = cur_codes[threadIdx.x + 1];
}

// Plain bf16 rows -> packed LL words (epoch 0: "written before launch") and back.  cols is even; ld_* in words / elements.
__global__ void fq3_pack_ll_kernel(LLWord* dst, int ld_dst, const bf16* src, int ld_src, int rows, int cols) {
  const int cw = cols >> 1;
  const size_t n = (size_t)rows * cw;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const size_t r = i / cw, c = i - r * cw;
    const uint32_t lo = __bfloat16_as_ushort(src[r * ld_src + 2 * c]), hi = __bfloat16_as_ushort(src[r * ld_src + 2 * c + 1]);
    dst[r * ld_dst + c] = make_uint2(lo | (hi << 16), 0u);
  }
}
__global__ void fq3_unpack_ll_bf16_kernel(bf16* dst, int ld_dst, const LLWord* src, int ld_src, int rows, int cols) {
  const int cw = cols >> 1;
  const size_t n = (size_t)rows * cw;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const size_t r = i / cw, c = i - r * cw;
    const uint32_t pay = src[r * ld_src + c].x;
    dst[r * ld_dst + 2 * c] = __ushort_as_bfloat16((unsigned short)(pay & 0xffffu));
    dst[r * ld_dst + 2 * c + 1] = __ushort_as_bfloat16((unsigned short)(pay >> 16));
  }
}
__global__ void fq3_unpack_ll_f32_kernel(float* dst, int ld_dst, const LLWord* src, int ld_src, int rows, int cols) {
  const int cw = cols >> 1;
  const size_t n = (size_t)rows * cw;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const size_t r = i / cw, c = i - r * cw;
    const uint32_t pay = src[r * ld_src + c].x;
    dst[r * ld_dst + 2 * c] = bf_lo(pay);
    dst[r * ld_dst + 2 * c + 1] = bf_hi(pay);
  }
}

}  // namespace fq3
