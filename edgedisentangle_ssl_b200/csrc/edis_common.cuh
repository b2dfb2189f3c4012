// Shared helpers for libedis (sm_100a).  Not part of the public ABI (see include/edis.h).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>

#include "edis.h"

namespace edis {

void set_error(const char* fmt, ...);

#define EDIS_CHECK_ARG(cond, ...)          \
  do {                                     \
    if (!(cond)) {                         \
      ::edis::set_error(__VA_ARGS__);      \
      return EDIS_ERR_ARG;                 \
    }                                      \
  } while (0)

#define EDIS_CUDA(call)                                                                  \
  do {                                                                                   \
    cudaError_t err__ = (call);                                                          \
    if (err__ != cudaSuccess) {                                                          \
      ::edis::set_error("%s failed at %s:%d: %s", #call, __FILE__, __LINE__,             \
                        cudaGetErrorString(err__));                                      \
      return EDIS_ERR_CUDA;                                                              \
    }                                                                                    \
  } while (0)

// One unit of row work: edges [beg, end) of `row`; slot < 0 when the chunk is the whole row,
// else the index of its partial-result slot (rows longer than max_chunk are split).
struct Item {
  int32_t row, beg, end, slot;
};
struct SplitRow {
  int32_t row, slot_beg, slot_cnt, pad;
};

struct Schedule {
  Item* items = nullptr;        // device
  SplitRow* split = nullptr;    // device
  int64_t n_items = 0, n_slots = 0, n_split = 0;
};

}  // namespace edis

struct edis_graph {
  int64_t n = 0, n_cols = 0, e = 0, e_in = 0;   // n = destination rows, n_cols = source columns
  int device = 0;
  int sm_count = 148;
  int64_t max_in = 0, max_out = 0;
  bool was_sorted = true;
  // device arrays
  int64_t* rowptr = nullptr;   // [n+1]
  int32_t* col = nullptr;      // [e]   source of CSR slot k
  int64_t* cscptr = nullptr;   // [n+1]
  int32_t* cscrow = nullptr;   // [e]   destination of CSC slot k
  int32_t* csceid = nullptr;   // [e]   CSR slot of CSC slot k
  edis::Schedule dst, src;
  // host mirrors (export / tests)
  int64_t* h_rowptr = nullptr;
  int32_t* h_col = nullptr;
  int64_t* h_perm = nullptr;
  int64_t* h_cscptr = nullptr;
  int32_t* h_cscrow = nullptr;
  int32_t* h_csceid = nullptr;
  // host copies of the two schedules (edis_graph_save) and the chunk size they were built with
  edis::Item* h_dst_items = nullptr;
  edis::SplitRow* h_dst_split = nullptr;
  edis::Item* h_src_items = nullptr;
  edis::SplitRow* h_src_split = nullptr;
  int max_chunk = 256;
};

namespace edis {

// ------------------------------------------------------------------ device helpers
__device__ __forceinline__ float4 ldg4(const float* p) {
  return __ldg(reinterpret_cast<const float4*>(p));
}
__device__ __forceinline__ float sigmoidf_fast(float x) {
  return __fdividef(1.0f, 1.0f + __expf(-x));
}
// Layer kernels: sigmoid and exp(sigmoid) straight on the MUFU units (ex2.approx / rcp.approx with
// flush-to-zero, no range fix-ups: 2^-22 relative).  Forward and backward use the SAME functions, so
// the softmax weights recomputed in the backward are bit-identical to the forward's row sums.
// EDIS_EXACT_MATH=1 (build-time, diagnostics): libm-accurate exp2 / division instead of the MUFU approximations
#ifndef EDIS_EXACT_MATH
#define EDIS_EXACT_MATH 0
#endif
__device__ __forceinline__ float ex2_fast(float x) {
#if EDIS_EXACT_MATH
  return exp2f(x);
#else
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
#endif
}
__device__ __forceinline__ float rcp_fast(float x) {
#if EDIS_EXACT_MATH
  return __frcp_rn(x);
#else
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
#endif
}
// s = sigmoid(e) and sp = s (1 - s) from u = exp(-|e|) in (0, 1]:  s = 1 / (1 + u) (e >= 0) or u / (1 + u),
// sp = u / (1 + u)^2.  The derivative never goes through "1 - s": with s rounded to fp32 that difference
// loses log2(1 / (1 - s)) bits, i.e. 1e-5 .. 1e-3 relative for logits of 3 .. 8 (chameleon's features reach
// |x| ~ 892, so such logits are common there), which showed up as 5e-5 on a score-weight gradient.
__device__ __forceinline__ void sigmoid_pair(float e, float& s, float& sp) {
  const float u = ex2_fast(-1.4426950408889634f * fabsf(e));
  const float r = rcp_fast(1.0f + u);
  const float ur = u * r;
  s = e >= 0.0f ? r : ur;
  sp = ur * r;
}
__device__ __forceinline__ float sigmoid_mufu(float e) {
  float s, sp;
  sigmoid_pair(e, s, sp);
  return s;
}
__device__ __forceinline__ float exp_mufu(float s) { return ex2_fast(1.4426950408889634f * s); }
__device__ __forceinline__ float lrelu01(float z) { return fmaxf(z, 0.01f * z); }

// Counter-based dropout mask: murmur3-style finaliser over (seed, element index).  Train-mode
// parity with the reference is "within seed noise" (its CPU and CUDA streams already differ),
// so the generator only has to be uniform and reproducible between fwd and bwd.
__device__ __forceinline__ float keep_scale(uint64_t seed, uint64_t idx, float p, float inv_keep) {
  uint32_t x = static_cast<uint32_t>(idx) ^ static_cast<uint32_t>(seed);
  x *= 0x9E3779B1u;
  x ^= static_cast<uint32_t>(idx >> 32) * 0x85EBCA77u + static_cast<uint32_t>(seed >> 32);
  x ^= x >> 16;
  x *= 0x85EBCA6Bu;
  x ^= x >> 13;
  x *= 0xC2B2AE35u;
  x ^= x >> 16;
  const float u = static_cast<float>(x >> 8) * (1.0f / 16777216.0f);
  return u >= p ? inv_keep : 0.0f;
}

__device__ __forceinline__ void red_add4(float* addr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c),
               "f"(d)
               : "memory");
}

// One instruction, one thread: pull `bytes` (multiple of 16, 16-byte aligned) from DRAM into L2.
// Used to run the gathers a few edges ahead of the consuming loads without registers or smem.
__device__ __forceinline__ void prefetch_l2_bulk(const void* p, unsigned bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}

// ---- L2 residency control for the gathers -------------------------------------------------
// The device copies of `col` / `cscrow` carry a 2-bit "heat" level of the neighbour in bits 30-31
// (3: among the 4K most-gathered nodes, 2: top 16K, 1: top 64K, 0: the rest).  Rows of hot
// neighbours are loaded with an evict_last L2 policy, all other gathered rows with evict_first,
// so the hub rows of a power-law graph stay resident in the 126 MB L2 instead of competing
// with the streaming rows under plain LRU.
constexpr int kHeatShift = 30;
constexpr int kIdMask = (1 << kHeatShift) - 1;
// Policy words of createpolicy.fractional.L2::evict_{first,last} with fraction 1.0, passed as
// IMMEDIATES: the cache-hint operand of ld / cp.async.bulk.prefetch must be warp-uniform, and a
// policy held in an ordinary register makes the compiler wrap every hinted access in a
// per-distinct-value loop (R2UR + BRA.U.ANY).  Hot / cold is therefore a BRANCH on the (warp-
// uniform) heat bits with a constant policy on either side.
constexpr uint64_t kPolEvictFirst = 0x12F0000000000000ull;
constexpr uint64_t kPolEvictLast = 0x14F0000000000000ull;
// cold (non-hub) gathered rows: 1 = evict_first hint, 0 = plain loads
#ifndef EDIS_COLD_HINT
#define EDIS_COLD_HINT 1
#endif
template <bool HOT>
__device__ __forceinline__ float4 ldg4_pol(const float* ptr) {
  if (!HOT && !EDIS_COLD_HINT) return __ldg(reinterpret_cast<const float4*>(ptr));
  float4 v;
  asm volatile("ld.global.nc.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(ptr), "l"(HOT ? kPolEvictLast : kPolEvictFirst));
  return v;
}
// Per-thread L2 prefetch of the 128-byte line at p.  (cp.async.bulk.prefetch runs on the uniform
// datapath: issued for a per-lane address the compiler serialises it over the lanes with an
// R2UR / BRA.U.ANY loop, ~12 instructions per call; this one is a single LSU instruction for 32
// different lines.)
template <bool HOT>
__device__ __forceinline__ void prefetch_l2_line(const void* p) {
  if (HOT) asm volatile("prefetch.global.L2::evict_last [%0];" ::"l"(p));
  else asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}
__device__ __forceinline__ bool is_hot(int raw, int hot_min) {
  return (static_cast<unsigned>(raw) >> kHeatShift) >= static_cast<unsigned>(hot_min);
}
// Per-edge records (logits, sign bits, (alpha, d logit)) are written once and read once per pass:
// streaming (evict-first) accesses keep them from displacing the gathered node rows in L2.
#ifndef EDIS_STREAM_HINT
#define EDIS_STREAM_HINT 1
#endif
template <class V>
__device__ __forceinline__ void st_stream(V* p, V v) {
  if (EDIS_STREAM_HINT) __stcs(p, v); else *p = v;
}
template <class V>
__device__ __forceinline__ V ld_stream(const V* p) {
  return EDIS_STREAM_HINT ? __ldcs(p) : __ldg(p);
}

// att-3 sign record: for each edge one bit per element of z = P_i + Q_j, bit set <=> z > 0.
// The forward works on w = (-P_i) - Q_j = -z (negations are free operand modifiers) and pushes the
// SIGN BIT of w into the record with one funnel shift per element, so element r of R ends up at bit
// R-1-r.  (z == +0 from P_i = Q_j = +0 reads as positive (w = -0), where torch's leaky_relu takes the
// 0.01 side; everything else, incl. an exact cancellation P_i = -Q_j != 0 (w = +0) and -0, matches
// z > 0.  Both operands are +0 for all-zero rows x_i = x_j = 0, which carry no gradient to W, but also
// when each dot product cancels exactly inside nonzero rows: there the element's gradient to W is taken
// with slope 1 instead of 0.01.  Matching torch would cost an instruction per element.)
__device__ __forceinline__ unsigned sign_push(unsigned mask, float w) {
  return __funnelshift_l(__float_as_uint(w), mask, 1);
}
template <int R>
__device__ __forceinline__ bool sign_pos(unsigned mask, int r) { return (mask & (1u << (R - 1 - r))) != 0u; }
// 1.0f if element r is positive, else 0.0f -- integer arithmetic only (AND + multiply by the constant
// that moves the bit onto 0x3f800000), no predicate registers: 16 of them live at once is more
// than ptxas can allocate in the whole-row kernels.
template <int R>
__device__ __forceinline__ float sign_pos_f(unsigned mask, int r) {
  static_assert(R <= 24, "sign record wider than the float-one trick supports");
  const int b = R - 1 - r;
  return __uint_as_float((mask & (1u << b)) * (0x3f800000u >> b));
}

// ---- asynchronous bulk staging (1-D TMA): global -> shared::cta, completion on an mbarrier --------
// SASS: UBLKCP.S.G + SYNCS.ARRIVE.TRANS64 / SYNCS.PHASECHK (B200_PROFILING.md).  One elected lane issues
// a whole gathered row (2-4 KB) with ONE instruction; the consumers read it with LDS.128 -- no per-lane
// 64-bit address chains, no registers held across the DRAM latency.
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// blocks (hardware sleep, not a spin on the LSU) until the phase with the given parity has completed
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "EDIS_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra EDIS_DONE;\n"
      "bra EDIS_WAIT;\n"
      "EDIS_DONE:\n"
      "}\n" ::"r"(bar), "r"(parity) : "memory");
}
// bytes: multiple of 16; dst / src 16-byte aligned.  HOT: keep the source lines in L2 (hub rows).
template <bool HOT>
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar), "l"(HOT ? kPolEvictLast : kPolEvictFirst) : "memory");
}

// same with the L2 policy in a register (issued by one lane, so the uniform-datapath move costs nothing extra
// and the hot / cold choice needs no branch)
__device__ __forceinline__ void bulk_g2s_pol(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar, uint64_t policy) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar), "l"(policy) : "memory");
}
__device__ __forceinline__ uint64_t l2_policy(int raw, int hot_min) { return is_hot(raw, hot_min) ? kPolEvictLast : kPolEvictFirst; }

int launch_grid(const void* kernel, int block, size_t smem, int sm_count);

}  // namespace edis
