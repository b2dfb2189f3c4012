// Fused DisGALayer kernels for sm_100a: all C channels of one DISGAT layer per launch.
//
// Replaces /root/reference/layers.py:349-416 (+ F.elu at 500/509), utils.py:192-207 and the
// aggregation of SageConv / GraphConvolution (layers.py:96-110, 38-54), forward and backward.
// HBM-bound gather / segment-reduce work: no tensor cores.  Scheduling:
//   * persistent grid (multiple of the SM count), one warp per (row chunk, channel group);
//   * rows longer than max_chunk are split into chunks whose partial sums go through a
//     small partial buffer + combine kernel (power-law hubs do not serialise a warp);
//   * per edge a warp gathers the source row with 128-bit coalesced loads (VecT) and reduces
//     the per-channel dot products with warp shuffles over the D/4 lanes of a channel;
//   * softmax is single pass: logits go through a sigmoid first (layers.py:392), so
//     exp(sigmoid(e)) is in (1, e) and needs no running max;
//   * backward = destination pass over CSR (dP, d logits) + source pass over CSC (dQ, dV):
//     pull on both sides, no float atomics on node tensors, deterministic.
// Template parameter RX selects the aggregated operand: RX == 0 -> per-channel V[N, C*D]
// (gnn_type AT / GCN); RX > 0 -> the raw input X[N, F <= 32*RX] shared by all channels
// (gnn_type SAGE, or AT / GCN run as aggregate-then-project), accumulated lane-strided;
// RX == -1 -> the same shared operand when F == D on the 128-bit layouts: one float4 of X_j per
// lane feeds all of the lane's channel slots (256 B gathered per edge instead of C*D*4).
#include <type_traits>

#include "edis_common.cuh"
#include "traits.cuh"

// Tuning knobs (build-time): edges in flight per warp for the 128-bit paths and the minimum
// resident CTAs per SM the register allocator must allow.
#ifndef EDIS_U_KV1
#define EDIS_U_KV1 4
#endif
#ifndef EDIS_U_KV2
#define EDIS_U_KV2 2
#endif
#ifndef EDIS_U_KV4
#define EDIS_U_KV4 1
#endif
// destination pass of att 3 (no Q gather): edges in flight on the whole-row path
#ifndef EDIS_UB_KV4
#define EDIS_UB_KV4 2
#endif
// source pass on the whole-row path: edges in flight
#ifndef EDIS_USRC_KV4
#define EDIS_USRC_KV4 2
#endif
// shared-operand 128-bit path (RX == -1), whole-row warps: edges in flight
#ifndef EDIS_US_KV4
#define EDIS_US_KV4 2
#endif
#ifndef EDIS_MINB
#define EDIS_MINB 2
#endif
#ifndef EDIS_MINB_DST
#define EDIS_MINB_DST EDIS_MINB
#endif
// L2 prefetch distance (edges ahead of the consuming loads) for the 128-bit paths; 0 = off
#ifndef EDIS_PF
#define EDIS_PF 2
#endif
#ifndef EDIS_PF_SRC
#define EDIS_PF_SRC 0
#endif
// ring (bulk-copy) variants: slots per warp
#ifndef EDIS_NS_DST
#define EDIS_NS_DST 4
#endif
#ifndef EDIS_NS_SRC
#define EDIS_NS_SRC 4
#endif
#ifndef EDIS_NS_FWD
#define EDIS_NS_FWD 3
#endif

namespace edis {

struct LayerArgs {
  const Item* items;
  int64_t n_edges;          // edges of the pass's index (CSR or CSC): items cover [0, n_edges) in order
  int64_t n_units;          // items * G
  int G;                    // channel groups per item
  const int32_t* nbr;       // CSR col (dst pass / fwd) or CSC row (src pass)
  const int32_t* eid;       // CSC -> CSR slot (src pass)
  const float *P, *Q, *a, *V, *bias;   // V doubles as X[N, F] in SAGE mode
  int64_t ldp, ldq, ldv;
  int C, D, F;
  // forward outputs / saved
  float *out, *hpre, *edge_e, *stats;  // SAGE: hpre = neigh[N, C*F], out unused
  // backward
  const float *g_out, *g_edge_e;
  float *gP, *gQ, *ga, *gV, *edge_rec, *gh;
  unsigned char* esign;              // att 3: sign bits of P_i + Q_j per edge (forward -> both backward passes)
  int64_t ldgp, ldgq, ldgv;          // row strides of gP, gQ, gV
  float* partial;
  int64_t pwidth;
  int hot_min;              // neighbours with heat >= hot_min get the evict_last L2 policy (4 = off)
  int training;
  int plain;                // shared-operand mode: 1 = plain softmax mean (AT/GCN aggregate-then-project),
                            // 0 = SAGE neighbour mean (divide by detached rowsum + 1)
  float p, inv_keep;
  uint64_t seed;
};

template <int RX>
__device__ __forceinline__ void load_x(float (&x)[RX > 0 ? RX : 1], const float* base, int lane, int F) {
#pragma unroll
  for (int k = 0; k < RX; ++k) x[k] = (k * 32 + lane < F) ? __ldg(base + k * 32 + lane) : 0.0f;
}
template <int RX>
__device__ __forceinline__ void store_x(float* base, const float (&x)[RX > 0 ? RX : 1], int lane, int F) {
#pragma unroll
  for (int k = 0; k < RX; ++k)
    if (k * 32 + lane < F) base[k * 32 + lane] = x[k];
}

// ------------------------------------------------------------------ forward
template <class T, int ATT, int RX, int U>
__global__ void __launch_bounds__(256, EDIS_MINB) k_disga_fwd(const LayerArgs A) {
  constexpr int R = T::R, NCH = T::NCH, RPC = T::RPC, CPW = T::CPW;
  constexpr int RXA = RX > 0 ? RX : 1, NACC = RX > 0 ? CPW * RX : 1;
  constexpr bool SHV = RX < 0;          // shared operand in the 128-bit layout (F == D)
  constexpr int PF = (T::kVec && RX <= 0) ? EDIS_PF : 0;
  constexpr int SBPL = (R + 7) / 8;   // sign bytes per lane per edge
  // The whole warp pulls the row parts of the edge PF steps ahead into L2, one 128-byte line per
  // lane: lanes [0, R) the score part Q_j, lanes [R, 2R) the value part V_j (R*128 bytes each);
  // shared operand: F*4 bytes of X_j.
  constexpr int QL = ATT >= 2 ? R : 0;                 // lines of the score part
  auto prefetch_src = [&](int raw, int off, int lane) {
    const int64_t j = raw & kIdMask;
    const int vl = lane - QL;                          // line of the value part
    const float* pp = nullptr;
    if (lane < QL) pp = A.Q + j * A.ldq + off + lane * 32;
    else if (SHV ? vl * 32 < A.D : vl < R) pp = A.V + j * A.ldv + (SHV ? 0 : off) + vl * 32;
    if (pp) {
      if (is_hot(raw, A.hot_min)) prefetch_l2_line<true>(pp); else prefetch_l2_line<false>(pp);
    }
  };
  const int lane = threadIdx.x & 31;
  const int xoff = (lane % T::LPCV) * 4;   // SHV: this lane's float4 of the shared operand
  const int64_t nwarps = static_cast<int64_t>(gridDim.x) * (blockDim.x >> 5);
  int64_t unit = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  for (; unit < A.n_units; unit += nwarps) {
    const int64_t item_id = unit / A.G;
    const int grp = static_cast<int>(unit - item_id * A.G);
    const Item it = A.items[item_id];
    const int c0 = grp * CPW;
    const int off = c0 * A.D;
    const int myc = c0 + T::own_ch(lane);   // the channel whose scalar math this lane owns
    const int64_t srow = static_cast<int64_t>(it.row);
    float pr[R], ar[R], sd = 0.0f;
    if (ATT >= 2) T::load(pr, A.P + srow * A.ldp + off, lane, A.D);
    if (ATT == 3) {
      T::load(ar, A.a + off, lane, A.D);
#pragma unroll
      for (int r = 0; r < R; ++r) ar[r] = -ar[r];
    }
    if (ATT == 1) sd = __ldg(A.P + srow * A.ldp + myc);
    float acc[R], accx[NACC], ws = 0.0f, wms = 0.0f;
    zero<T>(acc);
#pragma unroll
    for (int k = 0; k < NACC; ++k) accx[k] = 0.0f;

    for (int eb = it.beg; eb < it.end; eb += 32) {
      const int cnt = min(32, it.end - eb);
      const int myj = lane < cnt ? __ldg(A.nbr + eb + lane) : 0;
      if (PF > 0) {
#pragma unroll
        for (int pq = 0; pq < PF; ++pq)
          if (pq < cnt) prefetch_src(__shfl_sync(FULL, myj, pq), off, lane);
      }
      for (int t = 0; t < cnt; t += U) {
        if (PF > 0) {
#pragma unroll
          for (int u = 0; u < U; ++u)
            if (t + u + PF < cnt) prefetch_src(__shfl_sync(FULL, myj, t + u + PF), off, lane);
        }
        float q[U][R], h[RX == 0 ? U : 1][R], qs[U], xj[U][RXA];
        float4 hx[SHV ? U : 1];
        // a short tail re-reads the last edge of the block (same cache lines) with weight 0
        // instead of guarding every load / FMA with a branch
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int raw = __shfl_sync(FULL, myj, min(t + u, cnt - 1));
          const int64_t j = raw & kIdMask;
          const float* qp = A.Q + j * A.ldq + off;
          const float* vp = A.V + j * A.ldv + (SHV ? xoff : off);
          auto go = [&](auto hot) {
            constexpr bool H = decltype(hot)::value;
            if (ATT >= 2) T::template load_pol<H>(q[u], qp, lane, A.D);
            if (RX == 0) T::template load_pol<H>(h[RX == 0 ? u : 0], vp, lane, A.D);
            else if (SHV) hx[SHV ? u : 0] = ldg4_pol<H>(vp);
          };
          if (is_hot(raw, A.hot_min)) go(std::true_type{}); else go(std::false_type{});
          if (ATT == 1) qs[u] = __ldg(A.Q + j * A.ldq + myc);
          if (RX > 0) load_x<RX>(xj[u], A.V + j * A.ldv, lane, A.F);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const bool valid = U == 1 || t + u < cnt;
          {
            const int64_t edge = eb + min(t + u, cnt - 1);
            float e;
            if (ATT == 1) {
              e = sd + qs[u];
            } else {
              float part[NCH];
              unsigned mask = 0u;
#pragma unroll
              for (int k = 0; k < NCH; ++k) part[k] = 0.0f;
#pragma unroll
              for (int r = 0; r < R; ++r) {
                if (ATT == 3) {
                  // w = -(P_i + Q_j); ar holds -a: a * lrelu(z) = (-a) * min(w, 0.01 w)
                  const float w = -pr[r] - q[u][r];
                  mask = sign_push(mask, w);
                  part[r / RPC] = fmaf(ar[r], fminf(w, 0.01f * w), part[r / RPC]);
                } else {
                  part[r / RPC] = fmaf(pr[r], q[u][r], part[r / RPC]);
                }
              }
              if (ATT == 3 && A.esign && valid) {
                // 1 bit per element of P_i + Q_j, saved for the backward: leaky-relu is piecewise
                // linear, so neither backward pass needs z itself, only lrelu'(z)
                const int64_t so = ((edge * A.G + grp) * 32 + lane) * SBPL;
                if (SBPL == 1) st_stream(A.esign + so, static_cast<unsigned char>(mask));
                else st_stream(reinterpret_cast<unsigned short*>(A.esign + so), static_cast<unsigned short>(mask));
              }
              e = T::reduce_own(part, lane);
            }
            const float w = valid ? exp_mufu(sigmoid_mufu(e)) : 0.0f;
            const float ms = A.training ? keep_scale(A.seed, edge * A.C + myc, A.p, A.inv_keep) : 1.0f;
            const float wm = w * ms;
            ws += w;
            wms += wm;
            if (RX == 0) {
#pragma unroll
              for (int k = 0; k < NCH; ++k) {
                const float wk = T::from_owner(wm, k, lane);
#pragma unroll
                for (int r = k * RPC; r < (k + 1) * RPC; ++r) acc[r] = fmaf(wk, h[RX == 0 ? u : 0][r], acc[r]);
              }
            } else if (SHV) {
              const float4 hv = hx[SHV ? u : 0];
              const float x4[4] = {hv.x, hv.y, hv.z, hv.w};
#pragma unroll
              for (int k = 0; k < NCH; ++k) {
                const float wk = T::from_owner(wm, k, lane);
#pragma unroll
                for (int i = 0; i < 4; ++i) acc[(k * 4 + i) % R] = fmaf(wk, x4[i], acc[(k * 4 + i) % R]);
              }
            } else {
#pragma unroll
              for (int cc = 0; cc < CPW; ++cc) {
                const float wcc = T::from_channel(wm, cc);
#pragma unroll
                for (int k = 0; k < RX; ++k) accx[cc * RXA + k] = fmaf(wcc, xj[u][k], accx[cc * RXA + k]);
              }
            }
            if (T::own_writer(lane) && valid) st_stream(A.edge_e + edge * A.C + myc, e);
          }
        }
      }
    }
    if (RX == 0) {
      if (it.slot < 0) {
        float o[R], hp[R], br[R];
        if (A.bias) T::load(br, A.bias + off, lane, A.D);
#pragma unroll
        for (int k = 0; k < NCH; ++k) {
          const float wsum = T::from_owner(ws, k, lane);
          const float inv = wsum > 0.0f ? 1.0f / wsum : 0.0f;
#pragma unroll
          for (int r = k * RPC; r < (k + 1) * RPC; ++r) {
            // hpre keeps the aggregate BEFORE the bias: the backward needs <gh, agg> and recomputing
            // agg as (agg + b) - b would put a cancellation into the softmax gradient
            float v = acc[r] * inv;
            hp[r] = v;
            if (A.bias) v += br[r];
            o[r] = v > 0.0f ? v : expm1f(v);
          }
        }
        T::store(A.hpre + srow * A.C * A.D + off, hp, lane, A.D);
        T::store(A.out + srow * A.C * A.D + off, o, lane, A.D);
      } else {
        T::store(A.partial + static_cast<int64_t>(it.slot) * A.pwidth + off, acc, lane, A.D);
      }
    } else if (SHV) {
      // agg[i, c, :] = acc / (sum w [+ sum w*mask: SAGE's detached "row sum + 1"])
      if (it.slot < 0) {
#pragma unroll
        for (int k = 0; k < NCH; ++k) {
          const float den = T::from_owner(ws, k, lane) + (A.plain ? 0.0f : T::from_owner(wms, k, lane));
          const float inv = den > 0.0f ? 1.0f / den : 0.0f;
#pragma unroll
          for (int r = k * RPC; r < (k + 1) * RPC; ++r) acc[r] *= inv;
        }
        T::store(A.hpre + srow * A.C * A.D + off, acc, lane, A.D);
      } else {
        T::store(A.partial + static_cast<int64_t>(it.slot) * A.pwidth + off, acc, lane, A.D);
      }
    } else {
      // SAGE: neigh = agg / (rowsum(alpha_drop) + 1) = acc / (sum w*mask + sum w); plain: acc / sum w
#pragma unroll
      for (int cc = 0; cc < CPW; ++cc) {
        const float den = T::from_channel(ws, cc) + (A.plain ? 0.0f : T::from_channel(wms, cc));
        float o[RXA];
#pragma unroll
        for (int k = 0; k < RX; ++k)
          o[k] = it.slot < 0 ? (den > 0.0f ? accx[cc * RXA + k] / den : 0.0f) : accx[cc * RXA + k];
        float* dst = it.slot < 0 ? A.hpre + (srow * A.C + c0 + cc) * A.F
                                 : A.partial + static_cast<int64_t>(it.slot) * A.pwidth + (c0 + cc) * A.F;
        store_x<RX>(dst, o, lane, A.F);
      }
    }
    if (T::own_writer(lane)) {
      const int aggw = RX <= 0 ? A.C * A.D : A.C * A.F;
      float* st = it.slot < 0 ? A.stats + srow * 2 * A.C : A.partial + static_cast<int64_t>(it.slot) * A.pwidth + aggw;
      st[myc] = ws;
      st[A.C + myc] = wms;
    }
  }
}

// Split rows: sum the chunk partials, then the same epilogue.  One thread per (row, column).
// W = width per channel (D, or F in SAGE mode).
__global__ void k_combine_fwd(const SplitRow* split, int64_t n_split, const float* partial,
                              int64_t pwidth, int C, int W, int sage, const float* bias, float* out,
                              float* hpre, float* stats) {
  const int CW = C * W;
  const int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= n_split * CW) return;
  const SplitRow s = split[idx / CW];
  const int x = static_cast<int>(idx % CW);
  const int c = x / W;
  float acc = 0.0f, ws = 0.0f, wms = 0.0f, sx = 0.0f;
  for (int k = 0; k < s.slot_cnt; ++k) {
    const float* pb = partial + static_cast<int64_t>(s.slot_beg + k) * pwidth;
    acc += pb[x];
    ws += pb[CW + c];
    wms += pb[CW + C + c];
    if (x < 2 * C) sx += pb[CW + x];
  }
  const int64_t o = static_cast<int64_t>(s.row) * CW + x;
  if (sage) {
    const float den = sage == 2 ? ws : ws + wms;   // 2 = plain mean
    hpre[o] = den > 0.0f ? acc / den : 0.0f;
  } else {
    float v = ws > 0.0f ? acc / ws : 0.0f;
    hpre[o] = v;                       // pre-bias aggregate (see k_disga_fwd)
    if (bias) v += bias[x];
    out[o] = v > 0.0f ? v : expm1f(v);
  }
  if (x < 2 * C) stats[static_cast<int64_t>(s.row) * 2 * C + x] = sx;
}

// out[row*ld + x] = sum_slots partial[slot*pwidth + seg_off + x], x < seg_len
__global__ void k_combine_rows(const SplitRow* split, int64_t n_split, const float* partial,
                               int64_t pwidth, int seg_off, int seg_len, float* out, int64_t ld) {
  const int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= n_split * seg_len) return;
  const SplitRow s = split[idx / seg_len];
  const int x = static_cast<int>(idx % seg_len);
  float acc = 0.0f;
  for (int k = 0; k < s.slot_cnt; ++k)
    acc += partial[static_cast<int64_t>(s.slot_beg + k) * pwidth + seg_off + x];
  out[static_cast<int64_t>(s.row) * ld + x] = acc;
}

// ------------------------------------------------------------------ backward, destination pass
// Per row i: gh_i = grad wrt the aggregate (AT/GCN: g_out * elu'(hpre); SAGE: g_neigh / div);
// t_c = <gh_i, agg_i>_c (== sum_k alpha_ik dalpha_ik); per edge: d alpha_drop = <gh_i, V_j>_c,
// d logit = alpha (d alpha - t) * s(1-s) [+ g_edge_e]; accumulates dP_i (registers) and da
// (registers, flushed with vector atomics once per warp).
template <class T, int ATT, int RX, int U>
__global__ void __launch_bounds__(256, EDIS_MINB_DST) k_disga_bwd_dst(const LayerArgs A) {
  constexpr int R = T::R, NCH = T::NCH, RPC = T::RPC, CPW = T::CPW;
  constexpr int RXA = RX > 0 ? RX : 1, NACC = RX > 0 ? CPW * RX : 1;
  constexpr bool SHV = RX < 0;          // shared operand in the 128-bit layout (F == D)
  constexpr int PF = (T::kVec && RX <= 0) ? EDIS_PF : 0;
  // whole-warp L2 prefetch of the edge PF steps ahead, one 128-byte line per lane (see the forward)
  constexpr int QL = ATT == 2 ? R : 0;
  auto prefetch_src = [&](int raw, int off, int lane) {
    const int64_t j = raw & kIdMask;
    const int vl = lane - QL;
    const float* pp = nullptr;
    if (lane < QL) pp = A.Q + j * A.ldq + off + lane * 32;
    else if (SHV ? vl * 32 < A.D : vl < R) pp = A.V + j * A.ldv + (SHV ? 0 : off) + vl * 32;
    if (pp) {
      if (is_hot(raw, A.hot_min)) prefetch_l2_line<true>(pp); else prefetch_l2_line<false>(pp);
    }
  };
  constexpr int SBPL = (R + 7) / 8;   // sign bytes per lane per edge
  const int lane = threadIdx.x & 31;
  const int xoff = (lane % T::LPCV) * 4;   // SHV: this lane's float4 of the shared operand
  const int64_t nwarps = static_cast<int64_t>(gridDim.x) * (blockDim.x >> 5);
  int64_t unit = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  // att 3: this warp's running da lives in shared memory (touched once per ROW), not in registers
  __shared__ float s_da[ATT == 3 ? 8 * 32 * R : 1];
  float* my_da = s_da + (ATT == 3 ? (threadIdx.x >> 5) * 32 * R + lane : 0);
  auto flush_da = [&](int g) {
    float da[R];
#pragma unroll
    for (int r = 0; r < R; ++r) da[r] = my_da[r * 32];
    T::atomic_add(A.ga + g * CPW * A.D, da, lane, A.D);
  };
  int da_grp = -1;
  const int CD = A.C * A.D;
  for (; unit < A.n_units; unit += nwarps) {
    const int64_t item_id = unit / A.G;
    const int grp = static_cast<int>(unit - item_id * A.G);
    const Item it = A.items[item_id];
    const int c0 = grp * CPW;
    const int off = c0 * A.D;
    if (ATT == 3 && grp != da_grp) {
      if (da_grp >= 0) flush_da(da_grp);
#pragma unroll
      for (int r = 0; r < R; ++r) my_da[r * 32] = 0.0f;
      da_grp = grp;
    }
    const int myc = c0 + T::own_ch(lane);
    const int64_t srow = static_cast<int64_t>(it.row);
    const int64_t rowoff = srow * CD + off;
    // every chunk of a split row computes the same gh; the first chunk (or the only one) stores it
    bool first_chunk = it.slot < 0;
    if (it.slot >= 0) first_chunk = item_id == 0 || A.items[item_id - 1].row != it.row;
    float dh[R], dhx[NACC], tc = 0.0f;
    const float wsum = __ldg(A.stats + srow * 2 * A.C + myc);
    const float inv = wsum > 0.0f ? 1.0f / wsum : 0.0f;
    if (RX == 0) {
      float go[R], hp[R], br[R], tpart[NCH];
      T::load(go, A.g_out + rowoff, lane, A.D);
      T::load(hp, A.hpre + rowoff, lane, A.D);
      if (A.bias) T::load(br, A.bias + off, lane, A.D);
#pragma unroll
      for (int k = 0; k < NCH; ++k) tpart[k] = 0.0f;
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const float v = A.bias ? hp[r] + br[r] : hp[r];      // same fp32 op as the forward: bit-identical
        dh[r] = v > 0.0f ? go[r] : go[r] * expf(v);
        tpart[r / RPC] = fmaf(dh[r], hp[r], tpart[r / RPC]);
      }
      if (first_chunk) T::store(A.gh + rowoff, dh, lane, A.D);
      tc = T::reduce_own(tpart, lane);
    } else if (SHV) {
      // shared operand: gh = g_agg / div (div detached; plain mean: 1), t = <g_agg, agg>
      const float wmsv = __ldg(A.stats + srow * 2 * A.C + A.C + myc);
      const float den = wsum + wmsv;
      const float rdiv_own = A.plain ? 1.0f : (den > 0.0f ? wsum / den : 0.0f);
      float go[R], ng[R], tpart[NCH];
      T::load(go, A.g_out + rowoff, lane, A.D);
      T::load(ng, A.hpre + rowoff, lane, A.D);
#pragma unroll
      for (int k = 0; k < NCH; ++k) {
        tpart[k] = 0.0f;
        const float rdiv = T::from_owner(rdiv_own, k, lane);
#pragma unroll
        for (int r = k * RPC; r < (k + 1) * RPC; ++r) {
          dh[r] = go[r] * rdiv;
          tpart[k] = fmaf(go[r], ng[r], tpart[k]);
        }
      }
      if (first_chunk) T::store(A.gh + rowoff, dh, lane, A.D);
      tc = T::reduce_own(tpart, lane);
    } else {
      // SAGE: div = rowsum(alpha_drop) + 1 = (sum w*mask + sum w) / sum w, detached (layers.py:103)
      const float wmsv = __ldg(A.stats + srow * 2 * A.C + A.C + myc);
#pragma unroll
      for (int cc = 0; cc < CPW; ++cc) {
        const float wsc = T::from_channel(wsum, cc), den = wsc + T::from_channel(wmsv, cc);
        const float rdiv = A.plain ? 1.0f : (den > 0.0f ? wsc / den : 0.0f);   // 1 / div
        float gn[RXA], ng[RXA], o[RXA];
        load_x<RX>(gn, A.g_out + (srow * A.C + c0 + cc) * A.F, lane, A.F);
        load_x<RX>(ng, A.hpre + (srow * A.C + c0 + cc) * A.F, lane, A.F);
        float tp = 0.0f;
#pragma unroll
        for (int k = 0; k < RX; ++k) {
          dhx[cc * RXA + k] = gn[k] * rdiv;
          o[k] = dhx[cc * RXA + k];
          tp = fmaf(gn[k], ng[k], tp);     // <g_agg, agg> = <g_neigh, neigh>
        }
        tp = warp_sum(tp);
        if (T::own_ch(lane) == cc) tc = tp;
        if (first_chunk) store_x<RX>(A.gh + (srow * A.C + c0 + cc) * A.F, o, lane, A.F);
      }
    }

    // att 3: dP = 0.01 * (sum of all d logit) + 0.99 * (sum over the edges with z > 0): the second
    // sum is a predicated add per element, the first one add per channel slot
    float dP[R], dsum[NCH], dsd = 0.0f;
    zero<T>(dP);
#pragma unroll
    for (int k = 0; k < NCH; ++k) dsum[k] = 0.0f;

    for (int eb = it.beg; eb < it.end; eb += 32) {
      const int cnt = min(32, it.end - eb);
      const int myj = lane < cnt ? __ldg(A.nbr + eb + lane) : 0;
      if (PF > 0) {
#pragma unroll
        for (int pq = 0; pq < PF; ++pq)
          if (pq < cnt) prefetch_src(__shfl_sync(FULL, myj, pq), off, lane);
      }
      for (int t = 0; t < cnt; t += U) {
        if (PF > 0) {
#pragma unroll
          for (int u = 0; u < U; ++u)
            if (t + u + PF < cnt) prefetch_src(__shfl_sync(FULL, myj, t + u + PF), off, lane);
        }
        float q[ATT == 2 ? U : 1][R], h[RX == 0 ? U : 1][R], ev[U], gx[U], xj[U][RXA];
        float4 hx[SHV ? U : 1];
        unsigned sg[U];
        // a short tail re-reads the last edge of the block with d logit forced to 0 (no guards)
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int raw = __shfl_sync(FULL, myj, min(t + u, cnt - 1));
          const int64_t j = raw & kIdMask;
          const int64_t edge = eb + min(t + u, cnt - 1);
          const float* qp = A.Q + j * A.ldq + off;
          const float* vp = A.V + j * A.ldv + (SHV ? xoff : off);
          auto go = [&](auto hot) {
            constexpr bool H = decltype(hot)::value;
            if (ATT == 2) T::template load_pol<H>(q[ATT == 2 ? u : 0], qp, lane, A.D);
            if (RX == 0) T::template load_pol<H>(h[RX == 0 ? u : 0], vp, lane, A.D);
            else if (SHV) hx[SHV ? u : 0] = ldg4_pol<H>(vp);
          };
          if (is_hot(raw, A.hot_min)) go(std::true_type{}); else go(std::false_type{});
          if (ATT == 3) {
            // the forward's sign record of P_i + Q_j replaces the gather of Q_j (2 KB -> 64 B per edge)
            const int64_t so = ((edge * A.G + grp) * 32 + lane) * SBPL;
            sg[u] = SBPL == 1 ? static_cast<unsigned>(ld_stream(A.esign + so))
                              : static_cast<unsigned>(ld_stream(reinterpret_cast<const unsigned short*>(A.esign + so)));
          }
          if (RX > 0) load_x<RX>(xj[u], A.V + j * A.ldv, lane, A.F);
          ev[u] = ld_stream(A.edge_e + edge * A.C + myc);
          gx[u] = A.g_edge_e ? ld_stream(A.g_edge_e + edge * A.C + myc) : 0.0f;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const bool valid = U == 1 || t + u < cnt;
          {
            const int64_t edge = eb + min(t + u, cnt - 1);
            float gdot = 0.0f;
            if (RX == 0) {
              float gpart[NCH];
#pragma unroll
              for (int k = 0; k < NCH; ++k) gpart[k] = 0.0f;
#pragma unroll
              for (int r = 0; r < R; ++r) gpart[r / RPC] = fmaf(dh[r], h[RX == 0 ? u : 0][r], gpart[r / RPC]);
              gdot = T::reduce_own(gpart, lane);
            } else if (SHV) {
              const float4 hv = hx[SHV ? u : 0];
              const float x4[4] = {hv.x, hv.y, hv.z, hv.w};
              float gpart[NCH];
#pragma unroll
              for (int k = 0; k < NCH; ++k) {
                gpart[k] = 0.0f;
#pragma unroll
                for (int i = 0; i < 4; ++i) gpart[k] = fmaf(dh[(k * 4 + i) % R], x4[i], gpart[k]);
              }
              gdot = T::reduce_own(gpart, lane);
            } else {
#pragma unroll
              for (int cc = 0; cc < CPW; ++cc) {
                float gp = 0.0f;
#pragma unroll
                for (int k = 0; k < RX; ++k) gp = fmaf(dhx[cc * RXA + k], xj[u][k], gp);
                gp = warp_sum(gp);
                if (T::own_ch(lane) == cc) gdot = gp;
              }
            }
            float s, sp;
            sigmoid_pair(ev[u], s, sp);
            const float alpha = exp_mufu(s) * inv;
            const float ms = A.training ? keep_scale(A.seed, edge * A.C + myc, A.p, A.inv_keep) : 1.0f;
            const float ds = alpha * (gdot * ms - tc);
            const float de = valid ? fmaf(ds, sp, gx[u]) : 0.0f;
            if (T::own_writer(lane) && valid) {
              st_stream(A.edge_rec + edge * 2 * A.C + myc, alpha * ms);
              st_stream(A.edge_rec + edge * 2 * A.C + A.C + myc, de);
            }
            if (ATT == 1) dsd += de;
            if (ATT >= 2) {
#pragma unroll
              for (int k = 0; k < NCH; ++k) {
                const float d = T::from_owner(de, k, lane);
                if (ATT == 3) dsum[k] += d;
#pragma unroll
                for (int r = k * RPC; r < (k + 1) * RPC; ++r) {
                  // att 3: dP accumulates the z > 0 part of U = sum_j de_ij lrelu'(z_ijd)
                  if (ATT == 3) {
                    dP[r] = fmaf(sign_pos_f<R>(sg[u], r), d, dP[r]);
                  } else {
                    dP[r] = fmaf(d, q[ATT == 2 ? u : 0][r], dP[r]);
                  }
                }
              }
            }
          }
        }
      }
    }
    if (ATT == 3) {
      // lrelu(z) = lrelu'(z) z  =>  da_d = sum_i P_i[d] U_i[d] + sum_j Q_j[d] U'_j[d]: per ROW, not per
      // edge (the source half is added by the src pass).  P_i and a are only needed here.
      float pr[R], ar[R];
      T::load(pr, A.P + srow * A.ldp + off, lane, A.D);
      T::load(ar, A.a + off, lane, A.D);
#pragma unroll
      for (int r = 0; r < R; ++r) {
        dP[r] = fmaf(0.99f, dP[r], 0.01f * dsum[r / RPC]);     // U_i = sum_j de_ij lrelu'(z_ijd)
        my_da[r * 32] = fmaf(pr[r], dP[r], my_da[r * 32]);
        dP[r] *= ar[r];                                        // scaled by a once per row
      }
    }
    if (it.slot < 0) {
      if (ATT >= 2) T::store(A.gP + srow * A.ldgp + off, dP, lane, A.D);
      if (ATT == 1 && T::own_writer(lane)) A.gP[srow * A.ldgp + myc] = dsd;
    } else {
      float* pb = A.partial + static_cast<int64_t>(it.slot) * A.pwidth;
      if (ATT >= 2) T::store(pb + off, dP, lane, A.D);
      if (ATT == 1 && T::own_writer(lane)) pb[myc] = dsd;
    }
  }
  if (ATT == 3 && da_grp >= 0) flush_da(da_grp);
}

// ------------------------------------------------------------------ backward, source pass
// Per source row j over its out-edges (CSC): dV_j = sum_i alpha_drop_ij gh_i (HASV),
// dQ_j = sum_i d logit_ij * d e_ij / d Q_j.  Pull: gathers gh_i (and, for att 2, P_i), no atomics
// on node tensors.  att 3 reads the forward's 1-bit-per-element sign record instead of P_i.
// HASV: 0 = score side only; 1 = per-channel operand (dV_j[C*D]); 2 = shared operand in the 128-bit
// layout (F == D, one channel group): dX_j[F] = sum_i sum_c alpha_drop_ij^c gh_i^c, summed over the
// lane's channel slots in registers and over the warp's channel groups with shuffles once per row.
template <class T, int ATT, int HASV, int U>
__global__ void __launch_bounds__(256, EDIS_MINB) k_disga_bwd_src(const LayerArgs A) {
  constexpr int R = T::R, NCH = T::NCH, RPC = T::RPC, CPW = T::CPW;
  constexpr int SBPL = (R + 7) / 8;
  constexpr int PF = T::kVec ? EDIS_PF_SRC : 0;
  constexpr int QL = ATT == 2 ? R : 0;
  auto prefetch_dst = [&](int raw, int off, int lane) {
    const int64_t i = raw & kIdMask;
    const int vl = lane - QL;
    const float* pp = nullptr;
    if (lane < QL) pp = A.P + i * A.ldp + off + lane * 32;
    else if (HASV && vl < R) pp = A.gh + i * A.C * A.D + off + vl * 32;
    if (pp) {
      if (is_hot(raw, A.hot_min)) prefetch_l2_line<true>(pp); else prefetch_l2_line<false>(pp);
    }
  };
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = static_cast<int64_t>(gridDim.x) * (blockDim.x >> 5);
  int64_t unit = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int CD = A.C * A.D;
  // att 3: this warp's running da lives in shared memory (touched once per ROW), not in registers
  __shared__ float s_da[ATT == 3 ? 8 * 32 * R : 1];
  float* my_da = s_da + (ATT == 3 ? (threadIdx.x >> 5) * 32 * R + lane : 0);
  auto flush_da = [&](int g) {
    float da[R];
#pragma unroll
    for (int r = 0; r < R; ++r) da[r] = my_da[r * 32];
    T::atomic_add(A.ga + g * CPW * A.D, da, lane, A.D);
  };
  int da_grp = -1;
  for (; unit < A.n_units; unit += nwarps) {
    const int64_t item_id = unit / A.G;
    const int grp = static_cast<int>(unit - item_id * A.G);
    const Item it = A.items[item_id];
    const int c0 = grp * CPW;
    const int off = c0 * A.D;
    if (ATT == 3 && grp != da_grp) {
      if (da_grp >= 0) flush_da(da_grp);
#pragma unroll
      for (int r = 0; r < R; ++r) my_da[r * 32] = 0.0f;
      da_grp = grp;
    }
    int cidx[NCH];
#pragma unroll
    for (int k = 0; k < NCH; ++k) cidx[k] = c0 + T::ch(k, lane);
    // att 3: accQ holds the z > 0 part (predicated adds), dss the sum of all d logit per slot:
    // U'_j = 0.01 * dss + 0.99 * accQ
    float accV[R], accQ[R], dss[NCH], accX[4] = {0.0f, 0.0f, 0.0f, 0.0f};
    zero<T>(accV);
    zero<T>(accQ);
#pragma unroll
    for (int k = 0; k < NCH; ++k) dss[k] = 0.0f;
    for (int eb = it.beg; eb < it.end; eb += 32) {
      const int cnt = min(32, it.end - eb);
      const int myi = lane < cnt ? __ldg(A.nbr + eb + lane) : 0;
      const int mye = lane < cnt ? __ldg(A.eid + eb + lane) : 0;
      if (PF > 0) {
#pragma unroll
        for (int pq = 0; pq < PF; ++pq)
          if (pq < cnt) prefetch_dst(__shfl_sync(FULL, myi, pq), off, lane);
      }
      for (int t = 0; t < cnt; t += U) {
        if (PF > 0) {
#pragma unroll
          for (int u = 0; u < U; ++u)
            if (t + u + PF < cnt) prefetch_dst(__shfl_sync(FULL, myi, t + u + PF), off, lane);
        }
        float pg[ATT == 2 ? U : 1][R], dh[HASV ? U : 1][R], ad[U][NCH], de[U][NCH];
        unsigned sg[U];
        // a short tail re-reads the last edge of the block with its weights forced to 0 (no guards)
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const bool valid = U == 1 || t + u < cnt;
          const int raw = __shfl_sync(FULL, myi, min(t + u, cnt - 1));
          const int64_t i = raw & kIdMask;
          const int64_t edge = __shfl_sync(FULL, mye, min(t + u, cnt - 1));
          const float* pp = A.P + i * A.ldp + off;
          const float* gp = A.gh + i * CD + off;
          auto go = [&](auto hot) {
            constexpr bool H = decltype(hot)::value;
            if (ATT == 2) T::template load_pol<H>(pg[ATT == 2 ? u : 0], pp, lane, A.D);
            if (HASV) T::template load_pol<H>(dh[HASV ? u : 0], gp, lane, A.D);
          };
          if (is_hot(raw, A.hot_min)) go(std::true_type{}); else go(std::false_type{});
          if (ATT == 3) {
            const int64_t so = ((edge * A.G + grp) * 32 + lane) * SBPL;
            sg[u] = SBPL == 1 ? static_cast<unsigned>(ld_stream(A.esign + so))
                              : static_cast<unsigned>(ld_stream(reinterpret_cast<const unsigned short*>(A.esign + so)));
          }
#pragma unroll
          for (int k = 0; k < NCH; ++k) {
            if (HASV) ad[u][k] = valid ? ld_stream(A.edge_rec + edge * 2 * A.C + cidx[k]) : 0.0f;
            de[u][k] = valid ? ld_stream(A.edge_rec + edge * 2 * A.C + A.C + cidx[k]) : 0.0f;
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
#pragma unroll
          for (int k = 0; k < NCH; ++k) {
            const float d = de[u][k];
#pragma unroll
            for (int r = k * RPC; r < (k + 1) * RPC; ++r) {
              if (HASV == 1) accV[r] = fmaf(ad[u][k], dh[HASV ? u : 0][r], accV[r]);
              if (HASV == 2) accX[r % 4] = fmaf(ad[u][k], dh[HASV ? u : 0][r], accX[r % 4]);
              if (ATT == 3) {
                accQ[r] = fmaf(sign_pos_f<R>(sg[u], r), d, accQ[r]);
              } else if (ATT == 2) {
                accQ[r] = fmaf(d, pg[ATT == 2 ? u : 0][r], accQ[r]);
              }
            }
            if (ATT != 2) dss[k] += d;
          }
        }
      }
    }
    if (ATT == 3 && it.end > it.beg) {
      float qr[R], ar[R];
      T::load(qr, A.Q + static_cast<int64_t>(it.row) * A.ldq + off, lane, A.D);
      T::load(ar, A.a + off, lane, A.D);
#pragma unroll
      for (int r = 0; r < R; ++r) {
        accQ[r] = fmaf(0.99f, accQ[r], 0.01f * dss[r / RPC]);
        my_da[r * 32] = fmaf(qr[r], accQ[r], my_da[r * 32]);   // source half of da (see the dst pass)
        accQ[r] *= ar[r];
      }
    }
    if (HASV == 2) {
#pragma unroll
      for (int o = T::LPCV; o < 32; o <<= 1) {
#pragma unroll
        for (int i = 0; i < 4; ++i) accX[i] += __shfl_xor_sync(FULL, accX[i], o);
      }
      float* dst = it.slot < 0 ? A.gV + static_cast<int64_t>(it.row) * A.ldgv
                               : A.partial + static_cast<int64_t>(it.slot) * A.pwidth;
      if (lane < T::LPCV) *reinterpret_cast<float4*>(dst + lane * 4) = make_float4(accX[0], accX[1], accX[2], accX[3]);
    }
    if (it.slot < 0) {
      if (HASV == 1) T::store(A.gV + static_cast<int64_t>(it.row) * A.ldgv + off, accV, lane, A.D);
      if (ATT >= 2) T::store(A.gQ + static_cast<int64_t>(it.row) * A.ldgq + off, accQ, lane, A.D);
      if (ATT == 1 && T::writer(lane)) {
#pragma unroll
        for (int k = 0; k < NCH; ++k) A.gQ[static_cast<int64_t>(it.row) * A.ldgq + cidx[k]] = dss[k];
      }
    } else {
      float* pb = A.partial + static_cast<int64_t>(it.slot) * A.pwidth;
      if (HASV == 1) T::store(pb + off, accV, lane, A.D);
      if (ATT >= 2) T::store(pb + CD + off, accQ, lane, A.D);
      if (ATT == 1 && T::writer(lane)) {
#pragma unroll
        for (int k = 0; k < NCH; ++k) pb[CD + cidx[k]] = dss[k];
      }
    }
  }
  if (ATT == 3 && da_grp >= 0) flush_da(da_grp);
}

// SAGE: gX_j = sum_i sum_c alpha_drop_ij^c gh_i^c.  One warp per source-row chunk, all channels.
template <int RX>
__global__ void __launch_bounds__(256) k_sage_bwd_src_x(const LayerArgs A) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = static_cast<int64_t>(gridDim.x) * (blockDim.x >> 5);
  int64_t unit = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  for (; unit < A.n_units; unit += nwarps) {
    const Item it = A.items[unit];
    float acc[RX];
#pragma unroll
    for (int k = 0; k < RX; ++k) acc[k] = 0.0f;
    for (int eb = it.beg; eb < it.end; eb += 32) {
      const int cnt = min(32, it.end - eb);
      const int myi = lane < cnt ? __ldg(A.nbr + eb + lane) : 0;
      const int mye = lane < cnt ? __ldg(A.eid + eb + lane) : 0;
      for (int t = 0; t < cnt; ++t) {
        const int64_t i = __shfl_sync(FULL, myi, t) & kIdMask;
        const int64_t edge = __shfl_sync(FULL, mye, t);
        for (int c = 0; c < A.C; ++c) {
          const float ad = __ldg(A.edge_rec + edge * 2 * A.C + c);
          float g[RX];
          load_x<RX>(g, A.gh + (i * A.C + c) * A.F, lane, A.F);
#pragma unroll
          for (int k = 0; k < RX; ++k) acc[k] = fmaf(ad, g[k], acc[k]);
        }
      }
    }
    float* dst = it.slot < 0 ? A.gV + static_cast<int64_t>(it.row) * A.F
                             : A.partial + static_cast<int64_t>(it.slot) * A.pwidth;
    store_x<RX>(dst, acc, lane, A.F);
  }
}

// ------------------------------------------------------------------ ring (1-D TMA) variants
// Same math as the kernels above for the layouts where one warp owns a node's WHOLE row (att 3,
// per-channel operand, C == channels per warp: C = 8 / 4 / 2 at D = 64), restructured around
// asynchronous bulk copies:
//   * every warp owns a CONTIGUOUS run of work items (and therefore of edges), balanced by
//     edges + kRowCost * rows, found by binary search on the item list -- so its gathers can run
//     ahead across row boundaries (median in-degree of a power-law graph is ~9: per-row pipeline
//     restarts were most of the exposed latency);
//   * lane 0 issues ONE cp.async.bulk per gathered row (2 KB of V_j / gh_i, 4 KB of Q_j | V_j) into
//     a private shared-memory ring of NS slots, NS edges ahead, each slot with its own mbarrier;
//     the warp waits on the slot's phase and reads the row with LDS.128.  Compared with the per-lane
//     LDG.128 path: 1 instruction instead of 16 LDG + 64-bit address chains per edge, no staging
//     registers held across the DRAM latency, and NS rows per warp in flight independent of the
//     consumer's progress.
#ifndef EDIS_ROW_COST
#define EDIS_ROW_COST 2
#endif
#ifndef EDIS_RPW
#define EDIS_RPW 2
#endif
constexpr int kRowCost = EDIS_ROW_COST;   // cost of one work item in units of edges (row prologue / epilogue)
constexpr int kRangesPerWarp = EDIS_RPW;  // contiguous runs per warp (tail balance vs pipeline restarts)

struct WarpRange {
  int64_t i0, i1;   // items [i0, i1)
};
// first item whose cost prefix  beg_i + kRowCost * i  is >= target  (items are in edge order)
__device__ __forceinline__ int64_t item_lower_bound(const Item* items, int64_t n_items, int64_t target) {
  int64_t lo = 0, hi = n_items;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    const int64_t c = static_cast<int64_t>(__ldg(&items[mid].beg)) + kRowCost * mid;
    if (c < target) lo = mid + 1; else hi = mid;
  }
  return lo;
}
__device__ __forceinline__ WarpRange warp_range(const LayerArgs& A, int64_t rg, int64_t n_ranges) {
  const int64_t total = A.n_edges + kRowCost * A.n_units;
  const int64_t lo = total / n_ranges * rg + min(rg, total % n_ranges);
  const int64_t hi = total / n_ranges * (rg + 1) + min(rg + 1, total % n_ranges);
  WarpRange r;
  r.i0 = item_lower_bound(A.items, A.n_units, lo);
  r.i1 = rg + 1 == n_ranges ? A.n_units : item_lower_bound(A.items, A.n_units, hi);
  return r;
}

// Per-warp producer / consumer state of the ring.  ROWB = bytes per slot.
template <int NS, int ROWB>
struct Ring {
  unsigned char* slots;
  uint32_t bar0;         // shared-space address of this warp's first mbarrier
  uint32_t slot0;        // shared-space address of this warp's first slot
  uint32_t kp, kc;       // rows issued / rows consumed so far (slot = k % NS, phase parity = (k / NS) & 1)
  __device__ __forceinline__ void init(unsigned char* dyn, int wid, int lane) {
    slots = dyn + static_cast<size_t>(wid) * NS * ROWB;
    uint64_t* bars = reinterpret_cast<uint64_t*>(dyn + static_cast<size_t>(8) * NS * ROWB) + wid * NS;
    bar0 = smem_u32(bars);
    slot0 = smem_u32(slots);
    kp = kc = 0;
    if (lane == 0) {
#pragma unroll
      for (int s = 0; s < NS; ++s) mbar_init(bar0 + 8 * s, 1);
    }
    mbar_fence_init();
    __syncwarp();
  }
  __device__ __forceinline__ const unsigned char* wait_next() {      // all lanes
    const uint32_t s = kc % NS;
    mbar_wait(bar0 + 8 * s, (kc / NS) & 1u);
    ++kc;
    return slots + s * ROWB;
  }
};

// Neighbour ids of the 32-edge blocks the consumer (block b0) and the producer (b0 or b0 + 1) are in, plus
// block b0 + 2 already in flight: the load of a block is issued a whole block (32 edges) before the
// producer first needs it.  (With only two blocks the first `at()` after a block crossing waited a full
// DRAM latency on the index load: 23 % of the destination pass's stall samples, profiles/r2a.)
// (edge indices fit int32: edis_graph_create rejects e >= 2^31 - 64)
struct NbrWindow {
  int b0;
  int j0, j1, j2;
  __device__ __forceinline__ int ld(const int32_t* nbr, int n_edges, int i) const {
    return i < n_edges ? __ldg(nbr + i) : 0;
  }
  __device__ __forceinline__ void load(const int32_t* nbr, int n_edges, int e, int lane) {
    b0 = e >> 5;
    const int i0 = (b0 << 5) + lane;
    j0 = ld(nbr, n_edges, i0);
    j1 = ld(nbr, n_edges, i0 + 32);
    j2 = ld(nbr, n_edges, i0 + 64);
  }
  __device__ __forceinline__ void advance_to(const int32_t* nbr, int n_edges, int e, int lane) {
    if ((e >> 5) != b0) {
      b0 = e >> 5;
      j0 = j1;
      j1 = j2;
      j2 = ld(nbr, n_edges, (b0 << 5) + 64 + lane);
    }
  }
  __device__ __forceinline__ int at(int e) const {      // e in block b0 or b0 + 1; all lanes
    return __shfl_sync(FULL, (e >> 5) == b0 ? j0 : j1, e & 31);
  }
};

// backward, destination pass (att 3, per-channel operand, whole-row warps): ring of V_j rows
template <class T, int NS, bool TRAIN, bool GX>
__global__ void __launch_bounds__(256, EDIS_MINB_DST) k_disga_bwd_dst_ring(const LayerArgs A) {
  constexpr int R = T::R, NCH = T::NCH, RPC = T::RPC;
  constexpr int ROWB = R * 128;         // C * D * 4 bytes with C == T::CPW
  constexpr int SBPL = (R + 7) / 8;
  extern __shared__ __align__(128) unsigned char dyn_smem[];
  __shared__ float s_da[8 * 32 * R];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  Ring<NS, ROWB> ring;
  ring.init(dyn_smem, wid, lane);
  float* my_da = s_da + wid * 32 * R + lane;
#pragma unroll
  for (int r = 0; r < R; ++r) my_da[r * 32] = 0.0f;
  const int64_t nwarps = static_cast<int64_t>(gridDim.x) * 8;
  const int64_t n_ranges = nwarps * kRangesPerWarp;
  const int CD = A.C * A.D;
  const int myc = T::own_ch(lane);
  bool touched = false;
  for (int64_t rg = static_cast<int64_t>(blockIdx.x) * 8 + wid; rg < n_ranges; rg += nwarps) {
    const WarpRange wr = warp_range(A, rg, n_ranges);
    if (wr.i0 >= wr.i1) continue;
    touched = true;
    const int e0 = __ldg(&A.items[wr.i0].beg), e1 = __ldg(&A.items[wr.i1 - 1].end);
    const int n_edges = static_cast<int>(A.n_edges);
    NbrWindow nw;
    nw.load(A.nbr, n_edges, e0, lane);
    int pe = e0;
    // all lanes; lane 0 issues the copy of edge pe's source row when pe < e1 (ONE predicate: the index is
    // clamped so that the shuffle is unconditional)
    auto issue = [&]() {
      const int raw = nw.at(min(pe, e1 - 1));
      if (lane == 0 && pe < e1) {
        const uint32_t s = ring.kp % NS;
        const uint32_t bar = ring.bar0 + 8 * s;
        mbar_expect_tx(bar, ROWB);
        bulk_g2s_pol(ring.slot0 + s * ROWB, A.V + static_cast<int64_t>(raw & kIdMask) * A.ldv, ROWB, bar,
                     l2_policy(raw, A.hot_min));
      }
      ring.kp += pe < e1 ? 1u : 0u;
      ++pe;
    };
    for (int q = 0; q < NS; ++q) issue();      // (a run of edge-less rows has e0 == e1: nothing is issued)
    int e = e0;
    unsigned sg_n = 0u;
    float ev_n = 0.0f, gx_n = 0.0f;
    auto load_edge = [&](int ee) {      // ee clamped by the caller: no branch
      const int64_t so = (static_cast<int64_t>(ee) * 32 + lane) * SBPL;
      sg_n = SBPL == 1 ? static_cast<unsigned>(ld_stream(A.esign + so))
                       : static_cast<unsigned>(ld_stream(reinterpret_cast<const unsigned short*>(A.esign + so)));
      ev_n = ld_stream(A.edge_e + static_cast<int64_t>(ee) * A.C + myc);
      if (GX) gx_n = ld_stream(A.g_edge_e + static_cast<int64_t>(ee) * A.C + myc);
    };
    if (e0 < e1) load_edge(e0);
    for (int64_t item_id = wr.i0; item_id < wr.i1; ++item_id) {
      const Item it = A.items[item_id];
      const int64_t srow = static_cast<int64_t>(it.row);
      const int64_t rowoff = srow * CD;
      bool first_chunk = it.slot < 0;
      if (it.slot >= 0) first_chunk = item_id == 0 || A.items[item_id - 1].row != it.row;
      // the next item's row data (g_out, hpre: 2 x ROWB bytes, consecutive rows) into L2 while this row runs
      if (item_id + 1 < wr.i1) {
        const int64_t nrow = static_cast<int64_t>(__ldg(&A.items[item_id + 1].row)) * CD;
        if (lane < R) {
          prefetch_l2_line<false>(A.g_out + nrow + lane * 32);
          prefetch_l2_line<false>(A.P + static_cast<int64_t>(__ldg(&A.items[item_id + 1].row)) * A.ldp + lane * 32);
        } else if (lane < 2 * R) {
          prefetch_l2_line<false>(A.hpre + nrow + (lane - R) * 32);
        }
      }
      float dh[R], tc;
      const float wsum = __ldg(A.stats + srow * 2 * A.C + myc);
      const float inv = wsum > 0.0f ? 1.0f / wsum : 0.0f;
      {
        float go[R], hp[R], br[R], tpart[NCH];
        T::load(go, A.g_out + rowoff, lane, A.D);
        T::load(hp, A.hpre + rowoff, lane, A.D);
        if (A.bias) T::load(br, A.bias, lane, A.D);
#pragma unroll
        for (int k = 0; k < NCH; ++k) tpart[k] = 0.0f;
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const float v = A.bias ? hp[r] + br[r] : hp[r];
          dh[r] = v > 0.0f ? go[r] : go[r] * expf(v);
          tpart[r / RPC] = fmaf(dh[r], hp[r], tpart[r / RPC]);
        }
        if (first_chunk) T::store(A.gh + rowoff, dh, lane, A.D);
        tc = T::reduce_own(tpart, lane);
      }
      float dP[R], dsum[NCH];
      zero<T>(dP);
#pragma unroll
      for (int k = 0; k < NCH; ++k) dsum[k] = 0.0f;
      for (; e < it.end; ++e) {
        nw.advance_to(A.nbr, n_edges, e, lane);
        // per-edge streams (coalesced, sequential in e): sign record, logit, upstream logit gradient --
        // loaded ONE EDGE AHEAD into registers so that their latency hides under this edge's math
        const unsigned sg = sg_n;
        const float ev = ev_n, gx = gx_n;
        load_edge(min(e + 1, e1 - 1));
        const float* sp = reinterpret_cast<const float*>(ring.wait_next());
        float h[R];
#pragma unroll
        for (int k = 0; k < T::KV; ++k) {
          const float4 v = *reinterpret_cast<const float4*>(sp + (k * 32 + lane) * 4);
          h[4 * k] = v.x; h[4 * k + 1] = v.y; h[4 * k + 2] = v.z; h[4 * k + 3] = v.w;
        }
        float gpart[NCH];
#pragma unroll
        for (int k = 0; k < NCH; ++k) gpart[k] = 0.0f;
#pragma unroll
        for (int r = 0; r < R; ++r) gpart[r / RPC] = fmaf(dh[r], h[r], gpart[r / RPC]);
        const float gdot = T::reduce_own(gpart, lane);     // shuffles: every lane has consumed its slot reads
        issue();                                           // refill the slot just read
        float s, sgrad;
        sigmoid_pair(ev, s, sgrad);
        const float alpha = exp_mufu(s) * inv;
        const float ms = TRAIN ? keep_scale(A.seed, static_cast<int64_t>(e) * A.C + myc, A.p, A.inv_keep) : 1.0f;
        const float ds = alpha * (gdot * ms - tc);
        const float de = fmaf(ds, sgrad, gx);
        if (T::own_writer(lane)) {
          st_stream(A.edge_rec + static_cast<int64_t>(e) * 2 * A.C + myc, alpha * ms);
          st_stream(A.edge_rec + static_cast<int64_t>(e) * 2 * A.C + A.C + myc, de);
        }
#pragma unroll
        for (int k = 0; k < NCH; ++k) {
          const float d = T::from_owner(de, k, lane);
          dsum[k] += d;
#pragma unroll
          for (int r = k * RPC; r < (k + 1) * RPC; ++r) dP[r] = fmaf(sign_pos_f<R>(sg, r), d, dP[r]);
        }
      }
      {
        float pr[R], ar[R];
        T::load(pr, A.P + srow * A.ldp, lane, A.D);
        T::load(ar, A.a, lane, A.D);
#pragma unroll
        for (int r = 0; r < R; ++r) {
          dP[r] = fmaf(0.99f, dP[r], 0.01f * dsum[r / RPC]);
          my_da[r * 32] = fmaf(pr[r], dP[r], my_da[r * 32]);
          dP[r] *= ar[r];
        }
      }
      if (it.slot < 0) T::store(A.gP + srow * A.ldgp, dP, lane, A.D);
      else T::store(A.partial + static_cast<int64_t>(it.slot) * A.pwidth, dP, lane, A.D);
    }
  }
  if (touched) {
    float da[R];
#pragma unroll
    for (int r = 0; r < R; ++r) da[r] = my_da[r * 32];
    T::atomic_add(A.ga, da, lane, A.D);
  }
}

// backward, source pass (att 3, per-channel operand): ring of {gh_i row, (alpha_drop, d logit) record,
// sign record} per out-edge of the source row -- the two per-edge records sit at the edge's CSR slot
// (random 64-byte reads over CSC): they ride the same mbarrier as the row
template <class T, int NS>
__global__ void __launch_bounds__(256, EDIS_MINB) k_disga_bwd_src_ring(const LayerArgs A) {
  constexpr int R = T::R, NCH = T::NCH, RPC = T::RPC;
  constexpr int ROWB = R * 128;
  constexpr int SBPL = (R + 7) / 8;
  constexpr int RECB = 2 * T::CPW * 4;          // (alpha_drop, d logit)[2C] floats
  constexpr int SIGNB = 32 * SBPL;
  constexpr int SLOTB = ROWB + RECB + SIGNB;
  static_assert(RECB % 16 == 0 && SIGNB % 16 == 0, "bulk copies move multiples of 16 bytes");
  extern __shared__ __align__(128) unsigned char dyn_smem[];
  __shared__ float s_da[8 * 32 * R];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  Ring<NS, SLOTB> ring;
  ring.init(dyn_smem, wid, lane);
  float* my_da = s_da + wid * 32 * R + lane;
#pragma unroll
  for (int r = 0; r < R; ++r) my_da[r * 32] = 0.0f;
  const int64_t nwarps = static_cast<int64_t>(gridDim.x) * 8;
  const int64_t n_ranges = nwarps * kRangesPerWarp;
  const int CD = A.C * A.D;
  int cidx[NCH];
#pragma unroll
  for (int k = 0; k < NCH; ++k) cidx[k] = T::ch(k, lane);
  bool touched = false;
  for (int64_t rg = static_cast<int64_t>(blockIdx.x) * 8 + wid; rg < n_ranges; rg += nwarps) {
    const WarpRange wr = warp_range(A, rg, n_ranges);
    if (wr.i0 >= wr.i1) continue;
    touched = true;
    const int e0 = __ldg(&A.items[wr.i0].beg), e1 = __ldg(&A.items[wr.i1 - 1].end);
    const int n_edges = static_cast<int>(A.n_edges);
    NbrWindow nw, ew;
    nw.load(A.nbr, n_edges, e0, lane);
    ew.load(A.eid, n_edges, e0, lane);
    int pe = e0;
    auto issue = [&]() {
      const int pc = min(pe, e1 - 1);
      const int raw = nw.at(pc);
      const int64_t edge = ew.at(pc);
      if (lane == 0 && pe < e1) {
        const uint32_t s = ring.kp % NS;
        const uint32_t bar = ring.bar0 + 8 * s;
        const uint32_t dst = ring.slot0 + s * SLOTB;
        mbar_expect_tx(bar, SLOTB);
        bulk_g2s_pol(dst, A.gh + static_cast<int64_t>(raw & kIdMask) * CD, ROWB, bar, l2_policy(raw, A.hot_min));
        bulk_g2s<false>(dst + ROWB, A.edge_rec + edge * 2 * A.C, RECB, bar);
        bulk_g2s<false>(dst + ROWB + RECB, A.esign + edge * SIGNB, SIGNB, bar);
      }
      ring.kp += pe < e1 ? 1u : 0u;
      ++pe;
    };
    for (int q = 0; q < NS; ++q) issue();      // (a run of edge-less rows has e0 == e1: nothing is issued)
    int e = e0;
    for (int64_t item_id = wr.i0; item_id < wr.i1; ++item_id) {
      const Item it = A.items[item_id];
      if (item_id + 1 < wr.i1 && lane < R)      // next source row's Q_j (row epilogue operand) into L2
        prefetch_l2_line<false>(A.Q + static_cast<int64_t>(__ldg(&A.items[item_id + 1].row)) * A.ldq + lane * 32);
      float accV[R], accQ[R], dss[NCH];
      zero<T>(accV);
      zero<T>(accQ);
#pragma unroll
      for (int k = 0; k < NCH; ++k) dss[k] = 0.0f;
      for (; e < it.end; ++e) {
        nw.advance_to(A.nbr, n_edges, e, lane);
        ew.advance_to(A.eid, n_edges, e, lane);
        const unsigned char* sp = ring.wait_next();
        const float* rowp = reinterpret_cast<const float*>(sp);
        const float* recp = reinterpret_cast<const float*>(sp + ROWB);
        float dh[R], ad[NCH], de[NCH];
#pragma unroll
        for (int k = 0; k < T::KV; ++k) {
          const float4 v = *reinterpret_cast<const float4*>(rowp + (k * 32 + lane) * 4);
          dh[4 * k] = v.x; dh[4 * k + 1] = v.y; dh[4 * k + 2] = v.z; dh[4 * k + 3] = v.w;
        }
#pragma unroll
        for (int k = 0; k < NCH; ++k) {
          ad[k] = recp[cidx[k]];
          de[k] = recp[A.C + cidx[k]];
        }
        const unsigned sg = SBPL == 1 ? static_cast<unsigned>(sp[ROWB + RECB + lane])
                                      : static_cast<unsigned>(reinterpret_cast<const unsigned short*>(sp + ROWB + RECB)[lane]);
#pragma unroll
        for (int k = 0; k < NCH; ++k) {
#pragma unroll
          for (int r = k * RPC; r < (k + 1) * RPC; ++r) {
            accV[r] = fmaf(ad[k], dh[r], accV[r]);
            accQ[r] = fmaf(sign_pos_f<R>(sg, r), de[k], accQ[r]);
          }
          dss[k] += de[k];
        }
        __syncwarp();                 // every lane has read the slot
        issue();
      }
      const int64_t jrow = static_cast<int64_t>(it.row);
      if (it.end > it.beg) {
        float qr[R], ar[R];
        T::load(qr, A.Q + jrow * A.ldq, lane, A.D);
        T::load(ar, A.a, lane, A.D);
#pragma unroll
        for (int r = 0; r < R; ++r) {
          accQ[r] = fmaf(0.99f, accQ[r], 0.01f * dss[r / RPC]);
          my_da[r * 32] = fmaf(qr[r], accQ[r], my_da[r * 32]);
          accQ[r] *= ar[r];
        }
      }
      if (it.slot < 0) {
        T::store(A.gV + jrow * A.ldgv, accV, lane, A.D);
        T::store(A.gQ + jrow * A.ldgq, accQ, lane, A.D);
      } else {
        float* pb = A.partial + static_cast<int64_t>(it.slot) * A.pwidth;
        T::store(pb, accV, lane, A.D);
        T::store(pb + CD, accQ, lane, A.D);
      }
    }
  }
  if (touched) {
    float da[R];
#pragma unroll
    for (int r = 0; r < R; ++r) da[r] = my_da[r * 32];
    T::atomic_add(A.ga, da, lane, A.D);
  }
}

// forward (att 3, per-channel operand): ring of Q_j | V_j (2 rows, contiguous in the projection buffer)
template <class T, int NS>
__global__ void __launch_bounds__(256, EDIS_MINB) k_disga_fwd_ring(const LayerArgs A) {
  constexpr int R = T::R, NCH = T::NCH, RPC = T::RPC;
  constexpr int ROWB = R * 128;
  constexpr int SLOTB = 2 * ROWB;
  constexpr int SBPL = (R + 7) / 8;
  extern __shared__ __align__(128) unsigned char dyn_smem[];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  Ring<NS, SLOTB> ring;
  ring.init(dyn_smem, wid, lane);
  const int64_t nwarps = static_cast<int64_t>(gridDim.x) * 8;
  const int64_t n_ranges = nwarps * kRangesPerWarp;
  const int CD = A.C * A.D;
  const int myc = T::own_ch(lane);
  float ar[R];
  T::load(ar, A.a, lane, A.D);
#pragma unroll
  for (int r = 0; r < R; ++r) ar[r] = -ar[r];
  for (int64_t rg = static_cast<int64_t>(blockIdx.x) * 8 + wid; rg < n_ranges; rg += nwarps) {
    const WarpRange wr = warp_range(A, rg, n_ranges);
    if (wr.i0 >= wr.i1) continue;
    const int e0 = __ldg(&A.items[wr.i0].beg), e1 = __ldg(&A.items[wr.i1 - 1].end);
    const int n_edges = static_cast<int>(A.n_edges);
    NbrWindow nw;
    nw.load(A.nbr, n_edges, e0, lane);
    int pe = e0;
    auto issue = [&]() {
      const int raw = nw.at(min(pe, e1 - 1));
      if (lane == 0 && pe < e1) {
        const uint32_t s = ring.kp % NS;
        const uint32_t bar = ring.bar0 + 8 * s;
        mbar_expect_tx(bar, SLOTB);
        bulk_g2s_pol(ring.slot0 + s * SLOTB, A.Q + static_cast<int64_t>(raw & kIdMask) * A.ldq, SLOTB, bar,
                     l2_policy(raw, A.hot_min));                                      // Q_j | V_j adjacent
      }
      ring.kp += pe < e1 ? 1u : 0u;
      ++pe;
    };
    for (int q = 0; q < NS; ++q) issue();      // (a run of edge-less rows has e0 == e1: nothing is issued)
    int e = e0;
    for (int64_t item_id = wr.i0; item_id < wr.i1; ++item_id) {
      const Item it = A.items[item_id];
      const int64_t srow = static_cast<int64_t>(it.row);
      if (item_id + 1 < wr.i1 && lane < R)
        prefetch_l2_line<false>(A.P + static_cast<int64_t>(__ldg(&A.items[item_id + 1].row)) * A.ldp + lane * 32);
      float pr[R];
      T::load(pr, A.P + srow * A.ldp, lane, A.D);
      float acc[R], ws = 0.0f, wms = 0.0f;
      zero<T>(acc);
      for (; e < it.end; ++e) {
        nw.advance_to(A.nbr, n_edges, e, lane);
        const float* sp = reinterpret_cast<const float*>(ring.wait_next());
        float q[R], h[R];
#pragma unroll
        for (int k = 0; k < T::KV; ++k) {
          const float4 v = *reinterpret_cast<const float4*>(sp + (k * 32 + lane) * 4);
          q[4 * k] = v.x; q[4 * k + 1] = v.y; q[4 * k + 2] = v.z; q[4 * k + 3] = v.w;
          const float4 u = *reinterpret_cast<const float4*>(sp + R * 32 + (k * 32 + lane) * 4);
          h[4 * k] = u.x; h[4 * k + 1] = u.y; h[4 * k + 2] = u.z; h[4 * k + 3] = u.w;
        }
        float part[NCH];
        unsigned mask = 0u;
#pragma unroll
        for (int k = 0; k < NCH; ++k) part[k] = 0.0f;
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const float w = -pr[r] - q[r];
          mask = sign_push(mask, w);
          part[r / RPC] = fmaf(ar[r], fminf(w, 0.01f * w), part[r / RPC]);
        }
        const float ev = T::reduce_own(part, lane);      // shuffles: q has been consumed by every lane
        // h is still only in registers of this lane: the slot is free once all lanes have loaded it
        issue();
        if (A.esign) {
          const int64_t so = (static_cast<int64_t>(e) * 32 + lane) * SBPL;
          if (SBPL == 1) st_stream(A.esign + so, static_cast<unsigned char>(mask));
          else st_stream(reinterpret_cast<unsigned short*>(A.esign + so), static_cast<unsigned short>(mask));
        }
        const float w = exp_mufu(sigmoid_mufu(ev));
        const float ms = A.training ? keep_scale(A.seed, static_cast<int64_t>(e) * A.C + myc, A.p, A.inv_keep) : 1.0f;
        const float wm = w * ms;
        ws += w;
        wms += wm;
#pragma unroll
        for (int k = 0; k < NCH; ++k) {
          const float wk = T::from_owner(wm, k, lane);
#pragma unroll
          for (int r = k * RPC; r < (k + 1) * RPC; ++r) acc[r] = fmaf(wk, h[r], acc[r]);
        }
        if (T::own_writer(lane)) st_stream(A.edge_e + static_cast<int64_t>(e) * A.C + myc, ev);
      }
      if (it.slot < 0) {
        float o[R], hp[R], br[R];
        if (A.bias) T::load(br, A.bias, lane, A.D);
#pragma unroll
        for (int k = 0; k < NCH; ++k) {
          const float wsum = T::from_owner(ws, k, lane);
          const float inv = wsum > 0.0f ? 1.0f / wsum : 0.0f;
#pragma unroll
          for (int r = k * RPC; r < (k + 1) * RPC; ++r) {
            float v = acc[r] * inv;
            hp[r] = v;
            if (A.bias) v += br[r];
            o[r] = v > 0.0f ? v : expm1f(v);
          }
        }
        T::store(A.hpre + srow * CD, hp, lane, A.D);
        T::store(A.out + srow * CD, o, lane, A.D);
      } else {
        T::store(A.partial + static_cast<int64_t>(it.slot) * A.pwidth, acc, lane, A.D);
      }
      if (T::own_writer(lane)) {
        float* st = it.slot < 0 ? A.stats + srow * 2 * A.C : A.partial + static_cast<int64_t>(it.slot) * A.pwidth + CD;
        st[myc] = ws;
        st[A.C + myc] = wms;
      }
    }
  }
}

// ------------------------------------------------------------------ host dispatch
enum class Pass { Fwd, BwdDst, BwdSrc };

template <class K>
static int launch_persistent(K kernel, const edis_graph* g, const LayerArgs& A, cudaStream_t st) {
  if (A.n_units == 0) return EDIS_OK;
  int blocks = launch_grid(reinterpret_cast<const void*>(kernel), 256, 0, g->sm_count);
  const int64_t need = (A.n_units + 7) / 8;
  if (need < blocks) blocks = static_cast<int>(need);
  kernel<<<blocks, 256, 0, st>>>(A);
  EDIS_CUDA(cudaGetLastError());
  return EDIS_OK;
}

// ring variants: whole-row warps (one channel group), 16-byte aligned rows, D == 64 layouts
template <class T>
static bool ring_ok(const LayerArgs& A) {
  static const int on = env_int("EDIS_RING", 1);
  return on && T::kRing && A.C == T::CPW && A.D == 64;
}

template <class K>
static int launch_ring(K kernel, int slot_bytes_per_warp, const edis_graph* g, const LayerArgs& A, cudaStream_t st) {
  if (A.n_units == 0) return EDIS_OK;
  const size_t smem = static_cast<size_t>(8) * slot_bytes_per_warp + 8 * 32 * sizeof(uint64_t);
  EDIS_CUDA(cudaFuncSetAttribute(reinterpret_cast<const void*>(kernel), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 static_cast<int>(smem)));
  int blocks = launch_grid(reinterpret_cast<const void*>(kernel), 256, smem, g->sm_count);
  const int64_t need = (A.n_units + 7) / 8;
  if (need < blocks) blocks = static_cast<int>(need);
  kernel<<<blocks, 256, smem, st>>>(A);
  EDIS_CUDA(cudaGetLastError());
  return EDIS_OK;
}

template <class T, int ATT, int RX, int U>
static int launch_pass(Pass pass, const edis_graph* g, LayerArgs A, cudaStream_t st) {
  A.G = A.C / T::CPW;
  const Schedule& s = pass == Pass::BwdSrc ? g->src : g->dst;
  A.items = s.items;
  A.n_edges = g->e;
  A.n_units = s.n_items * A.G;
  if (pass == Pass::Fwd) {
    if constexpr (ATT == 3 && RX == 0 && T::kRing) {
      // Q_j | V_j must be one contiguous 2-row block of the projection buffer
      static const int ring_fwd = env_int("EDIS_RING_FWD", 1);
      if (ring_fwd && ring_ok<T>(A) && A.ldq == A.ldv && A.V == A.Q + A.C * A.D)
        return launch_ring(&k_disga_fwd_ring<T, EDIS_NS_FWD>, EDIS_NS_FWD * 2 * T::R * 128, g, A, st);
    }
    return launch_persistent(&k_disga_fwd<T, ATT, RX, U>, g, A, st);
  }
  if (pass == Pass::BwdDst) {
    if constexpr (ATT == 3 && RX == 0 && T::kRing) {
      static const int ring_dst = env_int("EDIS_RING_DST", 1);
      if (ring_dst && ring_ok<T>(A)) {
        constexpr int sb = EDIS_NS_DST * T::R * 128;
        if (A.training) {
          if (A.g_edge_e) return launch_ring(&k_disga_bwd_dst_ring<T, EDIS_NS_DST, true, true>, sb, g, A, st);
          return launch_ring(&k_disga_bwd_dst_ring<T, EDIS_NS_DST, true, false>, sb, g, A, st);
        }
        if (A.g_edge_e) return launch_ring(&k_disga_bwd_dst_ring<T, EDIS_NS_DST, false, true>, sb, g, A, st);
        return launch_ring(&k_disga_bwd_dst_ring<T, EDIS_NS_DST, false, false>, sb, g, A, st);
      }
    }
    constexpr int UB = (ATT == 3 && RX == 0 && T::kVec && T::KV == 4) ? EDIS_UB_KV4 : U;
    return launch_persistent(&k_disga_bwd_dst<T, ATT, RX, UB>, g, A, st);
  }
  constexpr int US = (T::kVec && T::KV == 4) ? EDIS_USRC_KV4 : U;
  if constexpr (ATT == 3 && RX == 0 && T::kRing) {
    static const int ring_src = env_int("EDIS_RING_SRC", 1);
    if (ring_src && ring_ok<T>(A)) {
      constexpr int slot = T::R * 128 + 2 * T::CPW * 4 + 32 * ((T::R + 7) / 8);
      return launch_ring(&k_disga_bwd_src_ring<T, EDIS_NS_SRC>, EDIS_NS_SRC * slot, g, A, st);
    }
  }
  if (RX == 0) return launch_persistent(&k_disga_bwd_src<T, ATT, 1, US>, g, A, st);
  if (RX < 0) {
    if (A.gV) return launch_persistent(&k_disga_bwd_src<T, ATT, 2, US>, g, A, st);
    return launch_persistent(&k_disga_bwd_src<T, ATT, 0, US>, g, A, st);
  }
  return launch_persistent(&k_disga_bwd_src<T, ATT, 0, 4>, g, A, st);
}

template <class T, int RX, int U>
static int launch_att(Pass pass, const edis_graph* g, const LayerArgs& A, int att, cudaStream_t st) {
  switch (att) {
    case 1: return launch_pass<T, 1, RX, U>(pass, g, A, st);
    case 2: return launch_pass<T, 2, RX, U>(pass, g, A, st);
    case 3: return launch_pass<T, 3, RX, U>(pass, g, A, st);
  }
  set_error("att must be 1, 2 or 3 (got %d)", att);
  return EDIS_ERR_ARG;
}

int env_int(const char* name, int dflt) {
  const char* v = getenv(name);
  return v ? atoi(v) : dflt;
}

// Layout choice: D == 64 and even C -> 128-bit path (2 or 4 channels per warp); other shapes ->
// lane-strided scalar path (still CUDA; covers any C and D <= 256).
static int launch_layer(Pass pass, const edis_graph* g, const LayerArgs& A, int att, cudaStream_t st) {
  const int C = A.C, D = A.D;
  static const int kv_env = env_int("EDIS_KV", 0);
  if (D == 64 && C % 2 == 0) {
    int kv = kv_env ? kv_env : (C % 8 == 0 ? 4 : (C % 4 == 0 ? 2 : 1));
    if (kv == 4 && C % 8 == 0) return launch_att<VecT<4, 16>, 0, EDIS_U_KV4>(pass, g, A, att, st);
    if (kv >= 2 && C % 4 == 0) return launch_att<VecT<2, 16>, 0, EDIS_U_KV2>(pass, g, A, att, st);
    return launch_att<VecT<1, 16>, 0, EDIS_U_KV1>(pass, g, A, att, st);
  }
  if (D == 32 && C % 4 == 0) return launch_att<VecT<1, 8>, 0, 4>(pass, g, A, att, st);
  if (D == 128) return launch_att<VecT<1, 32>, 0, 4>(pass, g, A, att, st);
  if (D <= 32) return launch_att<ScaT<1>, 0, 4>(pass, g, A, att, st);
  if (D <= 64) return launch_att<ScaT<2>, 0, 4>(pass, g, A, att, st);
  if (D <= 128) return launch_att<ScaT<4>, 0, 2>(pass, g, A, att, st);
  if (D <= 256) return launch_att<ScaT<8>, 0, 1>(pass, g, A, att, st);
  set_error("unsupported channel width D=%d (max 256)", D);
  return EDIS_ERR_UNSUPPORTED;
}

template <class T>
static int launch_sage_rx(Pass pass, const edis_graph* g, const LayerArgs& A, int att, cudaStream_t st) {
  constexpr int U = T::R >= 8 ? 1 : 2;
  if (A.F <= 64) return launch_att<T, 2, U>(pass, g, A, att, st);
  if (A.F <= 128) return launch_att<T, 4, U>(pass, g, A, att, st);
  if (A.F <= 256) return launch_att<T, 8, 1>(pass, g, A, att, st);
  set_error("unsupported SAGE input width F=%d (max 256)", A.F);
  return EDIS_ERR_UNSUPPORTED;
}

// Shared operand on the 128-bit layouts: F == D == 64 and all channels in one warp (C = 2, 4, 8).
static bool sage_shared_vec(int C, int D, int F) {
  static const int on = env_int("EDIS_SHV", 1);
  return on && F == D && D == 64 && (C == 2 || C == 4 || C == 8);
}

static int launch_sage(Pass pass, const edis_graph* g, const LayerArgs& A, int att, cudaStream_t st) {
  const int C = A.C, D = A.D;
  if (sage_shared_vec(C, D, A.F)) {
    if (C == 8) return launch_att<VecT<4, 16>, -1, EDIS_US_KV4>(pass, g, A, att, st);
    if (C == 4) return launch_att<VecT<2, 16>, -1, 2>(pass, g, A, att, st);
    return launch_att<VecT<1, 16>, -1, 4>(pass, g, A, att, st);
  }
  if (D == 64 && C % 8 == 0) return launch_sage_rx<VecT<4, 16>>(pass, g, A, att, st);
  if (D == 64 && C % 4 == 0) return launch_sage_rx<VecT<2, 16>>(pass, g, A, att, st);
  if (D == 64 && C % 2 == 0) return launch_sage_rx<VecT<1, 16>>(pass, g, A, att, st);
  if (D <= 64) return launch_sage_rx<ScaT<2>>(pass, g, A, att, st);
  if (D <= 256) return launch_sage_rx<ScaT<8>>(pass, g, A, att, st);
  set_error("unsupported channel width D=%d (max 256)", D);
  return EDIS_ERR_UNSUPPORTED;
}

static int check_desc(const edis_layer_desc* d, const char* who) {
  EDIS_CHECK_ARG(d, "%s: null descriptor", who);
  EDIS_CHECK_ARG(d->att >= 1 && d->att <= 3, "%s: att=%d", who, d->att);
  EDIS_CHECK_ARG(d->C >= 1 && d->D >= 2, "%s: C=%d D=%d", who, d->C, d->D);
  EDIS_CHECK_ARG(!d->training || (d->p >= 0.0f && d->p < 1.0f), "%s: dropout p=%f", who, d->p);
  return EDIS_OK;
}

static bool vec_ok(const void* p, int64_t ld) {
  // the 128-bit path needs 16-byte aligned rows
  return (reinterpret_cast<uintptr_t>(p) % 16 == 0) && (ld % 4 == 0);
}

static void fill_common(LayerArgs& A, const edis_layer_desc* d, const float* P, int64_t ldp,
                        const float* Q, int64_t ldq, const float* a, const float* V, int64_t ldv,
                        void* workspace) {
  A.P = P; A.Q = Q; A.a = a; A.V = V;
  A.ldp = ldp; A.ldq = ldq; A.ldv = ldv;
  A.C = d->C; A.D = d->D; A.F = d->Dv;
  A.partial = static_cast<float*>(workspace);
  A.training = d->training && d->p > 0.0f;
  A.plain = (d->flags & EDIS_FLAG_PLAIN_MEAN) ? 1 : 0;
  static const int hot_env = env_int("EDIS_HOT_MIN", 2);
  A.hot_min = hot_env;
  A.p = d->p;
  A.inv_keep = 1.0f / (1.0f - d->p);
  A.seed = d->seed;
}

static int check_ws(const edis_graph* g, int64_t pw, void* workspace, int64_t bytes, const char* who) {
  if (g->device < 0) {
    set_error("%s: structure-only graph handle (created with device -1): nothing is resident on a GPU", who);
    return EDIS_ERR_ARG;
  }
  if ((g->dst.n_slots > 0 || g->src.n_slots > 0) &&
      (!workspace || bytes < edis_graph_workspace_bytes(g, pw))) {
    set_error("%s: workspace too small (%lld < %lld)", who, (long long)bytes,
              (long long)edis_graph_workspace_bytes(g, pw));
    return EDIS_ERR_WORKSPACE;
  }
  return EDIS_OK;
}

static unsigned nblk(int64_t total) { return static_cast<unsigned>((total + 255) / 256); }

// Edge scratch `edge_rec` (dst pass -> src pass): E x 2C floats (alpha_drop, d logit).
static int64_t rec_total_bytes(const edis_graph* g, const edis_layer_desc* d) {
  return g->e * 2 * static_cast<int64_t>(d->C) * static_cast<int64_t>(sizeof(float)) + 64;
}
// Sign record `esign` (att 3, forward -> backward): one bit per element of P_i + Q_j, stored per
// (edge, channel group, lane); at most E*C*32 bytes (the lane-strided layouts pad D to 32*ND).
static int64_t sign_total_bytes(const edis_graph* g, const edis_layer_desc* d) {
  return d->att == 3 ? g->e * static_cast<int64_t>(d->C) * 32 + 64 : 0;
}

// shared tail of the two backward entry points: score-side source pass + combines
static int bwd_score_src(const edis_graph* g, const edis_layer_desc* d, LayerArgs& A, bool sage,
                         float* gQ, float* gV, cudaStream_t st) {
  const int CD = d->C * d->D;
  A.nbr = g->cscrow;
  A.eid = g->csceid;
  int rc = sage ? launch_sage(Pass::BwdSrc, g, A, d->att, st) : launch_layer(Pass::BwdSrc, g, A, d->att, st);
  if (rc) return rc;
  if (g->src.n_split > 0) {
    if (!sage) {
      k_combine_rows<<<nblk(g->src.n_split * CD), 256, 0, st>>>(g->src.split, g->src.n_split, A.partial,
                                                               A.pwidth, 0, CD, gV, A.ldgv);
    }
    const int seg = d->att == 1 ? d->C : CD;
    k_combine_rows<<<nblk(g->src.n_split * seg), 256, 0, st>>>(g->src.split, g->src.n_split, A.partial,
                                                              A.pwidth, CD, seg, gQ, A.ldgq);
    if (sage && gV && sage_shared_vec(d->C, d->D, d->Dv)) {
      // fused dX of the 128-bit shared-operand path: its partials sit at the head of each slot
      k_combine_rows<<<nblk(g->src.n_split * d->Dv), 256, 0, st>>>(g->src.split, g->src.n_split, A.partial,
                                                                  A.pwidth, 0, d->Dv, gV, d->Dv);
    }
    EDIS_CUDA(cudaGetLastError());
  }
  return EDIS_OK;
}

}  // namespace edis

using namespace edis;

extern "C" int64_t edis_disga_rec_bytes(const edis_graph* g, const edis_layer_desc* d) {
  if (!g || !d || d->C < 1) return EDIS_ERR_ARG;
  return rec_total_bytes(g, d);
}

extern "C" int edis_disga_sage_fused_gx(const edis_layer_desc* d) {
  return d && sage_shared_vec(d->C, d->D, d->Dv) ? 1 : 0;
}

extern "C" int64_t edis_disga_sign_bytes(const edis_graph* g, const edis_layer_desc* d) {
  if (!g || !d || d->C < 1) return EDIS_ERR_ARG;
  return sign_total_bytes(g, d);
}

extern "C" int edis_disga_fwd(const edis_graph* g, const edis_layer_desc* d, const float* P,
                              int64_t ldp, const float* Q, int64_t ldq, const float* a,
                              const float* V, int64_t ldv, const float* bias, float* out,
                              float* hpre, float* edge_e, float* stats, uint8_t* esign,
                              void* workspace, int64_t workspace_bytes, void* stream) {
  int rc = check_desc(d, "edis_disga_fwd");
  if (rc) return rc;
  EDIS_CHECK_ARG(g && P && Q && V && out && hpre && edge_e && stats, "edis_disga_fwd: null pointer");
  EDIS_CHECK_ARG(d->Dv == d->D, "edis_disga_fwd: Dv (%d) must equal D (%d)", d->Dv, d->D);
  EDIS_CHECK_ARG(d->att != 3 || a, "edis_disga_fwd: att=3 needs a[C,D]");
  EDIS_CHECK_ARG(d->D % 4 != 0 || (vec_ok(V, ldv) && (d->att == 1 || (vec_ok(P, ldp) && vec_ok(Q, ldq))) &&
                                   vec_ok(out, 4) && vec_ok(hpre, 4)),
                 "edis_disga_fwd: node tensors must be 16-byte aligned with ld %% 4 == 0");
  const int64_t pw = static_cast<int64_t>(d->C) * d->D + 2 * d->C;
  if ((rc = check_ws(g, pw, workspace, workspace_bytes, "edis_disga_fwd"))) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  LayerArgs A = {};
  fill_common(A, d, P, ldp, Q, ldq, a, V, ldv, workspace);
  A.nbr = g->col;
  A.bias = bias;
  A.out = out; A.hpre = hpre; A.edge_e = edge_e; A.stats = stats;
  A.esign = esign;
  A.pwidth = pw;
  rc = launch_layer(Pass::Fwd, g, A, d->att, st);
  if (rc) return rc;
  if (g->dst.n_split > 0) {
    k_combine_fwd<<<nblk(g->dst.n_split * d->C * d->D), 256, 0, st>>>(
        g->dst.split, g->dst.n_split, A.partial, pw, d->C, d->D, 0, bias, out, hpre, stats);
    EDIS_CUDA(cudaGetLastError());
  }
  return EDIS_OK;
}

static int disga_bwd_impl(int phases, const edis_graph* g, const edis_layer_desc* d, const float* P,
                              int64_t ldp, const float* Q, int64_t ldq, const float* a,
                              const float* V, int64_t ldv, const float* bias, const float* hpre,
                              const float* edge_e, const float* stats, const uint8_t* esign,
                              const float* g_out,
                              const float* g_edge_e, float* gP, int64_t ldgp, float* gQ, int64_t ldgq, float* ga, float* gV, int64_t ldgv,
                              float* edge_rec, float* gh, void* workspace, int64_t workspace_bytes,
                              void* stream) {
  int rc = check_desc(d, "edis_disga_bwd");
  if (rc) return rc;
  EDIS_CHECK_ARG(g && P && Q && V && hpre && edge_e && stats && g_out && gP && gQ && gV && edge_rec && gh,
                 "edis_disga_bwd: null pointer");
  EDIS_CHECK_ARG(d->Dv == d->D, "edis_disga_bwd: Dv must equal D");
  EDIS_CHECK_ARG(d->att != 3 || (a && ga), "edis_disga_bwd: att=3 needs a and ga");
  EDIS_CHECK_ARG(d->att != 3 || esign, "edis_disga_bwd: att=3 needs the forward's sign record (esign)");
  EDIS_CHECK_ARG(d->D % 4 != 0 || (vec_ok(V, ldv) && (d->att == 1 || (vec_ok(P, ldp) && vec_ok(Q, ldq))) &&
                                   vec_ok(g_out, 4) && vec_ok(gV, ldgv) && vec_ok(gh, 4) &&
                                   (d->att == 1 || (vec_ok(gP, ldgp) && vec_ok(gQ, ldgq)))),
                 "edis_disga_bwd: node tensors must be 16-byte aligned with ld %% 4 == 0");
  const int CD = d->C * d->D;
  const int64_t pw = 2 * static_cast<int64_t>(CD) + 2 * d->C;
  if ((rc = check_ws(g, pw, workspace, workspace_bytes, "edis_disga_bwd"))) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  LayerArgs A = {};
  fill_common(A, d, P, ldp, Q, ldq, a, V, ldv, workspace);
  A.bias = bias;
  A.hpre = const_cast<float*>(hpre); A.edge_e = const_cast<float*>(edge_e); A.stats = const_cast<float*>(stats);
  A.g_out = g_out; A.g_edge_e = g_edge_e;
  A.gP = gP; A.gQ = gQ; A.ga = ga; A.gV = gV; A.edge_rec = edge_rec; A.gh = gh;
  A.esign = const_cast<uint8_t*>(esign);
  A.ldgp = ldgp; A.ldgq = ldgq; A.ldgv = ldgv;
  A.pwidth = pw;
  // heat level from which a gathered row is held in L2 (evict_last): the forward gathers 4 KB per
  // source (Q_j | V_j), the backward passes 2 KB (V_j resp. gh_i), so they can afford a larger hot set
  static const int hot_dst = env_int("EDIS_HOT_MIN_DST", 2);
  static const int hot_src = env_int("EDIS_HOT_MIN_SRC", 2);
  if (phases & 1) {
    A.nbr = g->col;
    A.hot_min = hot_dst;
    rc = launch_layer(Pass::BwdDst, g, A, d->att, st);
    if (rc) return rc;
    if (g->dst.n_split > 0) {
      const int seg = d->att == 1 ? d->C : CD;
      k_combine_rows<<<nblk(g->dst.n_split * seg), 256, 0, st>>>(g->dst.split, g->dst.n_split, A.partial, pw,
                                                                0, seg, gP, A.ldgp);
      EDIS_CUDA(cudaGetLastError());
    }
  }
  if (phases & 2) {
    A.hot_min = hot_src;
    return bwd_score_src(g, d, A, false, gQ, gV, st);
  }
  return EDIS_OK;
}

#define EDIS_BWD_ARGS                                                                               \
  const edis_graph *g, const edis_layer_desc *d, const float *P, int64_t ldp, const float *Q,       \
      int64_t ldq, const float *a, const float *V, int64_t ldv, const float *bias,                  \
      const float *hpre, const float *edge_e, const float *stats, const uint8_t *esign,             \
      const float *g_out,                                                                           \
      const float *g_edge_e, float *gP, int64_t ldgp, float *gQ, int64_t ldgq, float *ga,         \
      float *gV, int64_t ldgv, float *edge_rec,                                                     \
      float *gh, void *workspace, int64_t workspace_bytes, void *stream
#define EDIS_BWD_PASS                                                                               \
  g, d, P, ldp, Q, ldq, a, V, ldv, bias, hpre, edge_e, stats, esign, g_out, g_edge_e, gP, ldgp, gQ, ldgq, ga, gV, ldgv, \
      edge_rec, gh, workspace, workspace_bytes, stream

extern "C" int edis_disga_bwd(EDIS_BWD_ARGS) { return disga_bwd_impl(3, EDIS_BWD_PASS); }
extern "C" int edis_disga_bwd_dst(EDIS_BWD_ARGS) { return disga_bwd_impl(1, EDIS_BWD_PASS); }
extern "C" int edis_disga_bwd_src(EDIS_BWD_ARGS) { return disga_bwd_impl(2, EDIS_BWD_PASS); }



extern "C" int edis_disga_sage_fwd(const edis_graph* g, const edis_layer_desc* d, const float* P,
                                   int64_t ldp, const float* Q, int64_t ldq, const float* a,
                                   const float* X, int64_t ldx, float* neigh, float* edge_e,
                                   float* stats, uint8_t* esign, void* workspace,
                                   int64_t workspace_bytes, void* stream) {
  int rc = check_desc(d, "edis_disga_sage_fwd");
  if (rc) return rc;
  EDIS_CHECK_ARG(g && P && Q && X && neigh && edge_e && stats, "edis_disga_sage_fwd: null pointer");
  EDIS_CHECK_ARG(d->Dv >= 1 && d->Dv <= 256, "edis_disga_sage_fwd: F=%d (Dv) must be in [1, 256]", d->Dv);
  EDIS_CHECK_ARG(d->att != 3 || a, "edis_disga_sage_fwd: att=3 needs a[C,D]");
  EDIS_CHECK_ARG(d->att == 1 || d->D % 4 != 0 || (vec_ok(P, ldp) && vec_ok(Q, ldq)),
                 "edis_disga_sage_fwd: score operands must be 16-byte aligned with ld %% 4 == 0");
  EDIS_CHECK_ARG(!sage_shared_vec(d->C, d->D, d->Dv) || (vec_ok(X, ldx) && vec_ok(neigh, 4)),
                 "edis_disga_sage_fwd: X / neigh must be 16-byte aligned with ld %% 4 == 0");
  const int64_t pw = static_cast<int64_t>(d->C) * d->Dv + 2 * d->C;
  if ((rc = check_ws(g, pw, workspace, workspace_bytes, "edis_disga_sage_fwd"))) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  LayerArgs A = {};
  fill_common(A, d, P, ldp, Q, ldq, a, X, ldx, workspace);
  A.nbr = g->col;
  A.hpre = neigh; A.edge_e = edge_e; A.stats = stats;
  A.esign = esign;
  A.pwidth = pw;
  rc = launch_sage(Pass::Fwd, g, A, d->att, st);
  if (rc) return rc;
  if (g->dst.n_split > 0) {
    k_combine_fwd<<<nblk(g->dst.n_split * d->C * d->Dv), 256, 0, st>>>(
        g->dst.split, g->dst.n_split, A.partial, pw, d->C, d->Dv, A.plain ? 2 : 1, nullptr, nullptr, neigh, stats);
    EDIS_CUDA(cudaGetLastError());
  }
  return EDIS_OK;
}

extern "C" int edis_disga_sage_bwd(const edis_graph* g, const edis_layer_desc* d, const float* P,
                                   int64_t ldp, const float* Q, int64_t ldq, const float* a,
                                   const float* X, int64_t ldx, const float* neigh,
                                   const float* edge_e, const float* stats, const uint8_t* esign,
                                   const float* g_neigh,
                                   const float* g_edge_e, float* gP, int64_t ldgp, float* gQ,
                                   int64_t ldgq, float* ga, float* gX, float* edge_rec, float* gh,
                                   void* workspace, int64_t workspace_bytes, void* stream) {
  int rc = check_desc(d, "edis_disga_sage_bwd");
  if (rc) return rc;
  const bool need_gx = !(d->flags & EDIS_FLAG_NO_GX);
  EDIS_CHECK_ARG(g && P && Q && X && neigh && edge_e && stats && g_neigh && gP && gQ && (gX || !need_gx) &&
                     edge_rec && gh, "edis_disga_sage_bwd: null pointer");
  EDIS_CHECK_ARG(d->Dv >= 1 && d->Dv <= 256, "edis_disga_sage_bwd: F=%d (Dv) must be in [1, 256]", d->Dv);
  EDIS_CHECK_ARG(d->att != 3 || (a && ga), "edis_disga_sage_bwd: att=3 needs a and ga");
  EDIS_CHECK_ARG(d->att != 3 || esign, "edis_disga_sage_bwd: att=3 needs the forward's sign record (esign)");
  EDIS_CHECK_ARG(!sage_shared_vec(d->C, d->D, d->Dv) ||
                     (vec_ok(X, ldx) && vec_ok(neigh, 4) && vec_ok(g_neigh, 4) && vec_ok(gh, 4) && vec_ok(gX, 4)),
                 "edis_disga_sage_bwd: node tensors must be 16-byte aligned with ld %% 4 == 0");
  const int CD = d->C * d->D;
  // rounded up to 4 floats: the 128-bit layouts store a split row's partials with float4 stores, so every
  // slot must start 16-byte aligned (an odd F left odd slots misaligned)
  const int64_t pw = (2 * static_cast<int64_t>(CD) + 2 * d->C + d->Dv + 3) / 4 * 4;
  if ((rc = check_ws(g, pw, workspace, workspace_bytes, "edis_disga_sage_bwd"))) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  LayerArgs A = {};
  fill_common(A, d, P, ldp, Q, ldq, a, X, ldx, workspace);
  A.hpre = const_cast<float*>(neigh); A.edge_e = const_cast<float*>(edge_e); A.stats = const_cast<float*>(stats);
  A.g_out = g_neigh; A.g_edge_e = g_edge_e;
  A.gP = gP; A.gQ = gQ; A.ga = ga; A.gV = gX; A.edge_rec = edge_rec; A.gh = gh;
  A.esign = const_cast<uint8_t*>(esign);
  A.ldgp = ldgp; A.ldgq = ldgq; A.ldgv = d->Dv;
  A.pwidth = pw;
  const int ph = d->flags & EDIS_FLAG_PHASE_MASK;   // 0 = all passes
  if (!ph || (ph & EDIS_FLAG_PHASE_DST)) {
    A.nbr = g->col;
    rc = launch_sage(Pass::BwdDst, g, A, d->att, st);
    if (rc) return rc;
    if (g->dst.n_split > 0) {
      const int seg = d->att == 1 ? d->C : CD;
      k_combine_rows<<<nblk(g->dst.n_split * seg), 256, 0, st>>>(g->dst.split, g->dst.n_split, A.partial, pw,
                                                                0, seg, gP, A.ldgp);
      EDIS_CUDA(cudaGetLastError());
    }
  }
  const bool shv = sage_shared_vec(d->C, d->D, d->Dv);
  if (!need_gx) A.gV = nullptr;
  if (!ph || (ph & EDIS_FLAG_PHASE_SRC)) {
    // 128-bit shared-operand path: the source pass also produces gX (no separate gX kernel)
    rc = bwd_score_src(g, d, A, true, gQ, shv ? A.gV : nullptr, st);
    if (rc) return rc;
  }
  if (!need_gx || shv || (ph && !(ph & EDIS_FLAG_PHASE_GX))) return EDIS_OK;
  // gX: one warp per source-row chunk, all channels
  A.nbr = g->cscrow;
  A.eid = g->csceid;
  A.items = g->src.items;
  A.n_units = g->src.n_items;
  A.G = 1;
  if (d->Dv <= 64) rc = launch_persistent(&k_sage_bwd_src_x<2>, g, A, st);
  else if (d->Dv <= 128) rc = launch_persistent(&k_sage_bwd_src_x<4>, g, A, st);
  else rc = launch_persistent(&k_sage_bwd_src_x<8>, g, A, st);
  if (rc) return rc;
  if (g->src.n_split > 0) {
    k_combine_rows<<<nblk(g->src.n_split * d->Dv), 256, 0, st>>>(g->src.split, g->src.n_split, A.partial, pw,
                                                                0, d->Dv, gX, d->Dv);
    EDIS_CUDA(cudaGetLastError());
  }
  return EDIS_OK;
}
