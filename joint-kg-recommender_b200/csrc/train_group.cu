// Group-compact fused training kernels for the KG families (TransE, TransH / KTUP KG branch).
//
// The reference samples each negative by corrupting the head OR the tail of a positive
// (utils/data.py:12-56), so a negative shares its relation and one entity with its positive.
// Here that is the data format: negative k of positive j is ONE int32,
//     corrupt[j*K + k] >= 0 : tail replaced by entity  corrupt
//     corrupt[j*K + k] <  0 : head replaced by entity ~corrupt
// One warp owns one positive and its K negatives.  The positive's rows are read once and kept
// in registers (as h + r and r - t, projected for TransH), each negative costs ONE row read, and
// in the backward the gradients of the shared rows are accumulated in registers across the
// group: (3 + K) rows read and (3 + K) rows written per group of (1 + K) scored triples --
// 481 + 481 bytes per triple at d = 100, K = 10 instead of 1216 + 1200.
//
// Reference arithmetic: transE.py:51-63, transH.py:58-71 (+ utils/misc.py:18-19),
// utils/loss.py:8-16, 29-31; CPU restatement: oracle/kg_oracle.py.
#include "train_dev.cuh"

namespace kgrec {

struct GroupArgs {
  kgrec_tables T;
  const void *ph, *pt, *pr;
  int is64;
  const int32_t* corrupt;
  LossCfg L;
  float keep;               // fraction of table lines loaded with the evict_last policy
};

__device__ __forceinline__ const float* row_ptr(const float* base, uint32_t row, uint32_t ld) {
  return base + static_cast<uint64_t>(row) * ld;        // one IMAD.WIDE.U32
}

template <int FAM, int NCH>
struct GroupPos {           // the positive of a group, reduced to what its negatives need
  using R = Row<NCH, true>;
  static constexpr int NE = R::NE;
  float h[NE], t[NE], w[NE];
  float base_h[NE];         // proj(h) + r
  float base_t[NE];         // r - proj(t)
  float a, b;               // h.w, t.w (TransH)
  float epos[NE];

  __device__ __forceinline__ void load(const kgrec_tables& T, uint32_t ih, uint32_t it, uint32_t ir, int lane, uint64_t pol) {
    const int d = T.dim;
    float r[NE];
    R::load_hint(h, row_ptr(T.ent, ih, T.ld), d, lane, pol);
    R::load_hint(t, row_ptr(T.ent, it, T.ld), d, lane, pol);
    R::load_hint(r, row_ptr(T.rel, ir, T.ld), d, lane, pol);
    a = b = 0.f;
    if (FAM == FAM_H) {
      R::load_hint(w, row_ptr(T.norm, ir, T.ld), d, lane, pol);
      a = R::dot(h, w);
      b = R::dot(t, w);
      warp_sum2(a, b);
    }
#pragma unroll
    for (int i = 0; i < NE; ++i) {
      const float ph = (FAM == FAM_H) ? h[i] - a * w[i] : h[i];
      const float pt = (FAM == FAM_H) ? t[i] - b * w[i] : t[i];
      base_h[i] = ph + r[i];
      base_t[i] = r[i] - pt;
      epos[i] = base_h[i] - pt;                 // (proj h + r) - proj t, the reference's order
    }
  }
  // residual of the negative whose corrupted row is x; ax = x.w (TransH, already reduced)
  __device__ __forceinline__ void residual(const float (&x)[NE], bool head, float ax, float (&e)[NE]) const {
#pragma unroll
    for (int i = 0; i < NE; ++i) {
      const float px = (FAM == FAM_H) ? x[i] - ax * w[i] : x[i];
      e[i] = head ? px + base_t[i] : base_h[i] - px;
    }
  }
};

template <int NE>
__device__ __forceinline__ float dist_sum(const float (&e)[NE], int l1) {
  float acc = 0.f;
#pragma unroll
  for (int i = 0; i < NE; ++i) acc += dist_term(e[i], l1);
  return warp_sum(acc);
}

__device__ __forceinline__ uint32_t group_idx(const void* p, int j, int is64, int64_t rows, int32_t* status) {
  const int64_t v = is64 ? __ldg(reinterpret_cast<const long long*>(p) + j)
                         : static_cast<int64_t>(__ldg(reinterpret_cast<const int*>(p) + j));
  if (static_cast<uint64_t>(v) >= static_cast<uint64_t>(rows)) {
    if (status) *status = 1;
    return 0u;
  }
  return static_cast<uint32_t>(v);
}

template <int FAM, int NCH, bool L1>
__global__ void __launch_bounds__(kThreads)
k_group_fwd(const GroupArgs G, float* __restrict__ pos_scores, float* __restrict__ neg_scores,
            float* __restrict__ group_loss, int32_t* status) {
  using R = Row<NCH, true>;
  constexpr int NE = NCH * 4;
  const kgrec_tables& T = G.T;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int K = G.L.n_neg, d = T.dim;
  constexpr int l1 = L1 ? 1 : 0;
  const int n_pos = static_cast<int>(G.L.n_pos);
  const uint32_t n_ent = static_cast<uint32_t>(T.n_ent), ld = static_cast<uint32_t>(T.ld);
  const uint64_t pol_keep = policy_evict_last(G.keep);
  for (int j = blockIdx.x * kWarpsPerCta + wid; j < n_pos; j += gridDim.x * kWarpsPerCta) {
    const int32_t* cj = G.corrupt + static_cast<int64_t>(j) * K;
    int32_t c = K > 0 ? __ldg(cj) : 0;                       // first negative's id, in flight with the rows
    const uint32_t ih = group_idx(G.ph, j, G.is64, T.n_ent, status);
    const uint32_t it = group_idx(G.pt, j, G.is64, T.n_ent, status);
    const uint32_t ir = group_idx(G.pr, j, G.is64, T.n_rel, status);
    GroupPos<FAM, NCH> P;
    P.load(T, ih, it, ir, lane, pol_keep);
    const float sp = dist_sum(P.epos, l1);
    float lsum = 0.f;
    // software pipeline over the negatives: row k+1 is requested before row k is consumed
    float x[NE], xn[NE];
    bool head = c < 0;
    uint32_t id = static_cast<uint32_t>(head ? ~c : c);
    if (id >= n_ent) { if (status) *status = 1; id = 0; }
    if (K > 0) R::load_hint(x, row_ptr(T.ent, id, ld), d, lane, pol_keep);
    for (int k = 0; k < K; ++k) {
      bool headn = false;
      if (k + 1 < K) {
        const int32_t cn = __ldg(cj + k + 1);
        headn = cn < 0;
        uint32_t idn = static_cast<uint32_t>(headn ? ~cn : cn);
        if (idn >= n_ent) { if (status) *status = 1; idn = 0; }
        R::load_hint(xn, row_ptr(T.ent, idn, ld), d, lane, pol_keep);
      }
      float ax = 0.f;
      if (FAM == FAM_H) ax = warp_sum(R::dot(x, P.w));
      float e[NE];
      P.residual(x, head, ax, e);
      const float sn = dist_sum(e, l1);
      if (lane == 0) neg_scores[static_cast<int64_t>(j) * K + k] = sn;
      lsum += loss_term(G.L, sp, sn);
      head = headn;
#pragma unroll
      for (int i = 0; i < NE; ++i) x[i] = xn[i];
    }
    if (lane == 0) {
      pos_scores[j] = sp;
      group_loss[j] = lsum;
    }
  }
}

// slots (mode 0): ent [n_pos * (2 + K), d] per group: h, t, c_1 .. c_K ; rel / norm [n_pos, d]
template <int FAM, int NCH, bool L1>
__global__ void __launch_bounds__(kThreads)
k_group_bwd(const GroupArgs G, const float* __restrict__ pos_scores, const float* __restrict__ neg_scores,
            const float grad_loss, const float* __restrict__ grad_loss_dev, const kgrec_grads Gr) {
  using R = Row<NCH, true>;
  constexpr int NE = NCH * 4;
  const kgrec_tables& T = G.T;
  const LossCfg& L = G.L;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int K = L.n_neg, d = T.dim;
  constexpr int l1 = L1 ? 1 : 0;
  const int n_pos = static_cast<int>(L.n_pos);
  const uint32_t n_ent = static_cast<uint32_t>(T.n_ent), ld = static_cast<uint32_t>(T.ld);
  const int bp = static_cast<int>(L.batch_pos < 0x7fffffff ? L.batch_pos : 0x7fffffff);
  const uint64_t pol_keep = policy_evict_last(G.keep), pol_stream = policy_evict_first();
  for (int j = blockIdx.x * kWarpsPerCta + wid; j < n_pos; j += gridDim.x * kWarpsPerCta) {
    const int32_t* cj = G.corrupt + static_cast<int64_t>(j) * K;
    const float* snj = neg_scores + static_cast<int64_t>(j) * K;
    int32_t c = K > 0 ? __ldg(cj) : 0;
    const uint32_t ih = group_idx(G.ph, j, G.is64, T.n_ent, nullptr);
    const uint32_t it = group_idx(G.pt, j, G.is64, T.n_ent, nullptr);
    const uint32_t ir = group_idx(G.pr, j, G.is64, T.n_rel, nullptr);
    GroupPos<FAM, NCH> P;
    P.load(T, ih, it, ir, lane, pol_keep);
    // upstream of this group: dLoss/d(loss term) = grad_loss * grad_loss_dev[batch] * (1 | 1/(cnt K))
    const int b = j / bp;
    float up = grad_loss * (grad_loss_dev ? __ldg(grad_loss_dev + b) : 1.f);
    if (L.kind == KGREC_LOSS_BPR) {
      const int cnt = min(bp, n_pos - b * bp);
      up /= static_cast<float>(cnt) * static_cast<float>(K);
    }
    const float sp = __ldg(pos_scores + j);
    float cpos = 0.f;
    for (int k = lane; k < K; k += 32) cpos += loss_dpos(L, sp, __ldg(snj + k));
    cpos = warp_sum(cpos) * up;

    float gh[NE], gt[NE], gr[NE], gw[NE];
    {
      float eps[NE];
#pragma unroll
      for (int i = 0; i < NE; ++i) eps[i] = cpos * ddist_term(P.epos[i], l1);
      float ew = 0.f;
      if (FAM == FAM_H) ew = warp_sum(R::dot(eps, P.w));
      const float xw = P.a - P.b;
#pragma unroll
      for (int i = 0; i < NE; ++i) {
        const float gx = (FAM == FAM_H) ? eps[i] - ew * P.w[i] : eps[i];
        gh[i] = gx;
        gt[i] = -gx;
        gr[i] = eps[i];
        gw[i] = (FAM == FAM_H) ? -(ew * (P.h[i] - P.t[i]) + xw * eps[i]) : 0.f;
      }
    }
    const int64_t slot0 = static_cast<int64_t>(j) * (2 + K);
    float x[NE], xn[NE];
    bool head = c < 0;
    uint32_t id = static_cast<uint32_t>(head ? ~c : c);
    if (id >= n_ent) id = 0;
    if (K > 0) R::load_hint(x, row_ptr(T.ent, id, ld), d, lane, pol_keep);
    for (int k = 0; k < K; ++k) {
      bool headn = false;
      uint32_t idn = 0;
      if (k + 1 < K) {
        const int32_t cn = __ldg(cj + k + 1);
        headn = cn < 0;
        idn = static_cast<uint32_t>(headn ? ~cn : cn);
        if (idn >= n_ent) idn = 0;
        R::load_hint(xn, row_ptr(T.ent, idn, ld), d, lane, pol_keep);
      }
      const float ck = -loss_dpos(L, sp, __ldg(snj + k)) * up;     // dLoss/d(neg score)
      float gc[NE];
      if (ck != 0.f) {                                             // warp-uniform: inactive hinges cost nothing
        float ax = 0.f;
        if (FAM == FAM_H) ax = warp_sum(R::dot(x, P.w));
        float e[NE], eps[NE];
        P.residual(x, head, ax, e);
#pragma unroll
        for (int i = 0; i < NE; ++i) eps[i] = ck * ddist_term(e[i], l1);
        float ew = 0.f;
        if (FAM == FAM_H) ew = warp_sum(R::dot(eps, P.w));
        const float xw = head ? ax - P.b : P.a - ax;               // (h' - t).w or (h - t').w
#pragma unroll
        for (int i = 0; i < NE; ++i) {
          const float gx = (FAM == FAM_H) ? eps[i] - ew * P.w[i] : eps[i];
          gr[i] += eps[i];
          if (head) { gc[i] = gx; gt[i] -= gx; }
          else { gc[i] = -gx; gh[i] += gx; }
          if (FAM == FAM_H) {
            const float xd = head ? x[i] - P.t[i] : P.h[i] - x[i];
            gw[i] -= ew * xd + xw * eps[i];
          }
        }
      } else {
#pragma unroll
        for (int i = 0; i < NE; ++i) gc[i] = 0.f;
      }
      if (Gr.mode == 0) R::store_hint(Gr.ent + (slot0 + 2 + k) * d, gc, d, lane, pol_stream);
      else if (ck != 0.f) R::red_add(Gr.ent + static_cast<uint64_t>(id) * d, gc, d, lane);
      head = headn;
      id = idn;
#pragma unroll
      for (int i = 0; i < NE; ++i) x[i] = xn[i];
    }
    if (Gr.mode == 0) {
      R::store_hint(Gr.ent + slot0 * d, gh, d, lane, pol_stream);
      R::store_hint(Gr.ent + (slot0 + 1) * d, gt, d, lane, pol_stream);
      R::store_hint(Gr.rel + static_cast<int64_t>(j) * d, gr, d, lane, pol_stream);
      if (FAM == FAM_H) R::store_hint(Gr.norm + static_cast<int64_t>(j) * d, gw, d, lane, pol_stream);
    } else {
      R::red_add(Gr.ent + static_cast<uint64_t>(ih) * d, gh, d, lane);
      R::red_add(Gr.ent + static_cast<uint64_t>(it) * d, gt, d, lane);
      R::red_add(Gr.rel + static_cast<uint64_t>(ir) * d, gr, d, lane);
      if (FAM == FAM_H) R::red_add(Gr.norm + static_cast<uint64_t>(ir) * d, gw, d, lane);
    }
  }
}

// ---- forward + loss + backward in one pass ------------------------------------------------
// d(sum of the per-batch losses)/d(tables) together with the scores and the losses: every
// reference driver calls backward() on the loss itself (knowledge_representation.py:207), so
// the upstream of each loss term is known (`up`, times 1/(cnt K) for the BPR mean) while the
// group is still in registers: one gather of (3 + K) rows, (3 + K) gradient rows written.
template <int FAM, int NCH, bool L1>
__global__ void __launch_bounds__(kThreads, (NCH == 1 && FAM == FAM_E) ? 4 : 1)
k_group_step(const GroupArgs G, const float up0, float* __restrict__ pos_scores, float* __restrict__ neg_scores,
             float* __restrict__ group_loss, const kgrec_grads Gr, int32_t* status) {
  using R = Row<NCH, true>;
  constexpr int NE = NCH * 4;
  constexpr int l1 = L1 ? 1 : 0;
  const kgrec_tables& T = G.T;
  const LossCfg& L = G.L;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int K = L.n_neg, d = T.dim;
  const int n_pos = static_cast<int>(L.n_pos);
  const uint32_t n_ent = static_cast<uint32_t>(T.n_ent), ld = static_cast<uint32_t>(T.ld);
  const int bp = static_cast<int>(L.batch_pos < 0x7fffffff ? L.batch_pos : 0x7fffffff);
  const uint64_t pol_keep = policy_evict_last(G.keep), pol_stream = policy_evict_first();
  for (int j = blockIdx.x * kWarpsPerCta + wid; j < n_pos; j += gridDim.x * kWarpsPerCta) {
    const int32_t* cj = G.corrupt + static_cast<int64_t>(j) * K;
    int32_t c = K > 0 ? __ldg(cj) : 0;
    const uint32_t ih = group_idx(G.ph, j, G.is64, T.n_ent, status);
    const uint32_t it = group_idx(G.pt, j, G.is64, T.n_ent, status);
    const uint32_t ir = group_idx(G.pr, j, G.is64, T.n_rel, status);
    GroupPos<FAM, NCH> P;
    P.load(T, ih, it, ir, lane, pol_keep);
    float up = up0;
    if (L.kind == KGREC_LOSS_BPR) {
      const int b = j / bp;
      up /= static_cast<float>(min(bp, n_pos - b * bp)) * static_cast<float>(K);
    }
    const float sp = dist_sum(P.epos, l1);
    float lsum = 0.f, cpos = 0.f;
    float gh[NE], gt[NE], gr[NE], gw[NE];
#pragma unroll
    for (int i = 0; i < NE; ++i) { gh[i] = 0.f; gt[i] = 0.f; gr[i] = 0.f; gw[i] = 0.f; }
    const int64_t slot0 = static_cast<int64_t>(j) * (2 + K);
    float x[NE], xn[NE];
    bool head = c < 0;
    uint32_t id = static_cast<uint32_t>(head ? ~c : c);
    if (id >= n_ent) { if (status) *status = 1; id = 0; }
    if (K > 0) R::load_hint(x, row_ptr(T.ent, id, ld), d, lane, pol_keep);
    for (int k = 0; k < K; ++k) {
      bool headn = false;
      uint32_t idn = 0;
      if (k + 1 < K) {
        const int32_t cn = __ldg(cj + k + 1);
        headn = cn < 0;
        idn = static_cast<uint32_t>(headn ? ~cn : cn);
        if (idn >= n_ent) { if (status) *status = 1; idn = 0; }
        R::load_hint(xn, row_ptr(T.ent, idn, ld), d, lane, pol_keep);
      }
      float ax = 0.f;
      if (FAM == FAM_H) ax = warp_sum(R::dot(x, P.w));
      float e[NE];
      P.residual(x, head, ax, e);
      const float sn = dist_sum(e, l1);
      if (lane == 0) neg_scores[static_cast<int64_t>(j) * K + k] = sn;
      lsum += loss_term(L, sp, sn);
      const float dp = loss_dpos(L, sp, sn);
      cpos += dp;
      const float ck = -dp * up;
      float gc[NE];
      if (ck != 0.f) {                     // warp-uniform: an inactive hinge has no gradient
        float eps[NE];
#pragma unroll
        for (int i = 0; i < NE; ++i) eps[i] = ck * ddist_term(e[i], l1);
        float ew = 0.f;
        if (FAM == FAM_H) ew = warp_sum(R::dot(eps, P.w));
        const float xw = head ? ax - P.b : P.a - ax;
#pragma unroll
        for (int i = 0; i < NE; ++i) {
          const float gx = (FAM == FAM_H) ? eps[i] - ew * P.w[i] : eps[i];
          gr[i] += eps[i];
          if (head) { gc[i] = gx; gt[i] -= gx; }
          else { gc[i] = -gx; gh[i] += gx; }
          if (FAM == FAM_H) {
            const float xd = head ? x[i] - P.t[i] : P.h[i] - x[i];
            gw[i] -= ew * xd + xw * eps[i];
          }
        }
      } else {
#pragma unroll
        for (int i = 0; i < NE; ++i) gc[i] = 0.f;
      }
      if (Gr.mode == 0) R::store_hint(Gr.ent + (slot0 + 2 + k) * d, gc, d, lane, pol_stream);
      else if (ck != 0.f) R::red_add(Gr.ent + static_cast<uint64_t>(id) * d, gc, d, lane);
      head = headn;
      id = idn;
#pragma unroll
      for (int i = 0; i < NE; ++i) x[i] = xn[i];
    }
    {   // the positive's own contribution, with the coefficient summed over its negatives
      const float cp = cpos * up;
      float eps[NE];
#pragma unroll
      for (int i = 0; i < NE; ++i) eps[i] = cp * ddist_term(P.epos[i], l1);
      float ew = 0.f;
      if (FAM == FAM_H) ew = warp_sum(R::dot(eps, P.w));
      const float xw = P.a - P.b;
#pragma unroll
      for (int i = 0; i < NE; ++i) {
        const float gx = (FAM == FAM_H) ? eps[i] - ew * P.w[i] : eps[i];
        gh[i] += gx;
        gt[i] -= gx;
        gr[i] += eps[i];
        if (FAM == FAM_H) gw[i] -= ew * (P.h[i] - P.t[i]) + xw * eps[i];
      }
    }
    if (lane == 0) {
      pos_scores[j] = sp;
      group_loss[j] = lsum;
    }
    if (Gr.mode == 0) {
      R::store_hint(Gr.ent + slot0 * d, gh, d, lane, pol_stream);
      R::store_hint(Gr.ent + (slot0 + 1) * d, gt, d, lane, pol_stream);
      R::store_hint(Gr.rel + static_cast<int64_t>(j) * d, gr, d, lane, pol_stream);
      if (FAM == FAM_H) R::store_hint(Gr.norm + static_cast<int64_t>(j) * d, gw, d, lane, pol_stream);
    } else {
      R::red_add(Gr.ent + static_cast<uint64_t>(ih) * d, gh, d, lane);
      R::red_add(Gr.ent + static_cast<uint64_t>(it) * d, gt, d, lane);
      R::red_add(Gr.rel + static_cast<uint64_t>(ir) * d, gr, d, lane);
      if (FAM == FAM_H) R::red_add(Gr.norm + static_cast<uint64_t>(ir) * d, gw, d, lane);
    }
  }
}

// --- TransE, d <= 128: the step kernel again, written for issue slots --------------------------
// k_group_step above is bound by instruction issue (ncu: 77 % issue-active, 159 warp-instructions per
// scored triple of which ~30 are the arithmetic).  This version removes the rest:
//   * the residual is kept as e' = B - x with B = h + r (tail replaced) or t - r (head replaced):
//     |e'| = |e|, the corrupted row's gradient is -eps' in both cases, and the shared rows collect
//     eps' in two accumulators (accT / accH) picked by one warp-uniform branch, so no per-element
//     head/tail select is left:  g_h = accT + eps_p, g_t = accH - eps_p, g_r = accT - accH + eps_p;
//   * loss kind, gradient layout and norm are template parameters (no constant-bank reloads and
//     branches on them inside the loop), the tail predicate lane*4 < d is hoisted, row / slot
//     addresses advance by one IMAD.WIDE each;
//   * the negative loop is unrolled by two with ping-pong row buffers (no register rotation);
//   * ids never sit between a row and its request: the K corrupted ids of a group are ONE coalesced
//     load held one per lane (and the positive's three ids one load in lanes 0-2), fetched a whole
//     group ahead and handed out by shuffles, so the request for row k+1 leaves as soon as row k's
//     arithmetic starts (with per-negative id loads the row request waited a full L2 round trip:
//     48 % of the stall samples).
template <bool L1, bool DENSE, bool MARGIN, bool REG, bool BWD, bool FWD = false>
__global__ void __launch_bounds__(kThreads, 4)
k_group_step_e(const GroupArgs G, const float up0, const float* __restrict__ up_dev, float* __restrict__ pos_scores,
               float* __restrict__ neg_scores, float* __restrict__ group_loss, const kgrec_grads Gr,
               int64_t* __restrict__ slot_ent, int64_t* __restrict__ slot_rel, int32_t* status) {
  // BWD: the autograd backward of kgrec_corrupt_loss_fwd -- the hinge / BPR coefficients come from the SAVED
  // scores (one coalesced load per group, handed out by shuffles), the upstream is up0 * up_dev[batch], and
  // nothing but the gradients is written.
  const kgrec_tables& T = G.T;
  const LossCfg& L = G.L;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int K = L.n_neg;
  const int n_pos = static_cast<int>(L.n_pos);
  const uint32_t n_ent = static_cast<uint32_t>(T.n_ent);
  const uint32_t ld4 = static_cast<uint32_t>(T.ld) * 4u, d4 = static_cast<uint32_t>(T.dim) * 4u;   // row pitches in bytes
  const int bp = static_cast<int>(L.batch_pos < 0x7fffffff ? L.batch_pos : 0x7fffffff);
  const uint64_t pol_keep = policy_evict_last(G.keep), pol_stream = policy_evict_first();
  const bool act = lane * 4 < T.dim;
  const char* ent_b = reinterpret_cast<const char*>(T.ent) + lane * 16;
  const char* rel_b = reinterpret_cast<const char*>(T.rel) + lane * 16;
  char* gent_b = reinterpret_cast<char*>(Gr.ent) + lane * 16;
  char* grel_b = reinterpret_cast<char*>(Gr.rel) + lane * 16;
  const float prm = L.param;
  const int stride = gridDim.x * kWarpsPerCta;
  const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
  auto row = [&](const char* base, uint32_t id) { return reinterpret_cast<const float4*>(base + static_cast<uint64_t>(id) * ld4); };
  bool bad = false;
  auto ent_id = [&](int32_t c, bool& head) {        // corrupted-entity id of one int32 of the compact format
    head = c < 0;
    uint32_t id = static_cast<uint32_t>(head ? ~c : c);
    if (id >= n_ent) { bad = true; id = 0; }
    return id;
  };

  int j = blockIdx.x * kWarpsPerCta + wid;
  // ids of a group, one per lane: cv = corrupt[j*K + lane] (lane < K), pv = (h, t, r)[lane] (lane < 3)
  const void* pcol = lane == 0 ? G.ph : (lane == 1 ? G.pt : G.pr);
  auto fetch_ids = [&](int jj, int32_t& cv, int64_t& pv) {
    cv = lane < K ? __ldg(G.corrupt + static_cast<uint32_t>(jj) * K + lane) : 0;
    pv = lane < 3 ? load_idx(pcol, jj, G.is64) : 0;
  };
  int32_t cv = 0, cvn = 0;
  int64_t pv = 0, pvn = 0;
  if (j < n_pos) fetch_ids(j, cvn, pvn);
  for (; j < n_pos; j += stride) {
    cv = cvn;
    pv = pvn;
    const int jn = j + stride;
    if (jn < n_pos) fetch_ids(jn, cvn, pvn);     // the next group's ids travel while this group computes
    const int64_t vh = __shfl_sync(FULL, pv, 0), vt = __shfl_sync(FULL, pv, 1), vr = __shfl_sync(FULL, pv, 2);
    uint32_t ih = static_cast<uint32_t>(vh), it = static_cast<uint32_t>(vt), ir = static_cast<uint32_t>(vr);
    if (static_cast<uint64_t>(vh) >= static_cast<uint64_t>(T.n_ent)) { bad = true; ih = 0; }
    if (static_cast<uint64_t>(vt) >= static_cast<uint64_t>(T.n_ent)) { bad = true; it = 0; }
    if (static_cast<uint64_t>(vr) >= static_cast<uint64_t>(T.n_rel)) { bad = true; ir = 0; }
    if (slot_ent) {      // row ids of the gradient slots: [h, t, corrupted_1..K] per group, r per group
      const uint32_t s0 = static_cast<uint32_t>(j) * (2 + K);
      if (lane < 2) slot_ent[s0 + lane] = pv;
      if (lane == 2) slot_rel[j] = pv;
      if (lane < K) slot_ent[s0 + 2 + lane] = cv < 0 ? ~cv : cv;
    }
    float4 h = z4, t = z4, r = z4, xa = z4, xb = z4;
    bool heada, headb = false;
    uint32_t ida = ent_id(__shfl_sync(FULL, cv, 0), heada), idb = 0;
    if (act) {
      h = ldg_f4_hint(row(ent_b, ih), pol_keep);
      t = ldg_f4_hint(row(ent_b, it), pol_keep);
      r = ldg_f4_hint(row(rel_b, ir), pol_keep);
      xa = ldg_f4_hint(row(ent_b, ida), pol_keep);
    }
    if (lane >= 2 && lane < K) {     // lane l holds the id of negative l: it pulls that row's lines towards the SM
      const uint32_t pid = static_cast<uint32_t>(cv < 0 ? ~cv : cv);
      if (pid < n_ent) {
        const char* pr = reinterpret_cast<const char*>(T.ent) + static_cast<uint64_t>(pid) * ld4;
        for (uint32_t o = 0; o < d4; o += 128) prefetch_l1(pr + o);
      }
    }
    [[maybe_unused]] const uint32_t ih0 = ih, it0 = it, ir0 = ir;
    float up = up0;
    if (BWD && up_dev) up *= __ldg(up_dev + j / bp);
    if (!MARGIN) {
      const int b = j / bp;
      up /= static_cast<float>(min(bp, n_pos - b * bp)) * static_cast<float>(K);
    }
    [[maybe_unused]] const float svec = (BWD && lane < K) ? __ldg(neg_scores + static_cast<uint32_t>(j) * K + lane) : 0.f;
    const float4 bh = make_float4(h.x + r.x, h.y + r.y, h.z + r.z, h.w + r.w);        // h + r
    const float4 bt = make_float4(t.x - r.x, t.y - r.y, t.z - r.z, t.w - r.w);        // t - r
    const float4 ep = make_float4(bh.x - t.x, bh.y - t.y, bh.z - t.z, bh.w - t.w);    // (h + r) - t
    const float sp = BWD ? __ldg(pos_scores + j)
                         : warp_sum(dist_term(ep.x, L1) + dist_term(ep.y, L1) + dist_term(ep.z, L1) + dist_term(ep.w, L1));
    float lsum = 0.f, cpos = 0.f, mys = 0.f;
    float4 accT = z4, accH = z4;
    uint32_t goff = (static_cast<uint32_t>(j) * (2 + K) + 2) * d4;      // byte offset of the first corrupted-row slot
    // REG: the drivers' regulariser normLoss over the rows the batch gathers (loss.py:21-23 on
    // cat[ph, pt, nh, nt] and cat[pr, nr], knowledge_representation.py:197-204): sum max(|row|^2 - 1, 0)
    // with the multiplicity each row has in those lists; the rows are in registers already.
    [[maybe_unused]] float nh2 = 0.f, nt2 = 0.f, nr2 = 0.f, lreg = 0.f, n_tail = 0.f;
    [[maybe_unused]] const float r2 = 2.f * up0;
    if (REG) {
      nh2 = h.x * h.x + h.y * h.y + h.z * h.z + h.w * h.w;
      nt2 = t.x * t.x + t.y * t.y + t.z * t.z + t.w * t.w;
      nr2 = r.x * r.x + r.y * r.y + r.z * r.z + r.w * r.w;
      warp_sum2(nh2, nt2);
      nr2 = warp_sum(nr2);
    }

    auto negative = [&](const float4& x, const bool head, const uint32_t id, const int k) {
      const float4 B = head ? bt : bh;
      const float4 e = make_float4(B.x - x.x, B.y - x.y, B.z - x.z, B.w - x.w);
      float sn = dist_term(e.x, L1) + dist_term(e.y, L1) + dist_term(e.z, L1) + dist_term(e.w, L1);
      [[maybe_unused]] float nx2 = 0.f;
      if (BWD) {
        sn = __shfl_sync(FULL, svec, k);
      } else if (REG) {
        nx2 = x.x * x.x + x.y * x.y + x.z * x.z + x.w * x.w;
        warp_sum2(sn, nx2);
        lreg += fmaxf(nx2 - 1.f, 0.f);
        n_tail += head ? 0.f : 1.f;
      } else {
        sn = warp_sum(sn);
      }
      if (!BWD && lane == k) mys = sn;
      float coef;      // -(dLoss/dsn): the corrupted row's gradient is coef * dL(e')/de'
      if (MARGIN) {
        const float tt = sp - sn + prm;
        lsum += fmaxf(tt, 0.f);
        coef = tt > 0.f ? up : 0.f;
        cpos += tt > 0.f ? 1.f : 0.f;
      } else {
        const float xx = prm * (sp - sn);
        lsum += fmaxf(-xx, 0.f) + log1pf(expf(-fabsf(xx)));
        const float dp = -prm / (1.f + expf(xx));
        cpos += dp;
        coef = dp * up;
      }
      if (FWD) return;                      // forward only (kgrec_corrupt_loss_fwd): scores and loss terms
      const bool regx = REG && nx2 > 1.f;
      if (coef != 0.f || regx) {            // warp-uniform: an inactive hinge has no gradient
        float4 gc = z4;                     // = -eps' (+ the regulariser's 2 x)
        if (coef != 0.f) {
          if (L1) {
            gc = make_float4(coef * ddist_term(e.x, 1), coef * ddist_term(e.y, 1), coef * ddist_term(e.z, 1), coef * ddist_term(e.w, 1));
          } else {
            const float c2 = 2.f * coef;
            gc = make_float4(c2 * e.x, c2 * e.y, c2 * e.z, c2 * e.w);
          }
          if (head) { accH.x -= gc.x; accH.y -= gc.y; accH.z -= gc.z; accH.w -= gc.w; }
          else { accT.x -= gc.x; accT.y -= gc.y; accT.z -= gc.z; accT.w -= gc.w; }
        }
        if (regx) { gc.x = fmaf(r2, x.x, gc.x); gc.y = fmaf(r2, x.y, gc.y); gc.z = fmaf(r2, x.z, gc.z); gc.w = fmaf(r2, x.w, gc.w); }
        if (act) {
          if (DENSE) red_add_f4(reinterpret_cast<float*>(gent_b + static_cast<uint64_t>(id) * d4), gc.x, gc.y, gc.z, gc.w);
          else stg_f4_hint(reinterpret_cast<float4*>(gent_b + goff), gc.x, gc.y, gc.z, gc.w, pol_stream);
        }
      } else if (!DENSE) {
        if (act) stg_f4_hint(reinterpret_cast<float4*>(gent_b + goff), 0.f, 0.f, 0.f, 0.f, pol_stream);
      }
      goff += d4;
    };

    for (int k = 0; k < K; k += 2) {
      if (k + 1 < K) {
        idb = ent_id(__shfl_sync(FULL, cv, k + 1), headb);
        if (act) xb = ldg_f4_hint(row(ent_b, idb), pol_keep);
      }
      negative(xa, heada, ida, k);
      if (k + 1 < K) {
        if (k + 2 < K) {
          ida = ent_id(__shfl_sync(FULL, cv, k + 2), heada);
          if (act) xa = ldg_f4_hint(row(ent_b, ida), pol_keep);
        }
        negative(xb, headb, idb, k + 1);
      }
    }
    // the positive's own contribution, with the coefficient summed over its negatives
    const float cp = cpos * up;
    const float4 eps = make_float4(cp * ddist_term(ep.x, L1), cp * ddist_term(ep.y, L1), cp * ddist_term(ep.z, L1), cp * ddist_term(ep.w, L1));
    float4 gh = make_float4(accT.x + eps.x, accT.y + eps.y, accT.z + eps.z, accT.w + eps.w);
    float4 gt = make_float4(accH.x - eps.x, accH.y - eps.y, accH.z - eps.z, accH.w - eps.w);
    float4 gr = make_float4(accT.x - accH.x + eps.x, accT.y - accH.y + eps.y, accT.z - accH.z + eps.z, accT.w - accH.w + eps.w);
    if (REG) {      // h is listed once as ph and once per tail-replaced negative (nh); t likewise; r once per triple
      const float mh = 1.f + n_tail, mt = 1.f + (static_cast<float>(K) - n_tail), mr = 1.f + static_cast<float>(K);
      lreg += mh * fmaxf(nh2 - 1.f, 0.f) + mt * fmaxf(nt2 - 1.f, 0.f) + mr * fmaxf(nr2 - 1.f, 0.f);
      const float ch = nh2 > 1.f ? mh * r2 : 0.f, ct = nt2 > 1.f ? mt * r2 : 0.f, cr = nr2 > 1.f ? mr * r2 : 0.f;
      gh.x = fmaf(ch, h.x, gh.x); gh.y = fmaf(ch, h.y, gh.y); gh.z = fmaf(ch, h.z, gh.z); gh.w = fmaf(ch, h.w, gh.w);
      gt.x = fmaf(ct, t.x, gt.x); gt.y = fmaf(ct, t.y, gt.y); gt.z = fmaf(ct, t.z, gt.z); gt.w = fmaf(ct, t.w, gt.w);
      gr.x = fmaf(cr, r.x, gr.x); gr.y = fmaf(cr, r.y, gr.y); gr.z = fmaf(cr, r.z, gr.z); gr.w = fmaf(cr, r.w, gr.w);
    }
    if (!BWD) {
      if (lane == 0) {
        pos_scores[j] = sp;
        group_loss[j] = lsum + (REG ? lreg : 0.f);
      }
      if (lane < K) neg_scores[static_cast<uint32_t>(j) * K + lane] = mys;
    }
    if (!FWD && act) {
      if (DENSE) {
        red_add_f4(reinterpret_cast<float*>(gent_b + static_cast<uint64_t>(ih0) * d4), gh.x, gh.y, gh.z, gh.w);
        red_add_f4(reinterpret_cast<float*>(gent_b + static_cast<uint64_t>(it0) * d4), gt.x, gt.y, gt.z, gt.w);
        red_add_f4(reinterpret_cast<float*>(grel_b + static_cast<uint64_t>(ir0) * d4), gr.x, gr.y, gr.z, gr.w);
      } else {
        const uint32_t g0 = static_cast<uint32_t>(j) * (2 + K) * d4;
        stg_f4_hint(reinterpret_cast<float4*>(gent_b + g0), gh.x, gh.y, gh.z, gh.w, pol_stream);
        stg_f4_hint(reinterpret_cast<float4*>(gent_b + g0 + d4), gt.x, gt.y, gt.z, gt.w, pol_stream);
        stg_f4_hint(reinterpret_cast<float4*>(grel_b + static_cast<uint32_t>(j) * d4), gr.x, gr.y, gr.z, gr.w, pol_stream);
      }
    }
  }
  if (bad && status) *status = 1;
}

// --- TransH (and the KTUP KG branch), d <= 128: the same treatment ------------------------------
// With proj(v) = v - (v.w) w the residual is e' = B - proj(x), B = proj(h) + r or proj(t) - r.  Writing
// g = -eps' for the gradient arriving at proj(x), the group needs per negative only
//   g_x = g - (g.w) w,   g_w -= (g.w) x + (x.w) g,   accT/accH -= g,   sT/sH -= g.w
// and everything that involves the shared rows is linear in (accT, accH, sT, sH), so it is applied once
// per group:  E_h = accT + eps_p, E_t = accH - eps_p,
//   g_h = E_h - (E_h.w) w,  g_t = E_t - (E_t.w) w,  g_r = accT - accH + eps_p,
//   g_w -= (E_h.w) h + (h.w) E_h + (E_t.w) t + (t.w) E_t.
// The two reductions a negative needs after its residual (the score and g.w) share one shuffle tree.
template <bool L1, bool DENSE, bool MARGIN, bool REG, bool BWD, bool FWD = false>
__global__ void __launch_bounds__(kThreads, 3)
k_group_step_h(const GroupArgs G, const float up0, const float* __restrict__ up_dev, float* __restrict__ pos_scores,
               float* __restrict__ neg_scores, float* __restrict__ group_loss, const kgrec_grads Gr,
               int64_t* __restrict__ slot_ent, int64_t* __restrict__ slot_rel, int32_t* status) {
  // BWD: the autograd backward of kgrec_corrupt_loss_fwd -- the hinge / BPR coefficients come from the SAVED
  // scores (one coalesced load per group, handed out by shuffles), the upstream is up0 * up_dev[batch], and
  // nothing but the gradients is written.
  const kgrec_tables& T = G.T;
  const LossCfg& L = G.L;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int K = L.n_neg;
  const int n_pos = static_cast<int>(L.n_pos);
  const uint32_t n_ent = static_cast<uint32_t>(T.n_ent);
  const uint32_t ld4 = static_cast<uint32_t>(T.ld) * 4u, d4 = static_cast<uint32_t>(T.dim) * 4u;
  const int bp = static_cast<int>(L.batch_pos < 0x7fffffff ? L.batch_pos : 0x7fffffff);
  const uint64_t pol_keep = policy_evict_last(G.keep), pol_stream = policy_evict_first();
  const bool act = lane * 4 < T.dim;
  const char* ent_b = reinterpret_cast<const char*>(T.ent) + lane * 16;
  const char* rel_b = reinterpret_cast<const char*>(T.rel) + lane * 16;
  const char* nrm_b = reinterpret_cast<const char*>(T.norm) + lane * 16;
  char* gent_b = reinterpret_cast<char*>(Gr.ent) + lane * 16;
  char* grel_b = reinterpret_cast<char*>(Gr.rel) + lane * 16;
  char* gnrm_b = reinterpret_cast<char*>(Gr.norm) + lane * 16;
  const float prm = L.param;
  const int stride = gridDim.x * kWarpsPerCta;
  const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
  auto row = [&](const char* base, uint32_t id) { return reinterpret_cast<const float4*>(base + static_cast<uint64_t>(id) * ld4); };
  auto dot4 = [](const float4& a, const float4& b) { return fmaf(a.x, b.x, fmaf(a.y, b.y, fmaf(a.z, b.z, a.w * b.w))); };
  bool bad = false;
  auto ent_id = [&](int32_t c, bool& head) {
    head = c < 0;
    uint32_t id = static_cast<uint32_t>(head ? ~c : c);
    if (id >= n_ent) { bad = true; id = 0; }
    return id;
  };
  int j = blockIdx.x * kWarpsPerCta + wid;
  const void* pcol = lane == 0 ? G.ph : (lane == 1 ? G.pt : G.pr);
  auto fetch_ids = [&](int jj, int32_t& cv, int64_t& pv) {
    cv = lane < K ? __ldg(G.corrupt + static_cast<uint32_t>(jj) * K + lane) : 0;
    pv = lane < 3 ? load_idx(pcol, jj, G.is64) : 0;
  };
  int32_t cv = 0, cvn = 0;
  int64_t pv = 0, pvn = 0;
  if (j < n_pos) fetch_ids(j, cvn, pvn);
  for (; j < n_pos; j += stride) {
    cv = cvn;
    pv = pvn;
    const int jn = j + stride;
    if (jn < n_pos) fetch_ids(jn, cvn, pvn);
    const int64_t vh = __shfl_sync(FULL, pv, 0), vt = __shfl_sync(FULL, pv, 1), vr = __shfl_sync(FULL, pv, 2);
    uint32_t ih = static_cast<uint32_t>(vh), it = static_cast<uint32_t>(vt), ir = static_cast<uint32_t>(vr);
    if (static_cast<uint64_t>(vh) >= static_cast<uint64_t>(T.n_ent)) { bad = true; ih = 0; }
    if (static_cast<uint64_t>(vt) >= static_cast<uint64_t>(T.n_ent)) { bad = true; it = 0; }
    if (static_cast<uint64_t>(vr) >= static_cast<uint64_t>(T.n_rel)) { bad = true; ir = 0; }
    if (slot_ent) {
      const uint32_t s0 = static_cast<uint32_t>(j) * (2 + K);
      if (lane < 2) slot_ent[s0 + lane] = pv;
      if (lane == 2) slot_rel[j] = pv;
      if (lane < K) slot_ent[s0 + 2 + lane] = cv < 0 ? ~cv : cv;
    }
    float4 h = z4, t = z4, r = z4, w = z4, xa = z4, xb = z4;
    bool heada, headb = false;
    uint32_t ida = ent_id(__shfl_sync(FULL, cv, 0), heada), idb = 0;
    if (act) {
      h = ldg_f4_hint(row(ent_b, ih), pol_keep);
      t = ldg_f4_hint(row(ent_b, it), pol_keep);
      r = ldg_f4_hint(row(rel_b, ir), pol_keep);
      w = ldg_f4_hint(row(nrm_b, ir), pol_keep);
      xa = ldg_f4_hint(row(ent_b, ida), pol_keep);
    }
    if (lane >= 2 && lane < K) {     // lane l holds the id of negative l: it pulls that row's lines towards the SM
      const uint32_t pid = static_cast<uint32_t>(cv < 0 ? ~cv : cv);
      if (pid < n_ent) {
        const char* pr = reinterpret_cast<const char*>(T.ent) + static_cast<uint64_t>(pid) * ld4;
        for (uint32_t o = 0; o < d4; o += 128) prefetch_l1(pr + o);
      }
    }
    float up = up0;
    if (BWD && up_dev) up *= __ldg(up_dev + j / bp);
    if (!MARGIN) {
      const int b = j / bp;
      up /= static_cast<float>(min(bp, n_pos - b * bp)) * static_cast<float>(K);
    }
    [[maybe_unused]] const float svec = (BWD && lane < K) ? __ldg(neg_scores + static_cast<uint32_t>(j) * K + lane) : 0.f;
    float a = dot4(h, w), b = dot4(t, w);
    warp_sum2(a, b);
    const float4 pt = make_float4(fmaf(-b, w.x, t.x), fmaf(-b, w.y, t.y), fmaf(-b, w.z, t.z), fmaf(-b, w.w, t.w));
    const float4 bh = make_float4(fmaf(-a, w.x, h.x) + r.x, fmaf(-a, w.y, h.y) + r.y, fmaf(-a, w.z, h.z) + r.z, fmaf(-a, w.w, h.w) + r.w);
    const float4 bt = make_float4(pt.x - r.x, pt.y - r.y, pt.z - r.z, pt.w - r.w);
    const float4 ep = make_float4(bh.x - pt.x, bh.y - pt.y, bh.z - pt.z, bh.w - pt.w);
    const float sp = BWD ? __ldg(pos_scores + j)
                         : warp_sum(dist_term(ep.x, L1) + dist_term(ep.y, L1) + dist_term(ep.z, L1) + dist_term(ep.w, L1));
    float lsum = 0.f, cpos = 0.f, mys = 0.f, sT = 0.f, sH = 0.f;
    float4 accT = z4, accH = z4, gwv = z4;
    uint32_t goff = (static_cast<uint32_t>(j) * (2 + K) + 2) * d4;
    // REG: normLoss over the gathered entity / relation rows and orthogonalLoss(rel, norm) (loss.py:18-23,
    // knowledge_representation.py:197-204), with each row's multiplicity in the driver's lists
    [[maybe_unused]] float nh2 = 0.f, nt2 = 0.f, nr2 = 0.f, wr = 0.f, lreg = 0.f, n_tail = 0.f;
    [[maybe_unused]] const float r2 = 2.f * up0;
    if (REG) {
      nh2 = dot4(h, h);
      nt2 = dot4(t, t);
      nr2 = dot4(r, r);
      wr = dot4(w, r);
      warp_sum2(nh2, nt2);
      warp_sum2(nr2, wr);
    }

    auto negative = [&](const float4& x, const bool head, const uint32_t id, const int k) {
      const float ax = warp_sum(dot4(x, w));
      const float4 B = head ? bt : bh;
      const float4 e = make_float4(B.x - fmaf(-ax, w.x, x.x), B.y - fmaf(-ax, w.y, x.y), B.z - fmaf(-ax, w.z, x.z), B.w - fmaf(-ax, w.w, x.w));
      const float4 dd = L1 ? make_float4(ddist_term(e.x, 1), ddist_term(e.y, 1), ddist_term(e.z, 1), ddist_term(e.w, 1)) : e;   // L2: x2 below
      float sn = dist_term(e.x, L1) + dist_term(e.y, L1) + dist_term(e.z, L1) + dist_term(e.w, L1);
      float dw = dot4(dd, w);
      if (BWD) {
        dw = warp_sum(dw);
        sn = __shfl_sync(FULL, svec, k);
      } else {
        warp_sum2(sn, dw);
      }
      [[maybe_unused]] float nx2 = 0.f;
      if (REG) {
        nx2 = warp_sum(dot4(x, x));
        lreg += fmaxf(nx2 - 1.f, 0.f);
        n_tail += head ? 0.f : 1.f;
      }
      if (!BWD && lane == k) mys = sn;
      float coef;
      if (MARGIN) {
        const float tt = sp - sn + prm;
        lsum += fmaxf(tt, 0.f);
        coef = tt > 0.f ? up : 0.f;
        cpos += tt > 0.f ? 1.f : 0.f;
      } else {
        const float xx = prm * (sp - sn);
        lsum += fmaxf(-xx, 0.f) + log1pf(expf(-fabsf(xx)));
        const float dp = -prm / (1.f + expf(xx));
        cpos += dp;
        coef = dp * up;
      }
      if (FWD) return;
      const bool regx = REG && nx2 > 1.f;
      if (coef != 0.f || regx) {
        float4 gx = z4;
        if (coef != 0.f) {
          const float c = L1 ? coef : 2.f * coef;
          const float4 g = make_float4(c * dd.x, c * dd.y, c * dd.z, c * dd.w);       // -eps' at proj(x)
          const float gdw = c * dw;                                                   // g . w
          gx = make_float4(fmaf(-gdw, w.x, g.x), fmaf(-gdw, w.y, g.y), fmaf(-gdw, w.z, g.z), fmaf(-gdw, w.w, g.w));
          gwv.x = fmaf(-gdw, x.x, fmaf(-ax, g.x, gwv.x));
          gwv.y = fmaf(-gdw, x.y, fmaf(-ax, g.y, gwv.y));
          gwv.z = fmaf(-gdw, x.z, fmaf(-ax, g.z, gwv.z));
          gwv.w = fmaf(-gdw, x.w, fmaf(-ax, g.w, gwv.w));
          if (head) { accH.x -= g.x; accH.y -= g.y; accH.z -= g.z; accH.w -= g.w; sH -= gdw; }
          else { accT.x -= g.x; accT.y -= g.y; accT.z -= g.z; accT.w -= g.w; sT -= gdw; }
        }
        if (regx) { gx.x = fmaf(r2, x.x, gx.x); gx.y = fmaf(r2, x.y, gx.y); gx.z = fmaf(r2, x.z, gx.z); gx.w = fmaf(r2, x.w, gx.w); }
        if (act) {
          if (DENSE) red_add_f4(reinterpret_cast<float*>(gent_b + static_cast<uint64_t>(id) * d4), gx.x, gx.y, gx.z, gx.w);
          else stg_f4_hint(reinterpret_cast<float4*>(gent_b + goff), gx.x, gx.y, gx.z, gx.w, pol_stream);
        }
      } else if (!DENSE) {
        if (act) stg_f4_hint(reinterpret_cast<float4*>(gent_b + goff), 0.f, 0.f, 0.f, 0.f, pol_stream);
      }
      goff += d4;
    };

    for (int k = 0; k < K; k += 2) {
      if (k + 1 < K) {
        idb = ent_id(__shfl_sync(FULL, cv, k + 1), headb);
        if (act) xb = ldg_f4_hint(row(ent_b, idb), pol_keep);
      }
      negative(xa, heada, ida, k);
      if (k + 1 < K) {
        if (k + 2 < K) {
          ida = ent_id(__shfl_sync(FULL, cv, k + 2), heada);
          if (act) xa = ldg_f4_hint(row(ent_b, ida), pol_keep);
        }
        negative(xb, headb, idb, k + 1);
      }
    }
    const float cp = cpos * up;
    const float4 eps = make_float4(cp * ddist_term(ep.x, L1), cp * ddist_term(ep.y, L1), cp * ddist_term(ep.z, L1), cp * ddist_term(ep.w, L1));
    const float epw = warp_sum(dot4(eps, w));
    const float4 EH = make_float4(accT.x + eps.x, accT.y + eps.y, accT.z + eps.z, accT.w + eps.w);
    const float4 ET = make_float4(accH.x - eps.x, accH.y - eps.y, accH.z - eps.z, accH.w - eps.w);
    const float eh = sT + epw, et = sH - epw;
    float4 gh = make_float4(fmaf(-eh, w.x, EH.x), fmaf(-eh, w.y, EH.y), fmaf(-eh, w.z, EH.z), fmaf(-eh, w.w, EH.w));
    float4 gt = make_float4(fmaf(-et, w.x, ET.x), fmaf(-et, w.y, ET.y), fmaf(-et, w.z, ET.z), fmaf(-et, w.w, ET.w));
    float4 gr = make_float4(accT.x - accH.x + eps.x, accT.y - accH.y + eps.y, accT.z - accH.z + eps.z, accT.w - accH.w + eps.w);
    gwv.x -= fmaf(eh, h.x, a * EH.x) + fmaf(et, t.x, b * ET.x);
    gwv.y -= fmaf(eh, h.y, a * EH.y) + fmaf(et, t.y, b * ET.y);
    gwv.z -= fmaf(eh, h.z, a * EH.z) + fmaf(et, t.z, b * ET.z);
    gwv.w -= fmaf(eh, h.w, a * EH.w) + fmaf(et, t.w, b * ET.w);
    if (REG) {
      const float mh = 1.f + n_tail, mt = 1.f + (static_cast<float>(K) - n_tail), mr = 1.f + static_cast<float>(K);
      const float inv = nr2 > 0.f ? 1.f / nr2 : 0.f, q = wr * inv;                       // (w.r) / |r|^2
      lreg += mh * fmaxf(nh2 - 1.f, 0.f) + mt * fmaxf(nt2 - 1.f, 0.f) + mr * (fmaxf(nr2 - 1.f, 0.f) + wr * q);
      const float ch = nh2 > 1.f ? mh * r2 : 0.f, ct = nt2 > 1.f ? mt * r2 : 0.f;
      const float cr = (nr2 > 1.f ? mr * r2 : 0.f) - mr * r2 * q * q, cw = mr * r2 * q;   // d/dr, d/dw of (w.r)^2 / |r|^2
      gh.x = fmaf(ch, h.x, gh.x); gh.y = fmaf(ch, h.y, gh.y); gh.z = fmaf(ch, h.z, gh.z); gh.w = fmaf(ch, h.w, gh.w);
      gt.x = fmaf(ct, t.x, gt.x); gt.y = fmaf(ct, t.y, gt.y); gt.z = fmaf(ct, t.z, gt.z); gt.w = fmaf(ct, t.w, gt.w);
      gr.x = fmaf(cr, r.x, fmaf(cw, w.x, gr.x)); gr.y = fmaf(cr, r.y, fmaf(cw, w.y, gr.y));
      gr.z = fmaf(cr, r.z, fmaf(cw, w.z, gr.z)); gr.w = fmaf(cr, r.w, fmaf(cw, w.w, gr.w));
      gwv.x = fmaf(cw, r.x, gwv.x); gwv.y = fmaf(cw, r.y, gwv.y); gwv.z = fmaf(cw, r.z, gwv.z); gwv.w = fmaf(cw, r.w, gwv.w);
    }
    if (!BWD) {
      if (lane == 0) {
        pos_scores[j] = sp;
        group_loss[j] = lsum + (REG ? lreg : 0.f);
      }
      if (lane < K) neg_scores[static_cast<uint32_t>(j) * K + lane] = mys;
    }
    if (!FWD && act) {
      if (DENSE) {
        red_add_f4(reinterpret_cast<float*>(gent_b + static_cast<uint64_t>(ih) * d4), gh.x, gh.y, gh.z, gh.w);
        red_add_f4(reinterpret_cast<float*>(gent_b + static_cast<uint64_t>(it) * d4), gt.x, gt.y, gt.z, gt.w);
        red_add_f4(reinterpret_cast<float*>(grel_b + static_cast<uint64_t>(ir) * d4), gr.x, gr.y, gr.z, gr.w);
        red_add_f4(reinterpret_cast<float*>(gnrm_b + static_cast<uint64_t>(ir) * d4), gwv.x, gwv.y, gwv.z, gwv.w);
      } else {
        const uint32_t g0 = static_cast<uint32_t>(j) * (2 + K) * d4;
        stg_f4_hint(reinterpret_cast<float4*>(gent_b + g0), gh.x, gh.y, gh.z, gh.w, pol_stream);
        stg_f4_hint(reinterpret_cast<float4*>(gent_b + g0 + d4), gt.x, gt.y, gt.z, gt.w, pol_stream);
        stg_f4_hint(reinterpret_cast<float4*>(grel_b + static_cast<uint32_t>(j) * d4), gr.x, gr.y, gr.z, gr.w, pol_stream);
        stg_f4_hint(reinterpret_cast<float4*>(gnrm_b + static_cast<uint32_t>(j) * d4), gwv.x, gwv.y, gwv.z, gwv.w, pol_stream);
      }
    }
  }
  if (bad && status) *status = 1;
}

// --- TransR, d <= 128: forward + ranking loss + backward of a group in one pass ------------------
// (transR.py:65-78, misc.py:21-26.)  The generic path re-reads the relation's d x d matrix M for every
// triple and adds its gradient with d*d atomics per triple.  A group shares one relation, so here a warp
//   * stages the 2 + K entity rows V = [h, t, c_1..c_K] in shared memory and computes Y = M V with every
//     lane owning rows of M (its own 3-4 rows, read once, 16 bytes at a time; V chunks are broadcast loads):
//     no cross-lane reduction for the projections, one shuffle tree per score only;
//   * forms residuals, losses and dL/dY = G in registers (row-owner layout), writes the relation-row gradient;
//   * adds the matrix gradient G V^T for the whole group with ONE set of d*d/4 vector atomics;
//   * transposes G through shared memory and computes the entity-row gradients M^T G with lanes owning
//     16-byte column chunks (coalesced second pass over M), storing the 2 + K slot rows.
// M is read twice per group instead of twice per triple, the atomics drop by 1 + K.
template <int NVT, bool MARGIN>
__global__ void __launch_bounds__(kThreads, 1)
k_group_step_r(const GroupArgs G, const float up0, float* __restrict__ pos_scores, float* __restrict__ neg_scores,
               float* __restrict__ group_loss, const kgrec_grads Gr, int64_t* __restrict__ slot_ent,
               int64_t* __restrict__ slot_rel, int32_t* status, const int32_t* __restrict__ order) {
  extern __shared__ __align__(16) float rsm[];
  const kgrec_tables& T = G.T;
  const LossCfg& L = G.L;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int K = L.n_neg, nv = 2 + K;
  const int d = T.dim, NC = d >> 2;
  const int n_pos = static_cast<int>(L.n_pos);
  const uint32_t n_ent = static_cast<uint32_t>(T.n_ent);
  const int l1 = T.l1;
  const int bp = static_cast<int>(L.batch_pos < 0x7fffffff ? L.batch_pos : 0x7fffffff);
  const float prm = L.param;
  float4* Vs = reinterpret_cast<float4*>(rsm) + static_cast<size_t>(wid) * (NVT * NC + d * (NVT / 4));   // [nv][NC]
  float4* GT = Vs + NVT * NC;                                                                            // [d][NVT / 4]
  const void* pcol = lane == 0 ? G.ph : (lane == 1 ? G.pt : G.pr);
  bool bad = false;
  // groups in relation order (`order`, k_rel_*): a CTA takes a CONTIGUOUS chunk of it, so its warps work on the same
  // relation and M_r (40 KB at d = 100) stays in this SM's L1 across the chunk
  const int chunk = ((n_pos + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x) + kWarpsPerCta - 1) / kWarpsPerCta * kWarpsPerCta;
  const int i_end = min(n_pos, (static_cast<int>(blockIdx.x) + 1) * chunk);

  for (int i = blockIdx.x * chunk + wid; i < i_end; i += kWarpsPerCta) {
    const int j = __ldg(order + i);
    const int32_t cv = lane < K ? __ldg(G.corrupt + static_cast<int64_t>(j) * K + lane) : 0;
    const int64_t pv = lane < 3 ? load_idx(pcol, j, G.is64) : 0;
    const int64_t vh = __shfl_sync(FULL, pv, 0), vt = __shfl_sync(FULL, pv, 1), vr = __shfl_sync(FULL, pv, 2);
    uint32_t ih = static_cast<uint32_t>(vh), it = static_cast<uint32_t>(vt), ir = static_cast<uint32_t>(vr);
    if (static_cast<uint64_t>(vh) >= static_cast<uint64_t>(T.n_ent)) { bad = true; ih = 0; }
    if (static_cast<uint64_t>(vt) >= static_cast<uint64_t>(T.n_ent)) { bad = true; it = 0; }
    if (static_cast<uint64_t>(vr) >= static_cast<uint64_t>(T.n_rel)) { bad = true; ir = 0; }
    const int64_t slot0 = static_cast<int64_t>(j) * nv;
    if (slot_ent) {
      if (lane < 2) slot_ent[slot0 + lane] = pv;
      if (lane == 2) slot_rel[j] = pv;
      if (lane < K) slot_ent[slot0 + 2 + lane] = cv < 0 ? ~cv : cv;
    }
    // ---- stage V = [h, t, c_1..c_K]
    __syncwarp();
    for (int v = 0; v < nv; ++v) {
      uint32_t id;
      if (v == 0) id = ih;
      else if (v == 1) id = it;
      else {
        const int32_t c = __shfl_sync(FULL, cv, v - 2);
        id = static_cast<uint32_t>(c < 0 ? ~c : c);
        if (id >= n_ent) { bad = true; id = 0; }
      }
      if (lane < NC) Vs[v * NC + lane] = ldg_f4(reinterpret_cast<const float4*>(T.ent + static_cast<uint64_t>(id) * T.ld) + lane);
    }
    __syncwarp();
    const float* M = T.proj + static_cast<uint64_t>(ir) * d * d;

    // ---- Y = M V, lane owns rows a = lane + 32 i
    float y[4][NVT];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int v = 0; v < NVT; ++v) y[i][v] = 0.f;
    for (int c = 0; c < NC; ++c) {
      float4 m[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int a = lane + 32 * i;
        m[i] = a < d ? __ldg(reinterpret_cast<const float4*>(M + static_cast<size_t>(a) * d) + c) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int v = 0; v < NVT; ++v) {
        if (v < nv) {
          const float4 x = Vs[v * NC + c];
#pragma unroll
          for (int i = 0; i < 4; ++i) y[i][v] = fmaf(m[i].x, x.x, fmaf(m[i].y, x.y, fmaf(m[i].z, x.z, fmaf(m[i].w, x.w, y[i][v]))));
        }
      }
    }
    float rr[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int a = lane + 32 * i;
      rr[i] = a < d ? __ldg(T.rel + static_cast<uint64_t>(ir) * T.ld + a) : 0.f;
    }
    // ---- scores, loss, coefficients
    float up = up0;
    if (!MARGIN) {
      const int b = j / bp;
      up /= static_cast<float>(min(bp, n_pos - b * bp)) * static_cast<float>(K);
    }
    float sp = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) sp += (lane + 32 * i < d) ? dist_term(y[i][0] + rr[i] - y[i][1], l1) : 0.f;
    sp = warp_sum(sp);
    float lsum = 0.f, cpos = 0.f, mys = 0.f;
    float gp[4] = {0.f, 0.f, 0.f, 0.f};       // sum of dLoss/de over the group's triples (= relation-row gradient), per owned row
    float gh[4] = {0.f, 0.f, 0.f, 0.f}, gt[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int v = 2; v < NVT; ++v) {
      if (v < nv) {
        const int k = v - 2;
        const bool head = __shfl_sync(FULL, cv, k) < 0;
        float e[4], sn = 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          e[i] = head ? y[i][v] + rr[i] - y[i][1] : y[i][0] + rr[i] - y[i][v];
          sn += (lane + 32 * i < d) ? dist_term(e[i], l1) : 0.f;
        }
        sn = warp_sum(sn);
        if (lane == k) mys = sn;
        float coef;                        // dLoss/dsn
        if (MARGIN) {
          const float tt = sp - sn + prm;
          lsum += fmaxf(tt, 0.f);
          coef = tt > 0.f ? -up : 0.f;
          cpos += tt > 0.f ? 1.f : 0.f;
        } else {
          const float xx = prm * (sp - sn);
          lsum += fmaxf(-xx, 0.f) + log1pf(expf(-fabsf(xx)));
          const float dp = -prm / (1.f + expf(xx));
          cpos += dp;
          coef = -dp * up;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float g = coef * ddist_term(e[i], l1);          // dLoss/de of this negative
          gp[i] += g;
          if (head) { y[i][v] = g; gt[i] -= g; }                   // e = y_c + r - y_t
          else { y[i][v] = -g; gh[i] += g; }                       // e = y_h + r - y_c
        }
      }
    }
    {
      const float cp = cpos * up;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float g = cp * ddist_term(y[i][0] + rr[i] - y[i][1], l1);
        gp[i] += g;
        y[i][0] = gh[i] + g;                                       // G for h
        y[i][1] = gt[i] - g;                                       // G for t
      }
    }
    if (lane == 0) {
      pos_scores[j] = sp;
      group_loss[j] = lsum;
    }
    if (lane < K) neg_scores[static_cast<int64_t>(j) * K + lane] = mys;
    // relation-row gradient
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int a = lane + 32 * i;
      if (a < d) {
        if (Gr.mode == 0) Gr.rel[static_cast<int64_t>(j) * d + a] = gp[i];
        else atomicAdd(Gr.rel + static_cast<uint64_t>(ir) * d + a, gp[i]);
      }
    }
    // ---- matrix gradient G V^T: one vector atomic per (row, chunk) for the whole group; and G^T to shared memory
    float* gM = Gr.proj + static_cast<uint64_t>(ir) * d * d;
    for (int c = 0; c < NC; ++c) {
      float4 acc[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int v = 0; v < NVT; ++v) {
        if (v < nv) {
          const float4 x = Vs[v * NC + c];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            acc[i].x = fmaf(y[i][v], x.x, acc[i].x); acc[i].y = fmaf(y[i][v], x.y, acc[i].y);
            acc[i].z = fmaf(y[i][v], x.z, acc[i].z); acc[i].w = fmaf(y[i][v], x.w, acc[i].w);
          }
        }
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int a = lane + 32 * i;
        if (a < d) red_add_f4(gM + static_cast<size_t>(a) * d + 4 * c, acc[i].x, acc[i].y, acc[i].z, acc[i].w);
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int a = lane + 32 * i;
      if (a < d) {
#pragma unroll
        for (int v4 = 0; v4 < NVT / 4; ++v4)
          GT[a * (NVT / 4) + v4] = make_float4(y[i][4 * v4], y[i][4 * v4 + 1], y[i][4 * v4 + 2], y[i][4 * v4 + 3]);
      }
    }
    __syncwarp();
    // ---- entity-row gradients M^T G, lane owns column chunk `lane`
    float4 gv[NVT];
#pragma unroll
    for (int v = 0; v < NVT; ++v) gv[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (lane < NC) {
      for (int a = 0; a < d; ++a) {
        const float4 mrow = __ldg(reinterpret_cast<const float4*>(M + static_cast<size_t>(a) * d) + lane);
#pragma unroll
        for (int v4 = 0; v4 < NVT / 4; ++v4) {
          const float4 g4 = GT[a * (NVT / 4) + v4];
          const float gs[4] = {g4.x, g4.y, g4.z, g4.w};
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int v = 4 * v4 + u;
            gv[v].x = fmaf(gs[u], mrow.x, gv[v].x); gv[v].y = fmaf(gs[u], mrow.y, gv[v].y);
            gv[v].z = fmaf(gs[u], mrow.z, gv[v].z); gv[v].w = fmaf(gs[u], mrow.w, gv[v].w);
          }
        }
      }
#pragma unroll
      for (int v = 0; v < NVT; ++v) {
        if (v < nv) {
          if (Gr.mode == 0) {
            __stcs(reinterpret_cast<float4*>(Gr.ent + (slot0 + v) * d) + lane, gv[v]);
          } else {
            uint32_t id;
            if (v == 0) id = ih;
            else if (v == 1) id = it;
            else {
              const int32_t c = G.corrupt[static_cast<int64_t>(j) * K + (v - 2)];
              id = static_cast<uint32_t>(c < 0 ? ~c : c);
              if (id >= n_ent) id = 0;
            }
            red_add_f4(Gr.ent + static_cast<uint64_t>(id) * d + 4 * lane, gv[v].x, gv[v].y, gv[v].z, gv[v].w);
          }
        }
      }
    }
    __syncwarp();
  }
  if (bad && status) *status = 1;
}

// --- TransR, relation runs: the CTA-level step ----------------------------------------------------------------
// The groups of a launch are visited in relation order (`order`, k_rel_*).  A CTA walks a contiguous chunk of that order
// tile by tile; a tile is up to (64 RB) / (2 + K) consecutive groups of ONE relation, i.e. up to 64 RB entity rows V.
// M_r and M_r^T stay in shared memory while the relation does not change, the gradient of M_r in registers (one flush per
// relation run and CTA), and the three products of the step are register-tiled FP32 GEMMs on shared-memory operands:
//     Y  = V M^T            [rows x d]  (warp = 8 rows of V, lane = rows a = lane + 32 q of M, dot form along b)
//     dM += G^T V           [d x d]     (thread = 4 QA rows a x 4 QB columns b, rank-1 form along the tile's rows)
//     dV = G M              [rows x d]  (warp = 8 rows of G, lane = rows b = lane + 32 q of M^T, dot form along a)
// with the scores / ranking loss / G = dL/dY stage of the warp kernel between the first and the other two (one warp per
// group, Y read from and G written to the same shared buffer).  Both [rows x d] products are one routine (run_tile_dot):
// two packed fma.rn.f32x2 per pair of 16-byte operands, no splats; QF = d / 32 full lane-rows, the d - 32 QF rows left
// (4 at d = 100) in a short (row, lane) pass instead of a quarter-empty fourth accumulator column.  The row pitch is an
// odd number of 16-byte units: the lane-per-row reads are conflict-free.
__host__ __device__ inline int run_pitch(int d) { return ((d >> 2) & 1) ? d : d + 4; }

template <int QF, typename Emit>
__device__ __forceinline__ void run_tile_dot(const float* __restrict__ A, const float* __restrict__ B, const int d, const int NC,
                                             const int pitch, const int lane, Emit emit) {
  f32x2 acc[8][QF];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int q = 0; q < QF; ++q) acc[i][q] = 0ull;
  const ulonglong2* pb[QF];
  const ulonglong2* pa[8];
#pragma unroll
  for (int q = 0; q < QF; ++q) pb[q] = reinterpret_cast<const ulonglong2*>(B + (lane + 32 * q) * pitch);
#pragma unroll
  for (int i = 0; i < 8; ++i) pa[i] = reinterpret_cast<const ulonglong2*>(A + i * pitch);
#pragma unroll 2
  for (int c = 0; c < NC; ++c) {
    ulonglong2 m[QF];
#pragma unroll
    for (int q = 0; q < QF; ++q) { m[q] = *pb[q]; ++pb[q]; }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const ulonglong2 x = *pa[i];
      ++pa[i];
#pragma unroll
      for (int q = 0; q < QF; ++q) acc[i][q] = fma2(m[q].x, x.x, fma2(m[q].y, x.y, acc[i][q]));
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int q = 0; q < QF; ++q) emit(i, lane + 32 * q, sum2(acc[i][q]));
  const int rem = d - 32 * QF;
  for (int p = lane; p < 8 * rem; p += 32) {
    const int i = p / rem, a = 32 * QF + p - i * rem;
    const ulonglong2* xa = reinterpret_cast<const ulonglong2*>(A + i * pitch);
    const ulonglong2* xb = reinterpret_cast<const ulonglong2*>(B + a * pitch);
    f32x2 s = 0ull;
    for (int c = 0; c < NC; ++c) s = fma2(xb[c].x, xa[c].x, fma2(xb[c].y, xa[c].y, s));
    emit(i, a, sum2(s));
  }
}

template <int QA, int QB, int QF, int RB, bool MARGIN>
__global__ void __launch_bounds__(kThreads, 1)
k_run_step_r(const GroupArgs G, const float up0, float* __restrict__ pos_scores, float* __restrict__ neg_scores,
             float* __restrict__ group_loss, const kgrec_grads Gr, int64_t* __restrict__ slot_ent,
             int64_t* __restrict__ slot_rel, int32_t* status, const int32_t* __restrict__ order) {
  extern __shared__ __align__(16) float rsm[];
  constexpr int ROWS = 64 * RB;
  const kgrec_tables& T = G.T;
  const LossCfg& L = G.L;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int K = L.n_neg, nv = 2 + K, GC = min(32, ROWS / nv);
  const int d = T.dim, NC = d >> 2, pitch = run_pitch(d);
  const int n_pos = static_cast<int>(L.n_pos);
  const int l1 = T.l1;
  const int bp = static_cast<int>(L.batch_pos < 0x7fffffff ? L.batch_pos : 0x7fffffff);
  const float prm = L.param;
  float* sM = rsm;                                   // [d][pitch]
  float* sMt = sM + d * pitch;                       // [d][pitch]  M^T
  float* sV = sMt + d * pitch;                       // [ROWS][pitch]
  float* sG = sV + ROWS * pitch;                     // [ROWS][pitch]  Y, then G
  float** sDst = reinterpret_cast<float**>(sG + ROWS * pitch);          // [2][ROWS] where the row's entity gradient goes
  const float** sSrc = const_cast<const float**>(sDst + 2 * ROWS);      // [ROWS] table rows of the NEXT tile (nullptr: zero row)
  int* sJ = reinterpret_cast<int*>(sSrc + ROWS);     // [2][36]: group index of the tile's groups; [32] relation, [33] groups
  bool bad = false;

  // dM tile of this thread: rows 4 (ta + nta q) .. + 3, column chunks tb + ntb q
  const int nta = (NC + QA - 1) / QA, ntb = (NC + QB - 1) / QB;
  const int ta = threadIdx.x % nta, tb = threadIdx.x / nta;
  const bool mt = tb < ntb;
  f32x2 accM[QA * 4][QB][2];
#pragma unroll
  for (int i = 0; i < QA * 4; ++i)
#pragma unroll
    for (int q = 0; q < QB; ++q) accM[i][q][0] = accM[i][q][1] = 0ull;
  auto flush = [&](int rel) {
    if (rel < 0 || !mt) return;
    float* gM = Gr.proj + static_cast<uint64_t>(rel) * d * d;
#pragma unroll
    for (int qa = 0; qa < QA; ++qa)
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int a = 4 * (ta + nta * qa) + r;
#pragma unroll
        for (int q = 0; q < QB; ++q) {
          const int cb = tb + ntb * q;
          f32x2(&v)[2] = accM[4 * qa + r][q];
          if (a < d && cb < NC) red_add_f4(gM + static_cast<size_t>(a) * d + 4 * cb, lo2(v[0]), hi2(v[0]), lo2(v[1]), hi2(v[1]));
          v[0] = v[1] = 0ull;
        }
      }
  };

  const int chunk = (n_pos + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);
  const int i_end = min(n_pos, (static_cast<int>(blockIdx.x) + 1) * chunk);
  int cur_rel = -1;
  float rr[4] = {0.f, 0.f, 0.f, 0.f};

  // The tile that starts at group i_from of the order (one warp): its groups -- the leading ones of the chunk's rest that
  // share a relation --, then per tile row the table row to copy from and the place its gradient goes to.
  auto plan = [&](int buf, int i_from) {
    int* J = sJ + 36 * buf;
    int j = -1;
    int64_t r = -1;
    if (lane < GC && i_from + lane < i_end) {
      j = __ldg(order + i_from + lane);
      r = load_idx(G.pr, j, G.is64);
      if (static_cast<uint64_t>(r) >= static_cast<uint64_t>(T.n_rel)) { bad = true; r = 0; }
    }
    const int64_t r0 = __shfl_sync(FULL, r, 0);
    const uint32_t same = __ballot_sync(FULL, j >= 0 && r == r0);
    const int ng = same == FULL ? 32 : __ffs(~same) - 1;          // leading ones; 0 past the chunk's end
    J[lane] = j;
    if (lane == 0) { J[32] = static_cast<int>(r0); J[33] = ng; }
    __syncwarp();
    const int rows = ng * nv;
    for (int n = lane; n < ROWS; n += 32) {
      const float* src = nullptr;
      if (n < rows) {
        const int gq = n / nv, v = n - gq * nv, jj = J[gq];
        int64_t id;
        if (v == 0) id = load_idx(G.ph, jj, G.is64);
        else if (v == 1) id = load_idx(G.pt, jj, G.is64);
        else { const int32_t c = __ldg(G.corrupt + static_cast<int64_t>(jj) * K + (v - 2)); id = c < 0 ? ~c : c; }
        if (slot_ent) {
          slot_ent[static_cast<int64_t>(jj) * nv + v] = id;
          if (v == 0) slot_rel[jj] = load_idx(G.pr, jj, G.is64);
        }
        if (static_cast<uint64_t>(id) >= static_cast<uint64_t>(T.n_ent)) { bad = true; id = 0; }
        sDst[buf * ROWS + n] = Gr.mode == 0 ? Gr.ent + (static_cast<int64_t>(jj) * nv + v) * d : Gr.ent + static_cast<uint64_t>(id) * d;
        src = T.ent + static_cast<uint64_t>(id) * T.ld;
      }
      sSrc[n] = src;
    }
  };
  // V of the planned tile: 16-byte asynchronous copies straight into shared memory (zero rows past the tile's last group)
  auto copy_rows = [&]() {
    for (int idx = threadIdx.x; idx < ROWS * NC; idx += kThreads) {
      const int n = idx / NC, c = idx - n * NC;
      const float* src = sSrc[n];
      float* dst = sV + n * pitch + 4 * c;
      if (src) {
        const uint32_t sa = static_cast<uint32_t>(__cvta_generic_to_shared(dst));
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(src + 4 * c) : "memory");
      } else {
        *reinterpret_cast<float4*>(dst) = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };

  int i0 = blockIdx.x * chunk, buf = 0;
  if (wid == 0) plan(0, i0);
  __syncthreads();
  copy_rows();
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();

  while (true) {
    const int* J = sJ + 36 * buf;
    const int rel = J[32], ng = J[33], rows = ng * nv;
    if (ng == 0) break;
    if (rel != cur_rel) {
      flush(cur_rel);
      cur_rel = rel;
      const float4* M4 = reinterpret_cast<const float4*>(T.proj + static_cast<uint64_t>(rel) * d * d);
      for (int idx = threadIdx.x; idx < d * NC; idx += kThreads) {
        const int c = idx / d, a = idx - c * d;                   // lanes along a: the transposed stores are conflict-free
        const float4 m = __ldg(M4 + a * NC + c);
        *reinterpret_cast<float4*>(sM + a * pitch + 4 * c) = m;
        sMt[(4 * c) * pitch + a] = m.x; sMt[(4 * c + 1) * pitch + a] = m.y;
        sMt[(4 * c + 2) * pitch + a] = m.z; sMt[(4 * c + 3) * pitch + a] = m.w;
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int a = lane + 32 * i;
        rr[i] = a < d ? __ldg(T.rel + static_cast<uint64_t>(rel) * T.ld + a) : 0.f;
      }
      __syncthreads();
    }
    // ---- Y = V M^T
#pragma unroll 1
    for (int rb = 0; rb < RB; ++rb) {
      const int base = 8 * (wid + kWarpsPerCta * rb);
      if (base >= rows) break;
      float* yrow = sG + base * pitch;
      run_tile_dot<QF>(sV + base * pitch, sM, d, NC, pitch, lane, [&](int i, int a, float v) { yrow[i * pitch + a] = v; });
    }
    __syncthreads();
    // ---- scores, ranking loss, G = dL/dY in place: one warp per group
    for (int gq = wid; gq < ng; gq += kWarpsPerCta) {
      const int j = J[gq];
      float* Y = sG + gq * nv * pitch;
      const int32_t cv = lane < K ? __ldg(G.corrupt + static_cast<int64_t>(j) * K + lane) : 0;
      float up = up0;
      if (!MARGIN) {
        const int b = j / bp;
        up /= static_cast<float>(min(bp, n_pos - b * bp)) * static_cast<float>(K);
      }
      float yh[4], yt[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int a = lane + 32 * i;
        yh[i] = a < d ? Y[a] : 0.f;
        yt[i] = a < d ? Y[pitch + a] : 0.f;
      }
      float sp = 0.f;
#pragma unroll
      for (int i = 0; i < 4; ++i) sp += (lane + 32 * i < d) ? dist_term(yh[i] + rr[i] - yt[i], l1) : 0.f;
      sp = warp_sum(sp);
      float lsum = 0.f, cpos = 0.f, mys = 0.f;
      float gp[4] = {0.f, 0.f, 0.f, 0.f}, gh[4] = {0.f, 0.f, 0.f, 0.f}, gt[4] = {0.f, 0.f, 0.f, 0.f};
      for (int k = 0; k < K; ++k) {
        const bool head = __shfl_sync(FULL, cv, k) < 0;
        float* Yc = Y + (2 + k) * pitch;
        float e[4], sn = 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int a = lane + 32 * i;
          const float yc = a < d ? Yc[a] : 0.f;
          e[i] = head ? yc + rr[i] - yt[i] : yh[i] + rr[i] - yc;
          sn += a < d ? dist_term(e[i], l1) : 0.f;
        }
        sn = warp_sum(sn);
        if (lane == k) mys = sn;
        float coef;
        if (MARGIN) {
          const float tt = sp - sn + prm;
          lsum += fmaxf(tt, 0.f);
          coef = tt > 0.f ? -up : 0.f;
          cpos += tt > 0.f ? 1.f : 0.f;
        } else {
          const float xx = prm * (sp - sn);
          lsum += fmaxf(-xx, 0.f) + log1pf(expf(-fabsf(xx)));
          const float dp = -prm / (1.f + expf(xx));
          cpos += dp;
          coef = -dp * up;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int a = lane + 32 * i;
          const float g = coef * ddist_term(e[i], l1);
          gp[i] += g;
          if (head) gt[i] -= g; else gh[i] += g;
          if (a < d) Yc[a] = head ? g : -g;
        }
      }
      const float cp = cpos * up;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int a = lane + 32 * i;
        const float g = cp * ddist_term(yh[i] + rr[i] - yt[i], l1);
        gp[i] += g;
        if (a < d) {
          Y[a] = gh[i] + g;
          Y[pitch + a] = gt[i] - g;
          if (Gr.mode == 0) Gr.rel[static_cast<int64_t>(j) * d + a] = gp[i];
          else atomicAdd(Gr.rel + static_cast<uint64_t>(rel) * d + a, gp[i]);
        }
      }
      if (lane == 0) { pos_scores[j] = sp; group_loss[j] = lsum; }
      if (lane < K) neg_scores[static_cast<int64_t>(j) * K + lane] = mys;
    }
    if (wid == kWarpsPerCta - 1) plan(buf ^ 1, i0 + ng);          // the next tile's rows, while the other warps finish their groups
    __syncthreads();
    // ---- dM += G^T V   (chunks past the row end are clamped: they accumulate values that are never flushed)
    if (mt) {
      const float4* gp[QA];
      const ulonglong2* vp[QB];
#pragma unroll
      for (int qa = 0; qa < QA; ++qa) gp[qa] = reinterpret_cast<const float4*>(sG + 4 * min(ta + nta * qa, NC - 1));
#pragma unroll
      for (int q = 0; q < QB; ++q) vp[q] = reinterpret_cast<const ulonglong2*>(sV + 4 * min(tb + ntb * q, NC - 1));
      const int p4 = pitch >> 2;
#pragma unroll 2
      for (int n = 0; n < rows; ++n) {
        float4 g[QA];
        ulonglong2 v[QB];
#pragma unroll
        for (int qa = 0; qa < QA; ++qa) { g[qa] = *gp[qa]; gp[qa] += p4; }
#pragma unroll
        for (int q = 0; q < QB; ++q) { v[q] = *vp[q]; vp[q] += p4; }
#pragma unroll
        for (int qa = 0; qa < QA; ++qa) {
          const float gs[4] = {g[qa].x, g[qa].y, g[qa].z, g[qa].w};
#pragma unroll
          for (int r = 0; r < 4; ++r) {
            const f32x2 s2 = splat2(gs[r]);
#pragma unroll
            for (int q = 0; q < QB; ++q) {
              accM[4 * qa + r][q][0] = fma2(s2, v[q].x, accM[4 * qa + r][q][0]);
              accM[4 * qa + r][q][1] = fma2(s2, v[q].y, accM[4 * qa + r][q][1]);
            }
          }
        }
      }
    }
    __syncthreads();
    copy_rows();                                                   // V of the next tile lands while dV is computed
    // ---- dV = G M
#pragma unroll 1
    for (int rb = 0; rb < RB; ++rb) {
      const int base = 8 * (wid + kWarpsPerCta * rb);
      if (base >= rows) break;
      const int dense = Gr.mode;
      float* const* dstp = sDst + buf * ROWS + base;
      run_tile_dot<QF>(sG + base * pitch, sMt, d, NC, pitch, lane, [&](int i, int b, float v) {
        if (base + i < rows) {
          float* dst = dstp[i] + b;
          if (dense) atomicAdd(dst, v); else __stcs(dst, v);
        }
      });
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
    i0 += ng;
    buf ^= 1;
  }
  flush(cur_rel);
  if (bad && status) *status = 1;
}

// slot row ids for the general step kernel (TransH, wide rows): one thread per slot
__global__ void __launch_bounds__(256)
k_group_slot_ids(const void* ph, const void* pt, const void* pr, const int is64, const int32_t* __restrict__ corrupt,
                 const int64_t n_pos, const int K, int64_t* __restrict__ slot_ent, int64_t* __restrict__ slot_rel) {
  const int64_t total = n_pos * (2 + K);
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t j = i / (2 + K);
    const int t = static_cast<int>(i - j * (2 + K));
    int64_t v;
    if (t == 0) { v = load_idx(ph, j, is64); slot_rel[j] = load_idx(pr, j, is64); }
    else if (t == 1) v = load_idx(pt, j, is64);
    else { const int32_t c = __ldg(corrupt + j * K + (t - 2)); v = c < 0 ? ~c : c; }
    slot_ent[i] = v;
  }
}

// --- groups in relation order (TransR): counting sort of the positives' relation ids --------------------------------
__global__ void __launch_bounds__(256)
k_rel_hist(const void* pr, const int is64, const int n_pos, const int64_t n_rel, int32_t* __restrict__ count) {
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n_pos; j += gridDim.x * blockDim.x) {
    int64_t r = load_idx(pr, j, is64);
    if (static_cast<uint64_t>(r) >= static_cast<uint64_t>(n_rel)) r = 0;          // the step kernel reports it
    atomicAdd(count + r, 1);
  }
}

// exclusive scan of count[0 .. n_rel) in place, one CTA (n_rel is a table height: thousands at most in practice)
__global__ void __launch_bounds__(1024)
k_rel_scan(int32_t* __restrict__ count, const int64_t n_rel) {
  __shared__ int32_t part[1024];
  const int64_t per = (n_rel + 1023) / 1024, lo = threadIdx.x * per, hi = lo + per < n_rel ? lo + per : n_rel;
  int32_t s = 0;
  for (int64_t r = lo; r < hi; ++r) s += count[r];
  part[threadIdx.x] = s;
  __syncthreads();
  for (int off = 1; off < 1024; off <<= 1) {
    const int32_t v = threadIdx.x >= off ? part[threadIdx.x - off] : 0;
    __syncthreads();
    part[threadIdx.x] += v;
    __syncthreads();
  }
  int32_t run = part[threadIdx.x] - s;
  for (int64_t r = lo; r < hi; ++r) { const int32_t c = count[r]; count[r] = run; run += c; }
}

__global__ void __launch_bounds__(256)
k_rel_scatter(const void* pr, const int is64, const int n_pos, const int64_t n_rel, int32_t* __restrict__ cursor,
              int32_t* __restrict__ order) {
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n_pos; j += gridDim.x * blockDim.x) {
    int64_t r = load_idx(pr, j, is64);
    if (static_cast<uint64_t>(r) >= static_cast<uint64_t>(n_rel)) r = 0;
    order[atomicAdd(cursor + r, 1)] = j;
  }
}

int make_plan(const kgrec_tables* T, int model, Plan* pl);

// Checks the arguments of a corrupt-format call and builds its kernel arguments.  small32: 32-bit slot offsets
// suffice and a group's scores fit in the lanes of a warp, as the d <= 128 step kernels need.
static int group_check(const kgrec_tables* T, int model, Plan* pl, const void* ph, const void* pt, const void* pr,
                       int idx_bytes, int64_t n_pos, const int32_t* corrupt, int32_t n_neg, int64_t batch_pos,
                       int loss_kind, float margin_or_target, GroupArgs* G, bool* small32, bool allow_r = false) {
  int rc = make_plan(T, model, pl);
  if (rc) return rc;
  if (pl->fam != FAM_E && pl->fam != FAM_H && !(allow_r && pl->fam == FAM_R)) {
    set_error("corrupt-format ranking loss is built for TransE / TransH (model %d)", model);
    return KGREC_ERR_UNSUPPORTED;
  }
  if (!pl->vec) { set_error("corrupt-format ranking loss needs embedding_size %% 4 == 0 and 16-byte aligned tables"); return KGREC_ERR_UNSUPPORTED; }
  if (idx_bytes != 4 && idx_bytes != 8) { set_error("idx_bytes must be 4 or 8"); return KGREC_ERR_INVALID; }
  if (!ph || !pt || !pr || !corrupt) { set_error("index array is NULL"); return KGREC_ERR_INVALID; }
  if (loss_kind != KGREC_LOSS_MARGIN && loss_kind != KGREC_LOSS_BPR) { set_error("unknown loss %d", loss_kind); return KGREC_ERR_INVALID; }
  if (n_pos < 0 || n_pos > 0x7fffffff || n_neg < 1 || batch_pos < 1) { set_error("bad n_pos / n_neg / batch_pos"); return KGREC_ERR_INVALID; }
  if (T->n_ent > 0x7fffffffll) { set_error("corrupt format holds entity ids in 31 bits"); return KGREC_ERR_UNSUPPORTED; }
  *G = GroupArgs{*T, ph, pt, pr, idx_bytes == 8, corrupt, LossCfg{loss_kind, margin_or_target, n_neg, n_pos, batch_pos},
                 l2_keep_fraction(static_cast<double>(T->n_ent) * T->ld * sizeof(float))};
  *small32 = n_neg <= 32 && static_cast<double>(n_pos) * (2 + n_neg) * T->dim * 4 < 4.0e9 &&
             static_cast<double>(n_pos) * n_neg < 2.0e9;
  return KGREC_OK;
}

}  // namespace kgrec

using namespace kgrec;

#define KGREC_GROUP_DISPATCH(CALL)                                            \
  if (pl.fam == FAM_E) {                                                      \
    if (pl.nch == 1) { CALL(FAM_E, 1) } else if (pl.nch == 2) { CALL(FAM_E, 2) } else { CALL(FAM_E, 4) } \
  } else {                                                                    \
    if (pl.nch == 1) { CALL(FAM_H, 1) } else if (pl.nch == 2) { CALL(FAM_H, 2) } else { CALL(FAM_H, 4) } \
  }

extern "C" int kgrec_corrupt_loss_fwd(const kgrec_tables* tables, int model, const void* ph, const void* pt,
                                      const void* pr, int idx_bytes, int64_t n_pos, const int32_t* corrupt,
                                      int32_t n_neg, int64_t batch_pos, int loss_kind, float margin_or_target,
                                      float* pos_scores, float* neg_scores, float* loss, void* workspace,
                                      int32_t* status, kgrec_stream_t stream) {
  Plan pl;
  GroupArgs G;
  bool small32;
  int rc = group_check(tables, model, &pl, ph, pt, pr, idx_bytes, n_pos, corrupt, n_neg, batch_pos, loss_kind,
                       margin_or_target, &G, &small32);
  if (rc) return rc;
  if (!pos_scores || !neg_scores || !loss || !workspace) { set_error("output / workspace pointer is NULL"); return KGREC_ERR_INVALID; }
  if (n_pos == 0) return KGREC_OK;
  float* group_loss = static_cast<float*>(workspace);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (pl.fam == FAM_E && pl.nch == 1 && small32) {
    // the TransE step kernel in forward-only mode (TransH: k_group_fwd measured faster, 1.06 vs 1.09 ms fwd+bwd)
    with_bools([&](auto l1, auto mg) {
      k_group_step_e<l1, false, mg, false, false, true><<<grid_for(n_pos), kThreads, 0, st>>>(
          G, 1.f, nullptr, pos_scores, neg_scores, group_loss, kgrec_grads{}, nullptr, nullptr, status);
    }, tables->l1 != 0, loss_kind == KGREC_LOSS_MARGIN);
  } else {
#define CALL(FAMV, NCHV)                                                                                             \
  with_bools([&](auto l1) {                                                                                          \
    k_group_fwd<FAMV, NCHV, l1><<<grid_for(n_pos), kThreads, 0, st>>>(G, pos_scores, neg_scores, group_loss, status); \
  }, tables->l1 != 0);
  KGREC_GROUP_DISPATCH(CALL)
#undef CALL
  }
  KGREC_CUDA_OK(cudaGetLastError());
  const int64_t n_batches = (n_pos + batch_pos - 1) / batch_pos;
  k_batch_loss<<<static_cast<unsigned>(n_batches), 256, 0, st>>>(group_loss, G.L, loss);
  KGREC_CUDA_OK(cudaGetLastError());
  return KGREC_OK;
}

extern "C" int kgrec_corrupt_loss_bwd(const kgrec_tables* tables, int model, const void* ph, const void* pt,
                                      const void* pr, int idx_bytes, int64_t n_pos, const int32_t* corrupt,
                                      int32_t n_neg, int64_t batch_pos, int loss_kind, float margin_or_target,
                                      const float* pos_scores, const float* neg_scores, float grad_loss,
                                      const float* grad_loss_dev, const kgrec_grads* grads, int64_t* slot_ent_ids,
                                      int64_t* slot_rel_ids, kgrec_stream_t stream) {
  Plan pl;
  GroupArgs G;
  bool small32;
  int rc = group_check(tables, model, &pl, ph, pt, pr, idx_bytes, n_pos, corrupt, n_neg, batch_pos, loss_kind,
                       margin_or_target, &G, &small32);
  if (rc) return rc;
  if (!pos_scores || !neg_scores) { set_error("saved scores are NULL"); return KGREC_ERR_INVALID; }
  if ((slot_ent_ids == nullptr) != (slot_rel_ids == nullptr)) { set_error("slot_ent_ids and slot_rel_ids go together"); return KGREC_ERR_INVALID; }
  if (!grads || (grads->mode != 0 && grads->mode != 1) || !grads->ent || !grads->rel || (pl.fam == FAM_H && !grads->norm)) {
    set_error("bad grads descriptor");
    return KGREC_ERR_INVALID;
  }
  if (n_pos == 0) return KGREC_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (pl.nch == 1 && small32) {
    // the step kernels in backward mode (coefficients from the saved scores, upstream per batch)
    float* ps = const_cast<float*>(pos_scores);
    float* ns = const_cast<float*>(neg_scores);
    with_bools([&](auto l1, auto dn, auto mg) {
      auto kern = pl.fam == FAM_E ? k_group_step_e<l1, dn, mg, false, true> : k_group_step_h<l1, dn, mg, false, true>;
      kern<<<grid_for(n_pos), kThreads, 0, st>>>(G, grad_loss, grad_loss_dev, ps, ns, nullptr, *grads, slot_ent_ids,
                                                   slot_rel_ids, nullptr);
    }, tables->l1 != 0, grads->mode == 1, loss_kind == KGREC_LOSS_MARGIN);
  } else {
#define CALL(FAMV, NCHV)                                                                                               \
  with_bools([&](auto l1) {                                                                                            \
    k_group_bwd<FAMV, NCHV, l1><<<grid_for(n_pos), kThreads, 0, st>>>(G, pos_scores, neg_scores, grad_loss, grad_loss_dev, *grads); \
  }, tables->l1 != 0);
  KGREC_GROUP_DISPATCH(CALL)
#undef CALL
    if (slot_ent_ids) {
      const int64_t total = n_pos * (2 + static_cast<int64_t>(n_neg));
      const int64_t ctas = (total + 255) / 256, cap = static_cast<int64_t>(sm_count()) * 16;
      k_group_slot_ids<<<static_cast<unsigned>(ctas < cap ? ctas : cap), 256, 0, st>>>(ph, pt, pr, idx_bytes == 8, corrupt, n_pos, n_neg,
                                                                                         slot_ent_ids, slot_rel_ids);
    }
  }
  KGREC_CUDA_OK(cudaGetLastError());
  return KGREC_OK;
}

extern "C" int64_t kgrec_corrupt_loss_step_workspace_bytes(const kgrec_tables* tables, int model, int64_t n_pos) {
  const int64_t n = n_pos > 0 ? n_pos : 1;
  if (model == KGREC_TRANSR && tables) return 4 * (2 * n + tables->n_rel + 1);      // + relation order and its cursors
  return 4 * n;
}

extern "C" int kgrec_corrupt_loss_step(const kgrec_tables* tables, int model, const void* ph, const void* pt,
                                       const void* pr, int idx_bytes, int64_t n_pos, const int32_t* corrupt,
                                       int32_t n_neg, int64_t batch_pos, int loss_kind, float margin_or_target,
                                       float grad_loss, int32_t reg_flags, float* pos_scores, float* neg_scores, float* loss,
                                       const kgrec_grads* grads, int64_t* slot_ent_ids, int64_t* slot_rel_ids,
                                       void* workspace, int32_t* status, kgrec_stream_t stream) {
  Plan pl;
  GroupArgs G;
  bool small32;
  int rc = group_check(tables, model, &pl, ph, pt, pr, idx_bytes, n_pos, corrupt, n_neg, batch_pos, loss_kind,
                       margin_or_target, &G, &small32, true);
  if (rc) return rc;
  if (!pos_scores || !neg_scores || !loss || !workspace) { set_error("output / workspace pointer is NULL"); return KGREC_ERR_INVALID; }
  if (!grads || (grads->mode != 0 && grads->mode != 1) || !grads->ent || !grads->rel || (pl.fam == FAM_H && !grads->norm) ||
      (pl.fam == FAM_R && !grads->proj)) {
    set_error("bad grads descriptor");
    return KGREC_ERR_INVALID;
  }
  if ((slot_ent_ids == nullptr) != (slot_rel_ids == nullptr)) { set_error("slot_ent_ids and slot_rel_ids go together"); return KGREC_ERR_INVALID; }
  if (pl.fam == FAM_R) {
    if (reg_flags) { set_error("fused regularisers are built for TransE / TransH"); return KGREC_ERR_UNSUPPORTED; }
    if (pl.nch != 1 || n_neg > 14) { set_error("TransR step kernel: embedding_size <= 128 and at most 14 negatives per positive"); return KGREC_ERR_UNSUPPORTED; }
    if (n_pos == 0) return KGREC_OK;
    float* gl = static_cast<float*>(workspace);
    cudaStream_t s2 = static_cast<cudaStream_t>(stream);
    // workspace: [group_loss n_pos | order n_pos | cursor n_rel]
    int32_t* order = reinterpret_cast<int32_t*>(gl + n_pos);
    int32_t* cursor = order + n_pos;
    KGREC_CUDA_OK(cudaMemsetAsync(cursor, 0, sizeof(int32_t) * tables->n_rel, s2));
    const int gs = static_cast<int>((n_pos + 255) / 256 < sm_count() * 4 ? (n_pos + 255) / 256 : sm_count() * 4);
    k_rel_hist<<<gs, 256, 0, s2>>>(pr, idx_bytes == 8, static_cast<int>(n_pos), tables->n_rel, cursor);
    k_rel_scan<<<1, 1024, 0, s2>>>(cursor, tables->n_rel);
    k_rel_scatter<<<gs, 256, 0, s2>>>(pr, idx_bytes == 8, static_cast<int>(n_pos), tables->n_rel, cursor, order);
    const bool mg = loss_kind == KGREC_LOSS_MARGIN;
    // short runs (fewer than ~4 groups per relation of the table): staging M_r per tile does not pay, the warp kernel stays
    if (tables->dim >= 32 && n_pos >= 4 * tables->n_rel) {
      // the CTA-level run kernel
      const int d = tables->dim, NC = d / 4, pitch = run_pitch(d), qf = d / 32;
      auto smem_for = [&](int rb) { return (2 * static_cast<size_t>(d) + 2 * 64 * rb) * pitch * 4 + 3 * 64 * rb * 8 + 72 * 4; };
      const int rb = (NC <= 27 && smem_for(2) <= 220 * 1024) ? 2 : 1;
      const size_t smem = smem_for(rb);
      const int64_t want = (n_pos + 3) / 4;                                  // at least ~4 groups per CTA
      const int grid = static_cast<int>(want < sm_count() ? want : sm_count());
#define CALL_RUN(QAV, QBV, QFV, RBV)                                                                                     \
  {                                                                                                                      \
    auto kern = mg ? k_run_step_r<QAV, QBV, QFV, RBV, true> : k_run_step_r<QAV, QBV, QFV, RBV, false>;                   \
    KGREC_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));       \
    kern<<<grid, kThreads, smem, s2>>>(G, grad_loss, pos_scores, neg_scores, gl, *grads, slot_ent_ids, slot_rel_ids, status, order); \
  }
      if (NC <= 16) { if (qf <= 1) CALL_RUN(1, 1, 1, 2) else CALL_RUN(1, 1, 2, 2) }
      else if (NC <= 27) { if (qf <= 2) CALL_RUN(1, 3, 2, 2) else CALL_RUN(1, 3, 3, 2) }
      else { if (qf <= 3) CALL_RUN(2, 2, 3, 1) else CALL_RUN(2, 2, 4, 1) }
#undef CALL_RUN
    } else {
    const int64_t want = (n_pos + kWarpsPerCta - 1) / kWarpsPerCta;
    const int grid_r = static_cast<int>(want < sm_count() ? want : sm_count());          // one resident CTA per SM
    const int nvt = n_neg <= 2 ? 4 : (n_neg <= 10 ? 12 : 16);
    const size_t smem = static_cast<size_t>(kWarpsPerCta) * (static_cast<size_t>(nvt) * (tables->dim / 4) + static_cast<size_t>(tables->dim) * (nvt / 4)) * 16;
#define CALL_R(NVTV, MV)                                                                                             \
  {                                                                                                                  \
    auto kern = k_group_step_r<NVTV, MV>;                                                                            \
    KGREC_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));   \
    kern<<<grid_r, kThreads, smem, s2>>>(G, grad_loss, pos_scores, neg_scores, gl, *grads, slot_ent_ids, slot_rel_ids, status, order); \
  }
    if (nvt == 4) { if (mg) CALL_R(4, true) else CALL_R(4, false) }
    else if (nvt == 12) { if (mg) CALL_R(12, true) else CALL_R(12, false) }
    else { if (mg) CALL_R(16, true) else CALL_R(16, false) }
#undef CALL_R
    }
    KGREC_CUDA_OK(cudaGetLastError());
    const int64_t nbt = (n_pos + batch_pos - 1) / batch_pos;
    k_batch_loss<<<static_cast<unsigned>(nbt), 256, 0, s2>>>(gl, G.L, loss);
    KGREC_CUDA_OK(cudaGetLastError());
    return KGREC_OK;
  }
  if (n_pos == 0) return KGREC_OK;
  float* group_loss = static_cast<float*>(workspace);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (reg_flags != 0 && reg_flags != 1) { set_error("reg_flags must be 0 or 1"); return KGREC_ERR_INVALID; }
  if (reg_flags && loss_kind != KGREC_LOSS_MARGIN) { set_error("fused regularisers go with the margin loss (the KG drivers' loss)"); return KGREC_ERR_UNSUPPORTED; }
  if (pl.nch == 1 && small32) {
    with_bools([&](auto l1, auto dn, auto mg) {
      const bool reg = mg && reg_flags;
      auto kern = pl.fam == FAM_E ? (reg ? k_group_step_e<l1, dn, true, true, false> : k_group_step_e<l1, dn, mg, false, false>)
                                  : (reg ? k_group_step_h<l1, dn, true, true, false> : k_group_step_h<l1, dn, mg, false, false>);
      kern<<<grid_for(n_pos), kThreads, 0, st>>>(G, grad_loss, nullptr, pos_scores, neg_scores, group_loss, *grads,
                                                   slot_ent_ids, slot_rel_ids, status);
    }, tables->l1 != 0, grads->mode == 1, loss_kind == KGREC_LOSS_MARGIN);
  } else {
    if (reg_flags) { set_error("fused regularisers are built for the d <= 128 margin-loss step kernels only"); return KGREC_ERR_UNSUPPORTED; }
#define CALL(FAMV, NCHV)                                                                                                \
  with_bools([&](auto l1) {                                                                                             \
    k_group_step<FAMV, NCHV, l1><<<grid_for(n_pos), kThreads, 0, st>>>(G, grad_loss, pos_scores, neg_scores, group_loss, *grads, status); \
  }, tables->l1 != 0);
  KGREC_GROUP_DISPATCH(CALL)
#undef CALL
    if (slot_ent_ids) {
      const int64_t total = n_pos * (2 + static_cast<int64_t>(n_neg));
      const int64_t ctas = (total + 255) / 256, cap = static_cast<int64_t>(sm_count()) * 16;
      k_group_slot_ids<<<static_cast<unsigned>(ctas < cap ? ctas : cap), 256, 0, st>>>(ph, pt, pr, idx_bytes == 8, corrupt, n_pos, n_neg,
                                                                                         slot_ent_ids, slot_rel_ids);
    }
  }
  KGREC_CUDA_OK(cudaGetLastError());
  const int64_t n_batches = (n_pos + batch_pos - 1) / batch_pos;
  k_batch_loss<<<static_cast<unsigned>(n_batches), 256, 0, st>>>(group_loss, G.L, loss);
  KGREC_CUDA_OK(cudaGetLastError());
  return KGREC_OK;
}
