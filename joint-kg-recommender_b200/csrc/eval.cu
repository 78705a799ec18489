// Full-catalog evaluation: every query (test (t,r) / (h,r) pair, or test user) scored against
// every catalog row (entity / item), reduced on chip to the full score matrix, the K best
// per query, or the count of rows ranked before a gold id.   sm_100a.
//
// Reference semantics restated (CPU form: oracle/kg_oracle.py):
//   transE.py:65-105, transH.py:73-121, transUP.py:84-102, jTransUP.py:163-247 (scores);
//   utils/misc.py:125-146, 213-229 (ranking walk the top-K / rank modes replace).
//
// Structure
//   * CTA = 8 warps; warp w owns 8 queries whose vectors (c, the hyperplane normal, or the
//     user row) live in registers for the whole kernel.
//   * The catalog streams once per 64-query tile: one elected lane moves tiles of TN
//     contiguous rows global -> shared with cp.async.bulk (TMA 1-D bulk copy) into a
//     4-stage ring guarded by full/empty mbarriers, two tiles ahead of the consumers.
//   * A row is spread over the warp (lane c owns float4 chunk c).  For each row the warp
//     forms the 8 per-query partial sums and folds them with one 8-way reduce-scatter
//     (9 shuffles): lanes 4q..4q+3 end up holding query q's score.  Rows are processed four
//     at a time so lane 4q+j holds (query q, row j): one candidate per lane.
//   * top-K: every lane compares its candidate key = score bits << 32 | id with its
//     query's current K-th best (a register); the rare survivors are inserted by the whole
//     warp into that query's sorted list in shared memory ("warp-local top-K").
#include <algorithm>
#include "common.cuh"

namespace kgrec {

enum { KIND_DIST = 0, KIND_HYPER = 1, KIND_PREF_HARD = 2, KIND_PREF_SOFT = 3, KIND_GUMBEL_L2 = 4 };
enum { MODE_FULL = 0, MODE_TOPK = 1, MODE_RANK = 2 };

constexpr int QW = 8;                       // queries per warp
constexpr int TQ = QW * kWarpsPerCta;       // queries per CTA
constexpr int kStages = 4;                 // ring depth
constexpr int kPrefetch = 2;               // tiles in flight ahead of the consumer
constexpr int kEvalThreads = kThreads;
constexpr uint64_t KEY_INF = ~0ull;

// ---- keys -------------------------------------------------------------------------------------
// scores are sums of |.| or squares: non-negative, so the IEEE bit pattern is monotone
__device__ __forceinline__ uint64_t make_key(float s, uint32_t id) {
  return (static_cast<uint64_t>(__float_as_uint(s)) << 32) | id;
}

// warp-cooperative insert of x into the ascending list[0..K) (x < list[K-1] is the caller's job)
__device__ __forceinline__ void list_insert(uint64_t* list, int K, uint64_t x, int lane) {
  int p = 0;
  for (int base = 0; base < K; base += 32) {
    const int j = base + lane;
    p += __popc(__ballot_sync(FULL, j < K && list[j] < x));
  }
  for (int base = ((K - 1) / 32) * 32; base >= 0; base -= 32) {
    const int j = base + lane;
    const uint64_t v = (j >= 1 && j < K) ? list[j - 1] : 0ull;
    __syncwarp();
    if (j < K && j > p) list[j] = v;
    __syncwarp();
  }
  if (lane == 0) list[p] = x;
  __syncwarp();
}

// is `id` in the ascending id list flt[lo, hi) ?
__device__ __forceinline__ bool filtered(const int32_t* __restrict__ flt, int64_t lo, int64_t hi, int32_t id) {
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    const int32_t v = __ldg(flt + mid);
    if (v == id) return true;
    if (v < id) lo = mid + 1; else hi = mid;
  }
  return false;
}

// cheap counter hash for the eval-time Gumbel draw (one 32-bit word per (query, row, k))
__device__ __forceinline__ uint32_t hash_bits(uint64_t seed, uint32_t q, uint32_t n, uint32_t k) {
  uint32_t x = static_cast<uint32_t>(seed) ^ (q * 0x9E3779B1u);
  x ^= x >> 16; x *= 0x21f0aaadu; x ^= x >> 15;
  x ^= n * 0x85EBCA77u + static_cast<uint32_t>(seed >> 32);
  x *= 0x735a2d97u; x ^= x >> 15;
  x ^= k * 0xC2B2AE3Du;
  x ^= x >> 16; x *= 0x21f0aaadu; x ^= x >> 15; x *= 0x735a2d97u; x ^= x >> 15;
  return x;
}

struct EvalArgs {
  kgrec_tables T;
  int ktup;                 // KTUP tables (pref + rel, halves)
  int side;
  const void* q;            // query ids (tail / head / user)
  const void* r;            // relation ids (KG sides)
  int is64;
  const float* qvec;        // optional explicit [nq, 2 dim] (c | w), overrides q / r (KG kinds)
  int64_t nq;
  const float* cat;         // first catalog row of this shard
  int64_t cat_ld;
  int64_t n_cat;
  int64_t id_base;          // global id of cat row 0
  const int32_t* cat_ids;   // optional explicit global id per catalog row (gathered sub-catalogs)
  int n_splits;             // catalog ranges (gridDim.y)
  int tn;                   // catalog rows per tile
  const float* gumbel_u;    // explicit [nq, n_cat, P] (PREF_HARD parity mode)
  uint64_t seed;
  int64_t qvec_ld;          // row stride of qvec (KG kinds: 2 dim; KIND_GUMBEL_L2: the augmented row length)
  const float* gconst;      // KIND_GUMBEL_L2: [3 P] |R_k|^2, |W_k|^2, R_k . W_k of the mixing tables
  // outputs
  float* out; int64_t ld_out;               // FULL
  uint64_t* part_keys; int k;               // TOPK: [n_splits][nq][k]
  uint32_t* thr_glob;                       // TOPK, tiled kernels: [nq] score bits no top-K entry of the call can exceed (shared by the pieces)
  const int64_t* filter_ptr; const int32_t* filter_ids;
  const float* gold_scores; const int32_t* gold_ids; int32_t* counts;   // RANK
};

// smem carve-up (floats unless noted), in this order:
//   bars        : 2 * kStages uint64
//   tiles       : kStages * tn * ld
//   [PREF] sP,sN: 2 * P * stride ; IP: tn * ppad ; UP: 8 warps * QW * ppad
//   [SOFT] IA,IB: 2 * tn * ld
//   [TOPK] lists: TQ * k uint64
struct EvalSmem {
  size_t bars, tiles, sP, sN, IP, UP, IA, IB, lists, total;
};
__host__ __device__ inline EvalSmem eval_smem_layout(int kind, int mode, int d, int64_t ld, int P, int tn, int k) {
  EvalSmem s{};
  size_t off = 0;
  s.bars = off; off += 2 * kStages * sizeof(uint64_t);
  off = (off + 127) & ~static_cast<size_t>(127);
  s.tiles = off; off += static_cast<size_t>(kStages) * tn * ld * sizeof(float);
  if (kind >= KIND_PREF_HARD) {
    const int stride = (d + 3) & ~3, ppad = (P + 3) & ~3;
    s.sP = off; off += static_cast<size_t>(P) * stride * sizeof(float);
    s.sN = off; off += static_cast<size_t>(P) * stride * sizeof(float);
    s.IP = off; off += static_cast<size_t>(tn) * ppad * sizeof(float);
    s.UP = off; off += static_cast<size_t>(kWarpsPerCta) * QW * ppad * sizeof(float);
    if (kind == KIND_PREF_SOFT) {
      s.IA = off; off += static_cast<size_t>(tn) * ld * sizeof(float);
      s.IB = off; off += static_cast<size_t>(tn) * ld * sizeof(float);
    }
  }
  if (mode == MODE_TOPK) {
    off = (off + 7) & ~static_cast<size_t>(7);
    s.lists = off; off += static_cast<size_t>(TQ) * k * sizeof(uint64_t);
  }
  s.total = off;
  return s;
}

template <int KIND, int NCH, int MODE, bool L1>
__global__ void __launch_bounds__(kEvalThreads)
k_eval(const EvalArgs A) {
  using R = Row<NCH, true>;
  constexpr int NE = NCH * 4;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const kgrec_tables& T = A.T;
  const int d = T.dim, P = T.n_pref;
  constexpr int l1 = L1 ? 1 : 0;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int tn = A.tn;
  const int64_t ld = A.cat_ld;
  const EvalSmem L = eval_smem_layout(KIND, MODE, d, ld, P, tn, A.k);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + L.bars);
  uint64_t* empty = full + kStages;
  float* tiles = reinterpret_cast<float*>(smem_raw + L.tiles);

  // catalog range of this CTA
  const int64_t n_tiles_all = (A.n_cat + tn - 1) / tn;
  const int64_t tiles_per_split = (n_tiles_all + A.n_splits - 1) / A.n_splits;
  const int64_t tile0 = static_cast<int64_t>(blockIdx.y) * tiles_per_split;
  const int64_t tile1 = min(n_tiles_all, tile0 + tiles_per_split);
  const int64_t my_tiles = max(static_cast<int64_t>(0), tile1 - tile0);

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, kWarpsPerCta); }
    mbar_fence_init();
  }
  [[maybe_unused]] float* sP = nullptr;
  [[maybe_unused]] float* sN = nullptr;
  [[maybe_unused]] int stride = 0, ppad = 0;
  if constexpr (KIND >= KIND_PREF_HARD) {
    stride = (d + 3) & ~3;
    ppad = (P + 3) & ~3;
    sP = reinterpret_cast<float*>(smem_raw + L.sP);
    sN = reinterpret_cast<float*>(smem_raw + L.sN);
    for (int idx = threadIdx.x; idx < P * stride; idx += blockDim.x) {
      const int k = idx / stride, j = idx - k * stride;
      float a = 0.f, b = 0.f;
      if (j < d) {
        a = __ldg(T.pref + static_cast<int64_t>(k) * T.ld + j);
        b = __ldg(T.pref_norm + static_cast<int64_t>(k) * T.ld + j);
        if (A.ktup) {
          a += __ldg(T.rel + static_cast<int64_t>(k) * T.ld + j);
          b += __ldg(T.norm + static_cast<int64_t>(k) * T.ld + j);
        }
      }
      sP[idx] = a;
      sN[idx] = b;
    }
  }
  __syncthreads();

  // The catalog tiles are moved by TMA bulk copies issued by one lane of warp 0, kPrefetch
  // tiles ahead; a stage is refilled kStages - kPrefetch tiles after its last reader, so the
  // issuing lane practically never waits on the empty barrier.
  auto issue_tile = [&](int64_t t) {
    const int s = static_cast<int>(t % kStages);
    if (t >= kStages) mbar_wait(empty + s, static_cast<uint32_t>(((t / kStages) - 1) & 1));
    const int64_t row0 = (tile0 + t) * tn;
    const int64_t rows = min(static_cast<int64_t>(tn), A.n_cat - row0);
    const uint32_t bytes = static_cast<uint32_t>(rows * ld * sizeof(float));
    mbar_arrive_expect_tx(full + s, bytes);
    bulk_g2s(tiles + static_cast<size_t>(s) * tn * ld, A.cat + row0 * ld, bytes, full + s);
  };
  if (threadIdx.x == 0)
    for (int64_t t = 0; t < kPrefetch && t < my_tiles; ++t) issue_tile(t);

  // ------------------------------------------------------------------ compute warps
  const float hf = A.ktup ? 0.5f : 1.f;
  const int64_t q0 = static_cast<int64_t>(blockIdx.x) * TQ + wid * QW;   // first query of this warp
  float qa[QW][NE];                    // DIST/HYPER: c ; PREF: user row
  [[maybe_unused]] float qb[QW][NE];   // HYPER: w ; SOFT: UA
  [[maybe_unused]] float qc[QW][NE];   // SOFT: UB
  [[maybe_unused]] float* UPw = nullptr;
#pragma unroll
  for (int qi = 0; qi < QW; ++qi) {
    const int64_t q = q0 + qi;
#pragma unroll
    for (int e = 0; e < NE; ++e) { qa[qi][e] = 0.f; if (KIND == KIND_HYPER || KIND == KIND_PREF_SOFT) qb[qi][e] = 0.f; if (KIND == KIND_PREF_SOFT) qc[qi][e] = 0.f; }
    if (q < A.nq) {
      if constexpr (KIND <= KIND_HYPER) {
        if (A.qvec) {
          R::load(qa[qi], A.qvec + q * 2 * d, d, lane);
          if (KIND == KIND_HYPER) R::load(qb[qi], A.qvec + q * 2 * d + d, d, lane);
        } else {
          const int64_t ie = load_idx(A.q, q, A.is64), ir = load_idx(A.r, q, A.is64);
          float ev[NE], rv[NE];
          R::load(ev, T.ent + ie * T.ld, d, lane);
          R::load(rv, T.rel + ir * T.ld, d, lane);
          if (KIND == KIND_HYPER) {
            R::load(qb[qi], T.norm + ir * T.ld, d, lane);
            const float a = warp_sum(R::dot(ev, qb[qi]));
#pragma unroll
            for (int e = 0; e < NE; ++e) ev[e] -= a * qb[qi][e];       // proj(E[q], w)
          }
#pragma unroll
          for (int e = 0; e < NE; ++e) qa[qi][e] = (A.side == KGREC_SIDE_HEAD) ? ev[e] - rv[e] : ev[e] + rv[e];
        }
      } else {
        R::load(qa[qi], T.user + load_idx(A.q, q, A.is64) * T.ld, d, lane);
      }
    }
  }
  if constexpr (KIND >= KIND_PREF_HARD) {
    // UP[qi][k] = u . P_k / 2 ; SOFT: UA = hf sum_k UP_k P_k, UB = hf sum_k UP_k N_k
    UPw = reinterpret_cast<float*>(smem_raw + L.UP) + wid * QW * ppad;
#pragma unroll
    for (int qi = 0; qi < QW; ++qi) {
      for (int g = 0; g < P; g += 8) {
        float vals[8];
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) {
          vals[kk] = 0.f;
          if (g + kk < P) {
            float row[NE];
            R::load_s(row, sP + (g + kk) * stride, d, lane);
            vals[kk] = R::dot(row, qa[qi]);
          }
        }
        const float rr = warp_reduce_scatter8(vals, lane);
        const int k = g + (lane >> 2);
        if ((lane & 3) == 0 && k < P) UPw[qi * ppad + k] = 0.5f * rr;
      }
    }
    __syncwarp();
    if constexpr (KIND == KIND_PREF_SOFT) {
#pragma unroll
      for (int qi = 0; qi < QW; ++qi) {
        for (int k = 0; k < P; ++k) {
          const float z = hf * UPw[qi * ppad + k];
          float row[NE];
          R::load_s(row, sP + k * stride, d, lane);
#pragma unroll
          for (int e = 0; e < NE; ++e) qb[qi][e] = fmaf(z, row[e], qb[qi][e]);
          R::load_s(row, sN + k * stride, d, lane);
#pragma unroll
          for (int e = 0; e < NE; ++e) qc[qi][e] = fmaf(z, row[e], qc[qi][e]);
        }
      }
    }
  }

  // per-lane candidate bookkeeping: lane 4 qi + j serves (query qi, row j of each 4-row group)
  const int myq = lane >> 2, myj = lane & 3;
  const int64_t my_query = q0 + myq;
  const bool q_valid = my_query < A.nq;
  [[maybe_unused]] uint64_t thr = KEY_INF;           // TOPK: current K-th best of my query
  [[maybe_unused]] uint64_t* lists = nullptr;
  [[maybe_unused]] uint64_t gold_key = 0;            // RANK
  [[maybe_unused]] int cnt = 0;
  [[maybe_unused]] int64_t f_lo = 0, f_hi = 0;
  if constexpr (MODE == MODE_TOPK) {
    lists = reinterpret_cast<uint64_t*>(smem_raw + L.lists) + static_cast<size_t>(wid) * QW * A.k;
    for (int i = lane; i < QW * A.k; i += 32) lists[i] = KEY_INF;
    __syncwarp();
    if (A.filter_ptr && q_valid) { f_lo = __ldg(A.filter_ptr + my_query); f_hi = __ldg(A.filter_ptr + my_query + 1); }
  }
  if constexpr (MODE == MODE_RANK) {
    if (q_valid) gold_key = make_key(__ldg(A.gold_scores + my_query), static_cast<uint32_t>(__ldg(A.gold_ids + my_query)));
  }

  for (int64_t t = 0; t < my_tiles; ++t) {
    const int s = static_cast<int>(t % kStages);
    const float* tile = tiles + static_cast<size_t>(s) * tn * ld;
    const int64_t row0 = (tile0 + t) * tn;
    const int rows = static_cast<int>(min(static_cast<int64_t>(tn), A.n_cat - row0));
    if (threadIdx.x == 0 && t + kPrefetch < my_tiles) issue_tile(t + kPrefetch);
    __syncwarp();
    mbar_wait(full + s, static_cast<uint32_t>((t / kStages) & 1));

    [[maybe_unused]] float* IP = nullptr;
    [[maybe_unused]] float* IA = nullptr;
    [[maybe_unused]] float* IB = nullptr;
    if constexpr (KIND >= KIND_PREF_HARD) {
      // catalog-side halves of the logits for this tile (rows split over the 8 warps):
      // IP[row][k] = i_row . P_k / 2 ; SOFT: IA[row] = hf sum_k IP_k P_k, IB likewise with N
      IP = reinterpret_cast<float*>(smem_raw + L.IP);
      if (KIND == KIND_PREF_SOFT) { IA = reinterpret_cast<float*>(smem_raw + L.IA); IB = reinterpret_cast<float*>(smem_raw + L.IB); }
      // all warps must be done with the previous tile's IP / IA / IB
      asm volatile("bar.sync 1, %0;" ::"r"(kThreads));
      for (int rr = wid; rr < rows; rr += kWarpsPerCta) {
        float x[NE];
        R::load_s(x, tile + rr * ld, d, lane);
        for (int g = 0; g < P; g += 8) {
          float vals[8];
#pragma unroll
          for (int kk = 0; kk < 8; ++kk) {
            vals[kk] = 0.f;
            if (g + kk < P) {
              float row[NE];
              R::load_s(row, sP + (g + kk) * stride, d, lane);
              vals[kk] = R::dot(row, x);
            }
          }
          const float v = warp_reduce_scatter8(vals, lane);
          const int k = g + (lane >> 2);
          if ((lane & 3) == 0 && k < P) IP[rr * ppad + k] = 0.5f * v;
        }
        if constexpr (KIND == KIND_PREF_SOFT) {
          __syncwarp();
          float ia[NE], ib[NE];
#pragma unroll
          for (int e = 0; e < NE; ++e) { ia[e] = 0.f; ib[e] = 0.f; }
          for (int k = 0; k < P; ++k) {
            const float z = hf * IP[rr * ppad + k];
            float row[NE];
            R::load_s(row, sP + k * stride, d, lane);
#pragma unroll
            for (int e = 0; e < NE; ++e) ia[e] = fmaf(z, row[e], ia[e]);
            R::load_s(row, sN + k * stride, d, lane);
#pragma unroll
            for (int e = 0; e < NE; ++e) ib[e] = fmaf(z, row[e], ib[e]);
          }
          R::store(IA + rr * ld, ia, d, lane);
          R::store(IB + rr * ld, ib, d, lane);
        }
      }
      asm volatile("bar.sync 1, %0;" ::"r"(kThreads));
    }

    for (int rg = 0; rg < rows; rg += 4) {
      float mine = 0.f;     // score of (query myq, row rg + myj)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int rr = rg + j;
        if (rr < rows) {   // warp-uniform
          float x[NE];
          R::load_s(x, tile + rr * ld, d, lane);
          float vals[QW];
          if constexpr (KIND == KIND_DIST) {
#pragma unroll
            for (int qi = 0; qi < QW; ++qi) {
              float acc = 0.f;
#pragma unroll
              for (int e = 0; e < NE; ++e) acc += dist_term(qa[qi][e] - x[e], l1);
              vals[qi] = acc;
            }
          } else if constexpr (KIND == KIND_HYPER) {
            // s_q = x . w_q for the 8 queries, reduced together and broadcast back
#pragma unroll
            for (int qi = 0; qi < QW; ++qi) vals[qi] = R::dot(x, qb[qi]);
            const float sr = warp_reduce_scatter8(vals, lane);
#pragma unroll
            for (int qi = 0; qi < QW; ++qi) {
              const float sq = __shfl_sync(FULL, sr, qi * 4);
              float acc = 0.f;
#pragma unroll
              for (int e = 0; e < NE; ++e) acc += dist_term(qa[qi][e] - (x[e] - sq * qb[qi][e]), l1);
              vals[qi] = acc;
            }
          } else if constexpr (KIND == KIND_PREF_HARD) {
            // arg-max preference of (query myq, this row): lane handles k = myj, myj + 4, ...
            float best = -INFINITY;
            int bk = 0x7fffffff;
            const uint32_t gn = static_cast<uint32_t>(A.id_base + row0 + rr);
            for (int k = myj; k < P; k += 4) {
              float gn_k;
              if (A.gumbel_u) gn_k = gumbel_from_uniform(q_valid ? __ldg(A.gumbel_u + (my_query * A.n_cat + (row0 + rr)) * P + k) : 0.5f);
              else gn_k = gumbel_fast(hash_bits(A.seed, static_cast<uint32_t>(my_query), gn, static_cast<uint32_t>(k)));
              const float v = UPw[myq * ppad + k] + IP[rr * ppad + k] + gn_k;
              if (v > best) { best = v; bk = k; }
            }
#pragma unroll
            for (int o = 1; o <= 2; o <<= 1) {
              const float ob = __shfl_xor_sync(FULL, best, o);
              const int ok = __shfl_xor_sync(FULL, bk, o);
              if (ob > best || (ob == best && ok < bk)) { best = ob; bk = ok; }
            }
            // phase 1: s_q = (u_q - x) . N[k*_q] ; phase 2: L((u_q - x) + hf (P[k*] - s N[k*]))
            int ks[QW];
#pragma unroll
            for (int qi = 0; qi < QW; ++qi) {
              ks[qi] = __shfl_sync(FULL, bk, qi * 4);
              float wv[NE];
              R::load_s(wv, sN + ks[qi] * stride, d, lane);
              float acc = 0.f;
#pragma unroll
              for (int e = 0; e < NE; ++e) acc = fmaf(qa[qi][e] - x[e], wv[e], acc);
              vals[qi] = acc;
            }
            const float sr = warp_reduce_scatter8(vals, lane);
#pragma unroll
            for (int qi = 0; qi < QW; ++qi) {
              const float sq = hf * __shfl_sync(FULL, sr, qi * 4);      // s = x . (hf N)
              float wv[NE], pv[NE];
              R::load_s(wv, sN + ks[qi] * stride, d, lane);
              R::load_s(pv, sP + ks[qi] * stride, d, lane);
              float acc = 0.f;
#pragma unroll
              for (int e = 0; e < NE; ++e) acc += dist_term((qa[qi][e] - x[e]) + hf * (pv[e] - sq * wv[e]), l1);
              vals[qi] = acc;
            }
          } else {
            float ia[NE], ib[NE];
            R::load_s(ia, IA + rr * ld, d, lane);
            R::load_s(ib, IB + rr * ld, d, lane);
#pragma unroll
            for (int qi = 0; qi < QW; ++qi) {
              float acc = 0.f;
#pragma unroll
              for (int e = 0; e < NE; ++e) acc = fmaf(qa[qi][e] - x[e], qc[qi][e] + ib[e], acc);
              vals[qi] = acc;
            }
            const float sr = warp_reduce_scatter8(vals, lane);
#pragma unroll
            for (int qi = 0; qi < QW; ++qi) {
              const float sq = __shfl_sync(FULL, sr, qi * 4);
              float acc = 0.f;
#pragma unroll
              for (int e = 0; e < NE; ++e)
                acc += dist_term((qa[qi][e] - x[e]) + (qb[qi][e] + ia[e]) - sq * (qc[qi][e] + ib[e]), l1);
              vals[qi] = acc;
            }
          }
          const float sc = warp_reduce_scatter8(vals, lane);
          if (myj == j) mine = sc;
        }
      }
      // one candidate per lane: (my_query, row rg + myj)
      const int rr = rg + myj;
      const bool valid = q_valid && rr < rows;
      const int64_t n_local = row0 + rr;
      if constexpr (MODE == MODE_FULL) {
        if (valid) A.out[my_query * A.ld_out + n_local] = mine;
      } else if constexpr (MODE == MODE_RANK) {
        if (valid && make_key(mine, static_cast<uint32_t>(A.id_base + n_local)) < gold_key) ++cnt;
      } else {
        const uint64_t key = make_key(mine, static_cast<uint32_t>(A.id_base + n_local));
        bool pass = valid && key < thr;
        if (pass && f_hi > f_lo) pass = !filtered(A.filter_ids, f_lo, f_hi, static_cast<int32_t>(A.id_base + n_local));
        unsigned mask = __ballot_sync(FULL, pass);
        while (mask) {
          const int src = __ffs(mask) - 1;
          mask &= mask - 1;
          const uint64_t ckey = __shfl_sync(FULL, key, src);
          const int cq = src >> 2;
          uint64_t* list = lists + cq * A.k;
          if (ckey < list[A.k - 1]) {        // re-check: the threshold may have tightened
            list_insert(list, A.k, ckey, lane);
            const uint64_t nthr = list[A.k - 1];
            if (myq == cq) thr = nthr;
          }
        }
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(empty + s);
  }

  if constexpr (MODE == MODE_TOPK) {
    __syncwarp();
    // partial lists of this catalog range: part_keys[split][q][k]
    for (int i = lane; i < QW * A.k; i += 32) {
      const int64_t q = q0 + i / A.k;
      if (q < A.nq) A.part_keys[(static_cast<int64_t>(blockIdx.y) * A.nq + q) * A.k + (i % A.k)] = lists[i];
    }
  }
  if constexpr (MODE == MODE_RANK) {
    cnt += __shfl_xor_sync(FULL, cnt, 1);
    cnt += __shfl_xor_sync(FULL, cnt, 2);
    if (myj == 0 && q_valid && cnt) atomicAdd(A.counts + my_query, cnt);
  }
}


// Cold path of the tiled kernel's top-K epilogue, kept out of line so the hot loop and the
// 32 unrolled threshold tests stay small enough for the instruction cache.  Returns the new
// score-bits threshold of the query.
__device__ __noinline__ uint32_t topk_insert_candidates(unsigned mask, uint32_t sb, uint32_t id_lane0, uint64_t* list, int k,
                                                        const int64_t* __restrict__ filter_ptr,
                                                        const int32_t* __restrict__ filter_ids, int64_t q, int lane) {
  while (mask) {
    const int src = __ffs(mask) - 1;
    mask &= mask - 1;
    const uint32_t cid = id_lane0 + static_cast<uint32_t>(src);
    const uint64_t ckey = (static_cast<uint64_t>(__shfl_sync(FULL, sb, src)) << 32) | cid;
    if (ckey < list[k - 1]) {
      bool skip = false;
      if (filter_ptr) skip = filtered(filter_ids, __ldg(filter_ptr + q), __ldg(filter_ptr + q + 1), static_cast<int32_t>(cid));
      if (!skip) list_insert(list, k, ckey, lane);
    }
  }
  return static_cast<uint32_t>(list[k - 1] >> 32);
}

// =============================================================================================
// Register-tiled kernel for the KG kinds (DIST: TransE / projected TransR; HYPER: TransH, KTUP).
//
// Every lane owns whole (query, row) pairs: warp w holds 8 queries, lane l holds rows
// l, l + 32, ... of the tile, so a thread accumulates an 8 x RN tile of distances over the
// d dimensions with NO cross-lane reduction and no idle lanes: 2 FP32 instructions per
// (pair, dim) for L1 / L2, 4 for the hyperplane form -- the issue-rate bound of the path.
// Query vectors sit in shared memory and are read as warp-wide broadcasts; catalog rows are
// read as one 128-bit load per lane.  Rows whose length in 16-byte units is even (d = 128)
// would put a quarter-warp on one bank group, so such tiles are stored with a row pitch of d + 4
// floats (tile_pitch(): one bulk copy per row): conflict-free, and every lane walks the dimensions in
// the same order, which keeps the query loads warp broadcasts.
//
// Work distribution: the (query tile x catalog tile) units are laid out query-tile-major and
// cut into gridDim.x equal contiguous ranges (one resident CTA per SM each), so every CTA
// streams the same number of tiles -- no tail wave.  A range may cross into the next query
// tile once; per-range top-K lists go to part_keys[piece][q][k] and are merged afterwards.
// =============================================================================================
constexpr int RQ = 8;                         // queries per warp

struct TiledSmem {
  size_t bars, q, w, gold, tiles, lists, total;
};
// Row pitch of a catalog tile in shared memory (floats).  A lane reads one 16-byte chunk of "its" row per step, so
// 8 consecutive rows must land on 8 different bank groups: true when the row is an odd number of 16-byte units long
// (d = 100); rows an even number of units long (d = 128, 64, 32) are stored one unit apart (pitch d + 4, one bulk copy
// per row instead of one per tile).  Every lane then walks the dimensions in the same order, so the query vectors stay
// warp broadcasts at immediate offsets.  (Round 1 walked such rows in a lane-skewed order instead; with the chunk-major
// query tile that turned every query load into an 8-way bank conflict: 0.23 of the FP32 bound at d = 128.)
__host__ __device__ inline int tile_pitch(int d) { return ((d >> 2) & 1) ? d : d + 4; }
// ST-Gumbel rec rows: [x (d) | A_k = x . P'_k / 2 (P) | C_k = x . W_k (P) | pad to a multiple of 4]
__host__ __device__ inline int gumbel_aug_ld(int d, int P) { return (d + 2 * P + 3) & ~3; }
__host__ __device__ inline TiledSmem tiled_smem_layout(int kind, int mode, int d, int tn, int stages, int k, int warps, int P = 0) {
  TiledSmem s{};
  const int TQT = RQ * warps;
  size_t off = 0;
  s.bars = off; off += 2 * 8 * sizeof(uint64_t);
  off = (off + 127) & ~static_cast<size_t>(127);
  s.q = off; off += static_cast<size_t>(TQT) * d * sizeof(float);
  if (kind == KIND_HYPER) { s.w = off; off += static_cast<size_t>(TQT) * d * sizeof(float); }
  if (kind == KIND_GUMBEL_L2) {           // per-query logit halves / normal dots [TQT][2 P], then the [3 P] table constants
    s.w = off; off += (static_cast<size_t>(TQT) * 2 * P + 3 * P) * sizeof(float);
    off = (off + 15) & ~static_cast<size_t>(15);
  }
  if (mode == MODE_RANK) { s.gold = off; off += static_cast<size_t>(TQT) * 2 * sizeof(uint32_t); }
  off = (off + 127) & ~static_cast<size_t>(127);
  s.tiles = off; off += static_cast<size_t>(stages) * tn * tile_pitch(kind == KIND_GUMBEL_L2 ? gumbel_aug_ld(d, P) : d) * sizeof(float);
  if (mode == MODE_TOPK) { s.lists = off; off += static_cast<size_t>(TQT) * k * sizeof(uint64_t); }
  s.total = off;
  return s;
}

template <int KIND, int MODE, bool L1, int RN, int W, bool IDS>
__global__ void __launch_bounds__(W * 32, 1)
k_eval_tiled(const EvalArgs A, const int stages, const int64_t units_per_cta) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr int TN = 32 * RN;
  constexpr int TQT = RQ * W;
  constexpr int kTiledWarps = W;
  const kgrec_tables& T = A.T;
  const int d = T.dim;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const TiledSmem L = tiled_smem_layout(KIND, MODE, d, TN, stages, A.k, W, T.n_pref);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + L.bars);
  uint64_t* empty = full + 8;
  float* sQ = reinterpret_cast<float*>(smem_raw + L.q);
  [[maybe_unused]] float* sW = reinterpret_cast<float*>(smem_raw + L.w);
  [[maybe_unused]] uint32_t* sGold = reinterpret_cast<uint32_t*>(smem_raw + L.gold);
  float* tiles = reinterpret_cast<float*>(smem_raw + L.tiles);
  const int rf = (KIND == KIND_GUMBEL_L2) ? gumbel_aug_ld(d, T.n_pref) : d;   // floats of a catalog row that travel
  const int pitch = tile_pitch(rf);
  const bool dense = A.cat_ld == rf && pitch == rf;   // strided catalogs / padded tiles need one copy per row

  const int64_t n_tiles = (A.n_cat + TN - 1) / TN;
  const int64_t n_qtiles = (A.nq + TQT - 1) / TQT;
  const int64_t total_units = n_tiles * n_qtiles;
  const int64_t u_begin = min(total_units, static_cast<int64_t>(blockIdx.x) * units_per_cta);
  const int64_t u_end = min(total_units, u_begin + units_per_cta);
  const int64_t my_units = u_end - u_begin;

  if (threadIdx.x == 0) {
    for (int s = 0; s < stages; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, kTiledWarps); }
    mbar_fence_init();
  }
  if constexpr (KIND == KIND_GUMBEL_L2)
    for (int i = threadIdx.x; i < 3 * T.n_pref; i += blockDim.x) sW[TQT * 2 * T.n_pref + i] = __ldg(A.gconst + i);
  __syncthreads();
  if (my_units <= 0) return;

  // unit g (0-based within this CTA) -> catalog tile (u_begin + g) % n_tiles -> stage g % stages
  auto issue_tile = [&](int64_t g) {          // called by all lanes of the issuing warp
    const int s = static_cast<int>(g % stages);
    const int64_t row0 = ((u_begin + g) % n_tiles) * TN;
    const int rows = static_cast<int>(min(static_cast<int64_t>(TN), A.n_cat - row0));
    float* dst = tiles + static_cast<size_t>(s) * TN * pitch;
    if (lane == 0) {
      if (g >= stages) mbar_wait(empty + s, static_cast<uint32_t>(((g / stages) - 1) & 1));
      mbar_arrive_expect_tx(full + s, static_cast<uint32_t>(rows) * rf * sizeof(float));
    }
    __syncwarp();
    if (dense) {
      if (lane == 0) bulk_g2s(dst, A.cat + row0 * A.cat_ld, static_cast<uint32_t>(rows) * rf * sizeof(float), full + s);
    } else {
      for (int r = lane; r < rows; r += 32)
        bulk_g2s(dst + r * pitch, A.cat + (row0 + r) * A.cat_ld, rf * sizeof(float), full + s);
    }
  };
  const int prefetch = stages - 1;
  if (wid == 0)
    for (int64_t g = 0; g < prefetch && g < my_units; ++g) issue_tile(g);

  [[maybe_unused]] uint32_t thr_hi[RQ];       // TOPK: score bits of the current K-th best
  [[maybe_unused]] uint64_t* lists = nullptr;
  [[maybe_unused]] int cnt[RQ];
  if constexpr (MODE == MODE_TOPK)
    lists = reinterpret_cast<uint64_t*>(smem_raw + L.lists) + static_cast<size_t>(wid) * RQ * A.k;
  const float* cq = sQ + wid * RQ * d;
  [[maybe_unused]] const float* wq = sW + wid * RQ * d;
  [[maybe_unused]] const uint32_t* gq = sGold + wid * RQ * 2;
  const int nk4 = d >> 2;
  // Every row is walked in the same dimension order, so a (query, row) score is bit-identical wherever the row
  // sits (tile, lane, shard, gathered sub-catalog).
  constexpr bool use_skew = false;            // see tile_pitch(): padded tiles replaced the skewed dimension walk
  const int skew0 = 0;
  int64_t cur_qt = -1, q0 = 0;

  // (re)load this warp's 8 query vectors and reset its per-query state
  auto begin_qtile = [&](int64_t qt) {
    using R = Row<2, true>;                   // d <= 256
    cur_qt = qt;
    q0 = qt * TQT + wid * RQ;
    __syncwarp();
    for (int qi = 0; qi < RQ; ++qi) {
      const int64_t q = q0 + qi;
      float cv[8], wv[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) { cv[e] = 0.f; wv[e] = 0.f; }
      if (q < A.nq) {
        if (A.qvec) {
          R::load(cv, A.qvec + q * A.qvec_ld, d, lane);
          if (KIND == KIND_HYPER) R::load(wv, A.qvec + q * A.qvec_ld + d, d, lane);
          if constexpr (KIND == KIND_GUMBEL_L2) {       // the query's logit halves and normal dots
            const int P2 = 2 * T.n_pref;
            for (int i = lane; i < P2; i += 32) sW[(wid * RQ + qi) * P2 + i] = __ldg(A.qvec + q * A.qvec_ld + d + i);
          }
        } else {
          const int64_t ie = load_idx(A.q, q, A.is64), ir = load_idx(A.r, q, A.is64);
          float rv[8];
          R::load(cv, T.ent + ie * T.ld, d, lane);
          R::load(rv, T.rel + ir * T.ld, d, lane);
          if (KIND == KIND_HYPER) {
            R::load(wv, T.norm + ir * T.ld, d, lane);
            const float a = warp_sum(R::dot(cv, wv));
#pragma unroll
            for (int e = 0; e < 8; ++e) cv[e] -= a * wv[e];       // proj(E[q], w)
          }
#pragma unroll
          for (int e = 0; e < 8; ++e) cv[e] = (A.side == KGREC_SIDE_HEAD) ? cv[e] - rv[e] : cv[e] + rv[e];
        }
      }
      // chunk-major: chunk c of query qi at [c * RQ + qi], so the eight queries of a chunk are immediate
      // offsets from one pointer inside the dimension loops (row-major cost one IMAD per query and load)
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const int c = lane + 32 * i;
        if (c * 4 < d) {
          reinterpret_cast<float4*>(sQ + wid * RQ * d)[c * RQ + qi] = make_float4(cv[4 * i], cv[4 * i + 1], cv[4 * i + 2], cv[4 * i + 3]);
          if (KIND == KIND_HYPER)
            reinterpret_cast<float4*>(sW + wid * RQ * d)[c * RQ + qi] = make_float4(wv[4 * i], wv[4 * i + 1], wv[4 * i + 2], wv[4 * i + 3]);
        }
      }
      if constexpr (MODE == MODE_RANK) {
        if (lane == 0) {
          sGold[(wid * RQ + qi) * 2] = q < A.nq ? __float_as_uint(__ldg(A.gold_scores + q)) : 0u;
          sGold[(wid * RQ + qi) * 2 + 1] = q < A.nq ? static_cast<uint32_t>(__ldg(A.gold_ids + q)) : 0u;
        }
      }
    }
#pragma unroll
    for (int qi = 0; qi < RQ; ++qi) { thr_hi[qi] = 0xffffffffu; cnt[qi] = 0; }
    if constexpr (MODE == MODE_TOPK)
      for (int i = lane; i < RQ * A.k; i += 32) lists[i] = KEY_INF;
    __syncwarp();
  };
  // write out what this warp accumulated for the query tile it is leaving
  auto end_qtile = [&]() {
    if constexpr (MODE == MODE_TOPK) {
      __syncwarp();
      // piece = index of this CTA among the CTAs that touch query tile cur_qt
      const int64_t first_cta = (cur_qt * n_tiles) / units_per_cta;
      const int64_t piece = static_cast<int64_t>(blockIdx.x) - first_cta;
      for (int i = lane; i < RQ * A.k; i += 32) {
        const int64_t q = q0 + i / A.k;
        if (q < A.nq) A.part_keys[(piece * A.nq + q) * A.k + (i % A.k)] = lists[i];
      }
    }
    if constexpr (MODE == MODE_RANK) {
#pragma unroll
      for (int qi = 0; qi < RQ; ++qi) {
        int c = cnt[qi];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(FULL, c, o);
        if (lane == 0 && q0 + qi < A.nq && c) atomicAdd(A.counts + q0 + qi, c);
      }
    }
  };

  int since = 0;                                 // tiles since this CTA entered its current query tile
  for (int64_t g = 0; g < my_units; ++g, ++since) {
    const int64_t u = u_begin + g;
    const int64_t qt = u / n_tiles, ti = u - qt * n_tiles;
    if (qt != cur_qt) {
      if (cur_qt >= 0) end_qtile();
      begin_qtile(qt);
      since = 0;
    }
    const int s = static_cast<int>(g % stages);
    if (wid == static_cast<int>(g % kTiledWarps) && g + prefetch < my_units) issue_tile(g + prefetch);   // the issue duty rotates: no warp is always the late one
    const float* tile = tiles + static_cast<size_t>(s) * TN * pitch;
    const int64_t row0 = ti * TN;
    const int rows = static_cast<int>(min(static_cast<int64_t>(TN), A.n_cat - row0));
    mbar_wait(full + s, static_cast<uint32_t>((g / stages) & 1));
    // The K-th best score any OTHER piece of these queries has reached bounds this piece's candidates too: one L2 load
    // per query and tile (lane qi holds query qi's), merged into the register thresholds in the epilogue.  A piece's
    // list costs K (1 + ln(rows / K)) insertions on its own; with the shared bound the pieces of a query warm up together.
    [[maybe_unused]] uint32_t gthr = 0xffffffffu;
    [[maybe_unused]] const bool refresh = since < 16 || (since & 15) == 0;     // every tile while the piece's lists warm up, then every 16th
    if constexpr (MODE == MODE_TOPK)
      if (refresh && A.thr_glob && lane < RQ && q0 + lane < A.nq) gthr = __ldcg(A.thr_glob + q0 + lane);

    // accumulators hold two partial sums each (even / odd dimension of every 8-byte pair)
    f32x2 acc2[RQ][RN];
#pragma unroll
    for (int qi = 0; qi < RQ; ++qi)
#pragma unroll
      for (int j = 0; j < RN; ++j) acc2[qi][j] = 0ull;
    const float* xrow = tile + lane * pitch;
    [[maybe_unused]] int skj[RN];
#pragma unroll
    for (int j = 0; j < RN; ++j) {
      skj[j] = skew0;
      if constexpr (IDS) {
        const int r = lane + 32 * j;
        skj[j] = (use_skew && r < rows) ? (__ldg(A.cat_ids + row0 + r) & 7) : 0;
      }
    }
    // chunk (16 bytes = two packed pairs) of row j / of query vector v at walk step k4
#define KGREC_LOAD_X(k4)                                                                   \
    int kk = (k4) + skew0; if (kk >= nk4) kk -= nk4;                                        \
    ulonglong2 xv[RN];                                                                      \
    int kj[RN];                                                                             \
    _Pragma("unroll")                                                                       \
    for (int j = 0; j < RN; ++j) {                                                          \
      kj[j] = kk;                                                                           \
      if constexpr (IDS) { kj[j] = (k4) + skj[j]; if (kj[j] >= nk4) kj[j] -= nk4; }         \
      xv[j] = *reinterpret_cast<const ulonglong2*>(xrow + j * 32 * pitch + 4 * kj[j]);      \
    }
#define KGREC_QVEC(base, qi, j) (reinterpret_cast<const ulonglong2*>(base)[(IDS ? kj[j] : kk) * RQ + (qi)])

    if constexpr (KIND == KIND_HYPER) {
      f32x2 sd2[RQ][RN];                       // phase 1: sd[q][n] = x_n . w_q
#pragma unroll
      for (int qi = 0; qi < RQ; ++qi)
#pragma unroll
        for (int j = 0; j < RN; ++j) sd2[qi][j] = 0ull;
#pragma unroll 1
      for (int k4 = 0; k4 < nk4; ++k4) {
        KGREC_LOAD_X(k4)
#pragma unroll
        for (int qi = 0; qi < RQ; ++qi) {
          ulonglong2 wv = KGREC_QVEC(wq, qi, 0);
#pragma unroll
          for (int j = 0; j < RN; ++j) {
            if constexpr (IDS) wv = KGREC_QVEC(wq, qi, j);
            sd2[qi][j] = fma2(xv[j].x, wv.x, fma2(xv[j].y, wv.y, sd2[qi][j]));
          }
        }
      }
      float sd[RQ][RN];
#pragma unroll
      for (int qi = 0; qi < RQ; ++qi)
#pragma unroll
        for (int j = 0; j < RN; ++j) sd[qi][j] = sum2(sd2[qi][j]);
#pragma unroll 1
      for (int k4 = 0; k4 < nk4; ++k4) {         // phase 2: L(c_q - x_n + s w_q)
        KGREC_LOAD_X(k4)
#pragma unroll
        for (int qi = 0; qi < RQ; ++qi) {
          ulonglong2 cv = KGREC_QVEC(cq, qi, 0), wv = KGREC_QVEC(wq, qi, 0);
#pragma unroll
          for (int j = 0; j < RN; ++j) {
            if constexpr (IDS) { cv = KGREC_QVEC(cq, qi, j); wv = KGREC_QVEC(wq, qi, j); }
            const f32x2 s2 = splat2(sd[qi][j]);
            const f32x2 e01 = fma2(s2, wv.x, sub2(cv.x, xv[j].x));
            const f32x2 e23 = fma2(s2, wv.y, sub2(cv.y, xv[j].y));
            if (L1) {
              const float t = abssum2(e01) + abssum2(e23);
              acc2[qi][j] = static_cast<f32x2>(__float_as_uint(__uint_as_float(static_cast<uint32_t>(acc2[qi][j])) + t));
            } else {
              acc2[qi][j] = fma2(e01, e01, fma2(e23, e23, acc2[qi][j]));
            }
          }
        }
      }
    } else {
#pragma unroll 1
      for (int k4 = 0; k4 < nk4; ++k4) {
        KGREC_LOAD_X(k4)
#pragma unroll
        for (int qi = 0; qi < RQ; ++qi) {
          ulonglong2 cv = KGREC_QVEC(cq, qi, 0);
#pragma unroll
          for (int j = 0; j < RN; ++j) {
            if constexpr (IDS) cv = KGREC_QVEC(cq, qi, j);
            const f32x2 e01 = sub2(cv.x, xv[j].x), e23 = sub2(cv.y, xv[j].y);
            if (L1) {
              const float t = abssum2(e01) + abssum2(e23);
              acc2[qi][j] = static_cast<f32x2>(__float_as_uint(__uint_as_float(static_cast<uint32_t>(acc2[qi][j])) + t));
            } else {
              acc2[qi][j] = fma2(e01, e01, fma2(e23, e23, acc2[qi][j]));
            }
          }
        }
      }
    }
#undef KGREC_LOAD_X
#undef KGREC_QVEC
    float acc[RQ][RN];
#pragma unroll
    for (int qi = 0; qi < RQ; ++qi)
#pragma unroll
      for (int j = 0; j < RN; ++j) acc[qi][j] = sum2(acc2[qi][j]);
    if constexpr (KIND == KIND_GUMBEL_L2) {
      // ST-Gumbel preference of every (query, row) pair (transUP.py:143-170 in evaluate, 84-102): k* = arg-max of
      // (u + i) . P'_k / 2 + g_k with fresh noise per (pair, k); then r = hf P'_k*, w = hf N'_k* and, for the squared L2
      // distance,  |a + r - s w|^2 = |a|^2 + |r|^2 + 2 a.r + s^2 (|w|^2 - 2) - 2 s r.w   with a = u - i, s = a.w:
      // |a|^2 is the accumulator, every other term comes from the rows' logit halves A = x.P'/2 and normal dots
      // C = x.w (k_gumbel_aug) and three per-preference constants.  No per-pair [P x d] work, no table gather.
      const int P = T.n_pref;
      const float* gc = sW + TQT * 2 * P;
      const float hf4 = A.ktup ? 2.f : 4.f;
#pragma unroll
      for (int j = 0; j < RN; ++j) {
        const int r = lane + 32 * j;
        const float* ia = tile + r * pitch + d;
        const int64_t n_local = row0 + r;
#pragma unroll 1
        for (int qi = 0; qi < RQ; ++qi) {
          const int64_t q = q0 + qi;
          if (q >= A.nq) continue;
          const float* ua = sW + (wid * RQ + qi) * 2 * P;
          float best = -INFINITY;
          int ks = 0;
          uint32_t x = hash_bits(A.seed, static_cast<uint32_t>(q), static_cast<uint32_t>(A.id_base + n_local), 0u);
          for (int k = 0; k < P; ++k) {
            float nz;
            if (A.gumbel_u) {
              nz = gumbel_from_uniform(r < rows ? __ldg(A.gumbel_u + (q * A.n_cat + n_local) * P + k) : 0.5f);
            } else {                                  // one hash per pair, then a PCG step per preference
              x = x * 747796405u + 2891336453u;
              uint32_t b = ((x >> ((x >> 28) + 4u)) ^ x) * 277803737u;
              b ^= b >> 22;
              nz = gumbel_fast(b);
            }
            const float v = ua[k] + ia[k] + nz;
            if (v > best) { best = v; ks = k; }
          }
          const float sd = ua[P + ks] - ia[P + ks];
          acc[qi][j] += gc[ks] + hf4 * (ua[ks] - ia[ks]) + sd * sd * (gc[P + ks] - 2.f) - 2.f * sd * gc[2 * P + ks];
        }
      }
    }
    // the tile is consumed: release the stage before the (register-only) epilogue
    __syncwarp();
    if (lane == 0) mbar_arrive(empty + s);

#pragma unroll
    for (int qi = 0; qi < RQ; ++qi) {
      const int64_t q = q0 + qi;
      if constexpr (MODE == MODE_TOPK)
        if (refresh) thr_hi[qi] = min(thr_hi[qi], __shfl_sync(FULL, gthr, qi));
      if (q >= A.nq) continue;                 // warp-uniform
#pragma unroll
      for (int j = 0; j < RN; ++j) {
        const int r = lane + 32 * j;
        const bool valid = r < rows;
        const int64_t n_local = row0 + r;
        const uint32_t sb = __float_as_uint(acc[qi][j]);
        if constexpr (MODE == MODE_FULL) {
          if (valid) __stcs(A.out + q * A.ld_out + n_local, acc[qi][j]);
        } else if constexpr (MODE == MODE_RANK) {
          const uint32_t id = static_cast<uint32_t>(A.id_base + n_local);
          const uint32_t gh = gq[qi * 2], gi = gq[qi * 2 + 1];
          if (valid && (sb < gh || (sb == gh && id < gi))) ++cnt[qi];
        } else {
          const unsigned mask = __ballot_sync(FULL, valid && sb <= thr_hi[qi]);
          if (mask) {                            // rare once the lists have warmed up
            const uint32_t nt = topk_insert_candidates(mask, sb, static_cast<uint32_t>(A.id_base + row0 + 32 * j), lists + qi * A.k,
                                                       A.k, A.filter_ptr, A.filter_ids, q, lane);
            if (nt < thr_hi[qi]) {
              thr_hi[qi] = nt;
              if (A.thr_glob && lane == 0) atomicMin(A.thr_glob + q, nt);
            }
          }
        }
      }
    }
  }
  end_qtile();
}

// =============================================================================================
// Soft-preference (no Gumbel) rec-side evaluation on the register-tiled structure.
//
// With raw logits as mixing weights (transUP.py:108-113) everything is linear in the logits:
//   z = (u + i) P'^T / 2 = zu + zi,  r = hf z P' = UA_q + IA_n,  w = hf z N' = UB_q + IB_n
// so with augmented rows built once per table by k_pref_aug
//   query   [ U = u | A = u + UA | -UB | c = u . UB ]      catalog [ I = i | B = i - IA | IB | dn = i . IB ]
// the pair score is  L( (A - s UB) - (B + s IB) ),  s = (u - i).(UB + IB) = c - dn + sum(U IB - I UB):
// two cross dots and one fused distance pass -- 6 FP32 lane-ops per (pair, dim), no per-pair
// mixing.  Rows are lda = 3 d + pad floats (pad makes lda / 4 odd: conflict-free 128-bit loads).
// =============================================================================================
__host__ __device__ inline int pref_aug_ld(int d) { return 3 * d + ((((3 * d) / 4) & 1) ? 8 : 4); }

// one warp per row: out[row] = augmented row (see above).  x rows come from `rows` (+ ids gather).
__global__ void __launch_bounds__(kThreads)
k_pref_aug(const kgrec_tables T, const int ktup, const int is_query, const void* ids, const int is64,
           const float* __restrict__ rows, const int64_t row_ld, const int64_t n, float* __restrict__ out, const int64_t lda) {
  using R = Row<2, true>;
  constexpr int NE = 8;
  extern __shared__ __align__(16) float aug_smem[];
  const int d = T.dim, P = T.n_pref, stride = (d + 3) & ~3;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  float* sP = aug_smem;
  float* sN = sP + P * stride;
  float* scr = sN + P * stride + wid * kMaxPref;
  for (int idx = threadIdx.x; idx < P * stride; idx += blockDim.x) {
    const int k = idx / stride, j = idx - k * stride;
    float a = 0.f, b = 0.f;
    if (j < d) {
      a = __ldg(T.pref + static_cast<int64_t>(k) * T.ld + j);
      b = __ldg(T.pref_norm + static_cast<int64_t>(k) * T.ld + j);
      if (ktup) { a += __ldg(T.rel + static_cast<int64_t>(k) * T.ld + j); b += __ldg(T.norm + static_cast<int64_t>(k) * T.ld + j); }
    }
    sP[idx] = a;
    sN[idx] = b;
  }
  __syncthreads();
  const float hf = ktup ? 0.5f : 1.f;
  for (int64_t row = static_cast<int64_t>(blockIdx.x) * kWarpsPerCta + wid; row < n; row += static_cast<int64_t>(gridDim.x) * kWarpsPerCta) {
    const int64_t src = ids ? load_idx(ids, row, is64) : row;
    float x[NE];
    R::load(x, rows + src * row_ld, d, lane);
    __syncwarp();
    for (int g = 0; g < P; g += 8) {               // XP_k = x . P'_k / 2
      float vals[8];
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) {
        vals[kk] = 0.f;
        if (g + kk < P) {
          float pr[NE];
          R::load_s(pr, sP + (g + kk) * stride, d, lane);
          vals[kk] = R::dot(pr, x);
        }
      }
      const float v = warp_reduce_scatter8(vals, lane);
      const int k = g + (lane >> 2);
      if ((lane & 3) == 0 && k < P) scr[k] = 0.5f * v;
    }
    __syncwarp();
    float xa[NE], xb[NE];
#pragma unroll
    for (int e = 0; e < NE; ++e) { xa[e] = 0.f; xb[e] = 0.f; }
    for (int k = 0; k < P; ++k) {
      const float z = hf * scr[k];
      float pr[NE];
      R::load_s(pr, sP + k * stride, d, lane);
#pragma unroll
      for (int e = 0; e < NE; ++e) xa[e] = fmaf(z, pr[e], xa[e]);
      R::load_s(pr, sN + k * stride, d, lane);
#pragma unroll
      for (int e = 0; e < NE; ++e) xb[e] = fmaf(z, pr[e], xb[e]);
    }
    const float sc = warp_sum(R::dot(x, xb));
    float seg1[NE], seg2[NE];
#pragma unroll
    for (int e = 0; e < NE; ++e) {
      seg1[e] = is_query ? x[e] + xa[e] : x[e] - xa[e];
      seg2[e] = is_query ? -xb[e] : xb[e];
    }
    float* o = out + row * lda;
    R::store(o, x, d, lane);
    R::store(o + d, seg1, d, lane);
    R::store(o + 2 * d, seg2, d, lane);
    for (int j = 3 * d + lane; j < lda; j += 32) o[j] = (j == 3 * d) ? sc : 0.f;
  }
}

struct SoftSmem { size_t bars, q, tiles, lists, total; };
__host__ __device__ inline SoftSmem soft_smem_layout(int mode, int lda, int stages, int k, int warps) {
  SoftSmem s{};
  size_t off = 0;
  s.bars = off; off += 2 * 8 * sizeof(uint64_t);
  off = (off + 127) & ~static_cast<size_t>(127);
  s.q = off; off += static_cast<size_t>(RQ) * warps * lda * sizeof(float);
  off = (off + 127) & ~static_cast<size_t>(127);
  s.tiles = off; off += static_cast<size_t>(stages) * 32 * lda * sizeof(float);
  if (mode == MODE_TOPK) { s.lists = off; off += static_cast<size_t>(RQ) * warps * k * sizeof(uint64_t); }
  s.total = off;
  return s;
}

template <int MODE, bool L1, int W>
__global__ void __launch_bounds__(W * 32, 1)
k_eval_soft(const EvalArgs A, const int stages, const int64_t units_per_cta) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr int TN = 32;
  constexpr int TQT = RQ * W;
  const int d = A.T.dim;
  const int lda = static_cast<int>(A.cat_ld);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const SoftSmem L = soft_smem_layout(MODE, lda, stages, A.k, W);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + L.bars);
  uint64_t* empty = full + 8;
  float* sQ = reinterpret_cast<float*>(smem_raw + L.q);
  float* tiles = reinterpret_cast<float*>(smem_raw + L.tiles);

  const int64_t n_tiles = (A.n_cat + TN - 1) / TN;
  const int64_t n_qtiles = (A.nq + TQT - 1) / TQT;
  const int64_t total_units = n_tiles * n_qtiles;
  const int64_t u_begin = min(total_units, static_cast<int64_t>(blockIdx.x) * units_per_cta);
  const int64_t u_end = min(total_units, u_begin + units_per_cta);
  const int64_t my_units = u_end - u_begin;
  if (threadIdx.x == 0) {
    for (int s = 0; s < stages; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, W); }
    mbar_fence_init();
  }
  __syncthreads();
  if (my_units <= 0) return;
  auto issue_tile = [&](int64_t g) {          // lane 0 of warp 0
    const int s = static_cast<int>(g % stages);
    const int64_t row0 = ((u_begin + g) % n_tiles) * TN;
    const int rows = static_cast<int>(min(static_cast<int64_t>(TN), A.n_cat - row0));
    if (g >= stages) mbar_wait(empty + s, static_cast<uint32_t>(((g / stages) - 1) & 1));
    const uint32_t bytes = static_cast<uint32_t>(rows) * lda * sizeof(float);
    mbar_arrive_expect_tx(full + s, bytes);
    bulk_g2s(tiles + static_cast<size_t>(s) * TN * lda, A.cat + row0 * lda, bytes, full + s);
  };
  const int prefetch = stages - 1;
  if (threadIdx.x == 0)
    for (int64_t g = 0; g < prefetch && g < my_units; ++g) issue_tile(g);

  [[maybe_unused]] uint32_t thr_hi[RQ];
  [[maybe_unused]] uint64_t* lists = nullptr;
  if constexpr (MODE == MODE_TOPK)
    lists = reinterpret_cast<uint64_t*>(smem_raw + L.lists) + static_cast<size_t>(wid) * RQ * A.k;
  const float* cq = sQ + wid * RQ * lda;
  const ulonglong2* cq2 = reinterpret_cast<const ulonglong2*>(cq);
  const int nk4 = d >> 2;
  int64_t cur_qt = -1, q0 = 0;
  auto begin_qtile = [&](int64_t qt) {
    cur_qt = qt;
    q0 = qt * TQT + wid * RQ;
    __syncwarp();
    // chunk-major: chunk e of query qi sits at cq4[e * RQ + qi], so inside the dimension loops the eight queries
    // of a chunk are immediate offsets from one pointer (row-major cost one IMAD per query and load)
    for (int qi = 0; qi < RQ; ++qi) {
      const int64_t q = q0 + qi;
      float4* dst = reinterpret_cast<float4*>(sQ + wid * RQ * lda);
      const float4* src = reinterpret_cast<const float4*>(A.qvec + q * lda);
      for (int c = lane; c < lda / 4; c += 32) dst[c * RQ + qi] = (q < A.nq) ? __ldg(src + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int qi = 0; qi < RQ; ++qi) thr_hi[qi] = 0xffffffffu;
    if constexpr (MODE == MODE_TOPK)
      for (int i = lane; i < RQ * A.k; i += 32) lists[i] = KEY_INF;
    __syncwarp();
  };
  auto end_qtile = [&]() {
    if constexpr (MODE == MODE_TOPK) {
      __syncwarp();
      const int64_t first_cta = (cur_qt * n_tiles) / units_per_cta;
      const int64_t piece = static_cast<int64_t>(blockIdx.x) - first_cta;
      for (int i = lane; i < RQ * A.k; i += 32) {
        const int64_t q = q0 + i / A.k;
        if (q < A.nq) A.part_keys[(piece * A.nq + q) * A.k + (i % A.k)] = lists[i];
      }
    }
  };

  int since = 0;                                 // tiles since this CTA entered its current query tile
  for (int64_t g = 0; g < my_units; ++g, ++since) {
    const int64_t u = u_begin + g;
    const int64_t qt = u / n_tiles, ti = u - qt * n_tiles;
    if (qt != cur_qt) {
      if (cur_qt >= 0) end_qtile();
      begin_qtile(qt);
      since = 0;
    }
    const int s = static_cast<int>(g % stages);
    if (threadIdx.x == 0 && g + prefetch < my_units) issue_tile(g + prefetch);   // (rotating the duty as in k_eval_tiled LOSES here: 7.3 -> 9.6 ms)
    __syncwarp();
    const float* xr = tiles + static_cast<size_t>(s) * TN * lda + lane * lda;   // this lane's catalog row
    const int64_t row0 = ti * TN;
    const int rows = static_cast<int>(min(static_cast<int64_t>(TN), A.n_cat - row0));
    mbar_wait(full + s, static_cast<uint32_t>((g / stages) & 1));
    [[maybe_unused]] uint32_t gthr = 0xffffffffu;          // the bound the other pieces of these queries have reached (k_eval_tiled)
    [[maybe_unused]] const bool refresh = since < 16 || (since & 15) == 0;
    if constexpr (MODE == MODE_TOPK)
      if (refresh && A.thr_glob && lane < RQ && q0 + lane < A.nq) gthr = __ldcg(A.thr_glob + q0 + lane);

    // pass 1: cross dots  sum_j ( U_q IB_n + I_n (-UB_q) )
    f32x2 sd2[RQ];
#pragma unroll
    for (int qi = 0; qi < RQ; ++qi) sd2[qi] = 0ull;
#pragma unroll 1
    for (int k4 = 0; k4 < nk4; ++k4) {
      const ulonglong2 xi = *reinterpret_cast<const ulonglong2*>(xr + 4 * k4);
      const ulonglong2 xw = *reinterpret_cast<const ulonglong2*>(xr + 2 * d + 4 * k4);
#pragma unroll
      for (int qi = 0; qi < RQ; ++qi) {
        const ulonglong2 qu = cq2[k4 * RQ + qi];
        const ulonglong2 qn = cq2[(2 * nk4 + k4) * RQ + qi];
        sd2[qi] = fma2(qu.x, xw.x, fma2(qu.y, xw.y, fma2(xi.x, qn.x, fma2(xi.y, qn.y, sd2[qi]))));
      }
    }
    const float dn = xr[3 * d];
    float sv[RQ];
#pragma unroll
    for (int qi = 0; qi < RQ; ++qi) sv[qi] = sum2(sd2[qi]) + cq[(3 * nk4 * RQ + qi) * 4] - dn;
    // pass 2: L( (A_q - s UB_q) - (B_n + s IB_n) )
    f32x2 acc2[RQ];
#pragma unroll
    for (int qi = 0; qi < RQ; ++qi) acc2[qi] = 0ull;
#pragma unroll 1
    for (int k4 = 0; k4 < nk4; ++k4) {
      const ulonglong2 xb = *reinterpret_cast<const ulonglong2*>(xr + d + 4 * k4);
      const ulonglong2 xw = *reinterpret_cast<const ulonglong2*>(xr + 2 * d + 4 * k4);
#pragma unroll
      for (int qi = 0; qi < RQ; ++qi) {
        const ulonglong2 qa = cq2[(nk4 + k4) * RQ + qi];
        const ulonglong2 qn = cq2[(2 * nk4 + k4) * RQ + qi];
        const f32x2 s2 = splat2(sv[qi]);
        const f32x2 e01 = sub2(fma2(s2, qn.x, qa.x), fma2(s2, xw.x, xb.x));
        const f32x2 e23 = sub2(fma2(s2, qn.y, qa.y), fma2(s2, xw.y, xb.y));
        if (L1) {
          const float t = abssum2(e01) + abssum2(e23);
          acc2[qi] = static_cast<f32x2>(__float_as_uint(__uint_as_float(static_cast<uint32_t>(acc2[qi])) + t));
        } else {
          acc2[qi] = fma2(e01, e01, fma2(e23, e23, acc2[qi]));
        }
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(empty + s);

    const bool valid = lane < rows;
    const int64_t n_local = row0 + lane;
#pragma unroll
    for (int qi = 0; qi < RQ; ++qi) {
      const int64_t q = q0 + qi;
      if constexpr (MODE == MODE_TOPK)
        if (refresh) thr_hi[qi] = min(thr_hi[qi], __shfl_sync(FULL, gthr, qi));
      if (q >= A.nq) continue;
      const float sc = sum2(acc2[qi]);
      if constexpr (MODE == MODE_FULL) {
        if (valid) __stcs(A.out + q * A.ld_out + n_local, sc);
      } else {
        const uint32_t sb = __float_as_uint(sc);
        const unsigned mask = __ballot_sync(FULL, valid && sb <= thr_hi[qi]);
        if (mask) {
          const uint32_t nt = topk_insert_candidates(mask, sb, static_cast<uint32_t>(A.id_base + row0), lists + qi * A.k, A.k,
                                                     A.filter_ptr, A.filter_ids, q, lane);
          if (nt < thr_hi[qi]) {
            thr_hi[qi] = nt;
            if (A.thr_glob && lane == 0) atomicMin(A.thr_glob + q, nt);
          }
        }
      }
    }
  }
  end_qtile();
}

// K-way merge: in [n_lists][nq][k] ascending lists -> out [nq][k].  One warp per query.
__global__ void __launch_bounds__(256)
k_merge_topk(const uint64_t* __restrict__ in, int n_lists, int64_t nq, int k, uint64_t* __restrict__ out) {
  extern __shared__ __align__(8) unsigned char merge_smem[];
  uint64_t* lists = reinterpret_cast<uint64_t*>(merge_smem);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int64_t q = static_cast<int64_t>(blockIdx.x) * 8 + wid;
  if (q >= nq) return;
  uint64_t* list = lists + wid * k;
  for (int i = lane; i < k; i += 32) list[i] = KEY_INF;
  __syncwarp();
  for (int l = 0; l < n_lists; ++l) {
    const uint64_t* src = in + (static_cast<int64_t>(l) * nq + q) * k;
    for (int i = 0; i < k; ++i) {
      const uint64_t x = __ldg(src + i);
      if (x >= list[k - 1]) break;     // ascending source: nothing further can enter
      list_insert(list, k, x, lane);
    }
  }
  for (int i = lane; i < k; i += 32) out[q * k + i] = list[i];
}

// KTUP catalog for evaluateRec: ie[i] = Item[i] + Ent[item2ent[i]]  (jTransUP.py:177-181)
__global__ void __launch_bounds__(256)
k_ktup_items(const kgrec_tables T, int64_t i0, int64_t n, float* __restrict__ out, int64_t ld_out) {
  const int64_t total = n * T.dim;
  for (int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; idx < total;
       idx += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t i = idx / T.dim;
    const int j = static_cast<int>(idx - i * T.dim);
    const int64_t a = __ldg(T.item2ent + i0 + i);
    out[i * ld_out + j] = __ldg(T.item + (i0 + i) * T.ld + j) + __ldg(T.ent + a * T.ld + j);
  }
}

// ===========================================================================================
// host side
// ===========================================================================================
// ST-Gumbel rec rows (KIND_GUMBEL_L2): out[row] = [x | A_k = x . P'_k / 2 | C_k = x . (hf N'_k) | 0 pad], one warp per row;
// P' = pref (+ rel for KTUP), N' = pref_norm (+ norm), hf = 1 (TUP) or 1/2 (KTUP): transUP.py:105-115, jTransUP.py:250-260.
// Block 0 also writes the three per-preference constants |hf P'_k|^2, |hf N'_k|^2, (hf P'_k).(hf N'_k) to gconst [3 P].
__global__ void __launch_bounds__(kThreads)
k_gumbel_aug(const kgrec_tables T, const int ktup, const void* ids, const int is64, const float* __restrict__ rows,
             const int64_t row_ld, const int64_t n, float* __restrict__ out, const int64_t lda, float* __restrict__ gconst) {
  extern __shared__ __align__(16) float aug_smem[];
  const int d = T.dim, P = T.n_pref, stride = (d + 3) & ~3;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  float* sP = aug_smem;
  float* sN = sP + P * stride;
  const float hf = ktup ? 0.5f : 1.f;
  for (int idx = threadIdx.x; idx < P * stride; idx += blockDim.x) {
    const int k = idx / stride, j = idx - k * stride;
    float a = 0.f, b = 0.f;
    if (j < d) {
      a = __ldg(T.pref + static_cast<int64_t>(k) * T.ld + j);
      b = __ldg(T.pref_norm + static_cast<int64_t>(k) * T.ld + j);
      if (ktup) { a += __ldg(T.rel + static_cast<int64_t>(k) * T.ld + j); b += __ldg(T.norm + static_cast<int64_t>(k) * T.ld + j); }
    }
    sP[idx] = a;
    sN[idx] = b;
  }
  __syncthreads();
  if (blockIdx.x == 0 && gconst) {
    for (int k = wid; k < P; k += kWarpsPerCta) {
      float pp = 0.f, nn = 0.f, pn = 0.f;
      for (int j = lane; j < d; j += 32) {
        const float a = hf * sP[k * stride + j], b = hf * sN[k * stride + j];
        pp = fmaf(a, a, pp); nn = fmaf(b, b, nn); pn = fmaf(a, b, pn);
      }
      warp_sum2(pp, nn);
      pn = warp_sum(pn);
      if (lane == 0) { gconst[k] = pp; gconst[P + k] = nn; gconst[2 * P + k] = pn; }
    }
  }
  for (int64_t row = static_cast<int64_t>(blockIdx.x) * kWarpsPerCta + wid; row < n; row += static_cast<int64_t>(gridDim.x) * kWarpsPerCta) {
    const int64_t src = ids ? load_idx(ids, row, is64) : row;
    const float* x = rows + src * row_ld;
    float* o = out + row * lda;
    for (int j = lane; j < d; j += 32) o[j] = __ldg(x + j);
    for (int k = 0; k < P; ++k) {
      float a = 0.f, c = 0.f;
      for (int j = lane; j < d; j += 32) {
        const float xv = __ldg(x + j);
        a = fmaf(xv, sP[k * stride + j], a);
        c = fmaf(xv, sN[k * stride + j], c);
      }
      warp_sum2(a, c);
      if (lane == 0) { o[d + k] = 0.5f * a; o[d + P + k] = hf * c; }
    }
    for (int j = d + 2 * P + lane; j < lda; j += 32) o[j] = 0.f;
  }
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

struct EvalPlan {
  int kind, nch, tn, n_splits;
  int64_t n_qtiles;
  size_t smem;
  bool tiled;       // register-tiled kernel (KG kinds)
  bool soft_aug;    // rec side, soft preferences, augmented rows (k_eval_soft)
  int rn, stages, grid, warps;
  int64_t units_per_cta;
};

static int eval_plan(const kgrec_tables* T, int model, int side, int mode, const float* cat, int64_t cat_ld,
                     int64_t nq, int64_t n_cat, int k, bool have_qvec, EvalArgs* A, EvalPlan* pl) {
  if (!T) { set_error("tables is NULL"); return KGREC_ERR_INVALID; }
  if (!cat || n_cat <= 0 || nq <= 0) { set_error("empty catalog / query set"); return KGREC_ERR_INVALID; }
  const int d = T->dim;
  if (d <= 0 || d > 256) { set_error("eval: embedding_size %d outside [1, 256]", d); return KGREC_ERR_UNSUPPORTED; }
  if (d % 4 || cat_ld % 4 || cat_ld < d || !aligned16(cat)) {
    set_error("eval: catalog must be 16-byte aligned with embedding_size and leading dimension multiples of 4");
    return KGREC_ERR_UNSUPPORTED;
  }
  A->ktup = 0;
  switch (model) {
    case KGREC_TRANSE: case KGREC_TRANSR: pl->kind = KIND_DIST; break;
    case KGREC_TRANSH: pl->kind = KIND_HYPER; break;
    case KGREC_KTUP: A->ktup = 1; /* fallthrough */
    case KGREC_TUP: pl->kind = (side == KGREC_SIDE_REC) ? (T->use_gumbel ? KIND_PREF_HARD : KIND_PREF_SOFT) : KIND_HYPER; break;
    default: set_error("unknown model %d", model); return KGREC_ERR_INVALID;
  }
  if (model == KGREC_TRANSR && !have_qvec) {
    set_error("TransR eval needs explicit query vectors and a catalog projected by the relation matrix");
    return KGREC_ERR_INVALID;
  }
  const bool rec = side == KGREC_SIDE_REC;
  if (rec != (pl->kind >= KIND_PREF_HARD)) { set_error("side %d does not fit model %d", side, model); return KGREC_ERR_INVALID; }
  pl->soft_aug = false;
  if (rec && have_qvec && pl->kind == KIND_PREF_HARD) {
    // ST-Gumbel on rows augmented by kgrec_gumbel_aug_rows: the register-tiled distance kernel + a per-pair epilogue
    if (T->l1) { set_error("augmented ST-Gumbel rows are built for the squared-L2 score (L1_flag = 0)"); return KGREC_ERR_UNSUPPORTED; }
    if (T->n_pref <= 0 || T->n_pref > 64) { set_error("augmented ST-Gumbel rows: preference_total must be <= 64"); return KGREC_ERR_UNSUPPORTED; }
    if (cat_ld != gumbel_aug_ld(d, T->n_pref)) { set_error("augmented ST-Gumbel catalog must have leading dimension %d", gumbel_aug_ld(d, T->n_pref)); return KGREC_ERR_INVALID; }
    if (mode == MODE_RANK) { set_error("rank counts are built for the KG sides"); return KGREC_ERR_UNSUPPORTED; }
    if (mode == MODE_TOPK && (k <= 0 || k > 128)) { set_error("topn %d outside [1, 128]", k); return KGREC_ERR_UNSUPPORTED; }
    pl->kind = KIND_GUMBEL_L2;
    pl->tiled = true;
    const bool wide = d > 128;
    pl->warps = wide ? 8 : 16;
    pl->rn = wide ? 1 : 2;
    const int tn_t = 32 * pl->rn;
    int stages = 4;
    while (stages > 2 && tiled_smem_layout(pl->kind, mode, d, tn_t, stages, k, pl->warps, T->n_pref).total > 210 * 1024) --stages;
    pl->stages = stages;
    pl->tn = tn_t;
    pl->smem = tiled_smem_layout(pl->kind, mode, d, tn_t, stages, k, pl->warps, T->n_pref).total;
    if (pl->smem > 225 * 1024) { set_error("eval: shared-memory budget exceeded (%zu bytes)", pl->smem); return KGREC_ERR_UNSUPPORTED; }
    const int64_t n_tiles_t = (n_cat + tn_t - 1) / tn_t;
    pl->n_qtiles = (nq + RQ * pl->warps - 1) / (RQ * pl->warps);
    const int64_t total_units = n_tiles_t * pl->n_qtiles;
    int64_t ctas = sm_count();
    if (ctas > total_units) ctas = total_units;
    pl->units_per_cta = (total_units + ctas - 1) / ctas;
    pl->grid = static_cast<int>((total_units + pl->units_per_cta - 1) / pl->units_per_cta);
    pl->n_splits = static_cast<int>((n_tiles_t + pl->units_per_cta - 1) / pl->units_per_cta + 1);
    A->T = *T; A->side = side; A->nq = nq; A->cat = cat; A->cat_ld = cat_ld; A->n_cat = n_cat;
    A->n_splits = pl->n_splits; A->tn = tn_t; A->k = k;
    return KGREC_OK;
  }
  if (rec && have_qvec) {
    // augmented-row evaluation of the soft preference model (rows built by kgrec_pref_aug_rows)
    if (pl->kind != KIND_PREF_SOFT) { set_error("augmented rec rows are for use_st_gumbel = 0"); return KGREC_ERR_INVALID; }
    if (cat_ld != pref_aug_ld(d)) { set_error("augmented catalog must have leading dimension %d", pref_aug_ld(d)); return KGREC_ERR_INVALID; }
    if (mode == MODE_RANK) { set_error("rank counts are built for the KG sides"); return KGREC_ERR_UNSUPPORTED; }
    if (mode == MODE_TOPK && (k <= 0 || k > 128)) { set_error("topn %d outside [1, 128]", k); return KGREC_ERR_UNSUPPORTED; }
    pl->soft_aug = true;
    pl->tiled = false;
    pl->warps = 8;
    int stages = 3;
    while (stages > 2 && soft_smem_layout(mode, static_cast<int>(cat_ld), stages, k, 8).total > 215 * 1024) --stages;
    pl->stages = stages;
    pl->smem = soft_smem_layout(mode, static_cast<int>(cat_ld), stages, k, 8).total;
    if (pl->smem > 225 * 1024) { set_error("eval: shared-memory budget exceeded (%zu bytes)", pl->smem); return KGREC_ERR_UNSUPPORTED; }
    const int64_t n_tiles_t = (n_cat + 31) / 32;
    pl->n_qtiles = (nq + RQ * 8 - 1) / (RQ * 8);
    const int64_t total_units = n_tiles_t * pl->n_qtiles;
    int64_t ctas = sm_count();
    if (ctas > total_units) ctas = total_units;
    pl->units_per_cta = (total_units + ctas - 1) / ctas;
    pl->grid = static_cast<int>((total_units + pl->units_per_cta - 1) / pl->units_per_cta);
    pl->n_splits = static_cast<int>((n_tiles_t + pl->units_per_cta - 1) / pl->units_per_cta + 1);
    A->T = *T; A->side = side; A->nq = nq; A->cat = cat; A->cat_ld = cat_ld; A->n_cat = n_cat;
    A->n_splits = pl->n_splits; A->tn = 32; A->k = k;
    return KGREC_OK;
  }
  bool al = true;
  auto chk = [&](const void* p) { if (!p || !aligned16(p)) al = false; };
  if (rec) { chk(T->user); chk(T->pref); chk(T->pref_norm); if (A->ktup) { chk(T->rel); chk(T->norm); } }
  else if (!have_qvec) { chk(T->ent); chk(T->rel); if (pl->kind == KIND_HYPER) chk(T->norm); }
  if (!al || T->ld % 4) { set_error("eval: a table this model needs is NULL or not 16-byte aligned"); return KGREC_ERR_INVALID; }
  if (rec && (T->n_pref <= 0 || T->n_pref > kMaxPref)) { set_error("preference_total out of range"); return KGREC_ERR_UNSUPPORTED; }
  if (mode == MODE_TOPK && (k <= 0 || k > 128)) { set_error("topn %d outside [1, 128]", k); return KGREC_ERR_UNSUPPORTED; }
  pl->nch = d <= 128 ? 1 : 2;
  pl->n_qtiles = (nq + TQ - 1) / TQ;
  pl->tiled = pl->kind <= KIND_HYPER;
  if (pl->tiled) {
    // register tile 8 x RN per thread, W warps per CTA.  d <= 128: 16 warps, DIST 8x4 / HYPER 8x2
    // (HYPER keeps two tiles: dots and distances); wider rows: 8 warps, 8x2 / 8x1 to fit smem.
    const bool wide = d > 128;
    pl->warps = wide ? 8 : 16;
    pl->rn = (pl->kind == KIND_DIST ? 4 : 2) / (wide ? 2 : 1);
    const int tn_t = 32 * pl->rn;
    int stages = 4;
    while (stages > 2 && tiled_smem_layout(pl->kind, mode, d, tn_t, stages, k, pl->warps).total > 210 * 1024) --stages;
    pl->stages = stages;
    pl->tn = tn_t;
    pl->smem = tiled_smem_layout(pl->kind, mode, d, tn_t, stages, k, pl->warps).total;
    if (pl->smem > 225 * 1024) { set_error("eval: shared-memory budget exceeded (%zu bytes)", pl->smem); return KGREC_ERR_UNSUPPORTED; }
    const int64_t n_tiles_t = (n_cat + tn_t - 1) / tn_t;
    const int tqt = RQ * pl->warps;
    pl->n_qtiles = (nq + tqt - 1) / tqt;
    const int64_t total_units = n_tiles_t * pl->n_qtiles;
    int64_t ctas = sm_count();                       // one resident CTA per SM
    if (ctas > total_units) ctas = total_units;
    pl->units_per_cta = (total_units + ctas - 1) / ctas;
    pl->grid = static_cast<int>((total_units + pl->units_per_cta - 1) / pl->units_per_cta);
    // pieces of partial top-K lists per query tile: CTAs whose ranges touch one query tile
    pl->n_splits = static_cast<int>((n_tiles_t + pl->units_per_cta - 1) / pl->units_per_cta + 1);
    A->T = *T; A->side = side; A->nq = nq; A->cat = cat; A->cat_ld = cat_ld; A->n_cat = n_cat;
    A->n_splits = pl->n_splits; A->tn = tn_t; A->k = k;
    return KGREC_OK;
  }
  // tile rows: ~16 KB per stage
  int tn = static_cast<int>((16 * 1024) / (cat_ld * sizeof(float)));
  tn = tn < 4 ? 4 : (tn > 64 ? 64 : tn);
  tn &= ~3;
  pl->tn = tn;
  const int64_t n_tiles = (n_cat + tn - 1) / tn;
  // catalog ranges per query tile: fill the resident CTA slots (3 per SM) without a second wave
  int64_t splits = (3 * static_cast<int64_t>(sm_count())) / pl->n_qtiles;
  splits = splits < 1 ? 1 : (splits > n_tiles ? n_tiles : splits);
  if (splits > 65535) splits = 65535;
  pl->n_splits = static_cast<int>(splits);
  pl->smem = eval_smem_layout(pl->kind, mode, d, cat_ld, T->n_pref, tn, k).total;
  if (pl->smem > 220 * 1024) { set_error("eval: shared-memory budget exceeded (%zu bytes)", pl->smem); return KGREC_ERR_UNSUPPORTED; }
  A->T = *T;
  A->side = side;
  A->nq = nq;
  A->cat = cat;
  A->cat_ld = cat_ld;
  A->n_cat = n_cat;
  A->n_splits = pl->n_splits;
  A->tn = tn;
  A->k = k;
  return KGREC_OK;
}

template <int MODE>
static int launch_eval(const EvalArgs& A, const EvalPlan& pl, cudaStream_t st) {
  const dim3 grid(static_cast<unsigned>(pl.n_qtiles), static_cast<unsigned>(pl.n_splits));
  if (pl.soft_aug) {
    if constexpr (MODE == MODE_RANK) {
      set_error("rank counts are built for the KG sides");
      return KGREC_ERR_UNSUPPORTED;
    } else {
      auto kern = A.T.l1 ? k_eval_soft<MODE, true, 8> : k_eval_soft<MODE, false, 8>;
      KGREC_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(pl.smem)));
      kern<<<pl.grid, 8 * 32, pl.smem, st>>>(A, pl.stages, pl.units_per_cta);
      KGREC_CUDA_OK(cudaGetLastError());
      return KGREC_OK;
    }
  }
  if (pl.tiled) {
#define KGREC_TILED_CASE(KINDV, RNV, WV)                                                                      \
  {                                                                                                           \
    auto kern = A.T.l1 ? k_eval_tiled<KINDV, MODE, true, RNV, WV, false> : k_eval_tiled<KINDV, MODE, false, RNV, WV, false>; \
    if constexpr (MODE == MODE_FULL) {                                                                        \
      if (A.cat_ids) kern = A.T.l1 ? k_eval_tiled<KINDV, MODE, true, RNV, WV, true> : k_eval_tiled<KINDV, MODE, false, RNV, WV, true>; \
    }                                                                                                         \
    KGREC_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(pl.smem))); \
    kern<<<pl.grid, WV * 32, pl.smem, st>>>(A, pl.stages, pl.units_per_cta);                                  \
  }
    if (pl.kind == KIND_DIST) { if (pl.warps == 16) KGREC_TILED_CASE(KIND_DIST, 4, 16) else KGREC_TILED_CASE(KIND_DIST, 2, 8) }
    else if (pl.kind == KIND_GUMBEL_L2) {
      if constexpr (MODE == MODE_RANK) { set_error("rank counts are built for the KG sides"); return KGREC_ERR_UNSUPPORTED; }
      else { if (pl.warps == 16) KGREC_TILED_CASE(KIND_GUMBEL_L2, 2, 16) else KGREC_TILED_CASE(KIND_GUMBEL_L2, 1, 8) }
    }
    else { if (pl.warps == 16) KGREC_TILED_CASE(KIND_HYPER, 2, 16) else KGREC_TILED_CASE(KIND_HYPER, 1, 8) }
#undef KGREC_TILED_CASE
    KGREC_CUDA_OK(cudaGetLastError());
    return KGREC_OK;
  }
#define KGREC_EVAL_CASE(KINDV, NCHV)                                                                          \
  {                                                                                                           \
    auto kern = A.T.l1 ? k_eval<KINDV, NCHV, MODE, true> : k_eval<KINDV, NCHV, MODE, false>;                  \
    KGREC_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(pl.smem))); \
    kern<<<grid, kEvalThreads, pl.smem, st>>>(A);                                                             \
  }
  switch (pl.kind * 2 + (pl.nch - 1)) {
    case 4: KGREC_EVAL_CASE(KIND_PREF_HARD, 1) break;
    case 5: KGREC_EVAL_CASE(KIND_PREF_HARD, 2) break;
    case 6: KGREC_EVAL_CASE(KIND_PREF_SOFT, 1) break;
    default: KGREC_EVAL_CASE(KIND_PREF_SOFT, 2) break;
  }
#undef KGREC_EVAL_CASE
  KGREC_CUDA_OK(cudaGetLastError());
  return KGREC_OK;
}

}  // namespace kgrec

using namespace kgrec;

extern "C" int64_t kgrec_eval_workspace_bytes(int64_t nq, int32_t k) {
  // worst case number of catalog splits is 2 * SMs (eval_plan)
  const int64_t splits = 3 * static_cast<int64_t>(sm_count());
  return splits * (nq > 0 ? nq : 1) * (k > 0 ? k : 1) * static_cast<int64_t>(sizeof(uint64_t)) + 4 * (nq > 0 ? nq : 1) + 16;
}

extern "C" int kgrec_eval_scores(const kgrec_tables* tables, int model, int side, const void* q, const void* r,
                                 int idx_bytes, const float* qvec, int64_t nq, const float* cat, int64_t cat_ld,
                                 int64_t n_cat, int64_t id_base, const int32_t* cat_ids, const float* gumbel_u,
                                 uint64_t seed, float* out, int64_t ld_out, kgrec_stream_t stream) {
  EvalArgs A{};
  EvalPlan pl{};
  int rc = eval_plan(tables, model, side, MODE_FULL, cat, cat_ld, nq, n_cat, 0, qvec != nullptr, &A, &pl);
  if (rc) return rc;
  if (!out || ld_out < n_cat) { set_error("bad out / ld_out"); return KGREC_ERR_INVALID; }
  if (!qvec && (!q || (side != KGREC_SIDE_REC && !r))) { set_error("query ids are NULL"); return KGREC_ERR_INVALID; }
  if (!qvec && idx_bytes != 4 && idx_bytes != 8) { set_error("idx_bytes must be 4 or 8"); return KGREC_ERR_INVALID; }
  A.q = q; A.r = r; A.is64 = idx_bytes == 8; A.qvec = qvec;
  A.qvec_ld = pl.kind == KIND_GUMBEL_L2 ? cat_ld : 2 * static_cast<int64_t>(tables->dim);
  A.gconst = pl.kind == KIND_GUMBEL_L2 ? qvec + nq * cat_ld : nullptr;     // the constants follow the query rows
  A.gumbel_u = gumbel_u; A.seed = seed; A.id_base = id_base; A.cat_ids = cat_ids;
  if (cat_ids && !pl.tiled) { set_error("eval_scores: cat_ids is for the KG sides only"); return KGREC_ERR_INVALID; }
  A.out = out; A.ld_out = ld_out;
  return launch_eval<MODE_FULL>(A, pl, static_cast<cudaStream_t>(stream));
}

extern "C" int kgrec_eval_topk(const kgrec_tables* tables, int model, int side, const void* q, const void* r,
                               int idx_bytes, const float* qvec, int64_t nq, const float* cat, int64_t cat_ld,
                               int64_t n_cat, int64_t id_base, int32_t k, const int64_t* filter_ptr,
                               const int32_t* filter_ids, const float* gumbel_u, uint64_t seed, uint64_t* out_keys,
                               void* workspace, int64_t workspace_bytes, kgrec_stream_t stream) {
  EvalArgs A{};
  EvalPlan pl{};
  int rc = eval_plan(tables, model, side, MODE_TOPK, cat, cat_ld, nq, n_cat, k, qvec != nullptr, &A, &pl);
  if (rc) return rc;
  if (!out_keys) { set_error("out_keys is NULL"); return KGREC_ERR_INVALID; }
  if (!qvec && (!q || (side != KGREC_SIDE_REC && !r))) { set_error("query ids are NULL"); return KGREC_ERR_INVALID; }
  if (!qvec && idx_bytes != 4 && idx_bytes != 8) { set_error("idx_bytes must be 4 or 8"); return KGREC_ERR_INVALID; }
  if (id_base < 0 || id_base + n_cat > 0xffffffffll) { set_error("catalog ids must fit 32 bits"); return KGREC_ERR_INVALID; }
  const int64_t need = static_cast<int64_t>(pl.n_splits) * nq * k * static_cast<int64_t>(sizeof(uint64_t));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  A.q = q; A.r = r; A.is64 = idx_bytes == 8; A.qvec = qvec;
  A.qvec_ld = pl.kind == KIND_GUMBEL_L2 ? cat_ld : 2 * static_cast<int64_t>(tables->dim);
  A.gconst = pl.kind == KIND_GUMBEL_L2 ? qvec + nq * cat_ld : nullptr;
  A.gumbel_u = gumbel_u; A.seed = seed; A.id_base = id_base;
  A.filter_ptr = filter_ptr; A.filter_ids = filter_ids;
  if (pl.n_splits == 1 && !pl.tiled && !pl.soft_aug) {
    A.part_keys = out_keys;
    return launch_eval<MODE_TOPK>(A, pl, st);
  }
  if (!workspace || workspace_bytes < need) {
    set_error("eval_topk workspace too small (%lld < %lld bytes)", static_cast<long long>(workspace_bytes), static_cast<long long>(need));
    return KGREC_ERR_INVALID;
  }
  A.part_keys = static_cast<uint64_t*>(workspace);
  if (pl.tiled || pl.soft_aug) {
    // unused pieces = empty lists; and, room permitting, the per-query bound the pieces share (0xffffffff = none yet)
    int64_t fill = need;
    if (pl.n_splits > 1 && workspace_bytes >= need + 4 * nq) {
      A.thr_glob = reinterpret_cast<uint32_t*>(static_cast<unsigned char*>(workspace) + need);
      fill = need + 4 * nq;
    }
    KGREC_CUDA_OK(cudaMemsetAsync(workspace, 0xff, static_cast<size_t>(fill), st));
  }
  if ((rc = launch_eval<MODE_TOPK>(A, pl, st))) return rc;
  return kgrec_merge_topk(A.part_keys, pl.n_splits, nq, k, out_keys, stream);
}

extern "C" int kgrec_merge_topk(const uint64_t* in_keys, int32_t n_lists, int64_t nq, int32_t k, uint64_t* out_keys,
                                kgrec_stream_t stream) {
  if (!in_keys || !out_keys || n_lists < 1 || nq < 0 || k < 1 || k > 128) { set_error("merge_topk: bad arguments"); return KGREC_ERR_INVALID; }
  if (nq == 0) return KGREC_OK;
  k_merge_topk<<<static_cast<unsigned>((nq + 7) / 8), 256, 8 * k * sizeof(uint64_t), static_cast<cudaStream_t>(stream)>>>(
      in_keys, n_lists, nq, k, out_keys);
  KGREC_CUDA_OK(cudaGetLastError());
  return KGREC_OK;
}

extern "C" int kgrec_eval_rank_count(const kgrec_tables* tables, int model, int side, const void* q, const void* r,
                                     int idx_bytes, const float* qvec, int64_t nq, const float* cat, int64_t cat_ld,
                                     int64_t n_cat, int64_t id_base, const float* gold_scores, const int32_t* gold_ids,
                                     int32_t* counts, kgrec_stream_t stream) {
  EvalArgs A{};
  EvalPlan pl{};
  int rc = eval_plan(tables, model, side, MODE_RANK, cat, cat_ld, nq, n_cat, 0, qvec != nullptr, &A, &pl);
  if (rc) return rc;
  if (!gold_scores || !gold_ids || !counts) { set_error("rank_count: NULL argument"); return KGREC_ERR_INVALID; }
  if (!qvec && (!q || (side != KGREC_SIDE_REC && !r))) { set_error("query ids are NULL"); return KGREC_ERR_INVALID; }
  if (!qvec && idx_bytes != 4 && idx_bytes != 8) { set_error("idx_bytes must be 4 or 8"); return KGREC_ERR_INVALID; }
  A.q = q; A.r = r; A.is64 = idx_bytes == 8; A.qvec = qvec;
  if (id_base < 0 || id_base + n_cat > 0xffffffffll) { set_error("catalog ids must fit 32 bits"); return KGREC_ERR_INVALID; }
  A.qvec_ld = 2 * static_cast<int64_t>(tables->dim);
  A.id_base = id_base; A.seed = 0;
  A.gold_scores = gold_scores; A.gold_ids = gold_ids; A.counts = counts;
  return launch_eval<MODE_RANK>(A, pl, static_cast<cudaStream_t>(stream));
}

extern "C" int kgrec_ktup_item_table(const kgrec_tables* tables, int64_t item_begin, int64_t n_items, float* out,
                                     int64_t ld_out, kgrec_stream_t stream) {
  if (!tables || !tables->item || !tables->ent || !tables->item2ent || !out || ld_out < tables->dim) {
    set_error("ktup_item_table: bad arguments");
    return KGREC_ERR_INVALID;
  }
  if (n_items <= 0) return KGREC_OK;
  const int64_t total = n_items * tables->dim;
  const int grid = static_cast<int>(std::min<int64_t>((total + 255) / 256, static_cast<int64_t>(sm_count()) * 16));
  k_ktup_items<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(*tables, item_begin, n_items, out, ld_out);
  KGREC_CUDA_OK(cudaGetLastError());
  return KGREC_OK;
}

extern "C" int32_t kgrec_gumbel_aug_ld(int32_t dim, int32_t n_pref) { return gumbel_aug_ld(dim, n_pref); }

extern "C" int32_t kgrec_gumbel_aug_supported(int32_t dim, int32_t n_pref, int32_t k) {
  if (dim <= 0 || dim > 256 || dim % 4 || n_pref <= 0 || n_pref > 64 || k < 0 || k > 128) return 0;
  const bool wide = dim > 128;
  return tiled_smem_layout(KIND_GUMBEL_L2, k > 0 ? MODE_TOPK : MODE_FULL, dim, wide ? 32 : 64, 2, k, wide ? 8 : 16, n_pref).total <= 225 * 1024;
}

extern "C" int kgrec_gumbel_aug_rows(const kgrec_tables* tables, int model, const void* ids, int idx_bytes, const float* rows,
                                     int64_t row_ld, int64_t n, float* out, int64_t ld_out, float* gconst, kgrec_stream_t stream) {
  if (!tables || !rows || !out || n < 0 || (model != KGREC_TUP && model != KGREC_KTUP)) { set_error("gumbel_aug_rows: bad arguments"); return KGREC_ERR_INVALID; }
  const int d = tables->dim, P = tables->n_pref;
  const bool ktup = model == KGREC_KTUP;
  if (d <= 0 || d > 256 || d % 4 || P <= 0 || P > 64 || ld_out != gumbel_aug_ld(d, P)) {
    set_error("gumbel_aug_rows: embedding_size must be a multiple of 4 (<= 256), preference_total <= 64, ld_out = %d", gumbel_aug_ld(d > 0 ? d : 4, P > 0 ? P : 1));
    return KGREC_ERR_UNSUPPORTED;
  }
  if (!tables->pref || !tables->pref_norm || (ktup && (!tables->rel || !tables->norm))) { set_error("gumbel_aug_rows: preference tables missing"); return KGREC_ERR_INVALID; }
  if (ids && idx_bytes != 4 && idx_bytes != 8) { set_error("idx_bytes must be 4 or 8"); return KGREC_ERR_INVALID; }
  if (n == 0 && !gconst) return KGREC_OK;
  const size_t smem = static_cast<size_t>(2) * P * ((d + 3) & ~3) * sizeof(float);
  KGREC_CUDA_OK(cudaFuncSetAttribute(k_gumbel_aug, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  int64_t ctas = (n + kWarpsPerCta - 1) / kWarpsPerCta;
  const int64_t cap = static_cast<int64_t>(sm_count()) * 4;
  ctas = ctas < 1 ? 1 : (ctas < cap ? ctas : cap);
  k_gumbel_aug<<<static_cast<int>(ctas), kThreads, smem, static_cast<cudaStream_t>(stream)>>>(*tables, ktup ? 1 : 0, ids, idx_bytes == 8, rows,
                                                                                         row_ld, n, out, ld_out, gconst);
  KGREC_CUDA_OK(cudaGetLastError());
  return KGREC_OK;
}

extern "C" int32_t kgrec_pref_aug_ld(int32_t dim) { return pref_aug_ld(dim); }

extern "C" int kgrec_pref_aug_rows(const kgrec_tables* tables, int model, int is_query, const void* ids, int idx_bytes,
                                   const float* rows, int64_t row_ld, int64_t n, float* out, int64_t ld_out,
                                   kgrec_stream_t stream) {
  if (!tables || !rows || !out || n < 0 || (model != KGREC_TUP && model != KGREC_KTUP)) { set_error("pref_aug_rows: bad arguments"); return KGREC_ERR_INVALID; }
  const int d = tables->dim;
  if (d <= 0 || d > 256 || d % 4 || row_ld % 4 || tables->ld % 4 || ld_out != pref_aug_ld(d)) {
    set_error("pref_aug_rows: embedding_size must be a multiple of 4 (<= 256) and ld_out = %d", pref_aug_ld(d > 0 ? d : 4));
    return KGREC_ERR_UNSUPPORTED;
  }
  const bool ktup = model == KGREC_KTUP;
  if (!tables->pref || !tables->pref_norm || (ktup && (!tables->rel || !tables->norm)) || tables->n_pref <= 0 || tables->n_pref > kMaxPref ||
      !aligned16(rows) || !aligned16(out) || !aligned16(tables->pref) || !aligned16(tables->pref_norm)) {
    set_error("pref_aug_rows: preference tables missing / misaligned");
    return KGREC_ERR_INVALID;
  }
  if (ids && idx_bytes != 4 && idx_bytes != 8) { set_error("idx_bytes must be 4 or 8"); return KGREC_ERR_INVALID; }
  if (n == 0) return KGREC_OK;
  const size_t smem = (static_cast<size_t>(2) * tables->n_pref * ((d + 3) & ~3) + kWarpsPerCta * kMaxPref) * sizeof(float);
  KGREC_CUDA_OK(cudaFuncSetAttribute(k_pref_aug, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  const int64_t ctas = (n + kWarpsPerCta - 1) / kWarpsPerCta, cap = static_cast<int64_t>(sm_count()) * 4;
  k_pref_aug<<<static_cast<int>(ctas < cap ? ctas : cap), kThreads, smem, static_cast<cudaStream_t>(stream)>>>(
      *tables, ktup ? 1 : 0, is_query ? 1 : 0, ids, idx_bytes == 8, rows, row_ld, n, out, ld_out);
  KGREC_CUDA_OK(cudaGetLastError());
  return KGREC_OK;
}
