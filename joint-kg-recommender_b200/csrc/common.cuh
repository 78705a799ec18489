// Shared device helpers for the kgrec_b200 kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <type_traits>
#include "../../include/kgrec_b200.h"

namespace kgrec {

constexpr unsigned FULL = 0xffffffffu;
constexpr int kWarpsPerCta = 8;
constexpr int kThreads = kWarpsPerCta * 32;
constexpr int kMaxPref = 128;             // preference_total limit (staging layout)

// ---- error plumbing (host) -------------------------------------------------
void set_error(const char* fmt, ...);
#define KGREC_CUDA_OK(expr)                                                        \
  do {                                                                             \
    cudaError_t e__ = (expr);                                                      \
    if (e__ != cudaSuccess) {                                                      \
      kgrec::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__),    \
                       __FILE__, __LINE__);                                        \
      return KGREC_ERR_CUDA;                                                       \
    }                                                                              \
  } while (0)
int sm_count();
float l2_keep_fraction(double table_bytes);   // share of a table's lines worth pinning in L2

// Launch dispatch on runtime flags: with_bools(f, a, b) calls f(std::integral_constant<bool, a>{}, ...), so f can
// name a kernel template with the flags as template arguments; f is instantiated once per combination.
template <typename F>
inline void with_bools(F&& f) { f(); }
template <typename F, typename... Bs>
inline void with_bools(F&& f, bool b, Bs... bs) {
  auto bind = [&](auto c) { with_bools([&](auto... cs) { f(c, cs...); }, bs...); };
  if (b) bind(std::true_type{}); else bind(std::false_type{});
}

// ---- warp reductions --------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
  return v;
}
__device__ __forceinline__ void warp_sum2(float& a, float& b) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_xor_sync(FULL, a, o);
    b += __shfl_xor_sync(FULL, b, o);
  }
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(FULL, v, o));
  return v;
}

// Reduce-scatter of 8 per-lane partials: on return every lane l holds the full warp sum of
// v[(l >> 2) & 7].  9 shuffles for 8 reductions (vs 40 with one tree each).
__device__ __forceinline__ float warp_reduce_scatter8(float (&v)[8], int lane) {
#pragma unroll
  for (int o = 16, n = 4; n > 0; o >>= 1, n >>= 1) {
    const bool up = (lane & o) != 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (j < n) {
        const float send = up ? v[j] : v[j + n];
        const float keep = up ? v[j + n] : v[j];
        v[j] = keep + __shfl_xor_sync(FULL, send, o);
      }
    }
  }
  float r = v[0];
  r += __shfl_xor_sync(FULL, r, 2);
  r += __shfl_xor_sync(FULL, r, 1);
  return r;
}

// ---- index loads --------------------------------------------------------------
__device__ __forceinline__ int64_t load_idx(const void* p, int64_t i, int is64) {
  return is64 ? __ldg(reinterpret_cast<const long long*>(p) + i)
              : static_cast<int64_t>(__ldg(reinterpret_cast<const int*>(p) + i));
}
__device__ __forceinline__ int64_t checked(int64_t row, int64_t rows, int32_t* status) {
  if (static_cast<uint64_t>(row) >= static_cast<uint64_t>(rows)) {
    if (status) *status = 1;
    return 0;
  }
  return row;
}

// ---- streaming loads / stores ------------------------------------------------------
__device__ __forceinline__ float4 ldg_f4(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void red_add_f4(float* p, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d)
               : "memory");
}

__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }

// ---- mbarrier / bulk-copy PTX ---------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity, uint32_t suspend_ns) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity), "r"(suspend_ns) : "memory");
  return ok != 0;
}
// Wait with a hardware suspend hint: a warp that finds the phase incomplete is parked by the
// barrier unit instead of re-issuing TRYWAIT back to back (which starves the async proxy).
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity, 20000u)) {}
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// ---- L2 cache policies ---------------------------------------------------------------------
// Embedding rows are re-read (by other triples, by the backward, by the next step) while
// gradient rows are written once and consumed later by a different kernel: table loads carry an
// evict_last policy on a fraction of their lines sized to fit L2, gradient stores evict_first,
// so the write stream does not push the tables out of the 126 MB L2.
__device__ __forceinline__ uint64_t policy_evict_last(float fraction) {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.L2::evict_unchanged.b64 %0, %1;" : "=l"(p) : "f"(fraction));
  return p;
}
__device__ __forceinline__ uint64_t policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ float4 ldg_f4_hint(const float4* p, uint64_t pol) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p), "l"(pol));
  return r;
}
__device__ __forceinline__ void stg_f4_hint(float4* p, float a, float b, float c, float d, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1,%2,%3,%4}, %5;" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d), "l"(pol)
               : "memory");
}

// One embedding row spread over a warp.  VEC: lane owns float4 chunks lane, lane+32, ...
// (128-bit loads, requires d % 4 == 0 and 16-byte aligned rows); otherwise lane owns
// scalars lane, lane+32, ...  Lanes / slots past d hold zeros so every reduction can run
// unmasked.
template <int NCH, bool VEC>
struct Row {
  static constexpr int NE = NCH * 4;
  __device__ __forceinline__ static int elem(int lane, int e) {
    return VEC ? ((lane + 32 * (e >> 2)) * 4 + (e & 3)) : (lane + 32 * e);
  }
  __device__ __forceinline__ static void load(float (&v)[NE], const float* __restrict__ row, int d, int lane) {
    if (VEC) {
#pragma unroll
      for (int i = 0; i < NCH; ++i) {
        const int c = lane + 32 * i;
        float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
        if (c * 4 < d) t = ldg_f4(reinterpret_cast<const float4*>(row) + c);
        v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
      }
    } else {
#pragma unroll
      for (int e = 0; e < NE; ++e) {
        const int j = lane + 32 * e;
        v[e] = (j < d) ? __ldg(row + j) : 0.f;
      }
    }
  }
  // vector path with an L2 cache policy (see policy_evict_last)
  __device__ __forceinline__ static void load_hint(float (&v)[NE], const float* __restrict__ row, int d, int lane, uint64_t pol) {
    static_assert(VEC, "cache-hinted loads are built for the 128-bit path");
#pragma unroll
    for (int i = 0; i < NCH; ++i) {
      const int c = lane + 32 * i;
      float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c * 4 < d) t = ldg_f4_hint(reinterpret_cast<const float4*>(row) + c, pol);
      v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
    }
  }
  __device__ __forceinline__ static void store_hint(float* __restrict__ row, const float (&v)[NE], int d, int lane, uint64_t pol) {
    static_assert(VEC, "cache-hinted stores are built for the 128-bit path");
#pragma unroll
    for (int i = 0; i < NCH; ++i) {
      const int c = lane + 32 * i;
      if (c * 4 < d) stg_f4_hint(reinterpret_cast<float4*>(row) + c, v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3], pol);
    }
  }
  // shared-memory variant (tables staged by the CTA)
  __device__ __forceinline__ static void load_s(float (&v)[NE], const float* row, int d, int lane) {
    if (VEC) {
#pragma unroll
      for (int i = 0; i < NCH; ++i) {
        const int c = lane + 32 * i;
        float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
        if (c * 4 < d) t = reinterpret_cast<const float4*>(row)[c];
        v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
      }
    } else {
#pragma unroll
      for (int e = 0; e < NE; ++e) {
        const int j = lane + 32 * e;
        v[e] = (j < d) ? row[j] : 0.f;
      }
    }
  }
  __device__ __forceinline__ static void store(float* __restrict__ row, const float (&v)[NE], int d, int lane) {
    if (VEC) {
#pragma unroll
      for (int i = 0; i < NCH; ++i) {
        const int c = lane + 32 * i;
        if (c * 4 < d)
          reinterpret_cast<float4*>(row)[c] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
      }
    } else {
#pragma unroll
      for (int e = 0; e < NE; ++e) {
        const int j = lane + 32 * e;
        if (j < d) row[j] = v[e];
      }
    }
  }
  // streaming store: gradient rows are written once and never re-read by the kernels, so they
  // should not displace the embedding tables from L2
  __device__ __forceinline__ static void store_cs(float* __restrict__ row, const float (&v)[NE], int d, int lane) {
    if (VEC) {
#pragma unroll
      for (int i = 0; i < NCH; ++i) {
        const int c = lane + 32 * i;
        if (c * 4 < d)
          __stcs(reinterpret_cast<float4*>(row) + c, make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]));
      }
    } else {
#pragma unroll
      for (int e = 0; e < NE; ++e) {
        const int j = lane + 32 * e;
        if (j < d) __stcs(row + j, v[e]);
      }
    }
  }
  __device__ __forceinline__ static void red_add(float* __restrict__ row, const float (&v)[NE], int d, int lane) {
    if (VEC) {
#pragma unroll
      for (int i = 0; i < NCH; ++i) {
        const int c = lane + 32 * i;
        if (c * 4 < d) red_add_f4(row + 4 * c, v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
      }
    } else {
#pragma unroll
      for (int e = 0; e < NE; ++e) {
        const int j = lane + 32 * e;
        if (j < d) atomicAdd(row + j, v[e]);
      }
    }
  }
  __device__ __forceinline__ static float dot(const float (&a)[NE], const float (&b)[NE]) {
    float s = 0.f;
#pragma unroll
    for (int e = 0; e < NE; ++e) s = fmaf(a[e], b[e], s);
    return s;
  }
};

// L(e) partial and its derivative (torch: d|x|/dx = sign(x), sign(0) = 0)
// ---- packed fp32x2 arithmetic (sm_100: one instruction, two lanes of the FMA pipe) ----------
typedef unsigned long long f32x2;     // two floats in one 64-bit register pair
__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b) { f32x2 r; asm("sub.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) { f32x2 r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
__device__ __forceinline__ f32x2 splat2(float v) { f32x2 r; asm("mov.b64 %0, {%1, %1};" : "=l"(r) : "f"(v)); return r; }
__device__ __forceinline__ float lo2(f32x2 v) { float a, b; asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); return a; }
__device__ __forceinline__ float hi2(f32x2 v) { float a, b; asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); return b; }
__device__ __forceinline__ float sum2(f32x2 v) { return lo2(v) + hi2(v); }
__device__ __forceinline__ float abssum2(f32x2 v) { return fabsf(lo2(v)) + fabsf(hi2(v)); }

__device__ __forceinline__ float dist_term(float e, int l1) { return l1 ? fabsf(e) : e * e; }
__device__ __forceinline__ float ddist_term(float e, int l1) {
  return l1 ? ((e > 0.f) ? 1.f : ((e < 0.f) ? -1.f : 0.f)) : 2.f * e;
}

// ---- Philox4x32-10 (counter-based; the in-kernel Gumbel uniform source) ---------------
__device__ __forceinline__ uint32_t philox_uniform_bits(uint64_t seed, uint64_t pair, uint32_t k) {
  uint32_t c0 = static_cast<uint32_t>(pair), c1 = static_cast<uint32_t>(pair >> 32), c2 = k, c3 = 0x4b47u;
  uint32_t k0 = static_cast<uint32_t>(seed), k1 = static_cast<uint32_t>(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return c0;
}
// all four words of one Philox4x32-10 block (counter = (ctr, blk, 0x4b47), key = seed)
__device__ __forceinline__ uint4 philox4(uint64_t seed, uint64_t ctr, uint32_t blk) {
  uint32_t c0 = static_cast<uint32_t>(ctr), c1 = static_cast<uint32_t>(ctr >> 32), c2 = blk, c3 = 0x4b47u;
  uint32_t k0 = static_cast<uint32_t>(seed), k1 = static_cast<uint32_t>(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return make_uint4(c0, c1, c2, c3);
}
__device__ __forceinline__ float philox_uniform(uint64_t seed, uint64_t pair, uint32_t k) {
  return static_cast<float>(philox_uniform_bits(seed, pair, k) >> 8) * (1.0f / 16777216.0f);  // [0,1)
}
// Gumbel noise exactly as transUP.py:159-161 builds it from a uniform draw
__device__ __forceinline__ float gumbel_from_uniform(float u) {
  const float eps = 1e-20f;
  return -logf(-logf(u + eps) + eps);
}

// In-kernel draws (no caller-supplied uniforms to reproduce): u in (0,1) strictly, so the two
// eps terms of the reference formula are not needed and the logs can be the 2-instruction
// lg2.approx form.  Same distribution; used only when the noise is generated on the device.
// 23 bits, not 24: n + 0.5 must be exact in fp32.  With bits >> 8 the top value 16777215.5 rounds to 2^24, u = 1, the
// noise +inf -- one draw in 2^24, i.e. a few per training step at configs[2] sizes -- and exp(inf - inf) in the
// straight-through soft-max turns the step's gradients, then the tables, into NaN.
__device__ __forceinline__ float gumbel_fast(uint32_t bits) {
  const float u = (static_cast<float>(bits >> 9) + 0.5f) * (1.0f / 8388608.0f);   // (0, 1) strictly
  return -__logf(-__logf(u));
}

}  // namespace kgrec
