// Row-wise epilogue kernels of the layer loop (SURVEY.md K9, K14), sm_100a, HBM-bound:
//   * LayerNorm + ReLU forward in one pass              (/root/reference/module/model.py:53-56)
//   * its backward, fused with the three column reductions the step needs (d gamma, d beta and the
//     bias gradient of the linear that produced the pre-norm tensor)
//   * summed soft-max cross-entropy forward / backward  (/root/reference/train.py:320,351)
// One warp owns one row; a row of up to 32 lanes x kMaxVec 16-byte vectors stays in registers between
// the statistics pass and the output pass, so every tensor is read once and written once.
// Column reductions are two-stage and deterministic: per-CTA partials, then a fixed-order sum.
#include <algorithm>
#include <type_traits>

#include "common.cuh"

namespace pg {

constexpr int kRowThreads = 256;
constexpr int kMaxVec = 4;          // vectors per lane kept in registers (bf16: d <= 1024, fp32: d <= 512)
// pg_set_option("ln_stage", 0|1|2): LayerNorm kernels read their rows through the cp.async ring never / when a lane
// holds one 16-byte vector per row (rows of up to 512 bytes: measured 0.237 -> 0.210 ms forward, 0.351 -> 0.312 ms
// backward on [1 M, 256] bf16; at two vectors per lane plain loads are 2-5 % faster) / always
int g_ln_stage = 1;
int g_ce_subwarp = 1;               // pg_set_option("ce_subwarp", 0|1): cross-entropy kernels with several rows per warp

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// K (1, 2 or 4) independent warp sums at once; every lane ends up with all K totals.  The first log2(K) butterfly
// steps halve the number of live values instead of doubling the traffic (a lane keeps the half selected by its own
// lane bit and ships the other half), so K = 4 costs 10 shuffles instead of 20 and K = 2 costs 7 instead of 10.
// The summation order is fixed by (K, lane), i.e. deterministic.
template <int K>
__device__ __forceinline__ void warp_sum_multi(float (&v)[K], int lane) {
  static_assert(K == 1 || K == 2 || K == 4, "warp_sum_multi: K must be 1, 2 or 4");
  constexpr unsigned kAll = 0xffffffffu;
  if constexpr (K == 1) {
    v[0] = warp_sum(v[0]);
  } else if constexpr (K == 2) {
    const bool up = (lane & 16) != 0;
    const float keep = up ? v[1] : v[0], send = up ? v[0] : v[1];
    float t = keep + __shfl_xor_sync(kAll, send, 16);
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) t += __shfl_xor_sync(kAll, t, o);
    v[0] = __shfl_sync(kAll, t, 0);
    v[1] = __shfl_sync(kAll, t, 16);
  } else {
    const bool up = (lane & 16) != 0;
    const float k0 = up ? v[2] : v[0], k1 = up ? v[3] : v[1];
    const float s0 = up ? v[0] : v[2], s1 = up ? v[1] : v[3];
    const float a0 = k0 + __shfl_xor_sync(kAll, s0, 16);     // value 2*bit4
    const float a1 = k1 + __shfl_xor_sync(kAll, s1, 16);     // value 2*bit4 + 1
    const bool up2 = (lane & 8) != 0;
    const float keep = up2 ? a1 : a0, send = up2 ? a0 : a1;
    float t = keep + __shfl_xor_sync(kAll, send, 8);          // value 2*bit4 + bit3
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) t += __shfl_xor_sync(kAll, t, o);
    v[0] = __shfl_sync(kAll, t, 0);
    v[1] = __shfl_sync(kAll, t, 8);
    v[2] = __shfl_sync(kAll, t, 16);
    v[3] = __shfl_sync(kAll, t, 24);
  }
}

// max(v, lo) that propagates NaN like torch's relu; lo = 0 (ReLU) or -inf (no activation)
__device__ __forceinline__ float max_nan(float v, float lo) {
  float r;
  asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(v), "f"(lo));
  return r;
}
// the affine LayerNorm output of one element; forward and backward (ReLU mask recomputation) MUST round identically
__device__ __forceinline__ float2 ln_affine2(float2 centered, float2 rstd, float2 g, float2 b) {
  return __ffma2_rn(__fmul2_rn(centered, rstd), g, b);
}

// ---- per-lane asynchronous staging ring ----------------------------------------------------------------------------
// A lane copies the 16-byte vectors IT will consume into its own shared-memory slots with cp.async (LDGSTS) several
// row groups ahead and reads back only its own slots after cp.async.wait_group: no barrier, no cross-lane hand-off,
// and the bytes in flight live in shared memory instead of registers (S - 1 stages per lane, whatever the register
// budget).  Slot layout [stage][vector][thread]: consecutive lanes, consecutive 16 bytes (conflict-free LDS.128).
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(static_cast<uint32_t>(__cvta_generic_to_shared(smem))), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// gamma / beta in shared memory, laid out so that lane l reads elements [4h, 4h+4) of its vector `vec` as ONE
// 16-byte word next to lane l+1's: index ((h * nv + vec) * 4 + e), h = (element in vector) / 4
template <int V>
__device__ __forceinline__ void stage_affine(float* sm, const float* __restrict__ src, int d, int nv) {
  for (int c = threadIdx.x; c < nv * V; c += kRowThreads) {
    const int vec = c / V, i = c % V;
    sm[((i / 4) * nv + vec) * 4 + (i % 4)] = c < d ? __ldg(src + c) : 0.f;
  }
}
template <int H>
__device__ __forceinline__ void load_affine(const float* sm, int nv, int vec, float2 (&f)[H]) {
#pragma unroll
  for (int h = 0; h < H / 2; ++h) {
    const float4 t = *reinterpret_cast<const float4*>(sm + (h * nv + vec) * 4);
    f[2 * h] = make_float2(t.x, t.y);
    f[2 * h + 1] = make_float2(t.z, t.w);
  }
}

// a 16-byte vector as H float2 pairs: the row kernels do their arithmetic with the packed fp32x2 instructions of
// sm_100 (FADD2 / FMUL2 / FFMA2: two IEEE round-to-nearest results per issue slot, bit-identical to the scalar ops)
template <typename T> struct Pair;
template <> struct Pair<float> {
  static constexpr int H = 2;
  __device__ __forceinline__ static void unpack(const uint4& r, float2 (&f)[2]) {
    f[0] = make_float2(__uint_as_float(r.x), __uint_as_float(r.y));
    f[1] = make_float2(__uint_as_float(r.z), __uint_as_float(r.w));
  }
  __device__ __forceinline__ static uint4 pack(const float2 (&f)[2]) {
    return make_uint4(__float_as_uint(f[0].x), __float_as_uint(f[0].y), __float_as_uint(f[1].x), __float_as_uint(f[1].y));
  }
  // what a store in T followed by a load gives back
  __device__ __forceinline__ static void round_trip(float2 (&)[2]) {}
};
template <> struct Pair<__nv_bfloat16> {
  static constexpr int H = 4;
  __device__ __forceinline__ static float2 widen(uint32_t w) { return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u)); }
  __device__ __forceinline__ static uint32_t narrow(float2 f) {
    const __nv_bfloat162 b = __floats2bfloat162_rn(f.x, f.y);
    return *reinterpret_cast<const uint32_t*>(&b);
  }
  __device__ __forceinline__ static void unpack(const uint4& r, float2 (&f)[4]) {
    f[0] = widen(r.x); f[1] = widen(r.y); f[2] = widen(r.z); f[3] = widen(r.w);
  }
  __device__ __forceinline__ static uint4 pack(const float2 (&f)[4]) {
    return make_uint4(narrow(f[0]), narrow(f[1]), narrow(f[2]), narrow(f[3]));
  }
  __device__ __forceinline__ static void round_trip(float2 (&f)[4]) {
#pragma unroll
    for (int k = 0; k < 4; ++k) f[k] = widen(narrow(f[k]));
  }
};
__device__ __forceinline__ float2 splat(float a) { return make_float2(a, a); }

// ---------------------------------------------------------------------------------------------------------
// VPL vectors per lane (d <= 32 * VPL * V), R rows per warp iteration.
// FULL: d == 32 * VPL * V, every lane owns VPL live vectors and no per-vector predicate is compiled in.
// S: stages of the staging ring (0: plain register loads, R * VPL of them in flight per lane).
// The kernel is issue-bound before it is HBM-bound (a row is ~20 instructions per element), so the row loop has
// no per-row branches (groups of R complete rows; the < R leftover rows run the R = 1 body on the first warps),
// the R row statistics are reduced together (warp_sum_multi), the mean is a multiply by 1/d and gamma / beta come
// from shared memory instead of 2 * VPL * V registers.
template <typename T, int VPL, int R, bool FULL, int S>
__global__ void __launch_bounds__(kRowThreads, (R * VPL * (16 / sizeof(T)) <= 16) ? 4 : 3)
ln_relu_fwd_kernel(const T* __restrict__ y, int64_t ldy, const float* __restrict__ gamma, const float* __restrict__ beta,
                   float eps, int relu, T* __restrict__ out, int64_t ldo, float* __restrict__ mean_out,
                   float* __restrict__ rstd_out, int n_rows, int d, T* __restrict__ out_clean, int64_t ldc, DropArg drop) {
  using Q = Pair<T>;
  using Raw = uint4;
  constexpr int H = Q::H, V = 2 * H;
  constexpr int NV = 32 * VPL;
  extern __shared__ uint4 ring[];                            // [S][R][VPL][kRowThreads]
  __shared__ __align__(16) float sg[NV * V], sb[NV * V];
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * kRowThreads + threadIdx.x) >> 5;
  const int warps = (gridDim.x * kRowThreads) >> 5;
  const int nvec = d / V;
  const float inv_d = 1.0f / static_cast<float>(d);
  const float lo = relu ? 0.f : -INFINITY;
  const bool dropping = drop.thresh16 != 0u;
  const uint32_t key = dropping ? drop_seed_hi(drop) : 0u;
  // 1 / (1 - p) a power of two (p = 0.5): scaling commutes with the rounding to T
  const bool exact_scale = (__float_as_uint(drop.scale) & 0x007fffffu) == 0u;
  bool act[VPL];
#pragma unroll
  for (int j = 0; j < VPL; ++j) act[j] = FULL || (lane + j * 32 < nvec);
  stage_affine<V>(sg, gamma, d, NV);
  stage_affine<V>(sb, beta, d, NV);
  __syncthreads();

  auto src = [&](int row, int j) { return y + static_cast<int64_t>(row) * ldy + static_cast<int64_t>(lane + j * 32) * V; };

  auto rows = [&](auto rc, int row0, const Raw (&raw)[decltype(rc)::value][VPL]) {
    constexpr int RR = decltype(rc)::value;
    float2 x[RR][VPL][H];
    float s[RR];
#pragma unroll
    for (int r = 0; r < RR; ++r) {
      float2 acc = make_float2(0.f, 0.f);
#pragma unroll
      for (int j = 0; j < VPL; ++j) {
        if (act[j]) {
          Q::unpack(raw[r][j], x[r][j]);
        } else {
#pragma unroll
          for (int k = 0; k < H; ++k) x[r][j][k] = make_float2(0.f, 0.f);
        }
#pragma unroll
        for (int k = 0; k < H; ++k) acc = __fadd2_rn(acc, x[r][j][k]);
      }
      s[r] = acc.x + acc.y;
    }
    warp_sum_multi<RR>(s, lane);
    float mean[RR], q[RR];
#pragma unroll
    for (int r = 0; r < RR; ++r) {
      mean[r] = s[r] * inv_d;
      const float2 neg = splat(-mean[r]);
      float2 acc = make_float2(0.f, 0.f);
#pragma unroll
      for (int j = 0; j < VPL; ++j)
#pragma unroll
        for (int k = 0; k < H; ++k) {
          const float2 c = act[j] ? __fadd2_rn(x[r][j][k], neg) : make_float2(0.f, 0.f);
          x[r][j][k] = c;
          acc = __ffma2_rn(c, c, acc);
        }
      q[r] = acc.x + acc.y;
    }
    warp_sum_multi<RR>(q, lane);
    float rstd[RR];
#pragma unroll
    for (int r = 0; r < RR; ++r) {
      rstd[r] = rsqrtf(q[r] * inv_d + eps);
      if (lane == 0) { mean_out[row0 + r] = mean[r]; rstd_out[row0 + r] = rstd[r]; }
    }
#pragma unroll
    for (int j = 0; j < VPL; ++j)
      if (act[j]) {
        float2 gm[H], bt[H];
        load_affine<H>(sg, NV, lane + j * 32, gm);
        load_affine<H>(sb, NV, lane + j * 32, bt);
#pragma unroll
        for (int r = 0; r < RR; ++r) {
          const int row = row0 + r;
          const float2 rs2 = splat(rstd[r]);
          float2 o[H];
#pragma unroll
          for (int k = 0; k < H; ++k) {
            const float2 v = ln_affine2(x[r][j][k], rs2, gm[k], bt[k]);
            o[k] = make_float2(max_nan(v.x, lo), max_nan(v.y, lo));
          }
          Raw packed = Q::pack(o);
          // the clean result (source of the halo push) when asked for, and dropout(result) for the next layer --
          // computed from the ROUNDED clean value, i.e. exactly what pg_dropout would make of the clean tensor
          // (a power-of-two 1 / (1 - p) commutes with the rounding: no second rounding needed)
          if (out_clean != nullptr)
            st_vec<16>(out_clean + static_cast<int64_t>(row) * ldc + static_cast<int64_t>(lane + j * 32) * V, packed);
          if (dropping) {
            if (!exact_scale) Q::round_trip(o);
            drop_apply2<H>(o, static_cast<uint64_t>(row) * nvec + (lane + j * 32), drop.thresh16, drop.scale, drop.seed_lo, key);
            packed = Q::pack(o);
          }
          st_vec<16>(out + static_cast<int64_t>(row) * ldo + static_cast<int64_t>(lane + j * 32) * V, packed);
        }
      }
  };

  const int n_groups = n_rows / R;
  if constexpr (S == 0) {
    for (int g = warp; g < n_groups; g += warps) {
      Raw raw[R][VPL];
#pragma unroll
      for (int r = 0; r < R; ++r)
#pragma unroll
        for (int j = 0; j < VPL; ++j)
          if (act[j]) raw[r][j] = *reinterpret_cast<const Raw*>(src(g * R + r, j));
      rows(std::integral_constant<int, R>{}, g * R, raw);
    }
  } else {
    const int n_it = warp < n_groups ? (n_groups - warp + warps - 1) / warps : 0;
    auto slot = [&](int it, int r, int j) { return ring + (((it % S) * R + r) * VPL + j) * kRowThreads + threadIdx.x; };
    auto issue = [&](int it) {
      const int row0 = (warp + it * warps) * R;
#pragma unroll
      for (int r = 0; r < R; ++r)
#pragma unroll
        for (int j = 0; j < VPL; ++j)
          if (act[j]) cp_async16(slot(it, r, j), src(row0 + r, j));
    };
#pragma unroll
    for (int it = 0; it < S - 1; ++it) {
      if (it < n_it) issue(it);
      cp_async_commit();
    }
    for (int it = 0; it < n_it; ++it) {
      // refills the stage consumed in iteration it - 1 (its reads completed: their values were used)
      if (it + S - 1 < n_it) issue(it + S - 1);
      cp_async_commit();
      cp_async_wait<S - 1>();
      Raw raw[R][VPL];
#pragma unroll
      for (int r = 0; r < R; ++r)
#pragma unroll
        for (int j = 0; j < VPL; ++j)
          if (act[j]) raw[r][j] = *slot(it, r, j);
      rows(std::integral_constant<int, R>{}, (warp + it * warps) * R, raw);
    }
  }
  if (R > 1 && warp < n_rows - n_groups * R) {
    const int row = n_groups * R + warp;
    Raw raw[1][VPL];
#pragma unroll
    for (int j = 0; j < VPL; ++j)
      if (act[j]) raw[0][j] = *reinterpret_cast<const Raw*>(src(row, j));
    rows(std::integral_constant<int, 1>{}, row, raw);
  }
}

// g_y = rstd * (gh*gamma - mean_d(gh*gamma) - xhat * mean_d(gh*gamma*xhat)),  gh = g_out * (out > 0)
// partial[blockIdx][0] += gh * xhat (d gamma), [1] += gh (d beta), [2] += g_y (bias gradient upstream)
// MODE 0: no activation, 1: ReLU mask read from the forward output `out`, 2: ReLU mask recomputed from y with the
// forward's own expression (ln_affine2) -- one [N, d] tensor less to read.  One row per warp iteration; S as above
// (stages hold the row's g_out and y vectors; MODE 1 only runs with S = 0).
template <typename T, int VPL, int MODE, bool FULL, int S>
__global__ void __launch_bounds__(kRowThreads, (VPL * (16 / sizeof(T)) <= 8) ? 3 : ((VPL * (16 / sizeof(T)) <= 16) ? 2 : 1))
ln_relu_bwd_kernel(const T* __restrict__ g_out, int64_t ldg, const T* __restrict__ out, int64_t ldo,
                   const T* __restrict__ y, int64_t ldy, const float* __restrict__ mean, const float* __restrict__ rstd,
                   const float* __restrict__ gamma, T* __restrict__ g_y, int64_t ldgy,
                   float* __restrict__ partial, int n_rows, int d, const float* __restrict__ beta) {
  using Q = Pair<T>;
  using Raw = uint4;
  constexpr int H = Q::H, V = 2 * H;
  constexpr int NV = 32 * VPL;
  static_assert(MODE != 1 || S == 0, "the ring holds two tensors");
  extern __shared__ uint4 ring[];                            // [S][2][VPL][kRowThreads], then red[3][d]
  __shared__ __align__(16) float sg[NV * V], sb[NV * V];
  float* red = reinterpret_cast<float*>(ring + S * 2 * VPL * kRowThreads);
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * kRowThreads + threadIdx.x) >> 5;
  const int warps = (gridDim.x * kRowThreads) >> 5;
  const int nvec = d / V;
  const float inv_d = 1.0f / static_cast<float>(d);
  bool act[VPL];
  float2 cg[VPL][H], cb[VPL][H], cy[VPL][H];                 // this lane's column partials
#pragma unroll
  for (int j = 0; j < VPL; ++j) {
    act[j] = FULL || (lane + j * 32 < nvec);
#pragma unroll
    for (int k = 0; k < H; ++k) cg[j][k] = cb[j][k] = cy[j][k] = make_float2(0.f, 0.f);
  }
  stage_affine<V>(sg, gamma, d, NV);
  if (MODE == 2) stage_affine<V>(sb, beta, d, NV);
  __syncthreads();

  auto off = [&](int row, int64_t ld, int j) { return static_cast<int64_t>(row) * ld + static_cast<int64_t>(lane + j * 32) * V; };

  auto one_row = [&](int row, float mu, float rs, const Raw (&rg)[VPL], const Raw (&ry)[VPL], const Raw (&ro)[VPL]) {
    float2 gx[VPL][H], xh[VPL][H], s1 = make_float2(0.f, 0.f), s2 = make_float2(0.f, 0.f);
    const float2 neg_mu = splat(-mu), rs2 = splat(rs);
#pragma unroll
    for (int j = 0; j < VPL; ++j) {
      if (!FULL && !act[j]) {
#pragma unroll
        for (int k = 0; k < H; ++k) gx[j][k] = xh[j][k] = make_float2(0.f, 0.f);
        continue;
      }
      float2 g[H], o[H], yy[H], gm[H], bt[H];
      Q::unpack(rg[j], g);
      Q::unpack(ry[j], yy);
      if (MODE == 1) Q::unpack(ro[j], o);
      load_affine<H>(sg, NV, lane + j * 32, gm);
      if (MODE == 2) load_affine<H>(sb, NV, lane + j * 32, bt);
#pragma unroll
      for (int k = 0; k < H; ++k) {
        const float2 c = __fadd2_rn(yy[k], neg_mu);
        const float2 xx = __fmul2_rn(c, rs2);
        float2 gg = g[k];
        if (MODE == 2) {
          const float2 v = __ffma2_rn(xx, gm[k], bt[k]);          // == ln_affine2(c, rs2, gm, bt): the forward's value
          gg.x = v.x > 0.f ? gg.x : 0.f;
          gg.y = v.y > 0.f ? gg.y : 0.f;
        }
        if (MODE == 1) {
          gg.x = o[k].x > 0.f ? gg.x : 0.f;
          gg.y = o[k].y > 0.f ? gg.y : 0.f;
        }
        const float2 gv = __fmul2_rn(gg, gm[k]);
        xh[j][k] = xx;
        gx[j][k] = gv;
        s1 = __fadd2_rn(s1, gv);
        s2 = __ffma2_rn(gv, xx, s2);
        cg[j][k] = __ffma2_rn(gg, xx, cg[j][k]);
        cb[j][k] = __fadd2_rn(cb[j][k], gg);
      }
    }
    float st[2] = {s1.x + s1.y, s2.x + s2.y};
    warp_sum_multi<2>(st, lane);
    // g_y = rs * gx - rs * c1 - xh * (rs * c2)
    const float2 k1 = splat(-rs * (st[0] * inv_d)), k2 = splat(-rs * (st[1] * inv_d));
#pragma unroll
    for (int j = 0; j < VPL; ++j)
      if (act[j]) {
        float2 o[H];
#pragma unroll
        for (int k = 0; k < H; ++k) o[k] = __ffma2_rn(xh[j][k], k2, __ffma2_rn(gx[j][k], rs2, k1));
        st_vec<16>(g_y + off(row, ldgy, j), Q::pack(o));
        // the tensor handed upstream is stored in T: reduce what is stored
        Q::round_trip(o);
#pragma unroll
        for (int k = 0; k < H; ++k) cy[j][k] = __fadd2_rn(cy[j][k], o[k]);
      }
  };

  const int n_it = warp < n_rows ? (n_rows - warp + warps - 1) / warps : 0;
  // mean / rstd of the NEXT row are fetched while the current one is processed (their latency is not behind the ring)
  float mu_n = 0.f, rs_n = 0.f;
  if (n_it > 0) { mu_n = __ldg(mean + warp); rs_n = __ldg(rstd + warp); }
  if constexpr (S == 0) {
    for (int it = 0; it < n_it; ++it) {
      const int row = warp + it * warps;
      Raw rg[VPL], ry[VPL], ro[VPL];
#pragma unroll
      for (int j = 0; j < VPL; ++j)
        if (act[j]) {
          rg[j] = *reinterpret_cast<const Raw*>(g_out + off(row, ldg, j));
          ry[j] = *reinterpret_cast<const Raw*>(y + off(row, ldy, j));
          if (MODE == 1) ro[j] = *reinterpret_cast<const Raw*>(out + off(row, ldo, j));
        }
      const float mu = mu_n, rs = rs_n;
      if (it + 1 < n_it) { mu_n = __ldg(mean + row + warps); rs_n = __ldg(rstd + row + warps); }
      one_row(row, mu, rs, rg, ry, ro);
    }
  } else {
    auto slot = [&](int it, int t, int j) { return ring + (((it % S) * 2 + t) * VPL + j) * kRowThreads + threadIdx.x; };
    auto issue = [&](int it) {
      const int row = warp + it * warps;
#pragma unroll
      for (int j = 0; j < VPL; ++j)
        if (act[j]) {
          cp_async16(slot(it, 0, j), g_out + off(row, ldg, j));
          cp_async16(slot(it, 1, j), y + off(row, ldy, j));
        }
    };
#pragma unroll
    for (int it = 0; it < S - 1; ++it) {
      if (it < n_it) issue(it);
      cp_async_commit();
    }
    for (int it = 0; it < n_it; ++it) {
      const int row = warp + it * warps;
      if (it + S - 1 < n_it) issue(it + S - 1);
      cp_async_commit();
      const float mu = mu_n, rs = rs_n;
      if (it + 1 < n_it) { mu_n = __ldg(mean + row + warps); rs_n = __ldg(rstd + row + warps); }
      cp_async_wait<S - 1>();
      Raw rg[VPL], ry[VPL], ro[VPL];
#pragma unroll
      for (int j = 0; j < VPL; ++j)
        if (act[j]) { rg[j] = *slot(it, 0, j); ry[j] = *slot(it, 1, j); }
      one_row(row, mu, rs, rg, ry, ro);
    }
  }

  // CTA-level reduction of the column partials in a fixed order (warp 0..7), then one partial row per CTA
  for (int i = threadIdx.x; i < 3 * d; i += kRowThreads) red[i] = 0.f;
  __syncthreads();
  for (int w = 0; w < kRowThreads / 32; ++w) {
    if ((threadIdx.x >> 5) == w) {
#pragma unroll
      for (int j = 0; j < VPL; ++j) {
        const int vi = lane + j * 32;
        if (vi < nvec)
#pragma unroll
          for (int k = 0; k < H; ++k) {
            const int c = vi * V + 2 * k;
            red[c] += cg[j][k].x;
            red[c + 1] += cg[j][k].y;
            red[d + c] += cb[j][k].x;
            red[d + c + 1] += cb[j][k].y;
            red[2 * d + c] += cy[j][k].x;
            red[2 * d + c + 1] += cy[j][k].y;
          }
      }
    }
    __syncthreads();
  }
  float* pp = partial + static_cast<int64_t>(blockIdx.x) * 3 * d;
  for (int i = threadIdx.x; i < 3 * d; i += kRowThreads) pp[i] = red[i];
}

// out[k] = sum over blocks of partial[b][k]: one warp per column, lanes stride over the blocks, fixed order
__global__ void colsum_final_kernel(const float* __restrict__ partial, int n_blocks, int width, float* __restrict__ out0,
                                    float* __restrict__ out1, float* __restrict__ out2, int d) {
  const int k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (k >= width) return;
  float s = 0.f;
  for (int b = lane; b < n_blocks; b += 32) s += partial[static_cast<int64_t>(b) * width + k];
  s = warp_sum(s);
  float* o = (k < d) ? out0 : (k < 2 * d ? out1 : out2);
  if (lane == 0 && o != nullptr) o[k % d] = s;
}

// ---------------------------------------------------------------------------------------------------------
// loss = sum_rows (logsumexp(z) - z[label]);  lse[row] kept for the backward
template <typename T>
__global__ void __launch_bounds__(kRowThreads)
ce_fwd_kernel(const T* __restrict__ z, int64_t ld, const int64_t* __restrict__ labels, int n_rows, int c,
              float* __restrict__ lse, float* __restrict__ partial) {
  __shared__ float wsum[kRowThreads / 32];
  const int lane = threadIdx.x & 31;
  const int warps = (gridDim.x * kRowThreads) >> 5;
  float acc = 0.f;
  for (int row = (blockIdx.x * kRowThreads + threadIdx.x) >> 5; row < n_rows; row += warps) {
    const T* zp = z + static_cast<int64_t>(row) * ld;
    float m = -INFINITY;
    for (int k = lane; k < c; k += 32) m = fmaxf(m, static_cast<float>(zp[k]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    float s = 0.f;
    for (int k = lane; k < c; k += 32) s += expf(static_cast<float>(zp[k]) - m);
    s = warp_sum(s);
    const float l = m + logf(s);
    if (lane == 0) {
      lse[row] = l;
      acc += l - static_cast<float>(zp[labels[row]]);
    }
  }
  if (lane == 0) wsum[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < kRowThreads / 32; ++w) s += wsum[w];
    partial[blockIdx.x] = s;
  }
}

// g[row, k] = (exp(z - lse) - [k == label]) * upstream   for row < n_rows, zero for n_rows <= row < n_total
template <typename T>
__global__ void __launch_bounds__(kRowThreads)
ce_bwd_kernel(const T* __restrict__ z, int64_t ld, const int64_t* __restrict__ labels, const float* __restrict__ lse,
              const float* __restrict__ upstream, int n_rows, int n_total, int c, T* __restrict__ g, int64_t ldg,
              float* __restrict__ partial) {
  extern __shared__ float red[];                             // [c]
  const int lane = threadIdx.x & 31;
  const int warps = (gridDim.x * kRowThreads) >> 5;
  const float up = upstream ? __ldg(upstream) : 1.f;
  for (int i = threadIdx.x; i < c; i += kRowThreads) red[i] = 0.f;
  __syncthreads();
  for (int row = (blockIdx.x * kRowThreads + threadIdx.x) >> 5; row < n_total; row += warps) {
    T* gp = g + static_cast<int64_t>(row) * ldg;
    if (row >= n_rows) {
      for (int k = lane; k < c; k += 32) gp[k] = static_cast<T>(0.f);
      continue;
    }
    const T* zp = z + static_cast<int64_t>(row) * ld;
    const float l = lse[row];
    const int lab = static_cast<int>(labels[row]);
    for (int k = lane; k < c; k += 32) {
      const float v = (expf(static_cast<float>(zp[k]) - l) - (k == lab ? 1.f : 0.f)) * up;
      const T t = static_cast<T>(v);
      gp[k] = t;
      atomicAdd(&red[k], static_cast<float>(t));             // shared-memory partial; order fixed within a warp only
    }
  }
  __syncthreads();
  float* pp = partial + static_cast<int64_t>(blockIdx.x) * c;
  for (int i = threadIdx.x; i < c; i += kRowThreads) pp[i] = red[i];
}

// ---- sub-warp versions: G lanes per row, 32 / G rows per warp at once, 16-byte vectors -----------------------
// A row of c logits is short (tens of classes): one warp per row leaves most lanes idle and serialises a row's
// load -> max -> exp -> sum -> log chain, so the kernels above are latency-bound at a fraction of HBM speed.  Here a
// row is held by G = 2^k >= ceil(c / V) lanes (NVL vectors per lane when G = 32 is not enough), the reductions are
// log2(G) shuffles, and 32 / G rows are in flight per warp.  Needs 16-byte aligned rows (checked by the caller).
template <typename T, int G, int NVL>
__global__ void __launch_bounds__(kRowThreads)
ce_fwd2_kernel(const T* __restrict__ z, int64_t ld, const int64_t* __restrict__ labels, int n_rows, int c,
               float* __restrict__ lse, float* __restrict__ partial) {
  using P = Pack<T, 16>;
  using Raw = typename P::Raw;
  constexpr int V = P::V;
  constexpr int RPW = 32 / G;
  __shared__ float wsum[kRowThreads / 32];
  const int lane = threadIdx.x & 31, lane_g = lane % G, sub = lane / G;
  const int warp = (blockIdx.x * kRowThreads + threadIdx.x) >> 5;
  const int warps = (gridDim.x * kRowThreads) >> 5;
  float acc = 0.f;
  for (int row0 = warp * RPW; row0 < n_rows; row0 += warps * RPW) {
    const bool valid = row0 + sub < n_rows;
    const int row = valid ? row0 + sub : n_rows - 1;            // idle sub-groups recompute the last row
    const T* zp = z + static_cast<int64_t>(row) * ld;
    float x[NVL][V];
    float zl = 0.f;
    if (lane_g == 0) zl = static_cast<float>(zp[__ldg(labels + row)]);
    float m = -INFINITY;
#pragma unroll
    for (int t = 0; t < NVL; ++t) {
      const int k0 = (lane_g + t * G) * V;
      if (k0 < c) {
        P::unpack(*reinterpret_cast<const Raw*>(zp + k0), x[t]);
      }
#pragma unroll
      for (int i = 0; i < V; ++i) {
        if (k0 + i >= c) x[t][i] = -INFINITY;
        m = fmaxf(m, x[t][i]);
      }
    }
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    float s = 0.f;
#pragma unroll
    for (int t = 0; t < NVL; ++t)
#pragma unroll
      for (int i = 0; i < V; ++i) s += expf(x[t][i] - m);        // exp(-inf) = 0 for the padding
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const float l = m + logf(s);
    if (lane_g == 0 && valid) {
      lse[row] = l;
      acc += l - zl;
    }
  }
  acc = warp_sum(acc);
  if (lane == 0) wsum[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < kRowThreads / 32; ++w) s += wsum[w];
    partial[blockIdx.x] = s;
  }
}

// the gradient, with deterministic column sums: a column is owned by one (lane_g, vector, element) slot, summed over
// the rows of the lane in registers, then over the sub-groups of the warp (shuffles) and the warps of the CTA (shared
// memory, fixed order)
template <typename T, int G, int NVL>
__global__ void __launch_bounds__(kRowThreads)
ce_bwd2_kernel(const T* __restrict__ z, int64_t ld, const int64_t* __restrict__ labels, const float* __restrict__ lse,
               const float* __restrict__ upstream, int n_rows, int n_total, int c, T* __restrict__ g, int64_t ldg,
               float* __restrict__ partial) {
  using P = Pack<T, 16>;
  using Raw = typename P::Raw;
  constexpr int V = P::V;
  constexpr int RPW = 32 / G;
  extern __shared__ float red[];                             // [c]
  const int lane = threadIdx.x & 31, lane_g = lane % G, sub = lane / G;
  const int warp = (blockIdx.x * kRowThreads + threadIdx.x) >> 5;
  const int warps = (gridDim.x * kRowThreads) >> 5;
  const float up = upstream ? __ldg(upstream) : 1.f;
  float col[NVL][V];
#pragma unroll
  for (int t = 0; t < NVL; ++t)
#pragma unroll
    for (int i = 0; i < V; ++i) col[t][i] = 0.f;
  for (int row0 = warp * RPW; row0 < n_total; row0 += warps * RPW) {
    const int row = row0 + sub;
    if (row >= n_total) continue;
    T* gp = g + static_cast<int64_t>(row) * ldg;
    const bool train = row < n_rows;
    const T* zp = z + static_cast<int64_t>(row) * ld;
    const float l = train ? __ldg(lse + row) : 0.f;
    const int lab = train ? static_cast<int>(__ldg(labels + row)) : -1;
#pragma unroll
    for (int t = 0; t < NVL; ++t) {
      const int k0 = (lane_g + t * G) * V;
      if (k0 >= c) continue;
      float v[V];
      if (train) {
        P::unpack(*reinterpret_cast<const Raw*>(zp + k0), v);
#pragma unroll
        for (int i = 0; i < V; ++i) v[i] = (expf(v[i] - l) - (k0 + i == lab ? 1.f : 0.f)) * up;
      } else {
#pragma unroll
        for (int i = 0; i < V; ++i) v[i] = 0.f;
      }
      const Raw packed = P::pack(v);
      if (k0 + V <= c) {
        st_vec<16>(gp + k0, packed);
      } else {                                                 // last, partial vector: element stores
        const T* pv = reinterpret_cast<const T*>(&packed);
#pragma unroll
        for (int i = 0; i < V; ++i)
          if (k0 + i < c) gp[k0 + i] = pv[i];
      }
      P::unpack(packed, v);                                    // reduce what is stored
#pragma unroll
      for (int i = 0; i < V; ++i) col[t][i] += v[i];
    }
  }
  // sub-groups of the warp hold the same columns: fold them (fixed order), then the warps of the CTA
#pragma unroll
  for (int t = 0; t < NVL; ++t)
#pragma unroll
    for (int i = 0; i < V; ++i)
#pragma unroll
      for (int o = G; o < 32; o <<= 1) col[t][i] += __shfl_xor_sync(0xffffffffu, col[t][i], o);
  for (int i = threadIdx.x; i < c; i += kRowThreads) red[i] = 0.f;
  __syncthreads();
  for (int w = 0; w < kRowThreads / 32; ++w) {
    if ((threadIdx.x >> 5) == w && sub == 0) {
#pragma unroll
      for (int t = 0; t < NVL; ++t)
#pragma unroll
        for (int i = 0; i < V; ++i) {
          const int k = (lane_g + t * G) * V + i;
          if (k < c) red[k] += col[t][i];
        }
    }
    __syncthreads();
  }
  float* pp = partial + static_cast<int64_t>(blockIdx.x) * c;
  for (int i = threadIdx.x; i < c; i += kRowThreads) pp[i] = red[i];
}

// ---------------------------------------------------------------------------------------------------------
// Multi-label (sigmoid) loss and micro-F1 counts over bit-packed 0/1 targets: label j of a row is bit j % 32 of word
// j / 32 of its lw words.  Same row mapping as the sub-warp cross-entropy kernels (G lanes per row, NVL 16-byte
// vectors per lane); a vector starts at a multiple of V, which divides 32, so its V label bits sit in one word.
template <int V>
__device__ __forceinline__ uint32_t label_bits(const uint32_t* __restrict__ y, int64_t row, int lw, int k0) {
  return (__ldg(y + row * lw + (k0 >> 5)) >> (k0 & 31)) & ((1u << V) - 1u);
}

// max(z, 0) - z * y + log1p(exp(-|z|)); the linear part is exact for y in {0, 1}
__device__ __forceinline__ float bce_term(float z, uint32_t y) {
  return fmaxf(y ? -z : z, 0.f) + log1pf(expf(-fabsf(z)));
}

// partial[block] = sum of bce_term over rows < n_rows, columns < c (fixed order: lane, warp, then CTA)
template <typename T, int G, int NVL>
__global__ void __launch_bounds__(kRowThreads)
bce_fwd_kernel(const T* __restrict__ z, int64_t ld, const uint32_t* __restrict__ y, int lw, int n_rows, int c,
               float* __restrict__ partial) {
  using P = Pack<T, 16>;
  using Raw = typename P::Raw;
  constexpr int V = P::V;
  constexpr int RPW = 32 / G;
  __shared__ float wsum[kRowThreads / 32];
  const int lane = threadIdx.x & 31, lane_g = lane % G, sub = lane / G;
  const int warp = (blockIdx.x * kRowThreads + threadIdx.x) >> 5;
  const int warps = (gridDim.x * kRowThreads) >> 5;
  float acc = 0.f;
  for (int row0 = warp * RPW; row0 < n_rows; row0 += warps * RPW) {
    const int row = row0 + sub;
    if (row >= n_rows) continue;
    const T* zp = z + static_cast<int64_t>(row) * ld;
#pragma unroll
    for (int t = 0; t < NVL; ++t) {
      const int k0 = (lane_g + t * G) * V;
      if (k0 >= c) continue;
      float v[V];
      P::unpack(*reinterpret_cast<const Raw*>(zp + k0), v);
      const uint32_t bits = label_bits<V>(y, row, lw, k0);
#pragma unroll
      for (int i = 0; i < V; ++i)
        if (k0 + i < c) acc += bce_term(v[i], (bits >> i) & 1u);
    }
  }
  acc = warp_sum(acc);
  if (lane == 0) wsum[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < kRowThreads / 32; ++w) s += wsum[w];
    partial[blockIdx.x] = s;
  }
}

// g[row, k] = (sigmoid(z) - y) * upstream for row < n_rows, zero for n_rows <= row < n_total; column sums of the stored
// gradient as in ce_bwd2_kernel (registers, then sub-groups, then the warps of the CTA in fixed order)
template <typename T, int G, int NVL>
__global__ void __launch_bounds__(kRowThreads, (NVL * (16 / sizeof(T)) <= 8) ? 4 : (NVL < 4 ? 3 : 2))
bce_bwd_kernel(const T* __restrict__ z, int64_t ld, const uint32_t* __restrict__ y, int lw,
               const float* __restrict__ upstream, int n_rows, int n_total, int c, T* __restrict__ g, int64_t ldg,
               float* __restrict__ partial) {
  using P = Pack<T, 16>;
  using Raw = typename P::Raw;
  constexpr int V = P::V;
  constexpr int RPW = 32 / G;
  extern __shared__ float red[];                             // [c]
  const int lane = threadIdx.x & 31, lane_g = lane % G, sub = lane / G;
  const int warp = (blockIdx.x * kRowThreads + threadIdx.x) >> 5;
  const int warps = (gridDim.x * kRowThreads) >> 5;
  const float up = upstream ? __ldg(upstream) : 1.f;
  float col[NVL][V];
#pragma unroll
  for (int t = 0; t < NVL; ++t)
#pragma unroll
    for (int i = 0; i < V; ++i) col[t][i] = 0.f;
  for (int row0 = warp * RPW; row0 < n_total; row0 += warps * RPW) {
    const int row = row0 + sub;
    if (row >= n_total) continue;
    T* gp = g + static_cast<int64_t>(row) * ldg;
    const bool train = row < n_rows;
    const T* zp = z + static_cast<int64_t>(row) * ld;
#pragma unroll
    for (int t = 0; t < NVL; ++t) {
      const int k0 = (lane_g + t * G) * V;
      if (k0 >= c) continue;
      float v[V];
      if (train) {
        P::unpack(*reinterpret_cast<const Raw*>(zp + k0), v);
        const uint32_t bits = label_bits<V>(y, row, lw, k0);
#pragma unroll
        for (int i = 0; i < V; ++i) v[i] = (1.f / (1.f + expf(-v[i])) - static_cast<float>((bits >> i) & 1u)) * up;
      } else {
#pragma unroll
        for (int i = 0; i < V; ++i) v[i] = 0.f;
      }
      const Raw packed = P::pack(v);
      P::unpack(packed, v);                                    // reduce what is stored
      if (k0 + V <= c) {
        st_vec<16>(gp + k0, packed);
      } else {                                                 // last, partial vector: element stores (exact)
#pragma unroll
        for (int i = 0; i < V; ++i)
          if (k0 + i < c) gp[k0 + i] = static_cast<T>(v[i]);
      }
#pragma unroll
      for (int i = 0; i < V; ++i) col[t][i] += v[i];            // columns >= c are never read out
    }
  }
#pragma unroll
  for (int t = 0; t < NVL; ++t)
#pragma unroll
    for (int i = 0; i < V; ++i)
#pragma unroll
      for (int o = G; o < 32; o <<= 1) col[t][i] += __shfl_xor_sync(0xffffffffu, col[t][i], o);
  for (int i = threadIdx.x; i < c; i += kRowThreads) red[i] = 0.f;
  __syncthreads();
  for (int w = 0; w < kRowThreads / 32; ++w) {
    if ((threadIdx.x >> 5) == w && sub == 0) {
#pragma unroll
      for (int t = 0; t < NVL; ++t)
#pragma unroll
        for (int i = 0; i < V; ++i) {
          const int k = (lane_g + t * G) * V + i;
          if (k < c) red[k] += col[t][i];
        }
    }
    __syncthreads();
  }
  float* pp = partial + static_cast<int64_t>(blockIdx.x) * c;
  for (int i = threadIdx.x; i < c; i += kRowThreads) pp[i] = red[i];
}

// counts[0..2] += micro TP, FP, FN of the prediction z > 0 over rows rows[0..n) (rows == NULL: 0..n), columns < c.
// Integer sums: the result does not depend on the order of the adds.
template <typename T, int G, int NVL>
__global__ void __launch_bounds__(kRowThreads)
f1_counts_kernel(const T* __restrict__ z, int64_t ld, const uint32_t* __restrict__ y, int lw,
                 const int32_t* __restrict__ rows, int n, int c, unsigned long long* __restrict__ counts) {
  using P = Pack<T, 16>;
  using Raw = typename P::Raw;
  constexpr int V = P::V;
  constexpr int RPW = 32 / G;
  __shared__ unsigned long long wred[3][kRowThreads / 32];
  const int lane = threadIdx.x & 31, lane_g = lane % G, sub = lane / G;
  const int warp = (blockIdx.x * kRowThreads + threadIdx.x) >> 5;
  const int warps = (gridDim.x * kRowThreads) >> 5;
  unsigned long long tp = 0, fp = 0, fn = 0;
  for (int i0 = warp * RPW; i0 < n; i0 += warps * RPW) {
    const int i = i0 + sub;
    if (i >= n) continue;
    const int64_t row = rows ? static_cast<int64_t>(__ldg(rows + i)) : static_cast<int64_t>(i);
    const T* zp = z + row * ld;
#pragma unroll
    for (int t = 0; t < NVL; ++t) {
      const int k0 = (lane_g + t * G) * V;
      if (k0 >= c) continue;
      float v[V];
      P::unpack(*reinterpret_cast<const Raw*>(zp + k0), v);
      const uint32_t bits = label_bits<V>(y, row, lw, k0);
      const uint32_t valid = (k0 + V <= c) ? ((1u << V) - 1u) : ((1u << (c - k0)) - 1u);
      uint32_t pred = 0;
#pragma unroll
      for (int e = 0; e < V; ++e) pred |= (v[e] > 0.f ? 1u : 0u) << e;
      pred &= valid;
      tp += __popc(pred & bits);
      fp += __popc(pred & ~bits);
      fn += __popc(~pred & bits & valid);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    tp += __shfl_xor_sync(0xffffffffu, tp, o);
    fp += __shfl_xor_sync(0xffffffffu, fp, o);
    fn += __shfl_xor_sync(0xffffffffu, fn, o);
  }
  if (lane == 0) {
    wred[0][threadIdx.x >> 5] = tp;
    wred[1][threadIdx.x >> 5] = fp;
    wred[2][threadIdx.x >> 5] = fn;
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    unsigned long long s = 0;
    for (int w = 0; w < kRowThreads / 32; ++w) s += wred[threadIdx.x][w];
    if (s) atomicAdd(counts + threadIdx.x, s);
  }
}

// ---------------------------------------------------------------------------------------------------------
// Dropout with a counter-based generator: keep(i) is a pure function of (seed, element index), so the backward
// regenerates the mask instead of storing it.  out = keep ? x / (1 - p) : 0.  16 random bits per element.
template <typename T>
__global__ void __launch_bounds__(256)
dropout_kernel(const T* __restrict__ x, int64_t ldx, T* __restrict__ out, int64_t ldo, int n_rows, int nvec,
               int64_t row0, DropArg drop) {
  using P = Pack<T, 16>;
  const uint32_t seed_hi = drop_seed_hi(drop);                         // device-side epoch counter (graph replay)
  const uint32_t thresh16 = drop.thresh16, seed_lo = drop.seed_lo;
  const float scale = drop.scale;
  constexpr int V = P::V;
  const int64_t total = static_cast<int64_t>(n_rows) * nvec;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int r = static_cast<int>(i / nvec), vi = static_cast<int>(i % nvec);
    float f[V];
    P::unpack(*reinterpret_cast<const typename P::Raw*>(x + static_cast<int64_t>(r) * ldx + static_cast<int64_t>(vi) * V), f);
    drop_apply<V>(f, static_cast<uint64_t>(i) + static_cast<uint64_t>(row0) * nvec, thresh16, scale, seed_lo, seed_hi);
    st_vec<16>(out + static_cast<int64_t>(r) * ldo + static_cast<int64_t>(vi) * V, P::pack(f));
  }
}

static int row_grid(int n_rows) {
  const int need = (n_rows + (kRowThreads / 32) - 1) / (kRowThreads / 32);
  return need < 148 * 8 ? (need > 0 ? need : 1) : 148 * 8;
}

}  // namespace pg

extern "C" int pg_row_grid(int32_t n_rows) { return pg::row_grid(n_rows); }

extern "C" int pg_dropout_rows(const void* x, int64_t ldx, void* out, int64_t ldo, int64_t row0, int32_t n_rows, int32_t d,
                               int dtype, const pg_drop* drop, void* stream) {
  using namespace pg;
  PG_REQUIRE(x && out && drop && drop->p >= 0.f && drop->p < 1.f, "pg_dropout: bad argument");
  const int es = elem_size(dtype), v = 16 / es;
  PG_REQUIRE(d > 0 && round_up(d, v) <= ldx && round_up(d, v) <= ldo && vec_bytes(x, ldx, es) == 16 && vec_bytes(out, ldo, es) == 16,
             "pg_dropout: rows must be 16-byte aligned and padded to the vector width");
  const int nvec = static_cast<int>(round_up(d, v) / v);
  const int64_t total = static_cast<int64_t>(n_rows) * nvec;
  if (total == 0) return PG_OK;
  const unsigned blocks = static_cast<unsigned>((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
  DropArg a = make_drop(drop);
  if (drop->p == 0.f) { a.thresh16 = 0u; a.scale = 1.f; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype == PG_F32)
    dropout_kernel<float><<<blocks, 256, 0, st>>>(static_cast<const float*>(x), ldx, static_cast<float*>(out), ldo, n_rows, nvec, row0, a);
  else
    dropout_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>(static_cast<const __nv_bfloat16*>(x), ldx, static_cast<__nv_bfloat16*>(out), ldo, n_rows, nvec, row0, a);
  PG_LAUNCH_CHECK();
  return PG_OK;
}

extern "C" int pg_dropout(const void* x, int64_t ldx, void* out, int64_t ldo, int32_t n_rows, int32_t d, int dtype,
                          float p, uint64_t seed, const uint32_t* step_dev, void* stream) {
  pg_drop dr{p, seed, step_dev, 0};
  return pg_dropout_rows(x, ldx, out, ldo, 0, n_rows, d, dtype, &dr, stream);
}

extern "C" int pg_ln_relu_fwd(const void* y, int64_t ldy, const float* gamma, const float* beta, float eps, int relu,
                              void* out, int64_t ldo, float* mean, float* rstd, int32_t n_rows, int32_t d, int dtype,
                              void* stream) {
  return pg_ln_relu_drop_fwd(y, ldy, gamma, beta, eps, relu, out, ldo, nullptr, 0, mean, rstd, n_rows, d, dtype, nullptr, stream);
}

extern "C" int pg_ln_relu_drop_fwd(const void* y, int64_t ldy, const float* gamma, const float* beta, float eps, int relu,
                                   void* out, int64_t ldo, void* out_clean, int64_t ldc, float* mean, float* rstd,
                                   int32_t n_rows, int32_t d, int dtype, const pg_drop* drop, void* stream) {
  using namespace pg;
  PG_REQUIRE(y && gamma && beta && out && mean && rstd, "pg_ln_relu_fwd: null argument");
  PG_REQUIRE(out_clean == nullptr || (ldc >= d && vec_bytes(out_clean, ldc, elem_size(dtype)) == 16),
             "pg_ln_relu_drop_fwd: out_clean rows must be 16-byte aligned");
  const DropArg da = make_drop(drop);
  const int v = 16 / elem_size(dtype);
  PG_REQUIRE(d > 0 && d % v == 0 && d / v <= 32 * kMaxVec, "pg_ln_relu_fwd: d=%d must be a multiple of %d and <= %d", d, v, 32 * kMaxVec * v);
  PG_REQUIRE(vec_bytes(y, ldy, elem_size(dtype)) == 16 && vec_bytes(out, ldo, elem_size(dtype)) == 16, "pg_ln_relu_fwd: rows must be 16-byte aligned");
  if (n_rows == 0) return PG_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int vpl = (d / v + 31) / 32;
  const bool full = d / v == 32 * vpl;
  // one resident wave (the kernels are compiled for 4 CTAs per SM, 3 when a lane holds more than 16 floats)
  const int grid = std::min(row_grid(n_rows), 148 * 4);
  // rows per warp iteration R and ring stages S by vectors per lane: R * VPL * S * 16 bytes per lane = 32 KB per CTA
#define PG_LNF__(T_, VPL_, R_, F_, S_) ln_relu_fwd_kernel<T_, VPL_, R_, F_, S_><<<grid, kRowThreads, (S_) * (R_) * (VPL_) * kRowThreads * 16, st>>>(static_cast<const T_*>(y), ldy, gamma, beta, eps, relu, static_cast<T_*>(out), ldo, mean, rstd, n_rows, d, static_cast<T_*>(out_clean), ldc, da)
#define PG_LNF_(T_, VPL_, R_, S_) do { if (full) PG_LNF__(T_, VPL_, R_, true, S_); else PG_LNF__(T_, VPL_, R_, false, S_); } while (0)
#define PG_LNF(T_) do { \
    if (g_ln_stage == 2) { if (vpl <= 1) PG_LNF_(T_, 1, 2, 4); else if (vpl <= 2) PG_LNF_(T_, 2, 1, 4); else PG_LNF_(T_, 4, 1, 2); } \
    else if (g_ln_stage == 1 && vpl <= 1) PG_LNF_(T_, 1, 2, 4); \
    else { if (vpl <= 1) PG_LNF_(T_, 1, 4, 0); else if (vpl <= 2) PG_LNF_(T_, 2, 2, 0); else PG_LNF_(T_, 4, 1, 0); } } while (0)
  if (dtype == PG_F32) PG_LNF(float); else PG_LNF(__nv_bfloat16);
#undef PG_LNF
#undef PG_LNF_
#undef PG_LNF__
  PG_LAUNCH_CHECK();
  return PG_OK;
}

extern "C" int pg_ln_relu_bwd(const void* g_out, int64_t ldg, const void* out, int64_t ldo, const void* y, int64_t ldy,
                              const float* mean, const float* rstd, const float* gamma, int relu, void* g_y,
                              int64_t ldgy, float* dgamma, float* dbeta, float* colsum, float* partial,
                              int32_t n_rows, int32_t d, int dtype, void* stream) {
  return pg_ln_relu_bwd2(g_out, ldg, out, ldo, y, ldy, mean, rstd, gamma, nullptr, relu, g_y, ldgy, dgamma, dbeta, colsum,
                         partial, n_rows, d, dtype, stream);
}

extern "C" int pg_ln_relu_bwd2(const void* g_out, int64_t ldg, const void* out, int64_t ldo, const void* y, int64_t ldy,
                               const float* mean, const float* rstd, const float* gamma, const float* beta, int relu,
                               void* g_y, int64_t ldgy, float* dgamma, float* dbeta, float* colsum, float* partial,
                               int32_t n_rows, int32_t d, int dtype, void* stream) {
  using namespace pg;
  PG_REQUIRE(g_out && y && mean && rstd && gamma && g_y && partial, "pg_ln_relu_bwd: null argument");
  PG_REQUIRE(!relu || out || beta, "pg_ln_relu_bwd: relu needs the forward output or beta");
  const int es = elem_size(dtype), v = 16 / es;
  PG_REQUIRE(d > 0 && d % v == 0 && d / v <= 32 * kMaxVec, "pg_ln_relu_bwd: unsupported d=%d", d);
  PG_REQUIRE(vec_bytes(g_out, ldg, es) == 16 && vec_bytes(y, ldy, es) == 16 && vec_bytes(g_y, ldgy, es) == 16 &&
             (!relu || beta || vec_bytes(out, ldo, es) == 16), "pg_ln_relu_bwd: rows must be 16-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t red_bytes = 3 * static_cast<size_t>(d) * sizeof(float);
  const int vpl = (d / v + 31) / 32;
  // one resident wave: every CTA pays the column-partial epilogue once (`partial` is sized for row_grid(n_rows) CTAs)
  const int grid = std::min(row_grid(n_rows), 148 * (vpl * v <= 8 ? 3 : (vpl * v <= 16 ? 2 : 1)));
  const bool full = d / v == 32 * vpl;
  const int mode = !relu ? 0 : (beta != nullptr ? 2 : 1);
#define PG_LNB___(T_, VPL_, M_, F_, S_) ln_relu_bwd_kernel<T_, VPL_, M_, F_, S_><<<grid, kRowThreads, (S_) * 2 * (VPL_) * kRowThreads * 16 + red_bytes, st>>>(static_cast<const T_*>(g_out), ldg, static_cast<const T_*>(out), ldo, static_cast<const T_*>(y), ldy, mean, rstd, gamma, static_cast<T_*>(g_y), ldgy, partial, n_rows, d, beta)
#define PG_LNB__(T_, VPL_, M_, S_) do { if (full) PG_LNB___(T_, VPL_, M_, true, S_); else PG_LNB___(T_, VPL_, M_, false, S_); } while (0)
#define PG_LNB_(T_, VPL_, S_) do { if (mode == 2) PG_LNB__(T_, VPL_, 2, S_); else if (mode == 1) PG_LNB__(T_, VPL_, 1, 0); else PG_LNB__(T_, VPL_, 0, S_); } while (0)
#define PG_LNB(T_) do { \
    if (g_ln_stage == 2) { if (vpl <= 1) PG_LNB_(T_, 1, 4); else if (vpl <= 2) PG_LNB_(T_, 2, 2); else PG_LNB_(T_, 4, 0); } \
    else if (g_ln_stage == 1 && vpl <= 1) PG_LNB_(T_, 1, 4); \
    else { if (vpl <= 1) PG_LNB_(T_, 1, 0); else if (vpl <= 2) PG_LNB_(T_, 2, 0); else PG_LNB_(T_, 4, 0); } } while (0)
  if (dtype == PG_F32) PG_LNB(float); else PG_LNB(__nv_bfloat16);
#undef PG_LNB
#undef PG_LNB_
#undef PG_LNB__
#undef PG_LNB___
  PG_LAUNCH_CHECK();
  colsum_final_kernel<<<(3 * d * 32 + 255) / 256, 256, 0, st>>>(partial, grid, 3 * d, dgamma, dbeta, colsum, d);
  PG_LAUNCH_CHECK();
  return PG_OK;
}

extern "C" int pg_ce_fwd(const void* z, int64_t ld, const int64_t* labels, int32_t n_rows, int32_t c, int dtype,
                         float* lse, float* partial, float* loss, void* stream) {
  using namespace pg;
  PG_REQUIRE(z && labels && lse && partial && loss && c > 0, "pg_ce_fwd: bad argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int grid = row_grid(n_rows);
  const int es = elem_size(dtype), nv = (c * es + 15) / 16;
  if (g_ce_subwarp && n_rows > 0 && vec_bytes(z, ld, es) == 16 && nv <= 128) {
#define PG_CEF(T_, G_, N_) ce_fwd2_kernel<T_, G_, N_><<<grid, kRowThreads, 0, st>>>(static_cast<const T_*>(z), ld, labels, n_rows, c, lse, partial)
#define PG_CEF_T(T_) do { \
    if (nv <= 1) PG_CEF(T_, 1, 1); else if (nv <= 2) PG_CEF(T_, 2, 1); else if (nv <= 4) PG_CEF(T_, 4, 1); \
    else if (nv <= 8) PG_CEF(T_, 8, 1); else if (nv <= 16) PG_CEF(T_, 16, 1); else if (nv <= 32) PG_CEF(T_, 32, 1); \
    else if (nv <= 64) PG_CEF(T_, 32, 2); else PG_CEF(T_, 32, 4); } while (0)
    if (dtype == PG_F32) PG_CEF_T(float); else PG_CEF_T(__nv_bfloat16);
#undef PG_CEF_T
#undef PG_CEF
  } else if (dtype == PG_F32) {
    ce_fwd_kernel<float><<<grid, kRowThreads, 0, st>>>(static_cast<const float*>(z), ld, labels, n_rows, c, lse, partial);
  } else {
    ce_fwd_kernel<__nv_bfloat16><<<grid, kRowThreads, 0, st>>>(static_cast<const __nv_bfloat16*>(z), ld, labels, n_rows, c, lse, partial);
  }
  PG_LAUNCH_CHECK();
  colsum_final_kernel<<<1, 32, 0, st>>>(partial, grid, 1, loss, nullptr, nullptr, 1);
  PG_LAUNCH_CHECK();
  return PG_OK;
}

extern "C" int pg_ce_bwd(const void* z, int64_t ld, const int64_t* labels, const float* lse, const float* upstream,
                         int32_t n_rows, int32_t n_total, int32_t c, int dtype, void* g, int64_t ldg, float* colsum,
                         float* partial, void* stream) {
  using namespace pg;
  PG_REQUIRE(z && labels && lse && g && partial && c > 0 && n_total >= n_rows, "pg_ce_bwd: bad argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int grid = row_grid(n_total);
  const size_t smem = static_cast<size_t>(c) * sizeof(float);
  const int es = elem_size(dtype), nv = (c * es + 15) / 16;
  if (g_ce_subwarp && vec_bytes(z, ld, es) == 16 && vec_bytes(g, ldg, es) == 16 && nv <= 128) {
#define PG_CEB(T_, G_, N_) ce_bwd2_kernel<T_, G_, N_><<<grid, kRowThreads, smem, st>>>(static_cast<const T_*>(z), ld, labels, lse, upstream, n_rows, n_total, c, static_cast<T_*>(g), ldg, partial)
#define PG_CEB_T(T_) do { \
    if (nv <= 1) PG_CEB(T_, 1, 1); else if (nv <= 2) PG_CEB(T_, 2, 1); else if (nv <= 4) PG_CEB(T_, 4, 1); \
    else if (nv <= 8) PG_CEB(T_, 8, 1); else if (nv <= 16) PG_CEB(T_, 16, 1); else if (nv <= 32) PG_CEB(T_, 32, 1); \
    else if (nv <= 64) PG_CEB(T_, 32, 2); else PG_CEB(T_, 32, 4); } while (0)
    if (dtype == PG_F32) PG_CEB_T(float); else PG_CEB_T(__nv_bfloat16);
#undef PG_CEB_T
#undef PG_CEB
  } else if (dtype == PG_F32) {
    ce_bwd_kernel<float><<<grid, kRowThreads, smem, st>>>(static_cast<const float*>(z), ld, labels, lse, upstream, n_rows, n_total, c, static_cast<float*>(g), ldg, partial);
  } else {
    ce_bwd_kernel<__nv_bfloat16><<<grid, kRowThreads, smem, st>>>(static_cast<const __nv_bfloat16*>(z), ld, labels, lse, upstream, n_rows, n_total, c, static_cast<__nv_bfloat16*>(g), ldg, partial);
  }
  PG_LAUNCH_CHECK();
  if (colsum != nullptr) {
    colsum_final_kernel<<<(c * 32 + 255) / 256, 256, 0, st>>>(partial, grid, c, colsum, nullptr, nullptr, c);
    PG_LAUNCH_CHECK();
  }
  return PG_OK;
}

namespace pg {
// Columns one launch of the multi-label kernels covers: 32 lanes x 4 vectors of 16 bytes (fp32 512, bf16 1024 classes,
// the row width the cross-entropy kernels keep in registers).  Wider rows are processed in chunks of this many columns,
// a multiple of 32, so a chunk starts on a label word.
static int ml_chunk(int es) { return 32 * 4 * (16 / es); }

static const char* ml_check(const void* z, int64_t ld, const uint32_t* ybits, int32_t lw, int32_t c, int dtype) {
  if (dtype != PG_F32 && dtype != PG_BF16) return "dtype must be PG_F32 or PG_BF16";
  if (c <= 0) return "c must be >= 1";
  if (z == nullptr || ybits == nullptr) return "null logits or labels";
  if (lw < (c + 31) / 32) return "lw must be >= ceil(c / 32)";
  if (ld < c || vec_bytes(z, ld, elem_size(dtype)) != 16) return "logit rows must be 16-byte aligned with ld >= c";
  return nullptr;
}
}  // namespace pg

#define PG_ML_DISPATCH(KERNEL, T_, NV_, GRID_, SMEM_, ST_, ...) do { \
    if ((NV_) <= 1) KERNEL<T_, 1, 1><<<GRID_, kRowThreads, SMEM_, ST_>>>(__VA_ARGS__); \
    else if ((NV_) <= 2) KERNEL<T_, 2, 1><<<GRID_, kRowThreads, SMEM_, ST_>>>(__VA_ARGS__); \
    else if ((NV_) <= 4) KERNEL<T_, 4, 1><<<GRID_, kRowThreads, SMEM_, ST_>>>(__VA_ARGS__); \
    else if ((NV_) <= 8) KERNEL<T_, 8, 1><<<GRID_, kRowThreads, SMEM_, ST_>>>(__VA_ARGS__); \
    else if ((NV_) <= 16) KERNEL<T_, 16, 1><<<GRID_, kRowThreads, SMEM_, ST_>>>(__VA_ARGS__); \
    else if ((NV_) <= 32) KERNEL<T_, 32, 1><<<GRID_, kRowThreads, SMEM_, ST_>>>(__VA_ARGS__); \
    else if ((NV_) <= 64) KERNEL<T_, 32, 2><<<GRID_, kRowThreads, SMEM_, ST_>>>(__VA_ARGS__); \
    else KERNEL<T_, 32, 4><<<GRID_, kRowThreads, SMEM_, ST_>>>(__VA_ARGS__); } while (0)

extern "C" int pg_bce_fwd(const void* z, int64_t ld, const uint32_t* ybits, int32_t lw, int32_t n_rows, int32_t c,
                          int dtype, float* partial, float* loss, void* stream) {
  using namespace pg;
  const char* bad = ml_check(z, ld, ybits, lw, c, dtype);
  PG_REQUIRE(bad == nullptr, "pg_bce_fwd: %s (c=%d, lw=%d, ld=%lld)", bad, c, lw, static_cast<long long>(ld));
  PG_REQUIRE(partial && loss && n_rows >= 0, "pg_bce_fwd: bad argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int grid = row_grid(n_rows), es = elem_size(dtype), cw = ml_chunk(es);
  int n_chunks = 0;
  for (int c0 = 0; c0 < c; c0 += cw, ++n_chunks) {
    const int cc = std::min(cw, c - c0), nv = (cc * es + 15) / 16;
    float* pp = partial + static_cast<int64_t>(n_chunks) * grid;
    if (dtype == PG_F32)
      PG_ML_DISPATCH(bce_fwd_kernel, float, nv, grid, 0, st, static_cast<const float*>(z) + c0, ld, ybits + c0 / 32, lw, n_rows, cc, pp);
    else
      PG_ML_DISPATCH(bce_fwd_kernel, __nv_bfloat16, nv, grid, 0, st, static_cast<const __nv_bfloat16*>(z) + c0, ld, ybits + c0 / 32, lw, n_rows, cc, pp);
    PG_LAUNCH_CHECK();
  }
  colsum_final_kernel<<<1, 32, 0, st>>>(partial, grid * n_chunks, 1, loss, nullptr, nullptr, 1);
  PG_LAUNCH_CHECK();
  return PG_OK;
}

extern "C" int pg_bce_bwd(const void* z, int64_t ld, const uint32_t* ybits, int32_t lw, const float* upstream,
                          int32_t n_rows, int32_t n_total, int32_t c, int dtype, void* g, int64_t ldg, float* colsum,
                          float* partial, void* stream) {
  using namespace pg;
  const char* bad = ml_check(z, ld, ybits, lw, c, dtype);
  PG_REQUIRE(bad == nullptr, "pg_bce_bwd: %s (c=%d, lw=%d, ld=%lld)", bad, c, lw, static_cast<long long>(ld));
  PG_REQUIRE(g && partial && n_rows >= 0 && n_total >= n_rows, "pg_bce_bwd: bad argument");
  const int es = elem_size(dtype);
  PG_REQUIRE(ldg >= c && vec_bytes(g, ldg, es) == 16, "pg_bce_bwd: gradient rows must be 16-byte aligned with ldg >= c");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int grid = row_grid(n_total), cw = ml_chunk(es);
  for (int c0 = 0; c0 < c; c0 += cw) {
    const int cc = std::min(cw, c - c0), nv = (cc * es + 15) / 16;
    const size_t smem = static_cast<size_t>(cc) * sizeof(float);
    float* pp = partial + static_cast<int64_t>(grid) * c0;
    if (dtype == PG_F32)
      PG_ML_DISPATCH(bce_bwd_kernel, float, nv, grid, smem, st, static_cast<const float*>(z) + c0, ld, ybits + c0 / 32, lw, upstream, n_rows, n_total, cc, static_cast<float*>(g) + c0, ldg, pp);
    else
      PG_ML_DISPATCH(bce_bwd_kernel, __nv_bfloat16, nv, grid, smem, st, static_cast<const __nv_bfloat16*>(z) + c0, ld, ybits + c0 / 32, lw, upstream, n_rows, n_total, cc, static_cast<__nv_bfloat16*>(g) + c0, ldg, pp);
    PG_LAUNCH_CHECK();
    if (colsum != nullptr) {
      colsum_final_kernel<<<(cc * 32 + 255) / 256, 256, 0, st>>>(pp, grid, cc, colsum + c0, nullptr, nullptr, cc);
      PG_LAUNCH_CHECK();
    }
  }
  return PG_OK;
}

extern "C" int pg_f1_counts(const void* z, int64_t ld, const uint32_t* ybits, int32_t lw, const int32_t* rows, int32_t n,
                            int32_t c, int dtype, unsigned long long* counts, void* stream) {
  using namespace pg;
  const char* bad = ml_check(z, ld, ybits, lw, c, dtype);
  PG_REQUIRE(bad == nullptr, "pg_f1_counts: %s (c=%d, lw=%d, ld=%lld)", bad, c, lw, static_cast<long long>(ld));
  PG_REQUIRE(counts && n >= 0, "pg_f1_counts: bad argument");
  if (n == 0) return PG_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int grid = row_grid(n), es = elem_size(dtype), cw = ml_chunk(es);
  for (int c0 = 0; c0 < c; c0 += cw) {
    const int cc = std::min(cw, c - c0), nv = (cc * es + 15) / 16;
    if (dtype == PG_F32)
      PG_ML_DISPATCH(f1_counts_kernel, float, nv, grid, 0, st, static_cast<const float*>(z) + c0, ld, ybits + c0 / 32, lw, rows, n, cc, counts);
    else
      PG_ML_DISPATCH(f1_counts_kernel, __nv_bfloat16, nv, grid, 0, st, static_cast<const __nv_bfloat16*>(z) + c0, ld, ybits + c0 / 32, lw, rows, n, cc, counts);
    PG_LAUNCH_CHECK();
  }
  return PG_OK;
}
#undef PG_ML_DISPATCH
