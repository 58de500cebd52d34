// Hyper-Connections pre-branch kernels for d <= 1024, fourth generation (forward and backward of
//     depth connection of the previous branch -> width connection of this branch -> pre-LayerNorm).
//
// One CTA of 128 threads works on one token at a time (grid stride over tokens); thread t owns the 8 channels
// [8t, 8t+8) of every row, so every row access is one 16-B vector per thread.  The kernels are instruction-issue
// bound, so the per-token work is cut down to what the arithmetic needs:
//   * packed fp32 pairs (fma.rn.f32x2) for all per-channel math;
//   * every per-token dot product of a pass goes through ONE warp reduce-scatter (31 shuffles for 32 sums instead
//     of 5 per sum) and one CTA barrier; all shuffles run with the whole warp converged;
//   * backward: the token's inputs are staged in shared memory with cp.async, double-buffered (the next token's
//     copies run under this token's math), so the second pass reads shared memory, never L2 / HBM;
//   * backward: the per-channel parameter gradients (gamma_hc, dyn_alpha, dyn_beta, ln_gamma) are accumulated in
//     fp32 registers of the thread that owns the channel, written once per CTA to a [grid, d, 8] partial buffer and
//     reduced in a fixed order by param_finish_kernel: bitwise deterministic, no atomics.
// Reference semantics: hyper_connections.HyperConnections width/depth connections as called from
// audiolm_pytorch.py:446-454, 524-551 (third-party dependency, restated in oracle/third_party.py).
#pragma once
#include "alm_common.cuh"

namespace alm {
namespace hc4 {

constexpr int S = 4, T = 5;
constexpr int AUX = S * T + S + S + (S * T + S) + 2;  // ta[20] tb[4] inv[4] z[24] (pre-tanh) mean rstd
constexpr int THREADS = 128, WARPS = THREADS / 32;
constexpr int Z_OFF = S * T + S + S;  // aux offset of the pre-activations z
constexpr int NSMALL = 8;             // per stream: d static_alpha[5], d static_beta, d alpha_scale, d beta_scale
constexpr int FWD_CTAS_PER_SM = 5, BWD_CTAS_PER_SM = 3;

struct Params {
  const float* gamma_hc; const float* dyn_alpha; const float* dyn_beta; const float* static_alpha;
  const float* static_beta; const float* alpha_scale; const float* beta_scale; const float* ln_gamma;
};
struct Grads {
  float* gamma_hc; float* dyn_alpha; float* dyn_beta; float* static_alpha; float* static_beta;
  float* alpha_scale; float* beta_scale; float* ln_gamma;
};

__device__ __forceinline__ uint32_t pk(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ float tanh_fast(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));  // MUFU.TANH, rel. err ~2^-11: far below the bf16 noise floor
  return y;
}
__device__ __forceinline__ float2 dup2(float a) { return make_float2(a, a); }
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ float2 add2(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 mul2(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 bf2(uint32_t u) { return make_float2(bf16_lo(u), bf16_hi(u)); }
__device__ __forceinline__ void unpack8p(const uint4& u, float2 (&f)[4]) {
  f[0] = bf2(u.x); f[1] = bf2(u.y); f[2] = bf2(u.z); f[3] = bf2(u.w);
}
__device__ __forceinline__ uint4 pack8p(const float2 (&f)[4]) {
  return make_uint4(pk(f[0].x, f[0].y), pk(f[1].x, f[1].y), pk(f[2].x, f[2].y), pk(f[3].x, f[3].y));
}
__device__ __forceinline__ void lds8p(const float* p, float2 (&f)[4]) {
  const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
  f[0] = make_float2(a.x, a.y); f[1] = make_float2(a.z, a.w); f[2] = make_float2(b.x, b.y); f[3] = make_float2(b.z, b.w);
}

// Warp reduce-scatter of N (power of two <= 32) per-lane values: returns, in lane l, the warp total of value l % N.
// N - 1 + log2(32 / N) shuffles in all, every lane taking part in every one.
template <int N>
__device__ __forceinline__ float warp_scatter_sum(float (&v)[N], int lane) {
#pragma unroll
  for (int h = N / 2; h >= 1; h >>= 1) {
    const bool up = (lane & h) != 0;
#pragma unroll
    for (int i = 0; i < h; ++i) {
      const float send = up ? v[i] : v[i + h];
      const float keep = up ? v[i + h] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, h);
    }
  }
  float r = v[0];
#pragma unroll
  for (int o = N; o < 32; o <<= 1) r += __shfl_xor_sync(0xffffffffu, r, o);
  return r;
}

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem)), "l"(gmem)
               : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_prev() { asm volatile("cp.async.wait_group 1;" ::: "memory"); }

// smem params: [0,d) ln_gamma; [d, 7d) P_c * g1 for c = dyn_alpha[:,0..4], dyn_beta;  g1 = (gamma + 1) * sqrt(d)
__device__ __forceinline__ void stage_param_rows(float* sm, const Params& p, int d) {
  const float sqrt_d = sqrtf((float)d);
  for (int i = threadIdx.x; i < d; i += blockDim.x) {
    const float g1 = (p.gamma_hc[i] + 1.f) * sqrt_d;
    sm[i] = p.ln_gamma[i];
#pragma unroll
    for (int t = 0; t < T; ++t) sm[(1 + t) * d + i] = g1 * p.dyn_alpha[(size_t)i * T + t];
    sm[(1 + T) * d + i] = g1 * p.dyn_beta[i];
  }
}
inline size_t param_smem(int d) { return (size_t)7 * d * sizeof(float); }

// ------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------
template <bool EXPAND>
__global__ void __launch_bounds__(THREADS, FWD_CTAS_PER_SM)
pre_fwd_kernel(const __nv_bfloat16* __restrict__ R_in, const __nv_bfloat16* __restrict__ Y,
               const float* __restrict__ beta_prev, const float* __restrict__ x_expand, Params prm,
               __nv_bfloat16* __restrict__ R_out, __nv_bfloat16* __restrict__ bin, __nv_bfloat16* __restrict__ xn,
               float* __restrict__ beta_out, float* __restrict__ aux, int M, int d) {
  extern __shared__ float sm[];
  __shared__ float mail[WARPS][32], mail2[WARPS][2];
  stage_param_rows(sm, prm, d);
  __syncthreads();
  const int lt = threadIdx.x, warp = lt >> 5, lane = lt & 31;
  const int c0 = lt * 8;
  const bool act = c0 < d;
  const float inv_d = 1.f / (float)d;
  // lane l < 24 finishes dynamic weight l (l = s*5+t: alpha, 20+s: beta); its stream is s(l)
  const int my_s = lane < S * T ? lane / T : (lane < S * T + S ? lane - S * T : 0);
  const float my_scale = lane < S * T ? *prm.alpha_scale : *prm.beta_scale;
  const float my_static = lane < S * T ? prm.static_alpha[lane] : (lane < S * T + S ? prm.static_beta[lane - S * T] : 0.f);

  for (int m = blockIdx.x; m < M; m += gridDim.x) {
    {  // pull the next token of this CTA towards L2 (one thread per 128-B line)
      const int mn = m + gridDim.x;
      if (mn < M && act && (lt & 7) == 0) {
        if (EXPAND) {
          prefetch_l2(x_expand + (size_t)mn * d + c0);
          prefetch_l2(x_expand + (size_t)mn * d + c0 + 32);
        } else {
          prefetch_l2(Y + (size_t)mn * d + c0);
#pragma unroll
          for (int s = 0; s < S; ++s) prefetch_l2(R_in + ((size_t)mn * S + s) * d + c0);
        }
      }
    }
    float2 r[S][4];
    if (act) {
      if (EXPAND) {
        float2 x[4];
        const float4 a = *reinterpret_cast<const float4*>(x_expand + (size_t)m * d + c0);
        const float4 b = *reinterpret_cast<const float4*>(x_expand + (size_t)m * d + c0 + 4);
        x[0] = make_float2(a.x, a.y); x[1] = make_float2(a.z, a.w); x[2] = make_float2(b.x, b.y); x[3] = make_float2(b.z, b.w);
#pragma unroll
        for (int s = 0; s < S; ++s)
#pragma unroll
          for (int p = 0; p < 4; ++p) r[s][p] = x[p];
      } else {
        float2 y[4];
        unpack8p(*reinterpret_cast<const uint4*>(Y + (size_t)m * d + c0), y);
        const float4 bp4 = *reinterpret_cast<const float4*>(beta_prev + (size_t)m * S);
        const float bp[S] = {bp4.x, bp4.y, bp4.z, bp4.w};
#pragma unroll
        for (int s = 0; s < S; ++s) {
          float2 rv[4];
          unpack8p(*reinterpret_cast<const uint4*>(R_in + ((size_t)m * S + s) * d + c0), rv);
#pragma unroll
          for (int p = 0; p < 4; ++p) r[s][p] = fma2(dup2(bp[s]), y[p], rv[p]);
        }
      }
    } else {
#pragma unroll
      for (int s = 0; s < S; ++s)
#pragma unroll
        for (int p = 0; p < 4; ++p) r[s][p] = make_float2(0.f, 0.f);
    }
    // one reduction for the 24 raw dots <R_s, g1*P_c> and the 4 squared norms (the dots do not wait for 1/|R_s|)
    float red[32];
    {
      float2 acc[S * T + S + S];
#pragma unroll
      for (int i = 0; i < S * T + S + S; ++i) acc[i] = make_float2(0.f, 0.f);
      if (act) {
#pragma unroll
        for (int c = 0; c < T + 1; ++c) {
          float2 pg[4];
          lds8p(sm + (1 + c) * d + c0, pg);
#pragma unroll
          for (int s = 0; s < S; ++s) {
            const int i = c < T ? s * T + c : S * T + s;
#pragma unroll
            for (int p = 0; p < 4; ++p) acc[i] = fma2(r[s][p], pg[p], acc[i]);
          }
        }
#pragma unroll
        for (int s = 0; s < S; ++s)
#pragma unroll
          for (int p = 0; p < 4; ++p) acc[S * T + S + s] = fma2(r[s][p], r[s][p], acc[S * T + S + s]);
      }
#pragma unroll
      for (int i = 0; i < S * T + S + S; ++i) red[i] = acc[i].x + acc[i].y;
#pragma unroll
      for (int i = S * T + S + S; i < 32; ++i) red[i] = 0.f;
    }
    mail[warp][lane] = warp_scatter_sum<32>(red, lane);
    __syncthreads();
    // every warp finishes the 24 dynamic weights redundantly (lane l owns weight l), then broadcasts alpha
    float tot = mail[0][lane];
#pragma unroll
    for (int w = 1; w < WARPS; ++w) tot += mail[w][lane];
    const float inv_l = 1.f / fmaxf(sqrtf(tot), 1e-12f);  // meaningful in lanes 24..27 (stream lane - 24)
    const float my_inv = __shfl_sync(0xffffffffu, inv_l, S * T + S + my_s);
    const float z = tot * my_inv;
    const float th = tanh_fast(z);
    const float wgt = fmaf(th, my_scale, my_static);  // alpha[s][t] (lane s*5+t) or beta[s] (lane 20+s)
    if (warp == 0) {
      float* a = aux + (size_t)m * AUX;
      if (lane < S * T + S) {
        a[lane] = th;
        a[Z_OFF + lane] = z;
      } else if (lane < S * T + S + S) {
        a[lane] = inv_l;  // inv[s] at S*T+S+s
      }
      if (lane >= S * T && lane < S * T + S) beta_out[(size_t)m * S + lane - S * T] = wgt;
    }
    float alpha[S][T];
#pragma unroll
    for (int s = 0; s < S; ++s)
#pragma unroll
      for (int t = 0; t < T; ++t) alpha[s][t] = __shfl_sync(0xffffffffu, wgt, s * T + t);
    // mixed streams out; branch input kept for the LayerNorm
    float2 bi[4];
    float2 st2[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
#pragma unroll
    for (int t = 0; t < T; ++t) {
      float2 o[4];
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        float2 a = mul2(dup2(alpha[0][t]), r[0][p]);
#pragma unroll
        for (int s = 1; s < S; ++s) a = fma2(dup2(alpha[s][t]), r[s][p], a);
        o[p] = a;
      }
      if (t == 0) {
#pragma unroll
        for (int p = 0; p < 4; ++p) {
          bi[p] = o[p];
          st2[0] = add2(st2[0], o[p]);
          st2[1] = fma2(o[p], o[p], st2[1]);
        }
        if (act) *reinterpret_cast<uint4*>(bin + (size_t)m * d + c0) = pack8p(o);
      } else if (act) {
        *reinterpret_cast<uint4*>(R_out + ((size_t)m * S + (t - 1)) * d + c0) = pack8p(o);
      }
    }
    float st[2] = {st2[0].x + st2[0].y, st2[1].x + st2[1].y};
    const float st_l = warp_scatter_sum<2>(st, lane);
    if (lane < 2) mail2[warp][lane] = st_l;
    __syncthreads();
    float s1 = mail2[0][0], s2 = mail2[0][1];
#pragma unroll
    for (int w = 1; w < WARPS; ++w) { s1 += mail2[w][0]; s2 += mail2[w][1]; }
    const float mean = s1 * inv_d;
    const float rstd = rsqrtf(fmaxf(s2 * inv_d - mean * mean, 0.f) + 1e-5f);
    if (act) {
      float2 lg[4], o[4];
      lds8p(sm + c0, lg);
      const float2 rs2 = dup2(rstd), nmr = dup2(-mean * rstd);
#pragma unroll
      for (int p = 0; p < 4; ++p) o[p] = mul2(fma2(bi[p], rs2, nmr), lg[p]);
      *reinterpret_cast<uint4*>(xn + (size_t)m * d + c0) = pack8p(o);
    }
    if (lt == 0) {
      aux[(size_t)m * AUX + AUX - 2] = mean;
      aux[(size_t)m * AUX + AUX - 1] = rstd;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// backward
// ------------------------------------------------------------------------------------------------
// staged 16-B chunks per thread and token: R_in[4] Y dR_out[4] dxn dbin_extra, or x (fp32, 2 chunks) dR_out[4] dxn
// dbin_extra when expanding.  Layout [chunk][THREADS] uint4: a warp's accesses are conflict-free.
template <bool EXPAND> struct Stage;
template <> struct Stage<false> { static constexpr int R = 0, Y = 4, DR = 5, DX = 9, EX = 10, N = 11; };
template <> struct Stage<true> { static constexpr int X = 0, DR = 2, DX = 6, EX = 7, N = 8; };

inline size_t bwd_smem(int d, bool expand) {
  return param_smem(d) + (size_t)2 * (expand ? Stage<true>::N : Stage<false>::N) * THREADS * 16;
}

template <bool EXPAND>
__device__ __forceinline__ void stage_token(uint4* buf, int m, int lt, int c0, int d, const __nv_bfloat16* R_in,
                                            const __nv_bfloat16* Y, const float* x_expand, const __nv_bfloat16* dR_out,
                                            const __nv_bfloat16* dxn, const __nv_bfloat16* dbin_extra) {
  using St = Stage<EXPAND>;
  if (EXPAND) {
    cp_async16(buf + Stage<true>::X * THREADS + lt, x_expand + (size_t)m * d + c0);
    cp_async16(buf + (Stage<true>::X + 1) * THREADS + lt, x_expand + (size_t)m * d + c0 + 4);
  } else {
#pragma unroll
    for (int s = 0; s < S; ++s) cp_async16(buf + (Stage<false>::R + s) * THREADS + lt, R_in + ((size_t)m * S + s) * d + c0);
    cp_async16(buf + Stage<false>::Y * THREADS + lt, Y + (size_t)m * d + c0);
  }
#pragma unroll
  for (int s = 0; s < S; ++s) cp_async16(buf + (St::DR + s) * THREADS + lt, dR_out + ((size_t)m * S + s) * d + c0);
  cp_async16(buf + St::DX * THREADS + lt, dxn + (size_t)m * d + c0);
  if (dbin_extra != nullptr) cp_async16(buf + St::EX * THREADS + lt, dbin_extra + (size_t)m * d + c0);
}

// R_s of the staged token: R_in + beta_prev (x) Y, or x for every stream
template <bool EXPAND>
__device__ __forceinline__ void staged_r(const uint4* buf, int lt, const float (&bp)[S], float2 (&r)[S][4], float2 (&y)[4]) {
  if (EXPAND) {
    const float4 a = reinterpret_cast<const float4*>(buf)[Stage<true>::X * THREADS + lt];
    const float4 b = reinterpret_cast<const float4*>(buf)[(Stage<true>::X + 1) * THREADS + lt];
    const float2 x[4] = {make_float2(a.x, a.y), make_float2(a.z, a.w), make_float2(b.x, b.y), make_float2(b.z, b.w)};
#pragma unroll
    for (int s = 0; s < S; ++s)
#pragma unroll
      for (int p = 0; p < 4; ++p) r[s][p] = x[p];
#pragma unroll
    for (int p = 0; p < 4; ++p) y[p] = make_float2(0.f, 0.f);
  } else {
    unpack8p(buf[Stage<false>::Y * THREADS + lt], y);
#pragma unroll
    for (int s = 0; s < S; ++s) {
      float2 rv[4];
      unpack8p(buf[(Stage<false>::R + s) * THREADS + lt], rv);
#pragma unroll
      for (int p = 0; p < 4; ++p) r[s][p] = fma2(dup2(bp[s]), y[p], rv[p]);
    }
  }
}

// Outputs dR_in [M,S,d], dY [M,d], dbeta_prev [M,S] (or dx_expand [M,d] fp32 = dx_scale * sum_s dR_s), and the
// CTA's parameter-gradient partial sums: part [gridDim.x][d][8] (dyn_alpha G[0..4], dyn_beta G[5], ln_gamma, 0) and
// part_small [gridDim.x][S][NSMALL].  G[c, j] = sum_{tokens, s} R_s[c] * inv_s * dz_s[j] (fp32, never rounded).
template <bool EXPAND>
__global__ void __launch_bounds__(THREADS, BWD_CTAS_PER_SM)
pre_bwd_kernel(const __nv_bfloat16* __restrict__ R_in, const __nv_bfloat16* __restrict__ Y,
               const float* __restrict__ beta_prev, const float* __restrict__ x_expand, Params prm,
               const float* __restrict__ aux, const __nv_bfloat16* __restrict__ dR_out,
               const __nv_bfloat16* __restrict__ dxn, const __nv_bfloat16* __restrict__ dbin_extra,
               const float* __restrict__ dbeta, __nv_bfloat16* __restrict__ dR_in, __nv_bfloat16* __restrict__ dY,
               float* __restrict__ dbeta_prev, float* __restrict__ dx_expand, float dx_scale,
               float* __restrict__ part, float* __restrict__ part_small, int M, int d) {
  using St = Stage<EXPAND>;
  extern __shared__ float sm[];
  __shared__ float mail[WARPS][34], mail2[WARPS][S];
  uint4* stage = reinterpret_cast<uint4*>(sm + 7 * d);  // [2][St::N][THREADS]
  stage_param_rows(sm, prm, d);
  const int lt = threadIdx.x, warp = lt >> 5, lane = lt & 31;
  const int c0 = lt * 8;
  const bool act = c0 < d;
  const float inv_d = 1.f / (float)d;
  const float a_scale = *prm.alpha_scale, b_scale = *prm.beta_scale;
  float astat0[S];
#pragma unroll
  for (int s = 0; s < S; ++s) astat0[s] = prm.static_alpha[s * T];
  // lane s < 4 of every warp finishes stream s's per-token scalars (lanes >= 4 compute a copy of stream 0's)
  const int ls = lane < S ? lane : 0;

  float2 gacc[T + 2][4];  // per owned channel pair: G[0..5], d ln_gamma
#pragma unroll
  for (int j = 0; j < T + 2; ++j)
#pragma unroll
    for (int p = 0; p < 4; ++p) gacc[j][p] = make_float2(0.f, 0.f);
  float small[NSMALL];
#pragma unroll
  for (int k = 0; k < NSMALL; ++k) small[k] = 0.f;

  int m = blockIdx.x;
  if (m < M && act) stage_token<EXPAND>(stage, m, lt, c0, d, R_in, Y, x_expand, dR_out, dxn, dbin_extra);
  cp_async_commit();
  // per-token scalars every thread needs, loaded one token ahead
  float nx_mean = 0.f, nx_rstd = 0.f, nx_ta0[S], nx_bp[S];
  auto load_scalars = [&](int mm) {
    const float* a = aux + (size_t)mm * AUX;
    nx_mean = a[AUX - 2];
    nx_rstd = a[AUX - 1];
#pragma unroll
    for (int s = 0; s < S; ++s) {
      nx_ta0[s] = a[s * T];
      nx_bp[s] = EXPAND ? 0.f : beta_prev[(size_t)mm * S + s];
    }
  };
  if (m < M) load_scalars(m);
  __syncthreads();  // params staged

  for (int it = 0; m < M; m += gridDim.x, ++it) {
    const uint4* buf = stage + (it & 1) * (St::N * THREADS);
    {
      const int mn = m + gridDim.x;
      if (mn < M && act)
        stage_token<EXPAND>(stage + ((it + 1) & 1) * (St::N * THREADS), mn, lt, c0, d, R_in, Y, x_expand, dR_out,
                            dxn, dbin_extra);
      cp_async_commit();
    }
    const float mean = nx_mean, rstd = nx_rstd;
    float bp[S], alpha0[S];
#pragma unroll
    for (int s = 0; s < S; ++s) {
      bp[s] = nx_bp[s];
      alpha0[s] = fmaf(nx_ta0[s], a_scale, astat0[s]);
    }
    // stream-owner lanes: this token's per-stream aux entries (used after the reduction)
    const float* a = aux + (size_t)m * AUX;
    float ta[T], zs[T + 1];
#pragma unroll
    for (int t = 0; t < T; ++t) { ta[t] = a[ls * T + t]; zs[t] = a[Z_OFF + ls * T + t]; }
    zs[T] = a[Z_OFF + S * T + ls];
    const float tb = a[S * T + ls], inv = a[S * T + S + ls], dbe = dbeta[(size_t)m * S + ls];
    {
      const int mn = m + gridDim.x;
      if (mn < M) load_scalars(mn);
    }
    cp_async_wait_prev();

    // ---------------- pass 1: every per-token sum in one reduction ----------------
    // red: 0+s sum gl*R_s | 4+s sum R_s | 8+s sum xhat*R_s | 12+s sum ex*R_s | 16+4s+(t-1) sum dR_out[t-1]*R_s;
    //      red2: sum gl, sum gl*xhat      (gl = dxn * ln_gamma, xhat = normalised branch input, ex = dbin_extra)
    float red[32], lnr[2];
    {
      float2 acc[32], lacc[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
#pragma unroll
      for (int i = 0; i < 32; ++i) acc[i] = make_float2(0.f, 0.f);
      if (act) {
        float2 r[S][4], y[4], dx[4], ex[4], lg[4];
        staged_r<EXPAND>(buf, lt, bp, r, y);
        unpack8p(buf[St::DX * THREADS + lt], dx);
        if (dbin_extra != nullptr) {
          unpack8p(buf[St::EX * THREADS + lt], ex);
        } else {
#pragma unroll
          for (int p = 0; p < 4; ++p) ex[p] = make_float2(0.f, 0.f);
        }
        lds8p(sm + c0, lg);
        const float2 rstd2 = dup2(rstd), nmr2 = dup2(-mean * rstd);
#pragma unroll
        for (int p = 0; p < 4; ++p) {
          float2 bsum = mul2(dup2(alpha0[0]), r[0][p]);
#pragma unroll
          for (int s = 1; s < S; ++s) bsum = fma2(dup2(alpha0[s]), r[s][p], bsum);
          const float2 xh = fma2(bsum, rstd2, nmr2);
          const float2 gl = mul2(dx[p], lg[p]);
          gacc[T + 1][p] = fma2(dx[p], xh, gacc[T + 1][p]);
          lacc[0] = add2(lacc[0], gl);
          lacc[1] = fma2(gl, xh, lacc[1]);
#pragma unroll
          for (int s = 0; s < S; ++s) {
            acc[s] = fma2(gl, r[s][p], acc[s]);
            acc[4 + s] = add2(acc[4 + s], r[s][p]);
            acc[8 + s] = fma2(xh, r[s][p], acc[8 + s]);
            acc[12 + s] = fma2(ex[p], r[s][p], acc[12 + s]);
          }
        }
#pragma unroll
        for (int t = 1; t < T; ++t) {
          float2 dm[4];
          unpack8p(buf[(St::DR + t - 1) * THREADS + lt], dm);
#pragma unroll
          for (int s = 0; s < S; ++s)
#pragma unroll
            for (int p = 0; p < 4; ++p) acc[16 + 4 * s + (t - 1)] = fma2(dm[p], r[s][p], acc[16 + 4 * s + (t - 1)]);
        }
      }
#pragma unroll
      for (int i = 0; i < 32; ++i) red[i] = acc[i].x + acc[i].y;
      lnr[0] = lacc[0].x + lacc[0].y;
      lnr[1] = lacc[1].x + lacc[1].y;
    }
    mail[warp][lane] = warp_scatter_sum<32>(red, lane);
    const float ln_l = warp_scatter_sum<2>(lnr, lane);
    if (lane < 2) mail[warp][32 + lane] = ln_l;
    __syncthreads();
    float tot = mail[0][lane], s_gl = mail[0][32], s_glx = mail[0][33];
#pragma unroll
    for (int w = 1; w < WARPS; ++w) { tot += mail[w][lane]; s_gl += mail[w][32]; s_glx += mail[w][33]; }
    const float m1 = s_gl * inv_d, m2 = s_glx * inv_d;

    // ---------------- per-token scalars: lane s < 4 owns stream s ----------------
    float coef[2 * T + 1];  // alpha[s][0..4], C[s][0..5] = inv_s * dz_s, then -kk_s (RMS-norm backward coefficient)
    {
      const float g_gl = __shfl_sync(0xffffffffu, tot, ls), g_r = __shfl_sync(0xffffffffu, tot, 4 + ls);
      const float g_xr = __shfl_sync(0xffffffffu, tot, 8 + ls), g_er = __shfl_sync(0xffffffffu, tot, 12 + ls);
      float dal[T];
      dal[0] = fmaf(rstd, g_gl - m1 * g_r - m2 * g_xr, g_er);
#pragma unroll
      for (int t = 1; t < T; ++t) dal[t] = __shfl_sync(0xffffffffu, tot, 16 + 4 * ls + (t - 1));
      const float dwb = dbe * b_scale * (1.f - tb * tb);
      float zsum = dwb * zs[T], ascale_acc = 0.f;
#pragma unroll
      for (int t = 0; t < T; ++t) {
        const float dw = dal[t] * a_scale * (1.f - ta[t] * ta[t]);
        zsum = fmaf(dw, zs[t], zsum);
        ascale_acc = fmaf(dal[t], ta[t], ascale_acc);
        coef[t] = fmaf(ta[t], a_scale, __ldg(prm.static_alpha + ls * T + t));
        coef[T + t] = inv * dw;
        small[t] += dal[t];
      }
      coef[2 * T] = inv * dwb;
      small[T] += dbe;
      small[T + 1] += ascale_acc;
      small[T + 2] = fmaf(dbe, tb, small[T + 2]);
      // -kk: with z = inv * <R, g1 P>, sum_c u_c R_c = (1 / inv) * sum_c dz_c z_c, so kk = inv^2 * sum dz z
      zsum = -inv * inv * zsum;
      // coefficient rows of all four streams to every lane
      float cf[S][2 * T + 2];
#pragma unroll
      for (int s = 0; s < S; ++s) {
#pragma unroll
        for (int k = 0; k < 2 * T + 1; ++k) cf[s][k] = __shfl_sync(0xffffffffu, coef[k], s);
        cf[s][2 * T + 1] = __shfl_sync(0xffffffffu, zsum, s);
      }

      // ---------------- pass 2: gradients (inputs re-read from shared memory) ----------------
      float2 dbp2[S];
#pragma unroll
      for (int s = 0; s < S; ++s) dbp2[s] = make_float2(0.f, 0.f);
      if (act) {
        float2 r[S][4], y[4], dm[T][4], pg[T + 1][4];
        staged_r<EXPAND>(buf, lt, bp, r, y);
        {
          float2 dx[4], ex[4], lg[4];
          unpack8p(buf[St::DX * THREADS + lt], dx);
          if (dbin_extra != nullptr) {
            unpack8p(buf[St::EX * THREADS + lt], ex);
          } else {
#pragma unroll
            for (int p = 0; p < 4; ++p) ex[p] = make_float2(0.f, 0.f);
          }
          lds8p(sm + c0, lg);
          const float2 rstd2 = dup2(rstd), nmr2 = dup2(-mean * rstd), nm1 = dup2(-m1), nm2 = dup2(-m2);
#pragma unroll
          for (int p = 0; p < 4; ++p) {
            float2 bsum = mul2(dup2(alpha0[0]), r[0][p]);
#pragma unroll
            for (int s = 1; s < S; ++s) bsum = fma2(dup2(alpha0[s]), r[s][p], bsum);
            const float2 xh = fma2(bsum, rstd2, nmr2);
            // d(branch input) = rstd * (dxn*ln_gamma - m1 - xhat*m2) + dbin_extra
            const float2 inner = fma2(xh, nm2, fma2(dx[p], lg[p], nm1));
            dm[0][p] = fma2(rstd2, inner, ex[p]);
          }
        }
#pragma unroll
        for (int t = 1; t < T; ++t) unpack8p(buf[(St::DR + t - 1) * THREADS + lt], dm[t]);
#pragma unroll
        for (int c = 0; c < T + 1; ++c) lds8p(sm + (1 + c) * d + c0, pg[c]);
        float2 dsum[4];
#pragma unroll
        for (int p = 0; p < 4; ++p) dsum[p] = make_float2(0.f, 0.f);
#pragma unroll
        for (int s = 0; s < S; ++s) {
          float2 dr[4];
#pragma unroll
          for (int p = 0; p < 4; ++p) {
            float2 acc = mul2(r[s][p], dup2(cf[s][2 * T + 1]));
#pragma unroll
            for (int t = 0; t < T; ++t) acc = fma2(dup2(cf[s][t]), dm[t][p], acc);
#pragma unroll
            for (int c = 0; c < T + 1; ++c) {
              acc = fma2(dup2(cf[s][T + c]), pg[c][p], acc);
              gacc[c][p] = fma2(dup2(cf[s][T + c]), r[s][p], gacc[c][p]);
            }
            dr[p] = acc;
            if (EXPAND) {
              dsum[p] = add2(dsum[p], acc);
            } else {
              dbp2[s] = fma2(acc, y[p], dbp2[s]);
              dsum[p] = fma2(dup2(bp[s]), acc, dsum[p]);
            }
          }
          if (!EXPAND) *reinterpret_cast<uint4*>(dR_in + ((size_t)m * S + s) * d + c0) = pack8p(dr);
        }
        if (EXPAND) {
          const float2 sc = dup2(dx_scale);
          float* dst = dx_expand + (size_t)m * d + c0;
          const float2 o0 = mul2(dsum[0], sc), o1 = mul2(dsum[1], sc), o2 = mul2(dsum[2], sc), o3 = mul2(dsum[3], sc);
          *reinterpret_cast<float4*>(dst) = make_float4(o0.x, o0.y, o1.x, o1.y);
          *reinterpret_cast<float4*>(dst + 4) = make_float4(o2.x, o2.y, o3.x, o3.y);
        } else {
          *reinterpret_cast<uint4*>(dY + (size_t)m * d + c0) = pack8p(dsum);
        }
      }
      if (!EXPAND) {
        float dbp[S];
#pragma unroll
        for (int s = 0; s < S; ++s) dbp[s] = dbp2[s].x + dbp2[s].y;
        const float dbp_l = warp_scatter_sum<S>(dbp, lane);
        if (lane < S) mail2[warp][lane] = dbp_l;
      }
    }
    if (!EXPAND) {
      __syncthreads();
      if (lt < S) dbeta_prev[(size_t)m * S + lt] = mail2[0][lt] + mail2[1][lt] + mail2[2][lt] + mail2[3][lt];
    } else {
      __syncthreads();  // mail is rewritten by the next token
    }
  }
  cp_async_wait_prev();  // nothing may still target shared memory when the CTA exits
  if (act) {
    float* dst = part + ((size_t)blockIdx.x * d + c0) * 8;
#pragma unroll
    for (int p = 0; p < 4; ++p)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        float v[8];
#pragma unroll
        for (int j = 0; j < T + 2; ++j) v[j] = h ? gacc[j][p].y : gacc[j][p].x;
        v[7] = 0.f;
        *reinterpret_cast<float4*>(dst + (2 * p + h) * 8) = make_float4(v[0], v[1], v[2], v[3]);
        *reinterpret_cast<float4*>(dst + (2 * p + h) * 8 + 4) = make_float4(v[4], v[5], v[6], v[7]);
      }
  }
  if (lt < S) {
#pragma unroll
    for (int k = 0; k < NSMALL; ++k) part_small[((size_t)blockIdx.x * S + lt) * NSMALL + k] = small[k];
  }
}

// Fixed-order reduction of the backward's per-CTA partial sums, then the chain rule through g1 = (gamma+1)*sqrt(d):
//   g_dyn_alpha[c,t] += g1 G[c,t], g_dyn_beta[c] += g1 G[c,5], g_gamma[c] += sqrt(d) sum_j P_j[c] G[c,j],
//   g_ln_gamma[c] += G[c,6], and the scalar parameters from part_small.
// One CTA per 32 partial columns (4 channels); its 16 warps sum interleaved rows, combined in warp order.
// The last CTA reduces part_small.
constexpr int FIN_WARPS = 16;
__global__ void __launch_bounds__(FIN_WARPS * 32)
param_finish_kernel(const float* __restrict__ part, const float* __restrict__ part_small, int nblk, Params prm,
                    Grads gr, int d) {
  __shared__ float rows[FIN_WARPS][32];
  __shared__ float tot[32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool small = blockIdx.x == gridDim.x - 1;
  const int ncol = small ? S * NSMALL : 8 * d;
  const float* src = small ? part_small : part;
  const int col = small ? lane : blockIdx.x * 32 + lane;
  float acc = 0.f;
#pragma unroll 4
  for (int b = warp; b < nblk; b += FIN_WARPS) acc += src[(size_t)b * ncol + col];
  rows[warp][lane] = acc;
  __syncthreads();
  if (warp == 0) {
    float v = rows[0][lane];
#pragma unroll
    for (int w = 1; w < FIN_WARPS; ++w) v += rows[w][lane];
    tot[lane] = v;
  }
  __syncthreads();
  if (small) {
    if (threadIdx.x < S * T) {
      const int s = threadIdx.x / T, t = threadIdx.x % T;
      gr.static_alpha[threadIdx.x] += tot[s * NSMALL + t];
    } else if (threadIdx.x < S * T + S) {
      const int s = threadIdx.x - S * T;
      gr.static_beta[s] += tot[s * NSMALL + T];
    } else if (threadIdx.x < S * T + S + 2) {
      const int k = threadIdx.x - (S * T + S);  // 0: alpha_scale, 1: beta_scale
      float v = 0.f;
#pragma unroll
      for (int s = 0; s < S; ++s) v += tot[s * NSMALL + T + 1 + k];
      *(k == 0 ? gr.alpha_scale : gr.beta_scale) += v;
    }
    return;
  }
  if (threadIdx.x < 4) {
    const int c = blockIdx.x * 4 + threadIdx.x;
    const float* G = tot + threadIdx.x * 8;
    const float sqrt_d = sqrtf((float)d);
    const float g1 = (prm.gamma_hc[c] + 1.f) * sqrt_d;
    float acc2 = G[T] * prm.dyn_beta[c];
    gr.dyn_beta[c] += g1 * G[T];
#pragma unroll
    for (int t = 0; t < T; ++t) {
      acc2 = fmaf(G[t], prm.dyn_alpha[(size_t)c * T + t], acc2);
      gr.dyn_alpha[(size_t)c * T + t] += g1 * G[t];
    }
    gr.gamma_hc[c] += sqrt_d * acc2;
    gr.ln_gamma[c] += G[T + 1];
  }
}

}  // namespace hc4
}  // namespace alm
