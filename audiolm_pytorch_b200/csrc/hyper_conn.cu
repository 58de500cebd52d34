// Hyper-Connections residual-stream kernels (S = 4 streams), fused with the neighbouring LayerNorm.
//
// Reference: audiolm_pytorch.py:446-454, 524-551 wraps every Attention / FeedForward branch in
// `hyper_connections.HyperConnections` (third-party; arithmetic restated in oracle/third_party.py).
// Per token the reference makes ~4 passes over the 4x-wide residual per branch.  Here one kernel does
//     depth connection of the PREVIOUS branch  ->  width connection of THIS branch  ->  pre-LayerNorm
// so the [M, S, d] residual is read once and written once per branch (HBM-bound, 16-B vector access).
//
// Layout (internal to Transformer.forward): residual streams R [M, S, d] bf16 with the S streams of a
// token contiguous; M = batch * seq.  One CTA walks tokens with a grid stride; thread t owns the 8
// contiguous channels [8t, 8t+8) of every stream, so d/8 threads are active (d % 8 == 0, d <= 8192).
#include "alm_common.cuh"
#include "hyper_conn_v4.cuh"

namespace alm {

constexpr int HC_S = 4;
constexpr int HC_T = HC_S + 1;
constexpr int HC_MAX_WARPS = 32;

struct HcParams {
  const float* gamma_hc;  // [d]      RMSNorm gain (applied as gamma + 1)
  const float* dyn_alpha; // [d, S+1]
  const float* dyn_beta;  // [d]
  const float* static_alpha;  // [S, S+1]
  const float* static_beta;   // [S]
  const float* alpha_scale;   // scalar
  const float* beta_scale;    // scalar
  const float* ln_gamma;  // [d] LayerNorm gain of the branch's pre-norm
};

struct HcGrads {  // fp32 accumulators (atomicAdd), same shapes as HcParams
  float* gamma_hc; float* dyn_alpha; float* dyn_beta; float* static_alpha; float* static_beta;
  float* alpha_scale; float* beta_scale; float* ln_gamma;
};

// sum N per-thread values over the whole CTA; every thread receives the totals.
// `buf` is a [2][N][HC_MAX_WARPS] smem scratch; alternating `which` removes the trailing barrier.
template <int N>
__device__ __forceinline__ void block_sum(float (&v)[N], float* buf, int& which) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
  for (int i = 0; i < N; ++i) v[i] = warp_sum(v[i]);
  float* b = buf + which * (N * HC_MAX_WARPS);
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < N; ++i) b[i * HC_MAX_WARPS + warp] = v[i];
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < N; ++i) {
    float s = 0.f;
    for (int w = 0; w < nw; ++w) s += b[i * HC_MAX_WARPS + w];
    v[i] = s;
  }
  which ^= 1;
}

__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
  f[0] = bf16_lo(u.x); f[1] = bf16_hi(u.x); f[2] = bf16_lo(u.y); f[3] = bf16_hi(u.y);
  f[4] = bf16_lo(u.z); f[5] = bf16_hi(u.z); f[6] = bf16_lo(u.w); f[7] = bf16_hi(u.w);
}
__device__ __forceinline__ uint32_t pk2(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  return make_uint4(pk2(f[0], f[1]), pk2(f[2], f[3]), pk2(f[4], f[5]), pk2(f[6], f[7]));
}
__device__ __forceinline__ void load8f(const float* p, float (&f)[8]) {
  const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
  f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
}

// Saved per token for the backward: tanh of the dynamic alpha/beta pre-activations, 1/|R_s|, LN stats.
//   aux [M, AUX] = { ta[S*(S+1)], tb[S], inv_nrm[S], mean, rstd }
constexpr int HC_AUX = hc4::AUX;  // same stride as the d <= 1024 kernels (z slots unused here)

// ---------------------------------------------------------------------------------------------
// forward:  R = R_in + beta_prev (x) Y   (or R_s = x for every s when expanding)
//           (bin, R_out) = width(R);  xn = LN(bin) * ln_gamma
// ---------------------------------------------------------------------------------------------
template <int MAXT>
__global__ void __launch_bounds__(MAXT)
hc_pre_fwd_kernel(const __nv_bfloat16* __restrict__ R_in, const __nv_bfloat16* __restrict__ Y,
                  const float* __restrict__ beta_prev, const float* __restrict__ x_expand, HcParams prm,
                  __nv_bfloat16* __restrict__ R_out, __nv_bfloat16* __restrict__ bin,
                  __nv_bfloat16* __restrict__ xn, float* __restrict__ beta_out, float* __restrict__ aux, int M,
                  int d) {
  __shared__ float red[2 * 24 * HC_MAX_WARPS];
  extern __shared__ float dyn_smem[];
  float* sA = dyn_smem;  // [HC_T][d] transposed copy of dyn_alpha
  int which = 0;
  const int c0 = threadIdx.x * 8;
  const bool act = c0 < d;
  const float sqrt_d = sqrtf((float)d);
  float g1[8], bfv[8], lng[8];
  if (act) {
    load8f(prm.gamma_hc + c0, g1);
    load8f(prm.dyn_beta + c0, bfv);
    load8f(prm.ln_gamma + c0, lng);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      g1[e] = (g1[e] + 1.f) * sqrt_d;
#pragma unroll
      for (int t = 0; t < HC_T; ++t) sA[t * d + c0 + e] = prm.dyn_alpha[(size_t)(c0 + e) * HC_T + t];
    }
  }
  const float a_scale = *prm.alpha_scale, b_scale = *prm.beta_scale;
  float Astat[HC_S][HC_T], Bstat[HC_S];
#pragma unroll
  for (int s = 0; s < HC_S; ++s) {
    Bstat[s] = prm.static_beta[s];
#pragma unroll
    for (int t = 0; t < HC_T; ++t) Astat[s][t] = prm.static_alpha[s * HC_T + t];
  }

  for (int m = blockIdx.x; m < M; m += gridDim.x) {
    float R[HC_S][8];
    if (act) {
      if (x_expand != nullptr) {
        float xv[8];
        load8f(x_expand + (size_t)m * d + c0, xv);
#pragma unroll
        for (int s = 0; s < HC_S; ++s)
#pragma unroll
          for (int e = 0; e < 8; ++e) R[s][e] = xv[e];
      } else {
        float yv[8];
        unpack8(*reinterpret_cast<const uint4*>(Y + (size_t)m * d + c0), yv);
#pragma unroll
        for (int s = 0; s < HC_S; ++s) {
          const float bp = beta_prev[(size_t)m * HC_S + s];
          float rv[8];
          unpack8(*reinterpret_cast<const uint4*>(R_in + ((size_t)m * HC_S + s) * d + c0), rv);
#pragma unroll
          for (int e = 0; e < 8; ++e) R[s][e] = rv[e] + bp * yv[e];
        }
      }
    } else {
#pragma unroll
      for (int s = 0; s < HC_S; ++s)
#pragma unroll
        for (int e = 0; e < 8; ++e) R[s][e] = 0.f;
    }
    // stream norms
    float ssq[HC_S];
#pragma unroll
    for (int s = 0; s < HC_S; ++s) {
      float a = 0.f;
#pragma unroll
      for (int e = 0; e < 8; ++e) a += R[s][e] * R[s][e];
      ssq[s] = a;
    }
    block_sum<HC_S>(ssq, red, which);
    float inv[HC_S];
#pragma unroll
    for (int s = 0; s < HC_S; ++s) inv[s] = 1.f / fmaxf(sqrtf(ssq[s]), 1e-12f);
    // dynamic alpha / beta pre-activations
    float w[HC_S * HC_T + HC_S];
#pragma unroll
    for (int i = 0; i < HC_S * HC_T + HC_S; ++i) w[i] = 0.f;
    if (act) {
#pragma unroll
      for (int s = 0; s < HC_S; ++s)
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float nv = R[s][e] * inv[s] * g1[e];
#pragma unroll
          for (int t = 0; t < HC_T; ++t) w[s * HC_T + t] += nv * sA[t * d + c0 + e];
          w[HC_S * HC_T + s] += nv * bfv[e];
        }
    }
    block_sum<HC_S * HC_T + HC_S>(w, red, which);
    float alpha[HC_S][HC_T], beta[HC_S];
#pragma unroll
    for (int s = 0; s < HC_S; ++s) {
#pragma unroll
      for (int t = 0; t < HC_T; ++t) {
        w[s * HC_T + t] = tanhf(w[s * HC_T + t]);
        alpha[s][t] = w[s * HC_T + t] * a_scale + Astat[s][t];
      }
      w[HC_S * HC_T + s] = tanhf(w[HC_S * HC_T + s]);
      beta[s] = w[HC_S * HC_T + s] * b_scale + Bstat[s];
    }
    // mix
    float mix[HC_T][8];
#pragma unroll
    for (int t = 0; t < HC_T; ++t)
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        float a = 0.f;
#pragma unroll
        for (int s = 0; s < HC_S; ++s) a += alpha[s][t] * R[s][e];
        mix[t][e] = a;
      }
    // LayerNorm of the branch input (two-pass variance)
    float st1[1] = {0.f};
#pragma unroll
    for (int e = 0; e < 8; ++e) st1[0] += mix[0][e];
    block_sum<1>(st1, red, which);
    const float mean = st1[0] / d;
    float st2[1] = {0.f};
    if (act) {
#pragma unroll
      for (int e = 0; e < 8; ++e) st2[0] += (mix[0][e] - mean) * (mix[0][e] - mean);
    }
    block_sum<1>(st2, red, which);
    const float rstd = rsqrtf(st2[0] / d + 1e-5f);
    if (act) {
#pragma unroll
      for (int s = 0; s < HC_S; ++s)
        *reinterpret_cast<uint4*>(R_out + ((size_t)m * HC_S + s) * d + c0) = pack8(mix[s + 1]);
      *reinterpret_cast<uint4*>(bin + (size_t)m * d + c0) = pack8(mix[0]);
      float xo[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) xo[e] = (mix[0][e] - mean) * rstd * lng[e];
      *reinterpret_cast<uint4*>(xn + (size_t)m * d + c0) = pack8(xo);
    }
    if (threadIdx.x == 0) {
      float* a = aux + (size_t)m * HC_AUX;
#pragma unroll
      for (int i = 0; i < HC_S * HC_T + HC_S; ++i) a[i] = w[i];
#pragma unroll
      for (int s = 0; s < HC_S; ++s) {
        a[HC_S * HC_T + HC_S + s] = inv[s];
        beta_out[(size_t)m * HC_S + s] = beta[s];
      }
      a[HC_AUX - 2] = mean;
      a[HC_AUX - 1] = rstd;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// backward of hc_pre.  Upstream: dR_out [M,S,d], dxn [M,d], dbin_extra [M,d] (optional), dbeta [M,S].
// Produces dR_in [M,S,d], dY [M,d], dbeta_prev [M,S]  (or dx [M,d] fp32 when expanding), plus
// parameter gradients (atomicAdd into fp32).
// ---------------------------------------------------------------------------------------------
template <int MAXT>
__global__ void __launch_bounds__(MAXT)
hc_pre_bwd_kernel(const __nv_bfloat16* __restrict__ R_in, const __nv_bfloat16* __restrict__ Y,
                  const float* __restrict__ beta_prev, const float* __restrict__ x_expand, HcParams prm,
                  const float* __restrict__ aux, const __nv_bfloat16* __restrict__ dR_out,
                  const __nv_bfloat16* __restrict__ dxn, const __nv_bfloat16* __restrict__ dbin_extra,
                  const float* __restrict__ dbeta, __nv_bfloat16* __restrict__ dR_in,
                  __nv_bfloat16* __restrict__ dY, float* __restrict__ dbeta_prev, float* __restrict__ dx_expand,
                  float dx_scale, HcGrads gr, int M, int d) {
  __shared__ float red[2 * 24 * HC_MAX_WARPS];
  extern __shared__ float dyn_smem[];
  float* sA = dyn_smem;             // [HC_T][d] transposed copy of dyn_alpha
  float* sGA = dyn_smem + HC_T * d; // [HC_T][d] gradient accumulator (each thread owns its columns)
  int which = 0;
  const int c0 = threadIdx.x * 8;
  const bool act = c0 < d;
  const float sqrt_d = sqrtf((float)d);
  float g1[8], bfv[8], lng[8];
  if (act) {
    load8f(prm.gamma_hc + c0, g1);
    load8f(prm.dyn_beta + c0, bfv);
    load8f(prm.ln_gamma + c0, lng);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      g1[e] = (g1[e] + 1.f) * sqrt_d;
#pragma unroll
      for (int t = 0; t < HC_T; ++t) {
        sA[t * d + c0 + e] = prm.dyn_alpha[(size_t)(c0 + e) * HC_T + t];
        sGA[t * d + c0 + e] = 0.f;
      }
    }
  }
  const float a_scale = *prm.alpha_scale, b_scale = *prm.beta_scale;
  float Astat[HC_S][HC_T];
#pragma unroll
  for (int s = 0; s < HC_S; ++s)
#pragma unroll
    for (int t = 0; t < HC_T; ++t) Astat[s][t] = prm.static_alpha[s * HC_T + t];
  // per-thread parameter-gradient accumulators over the tokens this CTA visits
  float gBf[8], gG[8], gLn[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) gBf[e] = gG[e] = gLn[e] = 0.f;
  float acc_small[HC_S * HC_T + HC_S + 2];
#pragma unroll
  for (int i = 0; i < HC_S * HC_T + HC_S + 2; ++i) acc_small[i] = 0.f;

  for (int m = blockIdx.x; m < M; m += gridDim.x) {
    const float* a = aux + (size_t)m * HC_AUX;
    float ta[HC_S][HC_T], tb[HC_S], inv[HC_S], alpha[HC_S][HC_T], bp[HC_S], dbe[HC_S];
#pragma unroll
    for (int s = 0; s < HC_S; ++s) {
#pragma unroll
      for (int t = 0; t < HC_T; ++t) {
        ta[s][t] = a[s * HC_T + t];
        alpha[s][t] = ta[s][t] * a_scale + Astat[s][t];
      }
      tb[s] = a[HC_S * HC_T + s];
      inv[s] = a[HC_S * HC_T + HC_S + s];
      dbe[s] = dbeta[(size_t)m * HC_S + s];
      bp[s] = (x_expand == nullptr) ? beta_prev[(size_t)m * HC_S + s] : 0.f;
    }
    const float mean = a[HC_AUX - 2], rstd = a[HC_AUX - 1];

    float R[HC_S][8], yv[8], dmix[HC_T][8];
#pragma unroll
    for (int e = 0; e < 8; ++e) yv[e] = 0.f;
    if (act) {
      if (x_expand != nullptr) {
        float xv[8];
        load8f(x_expand + (size_t)m * d + c0, xv);
#pragma unroll
        for (int s = 0; s < HC_S; ++s)
#pragma unroll
          for (int e = 0; e < 8; ++e) R[s][e] = xv[e];
      } else {
        unpack8(*reinterpret_cast<const uint4*>(Y + (size_t)m * d + c0), yv);
#pragma unroll
        for (int s = 0; s < HC_S; ++s) {
          float rv[8];
          unpack8(*reinterpret_cast<const uint4*>(R_in + ((size_t)m * HC_S + s) * d + c0), rv);
#pragma unroll
          for (int e = 0; e < 8; ++e) R[s][e] = rv[e] + bp[s] * yv[e];
        }
      }
#pragma unroll
      for (int s = 0; s < HC_S; ++s)
        unpack8(*reinterpret_cast<const uint4*>(dR_out + ((size_t)m * HC_S + s) * d + c0), dmix[s + 1]);
    } else {
#pragma unroll
      for (int s = 0; s < HC_S; ++s)
#pragma unroll
        for (int e = 0; e < 8; ++e) { R[s][e] = 0.f; dmix[s + 1][e] = 0.f; }
    }
    // ---- LayerNorm backward on bin = sum_s alpha[s][0] R[s] ----
    float xhat[8], gl[8];
    float lnred[2] = {0.f, 0.f};
    if (act) {
      float dx8[8];
      unpack8(*reinterpret_cast<const uint4*>(dxn + (size_t)m * d + c0), dx8);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        float b = 0.f;
#pragma unroll
        for (int s = 0; s < HC_S; ++s) b += alpha[s][0] * R[s][e];
        xhat[e] = (b - mean) * rstd;
        gl[e] = dx8[e] * lng[e];
        gLn[e] += dx8[e] * xhat[e];
        lnred[0] += gl[e];
        lnred[1] += gl[e] * xhat[e];
      }
    }
    block_sum<2>(lnred, red, which);
    const float m1 = lnred[0] / d, m2 = lnred[1] / d;
    if (act) {
      float ex[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) ex[e] = 0.f;
      if (dbin_extra != nullptr) unpack8(*reinterpret_cast<const uint4*>(dbin_extra + (size_t)m * d + c0), ex);
#pragma unroll
      for (int e = 0; e < 8; ++e) dmix[0][e] = rstd * (gl[e] - m1 - xhat[e] * m2) + ex[e];
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) dmix[0][e] = 0.f;
    }
    // ---- d alpha[s][t] = <dmix[t], R[s]> ----
    float dal[HC_S * HC_T];
#pragma unroll
    for (int s = 0; s < HC_S; ++s)
#pragma unroll
      for (int t = 0; t < HC_T; ++t) {
        float acc = 0.f;
#pragma unroll
        for (int e = 0; e < 8; ++e) acc += dmix[t][e] * R[s][e];
        dal[s * HC_T + t] = acc;
      }
    block_sum<HC_S * HC_T>(dal, red, which);
    float dwa[HC_S][HC_T], dwb[HC_S];
#pragma unroll
    for (int s = 0; s < HC_S; ++s) {
#pragma unroll
      for (int t = 0; t < HC_T; ++t) {
        const float g = dal[s * HC_T + t];
        dwa[s][t] = g * a_scale * (1.f - ta[s][t] * ta[s][t]);
        acc_small[s * HC_T + t] += g;                       // d static_alpha
        acc_small[HC_S * HC_T + HC_S] += g * ta[s][t];      // d alpha_scale
      }
      dwb[s] = dbe[s] * b_scale * (1.f - tb[s] * tb[s]);
      acc_small[HC_S * HC_T + s] += dbe[s];                 // d static_beta
      acc_small[HC_S * HC_T + HC_S + 1] += dbe[s] * tb[s];  // d beta_scale
    }
    // ---- dR = alpha . dmix  +  RMSNorm backward of the dynamic-weight path ----
    float dR[HC_S][8], udot[HC_S];
#pragma unroll
    for (int s = 0; s < HC_S; ++s) {
      udot[s] = 0.f;
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        float acc = 0.f;
#pragma unroll
        for (int t = 0; t < HC_T; ++t) acc += alpha[s][t] * dmix[t][e];
        float dn = dwb[s] * bfv[e];
#pragma unroll
        for (int t = 0; t < HC_T; ++t) dn += dwa[s][t] * sA[t * d + c0 + e];
        const float rn = R[s][e] * inv[s];             // unit-normalised residual
        const float nv = rn * g1[e];                   // normed value
        gG[e] += dn * rn * sqrt_d;
        gBf[e] += nv * dwb[s];
        if (act) {
#pragma unroll
          for (int t = 0; t < HC_T; ++t) sGA[t * d + c0 + e] += nv * dwa[s][t];
        }
        const float u = dn * g1[e];
        udot[s] += u * R[s][e];
        dR[s][e] = acc + u * inv[s];
      }
    }
    block_sum<HC_S>(udot, red, which);
#pragma unroll
    for (int s = 0; s < HC_S; ++s) {
      const float k = udot[s] * inv[s] * inv[s] * inv[s];
#pragma unroll
      for (int e = 0; e < 8; ++e) dR[s][e] -= R[s][e] * k;
    }
    // ---- depth connection of the previous branch / stream expansion ----
    if (x_expand != nullptr) {
      if (act) {
        float o[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          float acc = 0.f;
#pragma unroll
          for (int s = 0; s < HC_S; ++s) acc += dR[s][e];
          o[e] = acc * dx_scale;
        }
        float* dst = dx_expand + (size_t)m * d + c0;
        *reinterpret_cast<float4*>(dst) = make_float4(o[0], o[1], o[2], o[3]);
        *reinterpret_cast<float4*>(dst + 4) = make_float4(o[4], o[5], o[6], o[7]);
      }
    } else {
      float dbp[HC_S];
#pragma unroll
      for (int s = 0; s < HC_S; ++s) {
        float acc = 0.f;
#pragma unroll
        for (int e = 0; e < 8; ++e) acc += dR[s][e] * yv[e];
        dbp[s] = acc;
      }
      block_sum<HC_S>(dbp, red, which);
      if (act) {
        float dy[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          float acc = 0.f;
#pragma unroll
          for (int s = 0; s < HC_S; ++s) acc += bp[s] * dR[s][e];
          dy[e] = acc;
        }
        *reinterpret_cast<uint4*>(dY + (size_t)m * d + c0) = pack8(dy);
#pragma unroll
        for (int s = 0; s < HC_S; ++s)
          *reinterpret_cast<uint4*>(dR_in + ((size_t)m * HC_S + s) * d + c0) = pack8(dR[s]);
      }
      if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < HC_S; ++s) dbeta_prev[(size_t)m * HC_S + s] = dbp[s];
      }
    }
  }
  // ---- flush parameter gradients ----
  if (act) {
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      atomicAdd(gr.gamma_hc + c0 + e, gG[e]);
      atomicAdd(gr.dyn_beta + c0 + e, gBf[e]);
      atomicAdd(gr.ln_gamma + c0 + e, gLn[e]);
#pragma unroll
      for (int t = 0; t < HC_T; ++t) atomicAdd(gr.dyn_alpha + (size_t)(c0 + e) * HC_T + t, sGA[t * d + c0 + e]);
    }
  }
  if (threadIdx.x == 0) {  // acc_small is identical in every thread (built from block-reduced values)
#pragma unroll
    for (int i = 0; i < HC_S * HC_T; ++i) atomicAdd(gr.static_alpha + i, acc_small[i]);
#pragma unroll
    for (int s = 0; s < HC_S; ++s) atomicAdd(gr.static_beta + s, acc_small[HC_S * HC_T + s]);
    atomicAdd(gr.alpha_scale, acc_small[HC_S * HC_T + HC_S]);
    atomicAdd(gr.beta_scale, acc_small[HC_S * HC_T + HC_S + 1]);
  }
}

// ---------------------------------------------------------------------------------------------
// end of the stack: depth connection of the last branch, sum over streams (reduce_streams,
// audiolm_pytorch.py:551) and the final LayerNorm (:555).
// ---------------------------------------------------------------------------------------------
template <int MAXT>
__global__ void __launch_bounds__(MAXT)
hc_post_fwd_kernel(const __nv_bfloat16* __restrict__ R_in, const __nv_bfloat16* __restrict__ Y,
                   const float* __restrict__ beta_prev, const float* __restrict__ ln_gamma,
                   __nv_bfloat16* __restrict__ out, float* __restrict__ stats, int M, int d) {
  __shared__ float red[2 * 24 * HC_MAX_WARPS];
  int which = 0;
  const int c0 = threadIdx.x * 8;
  const bool act = c0 < d;
  float lng[8];
  if (act) load8f(ln_gamma + c0, lng);
  for (int m = blockIdx.x; m < M; m += gridDim.x) {
    float xs[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) xs[e] = 0.f;
    if (act) {
      float yv[8];
      unpack8(*reinterpret_cast<const uint4*>(Y + (size_t)m * d + c0), yv);
      float bsum = 0.f;
#pragma unroll
      for (int s = 0; s < HC_S; ++s) {
        bsum += beta_prev[(size_t)m * HC_S + s];
        float rv[8];
        unpack8(*reinterpret_cast<const uint4*>(R_in + ((size_t)m * HC_S + s) * d + c0), rv);
#pragma unroll
        for (int e = 0; e < 8; ++e) xs[e] += rv[e];
      }
#pragma unroll
      for (int e = 0; e < 8; ++e) xs[e] += bsum * yv[e];
    }
    float s1[1] = {0.f};
#pragma unroll
    for (int e = 0; e < 8; ++e) s1[0] += xs[e];
    block_sum<1>(s1, red, which);
    const float mean = s1[0] / d;
    float s2[1] = {0.f};
    if (act) {
#pragma unroll
      for (int e = 0; e < 8; ++e) s2[0] += (xs[e] - mean) * (xs[e] - mean);
    }
    block_sum<1>(s2, red, which);
    const float rstd = rsqrtf(s2[0] / d + 1e-5f);
    if (act) {
      float o[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) o[e] = (xs[e] - mean) * rstd * lng[e];
      *reinterpret_cast<uint4*>(out + (size_t)m * d + c0) = pack8(o);
    }
    if (threadIdx.x == 0) {
      stats[(size_t)m * 2] = mean;
      stats[(size_t)m * 2 + 1] = rstd;
    }
  }
}

template <int MAXT>
__global__ void __launch_bounds__(MAXT)
hc_post_bwd_kernel(const __nv_bfloat16* __restrict__ R_in, const __nv_bfloat16* __restrict__ Y,
                   const float* __restrict__ beta_prev, const float* __restrict__ ln_gamma,
                   const float* __restrict__ stats, const __nv_bfloat16* __restrict__ dout,
                   __nv_bfloat16* __restrict__ dR_in, __nv_bfloat16* __restrict__ dY,
                   float* __restrict__ dbeta_prev, float* __restrict__ g_ln_gamma, int M, int d) {
  __shared__ float red[2 * 24 * HC_MAX_WARPS];
  int which = 0;
  const int c0 = threadIdx.x * 8;
  const bool act = c0 < d;
  float lng[8], gLn[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) gLn[e] = 0.f;
  if (act) load8f(ln_gamma + c0, lng);
  for (int m = blockIdx.x; m < M; m += gridDim.x) {
    const float mean = stats[(size_t)m * 2], rstd = stats[(size_t)m * 2 + 1];
    float xs[8], yv[8], gl[8], xhat[8];
    float bsum = 0.f;
    float r2[2] = {0.f, 0.f};
#pragma unroll
    for (int e = 0; e < 8; ++e) { xs[e] = 0.f; yv[e] = 0.f; }
    if (act) {
      unpack8(*reinterpret_cast<const uint4*>(Y + (size_t)m * d + c0), yv);
#pragma unroll
      for (int s = 0; s < HC_S; ++s) {
        bsum += beta_prev[(size_t)m * HC_S + s];
        float rv[8];
        unpack8(*reinterpret_cast<const uint4*>(R_in + ((size_t)m * HC_S + s) * d + c0), rv);
#pragma unroll
        for (int e = 0; e < 8; ++e) xs[e] += rv[e];
      }
      float dv[8];
      unpack8(*reinterpret_cast<const uint4*>(dout + (size_t)m * d + c0), dv);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        xs[e] += bsum * yv[e];
        xhat[e] = (xs[e] - mean) * rstd;
        gl[e] = dv[e] * lng[e];
        gLn[e] += dv[e] * xhat[e];
        r2[0] += gl[e];
        r2[1] += gl[e] * xhat[e];
      }
    }
    block_sum<2>(r2, red, which);
    const float m1 = r2[0] / d, m2 = r2[1] / d;
    float dxs[8];
    float db[1] = {0.f};
#pragma unroll
    for (int e = 0; e < 8; ++e) dxs[e] = 0.f;
    if (act) {
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        dxs[e] = rstd * (gl[e] - m1 - xhat[e] * m2);
        db[0] += dxs[e] * yv[e];
      }
    }
    block_sum<1>(db, red, which);
    if (act) {
      const uint4 pk = pack8(dxs);
#pragma unroll
      for (int s = 0; s < HC_S; ++s) *reinterpret_cast<uint4*>(dR_in + ((size_t)m * HC_S + s) * d + c0) = pk;
      float dy[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) dy[e] = bsum * dxs[e];
      *reinterpret_cast<uint4*>(dY + (size_t)m * d + c0) = pack8(dy);
    }
    if (threadIdx.x == 0) {
#pragma unroll
      for (int s = 0; s < HC_S; ++s) dbeta_prev[(size_t)m * HC_S + s] = db[0];
    }
  }
  if (act) {
#pragma unroll
    for (int e = 0; e < 8; ++e) atomicAdd(g_ln_gamma + c0 + e, gLn[e]);
  }
}

static inline int hc_threads(int d) { return ((d / 8 + 31) / 32) * 32; }
// launch kernel template K<MAXT> with the smallest MAXT in {128,256,512,1024} that covers `threads`
// (dims above 1024 need more than the default 48 KB of dynamic shared memory: opt in per instantiation)
#define HC_LAUNCH_ONE(K, T_, grid, threads, smem, stream, ...)                                             \
  do {                                                                                                     \
    if ((size_t)(smem) > 48 * 1024)                                                                        \
      ALM_CUDA_OK(cudaFuncSetAttribute(K<T_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(smem)));  \
    K<T_><<<(grid), (threads), (smem), (stream)>>>(__VA_ARGS__);                                           \
  } while (0)
#define HC_DISPATCH(K, grid, threads, smem, stream, ...)                                      \
  do {                                                                                        \
    if ((threads) <= 128) HC_LAUNCH_ONE(K, 128, grid, threads, smem, stream, __VA_ARGS__);      \
    else if ((threads) <= 256) HC_LAUNCH_ONE(K, 256, grid, threads, smem, stream, __VA_ARGS__); \
    else if ((threads) <= 512) HC_LAUNCH_ONE(K, 512, grid, threads, smem, stream, __VA_ARGS__); \
    else HC_LAUNCH_ONE(K, 1024, grid, threads, smem, stream, __VA_ARGS__);                      \
  } while (0)
static inline int hc_grid(int M, int threads) {
  const int per_sm = max(1, 1024 / threads);
  const int g = num_sms() * min(per_sm, 4);
  return M < g ? M : g;
}

}  // namespace alm

using namespace alm;

extern "C" int alm_hc_pre_fwd(const void* R_in, const void* Y, const float* beta_prev, const float* x_expand,
                              const float* gamma_hc, const float* dyn_alpha, const float* dyn_beta,
                              const float* static_alpha, const float* static_beta, const float* alpha_scale,
                              const float* beta_scale, const float* ln_gamma, void* R_out, void* bin, void* xn,
                              float* beta_out, float* aux, int M, int d, int streams, alm_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  ALM_REQUIRE(streams == HC_S, ALM_ERR_UNSUPPORTED);
  ALM_REQUIRE(d % 8 == 0 && d >= 8 && d <= 8192 && M > 0, ALM_ERR_ARG);
  ALM_REQUIRE((x_expand != nullptr) != (R_in != nullptr), ALM_ERR_ARG);
  if (d <= 1024) {
    hc4::Params p4{gamma_hc, dyn_alpha, dyn_beta, static_alpha, static_beta, alpha_scale, beta_scale, ln_gamma};
    const int grid = min(M, hc4::FWD_CTAS_PER_SM * num_sms());
    const size_t smem = hc4::param_smem(d);
    if (x_expand != nullptr)
      hc4::pre_fwd_kernel<true><<<grid, hc4::THREADS, smem, stream>>>(nullptr, nullptr, nullptr, x_expand, p4,
          (__nv_bfloat16*)R_out, (__nv_bfloat16*)bin, (__nv_bfloat16*)xn, beta_out, aux, M, d);
    else
      hc4::pre_fwd_kernel<false><<<grid, hc4::THREADS, smem, stream>>>((const __nv_bfloat16*)R_in,
          (const __nv_bfloat16*)Y, beta_prev, nullptr, p4, (__nv_bfloat16*)R_out, (__nv_bfloat16*)bin,
          (__nv_bfloat16*)xn, beta_out, aux, M, d);
    ALM_CHECK_LAUNCH();
    ALM_LAUNCHED(1);
    return ALM_OK;
  }
  HcParams prm{gamma_hc, dyn_alpha, dyn_beta, static_alpha, static_beta, alpha_scale, beta_scale, ln_gamma};
  const int threads = hc_threads(d);
  HC_DISPATCH(hc_pre_fwd_kernel, hc_grid(M, threads), threads, HC_T * d * sizeof(float), stream,
              (const __nv_bfloat16*)R_in, (const __nv_bfloat16*)Y, beta_prev, x_expand, prm, (__nv_bfloat16*)R_out,
              (__nv_bfloat16*)bin, (__nv_bfloat16*)xn, beta_out, aux, M, d);
  ALM_CHECK_LAUNCH();
  ALM_LAUNCHED(1);
  return ALM_OK;
}

extern "C" int alm_hc_pre_bwd(const void* R_in, const void* Y, const float* beta_prev, const float* x_expand,
                              const float* gamma_hc, const float* dyn_alpha, const float* dyn_beta,
                              const float* static_alpha, const float* static_beta, const float* alpha_scale,
                              const float* beta_scale, const float* ln_gamma, const float* aux, const void* dR_out,
                              const void* dxn, const void* dbin_extra, const float* dbeta, void* dR_in, void* dY,
                              float* dbeta_prev, float* dx_expand, float dx_scale, float* g_gamma_hc,
                              float* g_dyn_alpha, float* g_dyn_beta, float* g_static_alpha, float* g_static_beta,
                              float* g_alpha_scale, float* g_beta_scale, float* g_ln_gamma, float* partial,
                              int partial_blocks, int M, int d, int streams, alm_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  ALM_REQUIRE(streams == HC_S, ALM_ERR_UNSUPPORTED);
  ALM_REQUIRE(d % 8 == 0 && d >= 8 && d <= 8192 && M > 0, ALM_ERR_ARG);
  if (d <= 1024) {
    const int grid = min(min(M, hc4::BWD_CTAS_PER_SM * num_sms()), partial_blocks);
    ALM_REQUIRE(partial != nullptr && grid > 0, ALM_ERR_ARG);
    hc4::Params p4{gamma_hc, dyn_alpha, dyn_beta, static_alpha, static_beta, alpha_scale, beta_scale, ln_gamma};
    hc4::Grads g4{g_gamma_hc, g_dyn_alpha, g_dyn_beta, g_static_alpha, g_static_beta, g_alpha_scale, g_beta_scale,
                  g_ln_gamma};
    float* part_small = partial + (size_t)grid * d * 8;
    const bool expand = x_expand != nullptr;
    const size_t smem = hc4::bwd_smem(d, expand);
    static bool attr4 = false;
    if (!attr4) {
      ALM_CUDA_OK(cudaFuncSetAttribute(hc4::pre_bwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)hc4::bwd_smem(1024, false)));
      ALM_CUDA_OK(cudaFuncSetAttribute(hc4::pre_bwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)hc4::bwd_smem(1024, true)));
      attr4 = true;
    }
#define HC4_BWD_ARGS (const __nv_bfloat16*)R_in, (const __nv_bfloat16*)Y, beta_prev, x_expand, p4, aux,          \
                        (const __nv_bfloat16*)dR_out, (const __nv_bfloat16*)dxn, (const __nv_bfloat16*)dbin_extra, \
                        dbeta, (__nv_bfloat16*)dR_in, (__nv_bfloat16*)dY, dbeta_prev, dx_expand, dx_scale, partial,  \
                        part_small, M, d
    if (expand) hc4::pre_bwd_kernel<true><<<grid, hc4::THREADS, smem, stream>>>(HC4_BWD_ARGS);
    else hc4::pre_bwd_kernel<false><<<grid, hc4::THREADS, smem, stream>>>(HC4_BWD_ARGS);
#undef HC4_BWD_ARGS
    ALM_CHECK_LAUNCH();
    hc4::param_finish_kernel<<<d / 4 + 1, hc4::FIN_WARPS * 32, 0, stream>>>(partial, part_small, grid, p4, g4, d);
    ALM_CHECK_LAUNCH();
    ALM_LAUNCHED(2);
    return ALM_OK;
  }
  HcParams prm{gamma_hc, dyn_alpha, dyn_beta, static_alpha, static_beta, alpha_scale, beta_scale, ln_gamma};
  HcGrads gr{g_gamma_hc, g_dyn_alpha, g_dyn_beta, g_static_alpha, g_static_beta, g_alpha_scale, g_beta_scale,
             g_ln_gamma};
  const int threads = hc_threads(d);
  const int grid = min(M, num_sms() * 2);
  HC_DISPATCH(hc_pre_bwd_kernel, grid, threads, 2 * HC_T * d * sizeof(float), stream,
              (const __nv_bfloat16*)R_in, (const __nv_bfloat16*)Y, beta_prev, x_expand, prm, aux,
              (const __nv_bfloat16*)dR_out, (const __nv_bfloat16*)dxn, (const __nv_bfloat16*)dbin_extra, dbeta,
              (__nv_bfloat16*)dR_in, (__nv_bfloat16*)dY, dbeta_prev, dx_expand, dx_scale, gr, M, d);
  ALM_CHECK_LAUNCH();
  ALM_LAUNCHED(1);
  return ALM_OK;
}

extern "C" int alm_hc_post_fwd(const void* R_in, const void* Y, const float* beta_prev, const float* ln_gamma,
                               void* out, float* stats, int M, int d, int streams, alm_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  ALM_REQUIRE(streams == HC_S, ALM_ERR_UNSUPPORTED);
  ALM_REQUIRE(d % 8 == 0 && d >= 8 && d <= 8192 && M > 0, ALM_ERR_ARG);
  const int threads = hc_threads(d);
  HC_DISPATCH(hc_post_fwd_kernel, hc_grid(M, threads), threads, 0, stream, (const __nv_bfloat16*)R_in,
              (const __nv_bfloat16*)Y, beta_prev, ln_gamma, (__nv_bfloat16*)out, stats, M, d);
  ALM_CHECK_LAUNCH();
  ALM_LAUNCHED(1);
  return ALM_OK;
}

extern "C" int alm_hc_post_bwd(const void* R_in, const void* Y, const float* beta_prev, const float* ln_gamma,
                               const float* stats, const void* dout, void* dR_in, void* dY, float* dbeta_prev,
                               float* g_ln_gamma, int M, int d, int streams, alm_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  ALM_REQUIRE(streams == HC_S, ALM_ERR_UNSUPPORTED);
  ALM_REQUIRE(d % 8 == 0 && d >= 8 && d <= 8192 && M > 0, ALM_ERR_ARG);
  const int threads = hc_threads(d);
  HC_DISPATCH(hc_post_bwd_kernel, min(M, num_sms() * 4), threads, 0, stream, (const __nv_bfloat16*)R_in,
              (const __nv_bfloat16*)Y, beta_prev, ln_gamma, stats, (const __nv_bfloat16*)dout,
              (__nv_bfloat16*)dR_in, (__nv_bfloat16*)dY, dbeta_prev, g_ln_gamma, M, d);
  ALM_CHECK_LAUNCH();
  ALM_LAUNCHED(1);
  return ALM_OK;
}
