// LayerNorm without bias (egom2p_utils.py:118-133) and, as a compile-time variant, nn.LayerNorm with a learnable bias (the
// GELU / bias family, egom2p_model.py:882-978); fp32 statistics. One warp per row, row held in registers,
// 16-byte vector loads/stores. HBM-bound: fwd moves 4*D bytes in + 2*D (bf16) out per row.
#include "common.cuh"

namespace egom2p {

constexpr int kLnMaxVec = 16;  // float4 per lane -> dim <= 2048

template <int NV, bool kBias>
__global__ void __launch_bounds__(256) ln_fwd_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                     const float* __restrict__ bias, int64_t rows, int dim, float eps, uint16_t* __restrict__ yb,
                                                     float* __restrict__ yf, float* __restrict__ mean_out,
                                                     float* __restrict__ rstd_out) {
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const int D4 = dim >> 2;
  const float4* xr = reinterpret_cast<const float4*>(x + row * dim);
  float4 v[NV];
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    const int i = lane + j * 32;
    if (i < D4) {
      v[j] = xr[i];
      s += (v[j].x + v[j].y) + (v[j].z + v[j].w);
    }
  }
  const float mean = warp_sum(s) / dim;
  float q = 0.f;
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    const int i = lane + j * 32;
    if (i < D4) {
      const float a = v[j].x - mean, b = v[j].y - mean, c = v[j].z - mean, d = v[j].w - mean;
      q += (a * a + b * b) + (c * c + d * d);
    }
  }
  const float rstd = rsqrtf(warp_sum(q) / dim + eps);
  if (lane == 0) {
    if (mean_out) mean_out[row] = mean;
    if (rstd_out) rstd_out[row] = rstd;
  }
  const float4* wr = reinterpret_cast<const float4*>(w);
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    const int i = lane + j * 32;
    if (i < D4) {
      const float4 g = __ldg(wr + i);
      float4 o;
      o.x = (v[j].x - mean) * rstd * g.x;
      o.y = (v[j].y - mean) * rstd * g.y;
      o.z = (v[j].z - mean) * rstd * g.z;
      o.w = (v[j].w - mean) * rstd * g.w;
      if (kBias) {
        const float4 b = __ldg(reinterpret_cast<const float4*>(bias) + i);
        o.x += b.x; o.y += b.y; o.z += b.z; o.w += b.w;
      }
      if (yf) reinterpret_cast<float4*>(yf + row * dim)[i] = o;
      if (yb) {
        uint2 pk;
        pk.x = pack_bf16(o.x, o.y);
        pk.y = pack_bf16(o.z, o.w);
        reinterpret_cast<uint2*>(yb + row * dim)[i] = pk;
      }
    }
  }
}

// dx = rstd * (g - mean(g) - xhat * mean(g * xhat)), g = dy * w ; dw += sum_rows dy * xhat ; (kBias) db += sum_rows dy.
// Each warp walks rows [row0 + warp, ...) with stride 8 inside its CTA's row chunk and keeps per-lane dw partials.
// Only the raw x / dy registers stay live across the two warp reductions (xhat and g are recomputed), which keeps the
// kernel at <= 80 registers -> 3 CTAs (24 warps) per SM to cover the load -> reduce -> store latency chain.
template <bool kBf16> struct DyVec;
template <> struct DyVec<true> {
  uint2 raw;
  __device__ __forceinline__ void load(const void* p, int64_t off4) { raw = reinterpret_cast<const uint2*>(p)[off4]; }
  __device__ __forceinline__ float4 get() const {
    const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&raw.x));
    const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&raw.y));
    return make_float4(a.x, a.y, b.x, b.y);
  }
};
template <> struct DyVec<false> {
  float4 raw;
  __device__ __forceinline__ void load(const void* p, int64_t off4) { raw = reinterpret_cast<const float4*>(p)[off4]; }
  __device__ __forceinline__ float4 get() const { return raw; }
};

template <bool kDyBf16, int NV, bool kBias>
__global__ void __launch_bounds__(128, 4) ln_bwd_kernel(const void* __restrict__ dy_, const float* __restrict__ x,
                                                        const float* __restrict__ w, const float* __restrict__ mean,
                                                        const float* __restrict__ rstd, const float* __restrict__ dx_in,
                                                        int64_t rows, int dim, int rows_per_cta, float* __restrict__ dx_out,
                                                        uint16_t* __restrict__ dx_bf16, float* __restrict__ dw,
                                                        float* __restrict__ db) {
  extern __shared__ float s_dw[];  // 4 warps x dim (kBias: then 4 warps x dim of db partials)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int D4 = dim >> 2;
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_cta;
  const int64_t r1 = min(r0 + (int64_t)rows_per_cta, rows);
  float4 acc[NV];
#pragma unroll
  for (int j = 0; j < NV; ++j) acc[j] = make_float4(0.f, 0.f, 0.f, 0.f);
  // kBias: the d_bias partials live in this warp's own shared-memory row (only its lanes touch it, each lane its own
  // columns), not in registers -- a second register accumulator spills at dim 768 under the 128-register bound.
  float4* s_db = reinterpret_cast<float4*>(s_dw + (4 + warp) * dim);
  if (kBias) {
    for (int i = lane; i < D4; i += 32) s_db[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const float4* wr = reinterpret_cast<const float4*>(w);
  for (int64_t row = r0 + warp; row < r1; row += 4) {
    const float mu = mean[row], rs = rstd[row];
    const float4* xr = reinterpret_cast<const float4*>(x + row * dim);
    float4 xv[NV], rv[NV];  // the residual-gradient row is fetched with the other two: one memory round trip per row
    DyVec<kDyBf16> dvr[NV];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      const int i = lane + j * 32;
      if (i < D4) {
        xv[j] = xr[i];
        dvr[j].load(dy_, row * D4 + i);
        rv[j] = dx_in ? reinterpret_cast<const float4*>(dx_in + row * dim)[i] : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      const int i = lane + j * 32;
      if (i < D4) {
        const float4 wv = __ldg(wr + i);
        const float4 d = dvr[j].get();
        const float hx = (xv[j].x - mu) * rs, hy = (xv[j].y - mu) * rs, hz = (xv[j].z - mu) * rs, hw = (xv[j].w - mu) * rs;
        acc[j].x += d.x * hx; acc[j].y += d.y * hy; acc[j].z += d.z * hz; acc[j].w += d.w * hw;
        if (kBias) {
          float4 t = s_db[i];
          t.x += d.x; t.y += d.y; t.z += d.z; t.w += d.w;
          s_db[i] = t;
        }
        const float gx = d.x * wv.x, gy = d.y * wv.y, gz = d.z * wv.z, gw = d.w * wv.w;
        s1 += (gx + gy) + (gz + gw);
        s2 += (gx * hx + gy * hy) + (gz * hz + gw * hw);
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {  // both reductions in one shuffle chain
      s1 += __shfl_xor_sync(0xffffffffu, s1, o);
      s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    }
    const float m1 = s1 / dim, m2 = s2 / dim;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      const int i = lane + j * 32;
      if (i < D4) {
        const float4 wv = __ldg(wr + i);
        const float4 d = dvr[j].get();
        const float hx = (xv[j].x - mu) * rs, hy = (xv[j].y - mu) * rs, hz = (xv[j].z - mu) * rs, hw = (xv[j].w - mu) * rs;
        float4 o;
        o.x = rs * (d.x * wv.x - m1 - hx * m2);
        o.y = rs * (d.y * wv.y - m1 - hy * m2);
        o.z = rs * (d.z * wv.z - m1 - hz * m2);
        o.w = rs * (d.w * wv.w - m1 - hw * m2);
        o.x += rv[j].x; o.y += rv[j].y; o.z += rv[j].z; o.w += rv[j].w;
        reinterpret_cast<float4*>(dx_out + row * dim)[i] = o;
        if (dx_bf16) {
          uint2 pk;
          pk.x = pack_bf16(o.x, o.y);
          pk.y = pack_bf16(o.z, o.w);
          reinterpret_cast<uint2*>(dx_bf16 + row * dim)[i] = pk;
        }
      }
    }
  }
  if (!dw && !db) return;  // a frozen LayerNorm: no reduction (db is null in the no-bias instantiation)
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    const int i = lane + j * 32;
    if (i < D4) reinterpret_cast<float4*>(s_dw + warp * dim)[i] = acc[j];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < dim; c += blockDim.x) {
    float t = 0.f;
#pragma unroll
    for (int wi = 0; wi < 4; ++wi) t += s_dw[wi * dim + c];
    if (dw) atomicAdd(dw + c, t);
    if (kBias && db) {
      float tb = 0.f;
#pragma unroll
      for (int wi = 4; wi < 8; ++wi) tb += s_dw[wi * dim + c];
      atomicAdd(db + c, tb);
    }
  }
}

}  // namespace egom2p

namespace egom2p {
template <bool kBias>
static int layernorm_fwd(const float* x, const float* weight, const float* bias, int64_t rows, int32_t dim, float eps,
                         uint16_t* y_bf16, float* y_f32, float* mean, float* rstd, void* stream) {
  EGO_REQUIRE(x && weight && rows > 0 && (!kBias || bias), "layernorm_fwd: null input");
  EGO_REQUIRE(dim % 4 == 0 && dim > 0 && dim <= kLnMaxVec * 128, "layernorm_fwd: dim %d unsupported (multiple of 4, <= %d)", dim, kLnMaxVec * 128);
  EGO_REQUIRE(y_bf16 || y_f32, "layernorm_fwd: no output");
  const int nv = (dim / 4 + 31) / 32;
#define EGO_LN_FWD(NV) ln_fwd_kernel<NV, kBias><<<(unsigned)((rows + 7) / 8), 256, 0, (cudaStream_t)stream>>>(x, weight, bias, rows, dim, eps, y_bf16, y_f32, mean, rstd)
  if (nv <= 2) EGO_LN_FWD(2); else if (nv <= 3) EGO_LN_FWD(3); else if (nv <= 4) EGO_LN_FWD(4); else if (nv <= 6) EGO_LN_FWD(6);
  else if (nv <= 8) EGO_LN_FWD(8); else EGO_LN_FWD(16);
#undef EGO_LN_FWD
  return check_launch("layernorm_fwd");
}

template <bool kBias>
static int layernorm_bwd(const uint16_t* dy_bf16, const float* dy_f32, const float* x, const float* weight, const float* mean,
                         const float* rstd, const float* dx_in, int64_t rows, int32_t dim, float* dx_out, uint16_t* dx_bf16,
                         float* d_weight, float* d_bias, void* stream) {
  EGO_REQUIRE((dy_bf16 != nullptr) != (dy_f32 != nullptr), "layernorm_bwd: exactly one of dy_bf16 / dy_f32");
  // d_weight / d_bias may each be null: the gradient of a frozen LayerNorm parameter is not reduced
  EGO_REQUIRE(x && weight && mean && rstd && dx_out && rows > 0, "layernorm_bwd: null argument");
  EGO_REQUIRE(dim % 4 == 0 && dim > 0 && dim <= kLnMaxVec * 128, "layernorm_bwd: dim %d unsupported", dim);
  const int rows_per_cta = 16;
  const unsigned grid = (unsigned)((rows + rows_per_cta - 1) / rows_per_cta);
  const size_t smem = (size_t)(kBias ? 8 : 4) * dim * sizeof(float);
  const int nv = (dim / 4 + 31) / 32;
#define EGO_LN_BWD(NV)                                                                                                  \
  do {                                                                                                                  \
    if (dy_bf16) {                                                                                                      \
      if (smem > 48 * 1024) cudaFuncSetAttribute(ln_bwd_kernel<true, NV, kBias>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
      ln_bwd_kernel<true, NV, kBias><<<grid, 128, smem, (cudaStream_t)stream>>>(dy_bf16, x, weight, mean, rstd, dx_in, rows, dim, rows_per_cta, dx_out, dx_bf16, d_weight, d_bias); \
    } else {                                                                                                            \
      if (smem > 48 * 1024) cudaFuncSetAttribute(ln_bwd_kernel<false, NV, kBias>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
      ln_bwd_kernel<false, NV, kBias><<<grid, 128, smem, (cudaStream_t)stream>>>(dy_f32, x, weight, mean, rstd, dx_in, rows, dim, rows_per_cta, dx_out, dx_bf16, d_weight, d_bias); \
    }                                                                                                                   \
  } while (0)
  if (nv <= 2) EGO_LN_BWD(2); else if (nv <= 3) EGO_LN_BWD(3); else if (nv <= 4) EGO_LN_BWD(4); else if (nv <= 6) EGO_LN_BWD(6);
  else if (nv <= 8) EGO_LN_BWD(8); else EGO_LN_BWD(16);
#undef EGO_LN_BWD
  return check_launch("layernorm_bwd");
}
}  // namespace egom2p

extern "C" int egom2p_layernorm_fwd(const float* x, const float* weight, int64_t rows, int32_t dim, float eps,
                                    uint16_t* y_bf16, float* y_f32, float* mean, float* rstd, void* stream) {
  return egom2p::layernorm_fwd<false>(x, weight, nullptr, rows, dim, eps, y_bf16, y_f32, mean, rstd, stream);
}

extern "C" int egom2p_layernorm_bias_fwd(const float* x, const float* weight, const float* bias, int64_t rows, int32_t dim,
                                         float eps, uint16_t* y_bf16, float* y_f32, float* mean, float* rstd, void* stream) {
  return egom2p::layernorm_fwd<true>(x, weight, bias, rows, dim, eps, y_bf16, y_f32, mean, rstd, stream);
}

extern "C" int egom2p_layernorm_bwd(const uint16_t* dy_bf16, const float* dy_f32, const float* x, const float* weight,
                                    const float* mean, const float* rstd, const float* dx_in, int64_t rows, int32_t dim,
                                    float* dx_out, uint16_t* dx_bf16, float* d_weight, void* stream) {
  return egom2p::layernorm_bwd<false>(dy_bf16, dy_f32, x, weight, mean, rstd, dx_in, rows, dim, dx_out, dx_bf16, d_weight,
                                      nullptr, stream);
}

extern "C" int egom2p_layernorm_bias_bwd(const uint16_t* dy_bf16, const float* dy_f32, const float* x, const float* weight,
                                         const float* mean, const float* rstd, const float* dx_in, int64_t rows, int32_t dim,
                                         float* dx_out, uint16_t* dx_bf16, float* d_weight, float* d_bias, void* stream) {
  return egom2p::layernorm_bwd<true>(dy_bf16, dy_f32, x, weight, mean, rstd, dx_in, rows, dim, dx_out, dx_bf16, d_weight,
                                     d_bias, stream);
}
