// HBM-bound elementwise kernels on the path: casts, residual add, row gather / scatter, and the optimizer tail
// (multi-tensor sum of squares for the global grad-norm clip + multi-tensor AdamW, torch.optim.AdamW semantics).
// 16-byte vectorised; grid-stride with grid = 148 SMs x 8 CTAs, or one block per chunk of a device-resident item table.
#include "common.cuh"

namespace egom2p {

constexpr int kEwThreads = 256;
static inline unsigned ew_grid(int64_t nvec) {
  int64_t g = (nvec + kEwThreads - 1) / kEwThreads;
  const int64_t cap = 148 * 8;
  return (unsigned)(g < 1 ? 1 : (g > cap ? cap : g));
}

__device__ __forceinline__ void unpack8(const uint4& r, float (&f)[8]) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&r);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 t = __bfloat1622float2(h[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  uint4 r;
  r.x = pack_bf16(f[0], f[1]); r.y = pack_bf16(f[2], f[3]); r.z = pack_bf16(f[4], f[5]); r.w = pack_bf16(f[6], f[7]);
  return r;
}

__global__ void __launch_bounds__(kEwThreads) cast_kernel(const float* __restrict__ src, uint16_t* __restrict__ dst, int64_t n) {
  const int64_t n4 = n >> 2;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 v = reinterpret_cast<const float4*>(src)[i];
    uint2 pk;
    pk.x = pack_bf16(v.x, v.y);
    pk.y = pack_bf16(v.z, v.w);
    reinterpret_cast<uint2*>(dst)[i] = pk;
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
    const int64_t i = (n4 << 2) + threadIdx.x;
    __nv_bfloat16 h = __float2bfloat16(src[i]);
    dst[i] = *reinterpret_cast<uint16_t*>(&h);
  }
}

// One launch that re-casts a whole list of fp32 master weights into their bf16 GEMM operands (the per-step refresh after the
// optimizer wrote the masters). A block = one chunk of rows of one tensor, found by bisection over the items' first chunks;
// group > 0 writes the rows into the interleaved [group x fc1 | group x fc3] layout the SwiGLU-epilogue GEMM consumes.
struct CastItem {
  const float* src;
  uint16_t* dst;
  int64_t rows;
  int64_t first_chunk;
  int32_t cols, dst_ld, group, slot, rows_per_chunk, pad_;
};
static_assert(sizeof(CastItem) == 56, "CastItem layout is part of the C ABI (egom2p_cast_item)");
__global__ void __launch_bounds__(kEwThreads) cast_multi_kernel(const CastItem* __restrict__ items, int n_items) {
  __shared__ CastItem it;
  if (threadIdx.x == 0) {
    int lo = 0, hi = n_items - 1;
    while (lo < hi) {  // last item with first_chunk <= blockIdx.x
      const int mid = (lo + hi + 1) >> 1;
      if (items[mid].first_chunk <= (int64_t)blockIdx.x) lo = mid; else hi = mid - 1;
    }
    it = items[lo];
  }
  __syncthreads();
  const int64_t r0 = ((int64_t)blockIdx.x - it.first_chunk) * it.rows_per_chunk;
  const int nr = (int)min((int64_t)it.rows_per_chunk, it.rows - r0);
  auto dst_row = [&](int64_t r) -> int64_t {
    return it.group > 0 ? (r / it.group) * 2 * it.group + (int64_t)it.slot * it.group + r % it.group : r;
  };
  if ((it.cols & 3) == 0 && (it.dst_ld & 3) == 0) {
    const int c4 = it.cols >> 2;
    for (int i = threadIdx.x; i < nr * c4; i += kEwThreads) {
      const int rr = i / c4, cc = i - rr * c4;
      const float4 v = reinterpret_cast<const float4*>(it.src + (r0 + rr) * it.cols)[cc];
      uint2 pk;
      pk.x = pack_bf16(v.x, v.y);
      pk.y = pack_bf16(v.z, v.w);
      reinterpret_cast<uint2*>(it.dst + dst_row(r0 + rr) * it.dst_ld)[cc] = pk;
    }
  } else {
    for (int i = threadIdx.x; i < nr * it.cols; i += kEwThreads) {
      const int rr = i / it.cols, cc = i - rr * it.cols;
      const __nv_bfloat16 h = __float2bfloat16(it.src[(r0 + rr) * it.cols + cc]);
      it.dst[dst_row(r0 + rr) * it.dst_ld + cc] = *reinterpret_cast<const uint16_t*>(&h);
    }
  }
}

__global__ void __launch_bounds__(kEwThreads) add_kernel(const float* __restrict__ a, const float* __restrict__ b, int64_t n,
                                                         float* __restrict__ out, uint16_t* __restrict__ outb) {
  const int64_t n4 = n >> 2;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 x = reinterpret_cast<const float4*>(a)[i], y = reinterpret_cast<const float4*>(b)[i];
    const float4 o = make_float4(x.x + y.x, x.y + y.y, x.z + y.z, x.w + y.w);
    if (out) reinterpret_cast<float4*>(out)[i] = o;
    if (outb) {
      uint2 pk;
      pk.x = pack_bf16(o.x, o.y);
      pk.y = pack_bf16(o.z, o.w);
      reinterpret_cast<uint2*>(outb)[i] = pk;
    }
  }
}

// ---- optimizer tail (the reference: NativeScalerWithGradNormCount.__call__, egom2p/utils/native_scaler.py:27-47 =
// clip_grad_norm_ + optimizer.step over 245 tensors; AdamW from egom2p/utils/optim_factory.py:206-226). Two launches over
// a device-resident table of all tensors: sum of squares of every gradient -> one scalar; then AdamW with the clip
// coefficient min(1, max_norm / (norm + 1e-6)) folded into the gradient read, so the gradients are never rewritten.
// A block = one chunk of kOptChunk elements of one tensor, found by bisection over the items' first chunks.
struct OptItem {
  float* p;
  const float* g;
  float* m;
  float* v;
  int64_t n;
  int64_t first_chunk;
  float lr, wd;
};
static_assert(sizeof(OptItem) == 56, "OptItem layout is part of the C ABI (egom2p_opt_item)");
constexpr int kOptChunk = 8192;

__device__ __forceinline__ OptItem find_item(const OptItem* __restrict__ items, int n_items, OptItem* sh, int* sh_idx = nullptr) {
  if (threadIdx.x == 0) {
    int lo = 0, hi = n_items - 1;
    while (lo < hi) {  // last item with first_chunk <= blockIdx.x
      const int mid = (lo + hi + 1) >> 1;
      if (items[mid].first_chunk <= (int64_t)blockIdx.x) lo = mid; else hi = mid - 1;
    }
    *sh = items[lo];
    if (sh_idx) *sh_idx = lo;
  }
  __syncthreads();
  return *sh;
}

// Deterministic: one partial sum per block, then a single block adds the partials in a fixed order. Under data parallelism
// every rank must compute the SAME clip coefficient from the same all-reduced gradients, or the replicas' weights drift apart
// in the last bits (nothing re-synchronises weights in DDP) -- so no floating-point atomics here.
__global__ void __launch_bounds__(kEwThreads) sumsq_multi_kernel(const OptItem* __restrict__ items, int n_items, float* __restrict__ partials) {
  __shared__ OptItem sh_it;
  const OptItem it = find_item(items, n_items, &sh_it);
  const int64_t e0 = ((int64_t)blockIdx.x - it.first_chunk) * kOptChunk;
  const int ne = (int)min((int64_t)kOptChunk, it.n - e0);
  const float* g = it.g + e0;
  float s = 0.f;
  if ((reinterpret_cast<uintptr_t>(g) & 15) == 0) {
    const int n4 = ne >> 2;
    for (int i = threadIdx.x; i < n4; i += kEwThreads) {
      const float4 x = reinterpret_cast<const float4*>(g)[i];
      s += x.x * x.x + x.y * x.y + x.z * x.z + x.w * x.w;
    }
    for (int i = (n4 << 2) + threadIdx.x; i < ne; i += kEwThreads) s += g[i] * g[i];
  } else {
    for (int i = threadIdx.x; i < ne; i += kEwThreads) s += g[i] * g[i];
  }
  s = warp_sum(s);
  __shared__ float sh[kEwThreads / 32];
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = threadIdx.x < kEwThreads / 32 ? sh[threadIdx.x] : 0.f;
    t = warp_sum(t);
    if (threadIdx.x == 0) partials[blockIdx.x] = t;
  }
}
__global__ void __launch_bounds__(1024) sumsq_finalize_kernel(const float* __restrict__ partials, int64_t n, float* __restrict__ out) {
  double acc = 0.0;   // thread t adds partials t, t + 1024, ... in order; the 1024 sums are then added in a fixed tree
  for (int64_t i = threadIdx.x; i < n; i += 1024) acc += (double)partials[i];
  __shared__ double sh[1024];
  sh[threadIdx.x] = acc;
  __syncthreads();
  for (int s = 512; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) sh[threadIdx.x] += sh[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) *out = (float)sh[0];
}

__device__ __forceinline__ void adamw_one(float& p, float g, float& m, float& v, float lr, float wd, float b1, float b2, float eps,
                                          float step_size, float inv_bc2_sqrt) {
  p *= 1.f - lr * wd;
  m = b1 * m + (1.f - b1) * g;
  v = b2 * v + (1.f - b2) * g * g;
  const float denom = sqrtf(v) * inv_bc2_sqrt + eps;
  p -= step_size * (m / denom);
}

// steps[i] holds the number of steps item i took BEFORE this one (torch.optim.AdamW counts per tensor: a tensor that sat out
// steps with no gradient starts its bias correction where it left off). steps_inc_kernel advances the counts afterwards, in a
// launch of its own because every chunk of an item reads its count; nothing host-side changes from step to step, so the
// whole tail is capturable in a CUDA graph.
__global__ void __launch_bounds__(kEwThreads) adamw_multi_kernel(const OptItem* __restrict__ items, int n_items, float b1, float b2,
                                                                 float eps, const int32_t* __restrict__ steps,
                                                                 const float* __restrict__ sumsq, float max_norm) {
  __shared__ OptItem sh_it;
  __shared__ int sh_idx;
  const OptItem it = find_item(items, n_items, &sh_it, &sh_idx);
  const float t = (float)(steps[sh_idx] + 1);
  const float bc1 = 1.f - powf(b1, t), inv_bc2_sqrt = rsqrtf(1.f - powf(b2, t));
  float gs = 1.f;
  if (sumsq) {   // torch.nn.utils.clip_grad_norm_: clamp(max = 1) keeps a NaN ratio NaN, so a NaN norm poisons every update
    const float c = max_norm / (sqrtf(*sumsq) + 1e-6f);
    gs = c > 1.f ? 1.f : c;
  }
  const float step_size = it.lr / bc1;
  const int64_t e0 = ((int64_t)blockIdx.x - it.first_chunk) * kOptChunk;
  const int ne = (int)min((int64_t)kOptChunk, it.n - e0);
  float* p = it.p + e0;
  const float* g = it.g + e0;
  float* m = it.m + e0;
  float* v = it.v + e0;
  const bool aligned = ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(m) |
                         reinterpret_cast<uintptr_t>(v)) & 15) == 0;
  int done = 0;
  if (aligned) {
    const int n4 = ne >> 2;
    for (int i = threadIdx.x; i < n4; i += kEwThreads) {
      float4 pv = reinterpret_cast<float4*>(p)[i], mv = reinterpret_cast<float4*>(m)[i], vv = reinterpret_cast<float4*>(v)[i];
      const float4 gv = reinterpret_cast<const float4*>(g)[i];
      adamw_one(pv.x, gv.x * gs, mv.x, vv.x, it.lr, it.wd, b1, b2, eps, step_size, inv_bc2_sqrt);
      adamw_one(pv.y, gv.y * gs, mv.y, vv.y, it.lr, it.wd, b1, b2, eps, step_size, inv_bc2_sqrt);
      adamw_one(pv.z, gv.z * gs, mv.z, vv.z, it.lr, it.wd, b1, b2, eps, step_size, inv_bc2_sqrt);
      adamw_one(pv.w, gv.w * gs, mv.w, vv.w, it.lr, it.wd, b1, b2, eps, step_size, inv_bc2_sqrt);
      reinterpret_cast<float4*>(p)[i] = pv;
      reinterpret_cast<float4*>(m)[i] = mv;
      reinterpret_cast<float4*>(v)[i] = vv;
    }
    done = n4 << 2;
  }
  for (int i = done + threadIdx.x; i < ne; i += kEwThreads) {
    float pi = p[i], mi = m[i], vi = v[i];
    adamw_one(pi, g[i] * gs, mi, vi, it.lr, it.wd, b1, b2, eps, step_size, inv_bc2_sqrt);
    p[i] = pi; m[i] = mi; v[i] = vi;
  }
}
__global__ void steps_inc_kernel(int32_t* __restrict__ steps, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) steps[i] += 1;
}

// out[c] += sum_r x[r, c]; each CTA reduces a 64-row slab, threads own columns (coalesced), one atomic per column.
__global__ void __launch_bounds__(kEwThreads) colsum_kernel(const float* __restrict__ x, int64_t rows, int cols, float* __restrict__ out) {
  const int64_t r0 = (int64_t)blockIdx.x * 64, r1 = min(r0 + 64, rows);
  for (int c = threadIdx.x; c < cols; c += blockDim.x) {
    float s = 0.f;
    for (int64_t r = r0; r < r1; ++r) s += x[r * cols + c];
    atomicAdd(out + c, s);
  }
}

// out[c] += sum_r x[r, c] for a bf16 (R, cols) matrix of row pitch ld: the bias gradients of the GELU / bias family (R up to
// 65 536 rows per call). A CTA owns 256 columns (8 per lane, one 16-byte load) and a slab of rows; its 8 warps stride the
// slab and meet in shared memory, so each column takes one atomic per slab. The slab height is chosen on the host so that
// the grid fills the machine about four times over: ~70 atomics per column at 65 536 rows.
__global__ void __launch_bounds__(kEwThreads) colsum_bf16_kernel(const uint16_t* __restrict__ x, int64_t rows, int cols, int64_t ld,
                                                                 int64_t rows_per_cta, float* __restrict__ out) {
  __shared__ float part[kEwThreads / 32][256];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c0 = blockIdx.x * 256 + lane * 8;
  const int64_t r0 = (int64_t)blockIdx.y * rows_per_cta, r1 = min(r0 + rows_per_cta, rows);
  float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (c0 < cols) {
#pragma unroll 4
    for (int64_t r = r0 + warp; r < r1; r += kEwThreads / 32) {
      const uint4 v = __ldg(reinterpret_cast<const uint4*>(x + r * ld + c0));
      const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[t]));
        s[2 * t] += f.x;
        s[2 * t + 1] += f.y;
      }
    }
  }
#pragma unroll
  for (int t = 0; t < 8; ++t) part[warp][lane * 8 + t] = s[t];
  __syncthreads();
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (threadIdx.x < 256 && c < cols) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < kEwThreads / 32; ++w) t += part[w][threadIdx.x];
    atomicAdd(out + c, t);
  }
}

// Row gather / scatter-add used to (un)compact the rows of one modality for its vocabulary head.
__global__ void __launch_bounds__(kEwThreads) gather_rows_bf16_kernel(const uint16_t* __restrict__ src, const int64_t* __restrict__ idx,
                                                                      int64_t n, int cols8, uint16_t* __restrict__ dst) {
  const int64_t total = n * cols8;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / cols8;
    const int c = (int)(i - r * cols8);
    reinterpret_cast<uint4*>(dst)[i] = reinterpret_cast<const uint4*>(src)[idx[r] * cols8 + c];
  }
}
__global__ void __launch_bounds__(kEwThreads) scatter_rows_f32_kernel(const float* __restrict__ src, const int64_t* __restrict__ idx,
                                                                      int64_t n, int cols4, float* __restrict__ dst) {
  const int64_t total = n * cols4;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / cols4;
    const int c = (int)(i - r * cols4);
    reinterpret_cast<float4*>(dst)[idx[r] * cols4 + c] = reinterpret_cast<const float4*>(src)[i];
  }
}

}  // namespace egom2p

extern "C" int egom2p_colsum_f32(const float* x, int64_t rows, int32_t cols, float* out, void* stream) {
  using namespace egom2p;
  EGO_REQUIRE(x && out && rows > 0 && cols > 0, "colsum_f32: bad argument");
  colsum_kernel<<<(unsigned)((rows + 63) / 64), kEwThreads, 0, (cudaStream_t)stream>>>(x, rows, cols, out);
  return check_launch("colsum_f32");
}
extern "C" int egom2p_colsum_bf16(const uint16_t* x, int64_t rows, int32_t cols, int64_t ld, float* out, void* stream) {
  using namespace egom2p;
  EGO_REQUIRE(x && out && rows > 0 && cols > 0 && cols % 8 == 0 && ld % 8 == 0 && ((uintptr_t)x & 15) == 0,
              "colsum_bf16: bad argument (cols, ld multiples of 8, 16-byte aligned rows)");
  const unsigned col_blocks = (unsigned)((cols + 255) / 256);
  const int64_t want = 4 * (int64_t)device_sm_count();                     // CTAs for the whole grid
  int64_t slabs = (want + col_blocks - 1) / col_blocks;
  const int64_t min_rows = 64;                                             // keep every warp busy for a few rows
  if (slabs > (rows + min_rows - 1) / min_rows) slabs = (rows + min_rows - 1) / min_rows;
  if (slabs < 1) slabs = 1;
  const int64_t rows_per_cta = (rows + slabs - 1) / slabs;
  slabs = (rows + rows_per_cta - 1) / rows_per_cta;
  colsum_bf16_kernel<<<dim3(col_blocks, (unsigned)slabs), kEwThreads, 0, (cudaStream_t)stream>>>(x, rows, cols, ld, rows_per_cta, out);
  return check_launch("colsum_bf16");
}
extern "C" int egom2p_gather_rows_bf16(const uint16_t* src, const int64_t* idx, int64_t n, int32_t cols, uint16_t* dst, void* stream) {
  using namespace egom2p;
  EGO_REQUIRE(src && idx && dst && n > 0 && cols > 0 && cols % 8 == 0, "gather_rows_bf16: bad argument (cols %% 8 == 0)");
  gather_rows_bf16_kernel<<<ew_grid(n * (cols / 8)), kEwThreads, 0, (cudaStream_t)stream>>>(src, idx, n, cols / 8, dst);
  return check_launch("gather_rows_bf16");
}
extern "C" int egom2p_scatter_rows_f32(const float* src, const int64_t* idx, int64_t n, int32_t cols, float* dst, void* stream) {
  using namespace egom2p;
  EGO_REQUIRE(src && idx && dst && n > 0 && cols > 0 && cols % 4 == 0, "scatter_rows_f32: bad argument (cols %% 4 == 0)");
  scatter_rows_f32_kernel<<<ew_grid(n * (cols / 4)), kEwThreads, 0, (cudaStream_t)stream>>>(src, idx, n, cols / 4, dst);
  return check_launch("scatter_rows_f32");
}

extern "C" int egom2p_cast_f32_to_bf16(const float* src, uint16_t* dst, int64_t n, void* stream) {
  using namespace egom2p;
  EGO_REQUIRE(src && dst && n > 0, "cast_f32_to_bf16: bad argument");
  EGO_REQUIRE(((uintptr_t)src & 15) == 0 && ((uintptr_t)dst & 7) == 0, "cast_f32_to_bf16: misaligned");
  cast_kernel<<<ew_grid(n / 4 + 1), kEwThreads, 0, (cudaStream_t)stream>>>(src, dst, n);
  return check_launch("cast_f32_to_bf16");
}
extern "C" int egom2p_cast_f32_to_bf16_multi(const void* items_dev, int32_t n_items, int64_t n_chunks, void* stream) {
  using namespace egom2p;
  EGO_REQUIRE(items_dev && n_items > 0 && n_chunks > 0 && n_chunks < (int64_t)INT32_MAX, "cast_f32_to_bf16_multi: bad argument");
  cast_multi_kernel<<<(unsigned)n_chunks, kEwThreads, 0, (cudaStream_t)stream>>>(reinterpret_cast<const CastItem*>(items_dev), n_items);
  return check_launch("cast_f32_to_bf16_multi");
}
extern "C" int egom2p_add_f32(const float* a, const float* b, int64_t n, float* out, uint16_t* out_bf16, void* stream) {
  using namespace egom2p;
  EGO_REQUIRE(a && b && (out || out_bf16) && n > 0 && n % 4 == 0, "add_f32: bad argument (n %% 4 == 0 required)");
  add_kernel<<<ew_grid(n / 4), kEwThreads, 0, (cudaStream_t)stream>>>(a, b, n, out, out_bf16);
  return check_launch("add_f32");
}
extern "C" int egom2p_sumsq_multi(const void* items_dev, int32_t n_items, int64_t n_chunks, float* partials, float* sumsq,
                                  void* stream) {
  using namespace egom2p;
  EGO_REQUIRE(items_dev && sumsq && partials && n_items > 0 && n_chunks > 0 && n_chunks < (int64_t)INT32_MAX, "sumsq_multi: bad argument");
  sumsq_multi_kernel<<<(unsigned)n_chunks, kEwThreads, 0, (cudaStream_t)stream>>>(reinterpret_cast<const OptItem*>(items_dev), n_items, partials);
  int rc = check_launch("sumsq_multi");
  if (rc) return rc;
  sumsq_finalize_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(partials, n_chunks, sumsq);
  return check_launch("sumsq_multi finalize");
}
extern "C" int egom2p_adamw_multi_steps(const void* items_dev, int32_t n_items, int64_t n_chunks, float beta1, float beta2,
                                        float eps, int32_t* steps, const float* sumsq, float max_norm, void* stream) {
  using namespace egom2p;
  EGO_REQUIRE(items_dev && steps && n_items > 0 && n_chunks > 0 && n_chunks < (int64_t)INT32_MAX, "adamw_multi_steps: bad argument");
  adamw_multi_kernel<<<(unsigned)n_chunks, kEwThreads, 0, (cudaStream_t)stream>>>(reinterpret_cast<const OptItem*>(items_dev), n_items,
                                                                                 beta1, beta2, eps, steps, sumsq, max_norm);
  int rc = check_launch("adamw_multi_steps");
  if (rc) return rc;
  steps_inc_kernel<<<(unsigned)((n_items + kEwThreads - 1) / kEwThreads), kEwThreads, 0, (cudaStream_t)stream>>>(steps, n_items);
  return check_launch("adamw_multi_steps increment");
}
