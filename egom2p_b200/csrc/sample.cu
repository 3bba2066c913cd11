// Fused token sampling for generation (SURVEY.md section 8(f) row 1): temperature + top-k + top-p (nucleus) filtering +
// one categorical draw per row, straight from fp32 logits, in ONE pass over each row.
//
// Reference: GenerationSampler.sample_tokens / top_k_top_p_filtering (egom2p/models/generate.py:332-371):
//   top-k : logits below the k-th largest value are removed;
//   top-p : sort descending, softmax (temperature 1) over what top-k left, cumulative sum; a token is removed when the
//           mass of the tokens ranked strictly above it exceeds top_p (the first token that crosses top_p is kept);
//   draw  : probs = softmax(kept / temperature), one sample (torch.multinomial); temperature ~ 0 -> argmax, prob 1.
// The reference does this with a full 64k-wide sort, a softmax, a cumsum, two gathers / argsorts and a second softmax over
// a (rows, V) fp32 tensor. Here one CTA owns one row and streams it a handful of times (the caller sizes row chunks to stay
// in the 126 MB L2): it finds the nucleus threshold with three rounds of a 2048-bin histogram over the value range that
// accumulates probability MASS per bin instead of counts -- no sort, no second copy of the logits. The draw is an
// inverse-CDF walk in ascending token order with a caller-supplied uniform u[row] (so the result is a deterministic
// function of logits and u).
#include <cfloat>

#include "common.cuh"

namespace egom2p {

constexpr int kSmpThreads = 1024;
constexpr int kSmpBins = 2048;

__device__ __forceinline__ float block_max_f(float v, float* sh) {
  v = warp_max(v);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) sh[warp] = v;
  __syncthreads();
  if (warp == 0) {
    float t = sh[lane];
    t = warp_max(t);
    if (lane == 0) sh[32] = t;
  }
  __syncthreads();
  return sh[32];
}
__device__ __forceinline__ float block_sum_f(float v, float* sh) {
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) sh[warp] = v;
  __syncthreads();
  if (warp == 0) {
    float t = sh[lane];
    t = warp_sum(t);
    if (lane == 0) sh[32] = t;
  }
  __syncthreads();
  return sh[32];
}
// exclusive prefix sum over the block in thread order; *total = block sum
__device__ __forceinline__ float block_excl_scan_f(float v, float* sh, float* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  __syncthreads();
  if (lane == 31) sh[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    const float w = sh[lane];
    float winc = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const float t = __shfl_up_sync(0xffffffffu, winc, o);
      if (lane >= o) winc += t;
    }
    sh[lane] = winc - w;
    if (lane == 31) sh[32] = winc;
  }
  __syncthreads();
  *total = sh[32];
  return inc - v + sh[warp];
}

// One row of logits, streamed from L2 / HBM in 16-byte pieces: element v = 4 * (t + kSmpThreads * k) + c.
struct RowReader {
  const float* src;
  int V;
  __device__ __forceinline__ int chunks() const { return (V + 4 * kSmpThreads - 1) / (4 * kSmpThreads); }
  __device__ __forceinline__ void load(int k, float (&q)[4], int& v0) const {
    v0 = 4 * ((int)threadIdx.x + kSmpThreads * k);
    if (v0 + 3 < V) {
      const float4 f = *reinterpret_cast<const float4*>(src + v0);
      q[0] = f.x; q[1] = f.y; q[2] = f.z; q[3] = f.w;
    } else {
#pragma unroll
      for (int c = 0; c < 4; ++c) q[c] = (v0 + c < V) ? src[v0 + c] : -FLT_MAX;
    }
  }
};

// A threshold found by up to three nested rounds of 2048 linear bins over the value range (bin 0 = largest logits). An
// element is classified by recomputing its bin chain with the very expressions the search used, so membership is exact and
// consistent between the search rounds and the later passes (no floating-point edge effects at bin borders).
struct Thresh {
  int n;          // rounds used; 0 = keep everything
  float hi[3], inv[3];
  int sel[3];
  __device__ __forceinline__ int bin(int r, float x) const { return min(kSmpBins - 1, max(0, (int)((hi[r] - x) * inv[r]))); }
  __device__ __forceinline__ bool keep(float x) const {   // x is at or above the threshold
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      if (r < n) {
        const int b = bin(r, x);
        if (b < sel[r]) return true;
        if (b > sel[r]) return false;
      }
    }
    return true;
  }
  __device__ __forceinline__ bool inside(int rounds, float x) const {   // x lies in the selected bins of the first `rounds` rounds
#pragma unroll
    for (int r = 0; r < 3; ++r)
      if (r < rounds && bin(r, x) != sel[r]) return false;
    return true;
  }
};

// Finds the first element -- in descending order of value -- whose inclusive cumulative weight reaches the target (MASS:
// weight = exp(x - gmax), reached when > target; else weight 1, reached when >= target), among the elements `base` keeps.
// The final bin is (gmax - gmin) / 2^33 wide: below one ulp of the logits for any realistic range, i.e. it holds one distinct
// value (ties are kept together). If the target is never reached, everything is kept (n = 0).
template <bool MASS>
__device__ Thresh find_threshold(const RowReader& rr, float gmax, float gmin, const Thresh& base, float target, float* hist,
                                 float* sh, float* s_f, int* s_i) {
  Thresh th;
  th.n = 0;
  float hi = gmax, lo = gmin;
  float above = 0.f;
  const int nchunk = rr.chunks();
  for (int r = 0; r < 3; ++r) {
    const float width = (hi - lo) / (float)kSmpBins;
    if (!(width > 0.f)) break;                  // interval collapsed to one value
    th.hi[r] = hi;
    th.inv[r] = 1.f / width;
    for (int i = threadIdx.x; i < kSmpBins; i += kSmpThreads) hist[i] = 0.f;
    __syncthreads();
    for (int k = 0; k < nchunk; ++k) {
      float q[4];
      int v0;
      rr.load(k, q, v0);
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const float x = q[c];
        if (v0 + c < rr.V && base.keep(x) && th.inside(r, x)) atomicAdd(&hist[th.bin(r, x)], MASS ? __expf(x - gmax) : 1.f);
      }
    }
    __syncthreads();
    // thread t owns bins 2t, 2t+1 (descending value order)
    const float h0 = hist[2 * threadIdx.x], h1 = hist[2 * threadIdx.x + 1];
    float tot;
    const float excl = block_excl_scan_f(h0 + h1, sh, &tot);
    if (threadIdx.x == 0) *s_i = -1;
    __syncthreads();
    const float c0 = above + excl, c1 = c0 + h0, c2 = c1 + h1;
    const bool hit0 = MASS ? (c0 <= target && c1 > target && h0 > 0.f) : (c0 < target && c1 >= target);
    const bool hit1 = MASS ? (c1 <= target && c2 > target && h1 > 0.f) : (c1 < target && c2 >= target);
    if (hit0) { *s_i = 2 * threadIdx.x; *s_f = c0; }
    else if (hit1) { *s_i = 2 * threadIdx.x + 1; *s_f = c1; }
    __syncthreads();
    const int bsel = *s_i;
    const float ab = *s_f;
    __syncthreads();
    if (bsel < 0) {                             // target never reached: keep everything `base` keeps
      th.n = 0;
      return th;
    }
    above = ab;
    th.sel[r] = bsel;
    th.n = r + 1;
    const float nhi = hi - (float)bsel * width;
    lo = hi - (float)(bsel + 1) * width;
    hi = nhi;
  }
  return th;
}

struct SampleParams {
  const float* logits;
  int64_t ld;
  int rows, V;
  float temperature, top_p;
  int top_k;
  const float* u;
  int64_t* token;
  float* prob;
  int32_t* n_kept;
};

__global__ void __launch_bounds__(kSmpThreads, 1) sample_rows_kernel(SampleParams p) {
  __shared__ float hist[kSmpBins];
  __shared__ float sh[33];
  __shared__ float s_f;
  __shared__ int s_i;
  __shared__ float s_chunk[64];
  const int row = blockIdx.x, t = threadIdx.x;
  RowReader rr{p.logits + (int64_t)row * p.ld, p.V};
  const int nchunk = rr.chunks();   // <= 16 for V <= 65536

  // ---- pass A: max (with the lowest index attaining it) and min
  float mx = -FLT_MAX, mn = FLT_MAX;
  int amax = 0x7fffffff;
  for (int k = 0; k < nchunk; ++k) {
    float q[4];
    int v0;
    rr.load(k, q, v0);
#pragma unroll
    for (int c = 0; c < 4; ++c)
      if (v0 + c < p.V) {
        if (q[c] > mx) { mx = q[c]; amax = v0 + c; }
        mn = fminf(mn, q[c]);
      }
  }
  const float gmax = block_max_f(mx, sh);
  const float gmin = -block_max_f(-mn, sh);
  const bool greedy = fabsf(p.temperature) <= 1e-10f;   // np.isclose(temperature, 0, atol=1e-10)
  if (greedy) {   // torch.argmax: the first maximal element
    if (t == 0) s_i = 0x7fffffff;
    __syncthreads();
    if (mx == gmax) atomicMin(&s_i, amax);
    __syncthreads();
    if (t == 0) {
      p.token[row] = s_i;
      if (p.prob) p.prob[row] = 1.f;
      if (p.n_kept) p.n_kept[row] = 1;
    }
    return;
  }

  // ---- top-k: the k-th largest logit (everything below it is removed)
  Thresh none;
  none.n = 0;
  Thresh tk = none, tp = none;
  if (p.top_k > 0 && p.top_k < p.V) tk = find_threshold<false>(rr, gmax, gmin, none, (float)p.top_k, hist, sh, &s_f, &s_i);

  // ---- top-p over what is left: mass = exp(logit - max) (temperature 1, as the reference)
  if (p.top_p > 0.f) {
    float zs = 0.f;
    for (int k = 0; k < nchunk; ++k) {
      float q[4];
      int v0;
      rr.load(k, q, v0);
#pragma unroll
      for (int c = 0; c < 4; ++c)
        if (v0 + c < p.V && tk.keep(q[c])) zs += __expf(q[c] - gmax);
    }
    const float Z = block_sum_f(zs, sh);
    tp = find_threshold<true>(rr, gmax, gmin, tk, p.top_p * Z, hist, sh, &s_f, &s_i);
  }

  // ---- draw from softmax(kept / temperature): inverse CDF in ascending token order, chunk by chunk
  const float invT = 1.f / p.temperature;
  float mine[16];
  int kept = 0;
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    mine[k] = 0.f;
    if (k < nchunk) {
      float q[4];
      int v0;
      rr.load(k, q, v0);
#pragma unroll
      for (int c = 0; c < 4; ++c)
        if (v0 + c < p.V && tk.keep(q[c]) && tp.keep(q[c])) { mine[k] += __expf((q[c] - gmax) * invT); ++kept; }
    }
  }
  // chunk totals: chunk k = tokens [4096 k, 4096 (k + 1))
  if (t < 64) s_chunk[t] = 0.f;
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    const float ws = warp_sum(mine[k]);
    if ((t & 31) == 0 && ws != 0.f) atomicAdd(&s_chunk[k], ws);
  }
  __syncthreads();
  float ZT = 0.f;
#pragma unroll
  for (int k = 0; k < 16; ++k) ZT += s_chunk[k];
  const float target = fminf(fmaxf(p.u[row], 0.f), 0.99999994f) * ZT;
  int ksel = -1;
  float before = 0.f;
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    if (ksel < 0 && s_chunk[k] > 0.f) {
      if (target < before + s_chunk[k]) ksel = k; else before += s_chunk[k];
    }
  }
  if (ksel < 0) {   // rounding at the very end: the last chunk that holds a kept token
#pragma unroll
    for (int k = 0; k < 16; ++k) if (s_chunk[k] > 0.f) ksel = k;
    before = 0.f;
#pragma unroll
    for (int k = 0; k < 16; ++k) if (k < ksel) before += s_chunk[k];
  }
  float myw = 0.f;
#pragma unroll
  for (int k = 0; k < 16; ++k) if (k == ksel) myw = mine[k];
  float tot;
  const float pre = before + block_excl_scan_f(myw, sh, &tot);
  if (t == 0) s_i = 0x7fffffff;
  __syncthreads();
  float q[4];
  int v0;
  rr.load(ksel, q, v0);
  float w4[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) w4[c] = (v0 + c < p.V && tk.keep(q[c]) && tp.keep(q[c])) ? __expf((q[c] - gmax) * invT) : 0.f;
  // The owner of the target is the first thread, in token order, with weight whose inclusive prefix pre + myw exceeds it
  // (searchsorted). Claiming pre <= target < pre + myw instead would leave gaps: the next thread's pre comes out of the scan
  // along a different rounding path than pre + myw and can exceed it by an ulp. The first candidate of every warp enters
  // a block min-reduction over token indices.
  const unsigned cand = __ballot_sync(0xffffffffu, myw > 0.f && target < pre + myw);
  if (cand != 0u && (t & 31) == __ffs(cand) - 1) {
    float cacc = pre;
    int pick = -1;
#pragma unroll
    for (int c = 0; c < 4; ++c)
      if (pick < 0 && w4[c] > 0.f) { cacc += w4[c]; if (target < cacc) pick = c; }
    if (pick < 0) {
#pragma unroll
      for (int c = 0; c < 4; ++c) if (w4[c] > 0.f) pick = c;
    }
    atomicMin(&s_i, v0 + pick);
  }
  __syncthreads();
  if (s_i == 0x7fffffff) {   // the target lies past the chunk's last bound (chunk sums and scan round differently): its last kept token
    __syncthreads();
    if (t == 0) s_i = -1;
    __syncthreads();
    int last = -1;
#pragma unroll
    for (int c = 0; c < 4; ++c) if (w4[c] > 0.f) last = v0 + c;
    if (last >= 0) atomicMax(&s_i, last);
    __syncthreads();
  }
  const int win = s_i;
  if (win >= v0 && win < v0 + 4) {
    p.token[row] = win;
    if (p.prob) p.prob[row] = w4[win - v0] / ZT;
  }
  if (p.n_kept) {
    const float kc = block_sum_f((float)kept, sh);
    if (t == 0) p.n_kept[row] = (int)(kc + 0.5f);
  }
}

// y = a + (b - a) * scale, fp32 -> bf16: classifier-free guidance applied to the decoder outputs BEFORE the vocabulary head.
// The head is linear without bias, so W(y_u + s (y_c - y_u)) == l_u + s (l_c - l_u) (generate.py:804): one head GEMM
// instead of two, and the combined logits are the only ones ever formed.
__global__ void __launch_bounds__(256) cfg_combine_kernel(const float* __restrict__ yu, const float* __restrict__ yc, int64_t n4,
                                                          float scale, uint16_t* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 a = reinterpret_cast<const float4*>(yu)[i], b = reinterpret_cast<const float4*>(yc)[i];
    uint2 pk;
    pk.x = pack_bf16(fmaf(b.x - a.x, scale, a.x), fmaf(b.y - a.y, scale, a.y));
    pk.y = pack_bf16(fmaf(b.z - a.z, scale, a.z), fmaf(b.w - a.w, scale, a.w));
    reinterpret_cast<uint2*>(out)[i] = pk;
  }
}

}  // namespace egom2p

extern "C" int egom2p_sample_rows(const float* logits, int64_t ld, int32_t rows, int32_t V, float temperature, float top_p,
                                  int32_t top_k, const float* u, int64_t* token, float* prob, int32_t* n_kept, void* stream) {
  using namespace egom2p;
  EGO_REQUIRE(logits && u && token && rows > 0 && V > 0, "sample_rows: bad argument");
  EGO_REQUIRE(V <= kSmpThreads * 64, "sample_rows: vocabulary %d exceeds %d", V, kSmpThreads * 64);
  EGO_REQUIRE(ld % 4 == 0 && ((uintptr_t)logits & 15) == 0, "sample_rows: logits must be 16-byte aligned with ld %% 4 == 0");
  EGO_REQUIRE(temperature >= 0.f && top_p >= 0.f && top_k >= 0, "sample_rows: negative temperature / top_p / top_k");
  SampleParams p{logits, ld, rows, V, temperature, top_p, top_k, u, token, prob, n_kept};
  sample_rows_kernel<<<rows, kSmpThreads, 0, (cudaStream_t)stream>>>(p);
  return check_launch("sample_rows");
}

extern "C" int egom2p_cfg_combine_bf16(const float* y_uncond, const float* y_cond, int64_t n, float scale, uint16_t* out,
                                       void* stream) {
  using namespace egom2p;
  EGO_REQUIRE(y_uncond && y_cond && out && n > 0 && n % 4 == 0, "cfg_combine_bf16: bad argument (n %% 4 == 0 required)");
  const int64_t n4 = n / 4;
  const int64_t g = (n4 + 255) / 256;
  cfg_combine_kernel<<<(unsigned)(g < 148 * 8 ? g : 148 * 8), 256, 0, (cudaStream_t)stream>>>(y_uncond, y_cond, n4, scale, out);
  return check_launch("cfg_combine_bf16");
}
