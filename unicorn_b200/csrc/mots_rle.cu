// MOTS mask tail on the device (unicorn/evaluators/mot_evaluator.py:804-805,858-866,882-888): the soft masks of the tracked
// instances are resized to the original frame (F.interpolate(scale_factor, bilinear, align_corners=False)[:img_h, :img_w]),
// thresholded, made overlap free in ascending track-id order and run-length encoded into COCO compressed RLE strings
// (results.rle_encode), so that only the strings leave the device.
//   mots_pack_kernel   resize + threshold + overlap-free; bit-packs every emitted mask column-major, one 32-pixel word per
//                      (column, 32-row group), bit b = row 32*wy + b (rows past the frame are zero)
//   mots_rle_kernel    one CTA per mask: run boundaries = set bits of w ^ (w << 1 | previous pixel), scanned into counts, each
//                      count's character length scanned into offsets; pass 1 measures the strings, pass 2 writes them
#include "uc_common.h"
#include "../../include/unicorn_b200.h"
#include <algorithm>
#include <climits>
#include <cmath>

namespace uc {

constexpr int kRleThreads = 1024;
constexpr int kRleSmem = (3 + 32 * kRleThreads) * 4;  // 3 carried boundaries + at most 32 per word of the chunk

// Source index of F.interpolate(bilinear, align_corners=False) with a given source scale (PyTorch's
// area_pixel_compute_source_index, the rule vos_aggregate_kernel and bilinear_kernel use).
__device__ __forceinline__ void bilinear_src(int d, float scale, int n, int& i0, int& i1, float& l) {
  const float f = fmaxf((d + 0.5f) * scale - 0.5f, 0.f);
  i0 = min(static_cast<int>(f), n - 1);
  i1 = min(i0 + 1, n - 1);
  l = f - i0;
}

// block (32 columns, 8 row groups); thread = one packed word of one column, all K masks in list order
__global__ void __launch_bounds__(256) mots_pack_kernel(const float* __restrict__ masks, int n_max, int Hin, int Win,
                                                         const int* __restrict__ rows, const int* __restrict__ emit, int K, int he,
                                                         int we, int WY, float thres, float scale, uint32_t* __restrict__ packed) {
  __shared__ int sy0[256], sy1[256];
  __shared__ float sly[256];
  pdl_wait();
  pdl_launch_dependents();
  const int tx = threadIdx.x, ty = threadIdx.y, i = ty * 32 + tx;
  {
    int y0, y1;
    float ly;
    bilinear_src(blockIdx.y * 256 + i, scale, Hin, y0, y1, ly);
    sy0[i] = y0 * Win;
    sy1[i] = y1 * Win;
    sly[i] = ly;
  }
  __syncthreads();
  const int x = blockIdx.x * 32 + tx, wy = blockIdx.y * 8 + ty;
  if (x >= we || wy >= WY) return;
  int x0, x1;
  float lx;
  bilinear_src(x, scale, Win, x0, x1, lx);
  const int nb = min(32, he - wy * 32);
  const long row_words = static_cast<long>(we) * WY;
  uint32_t claimed = 0;
#pragma unroll 1
  for (int k = 0; k < K; ++k) {
    const int r = rows[k];
    uint32_t bits = 0;
    if (r >= 0 && r < n_max) {
      const float* s = masks + static_cast<long>(r) * Hin * Win;
#pragma unroll 4
      for (int b = 0; b < nb; ++b) {
        const int j = ty * 32 + b;
        const float* s0 = s + sy0[j];
        const float* s1 = s + sy1[j];
        const float ly = sly[j];
        const float v = (1.f - ly) * ((1.f - lx) * s0[x0] + lx * s0[x1]) + ly * ((1.f - lx) * s1[x0] + lx * s1[x1]);
        bits |= static_cast<uint32_t>(v > thres) << b;
      }
    }
    if (emit[k]) packed[k * row_words + static_cast<long>(x) * WY + wy] = bits & ~claimed;
    claimed |= bits;  // rows outside the area filter still claim their pixels (mot_evaluator.py:860-866 runs before :882)
  }
}

template <typename T>
__device__ __forceinline__ T block_exclusive_scan(T v, T* tmp, T& total) {  // tmp: 33 elements of shared memory
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  T inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const T n = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += n;
  }
  if (lane == 31) tmp[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    const T own = lane < static_cast<int>(blockDim.x >> 5) ? tmp[lane] : T(0);
    T s = own;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const T n = __shfl_up_sync(0xffffffffu, s, o);
      if (lane >= o) s += n;
    }
    tmp[lane] = s - own;
    if (lane == 31) tmp[32] = s;
  }
  __syncthreads();
  const T r = inc - v + tmp[warp];
  total = tmp[32];
  __syncthreads();
  return r;
}

// one count of maskApi.c rleToString: 5 data bits per character, continuation bit 0x20, offset 48; returns the length
__device__ __forceinline__ int rle_put(long long x, char* out) {
  int n = 0;
  bool more = true;
  while (more) {
    int ch = static_cast<int>(x & 0x1f);
    x >>= 5;
    more = (ch & 0x10) ? x != -1 : x != 0;
    if (more) ch |= 0x20;
    if (out) out[n] = static_cast<char>(ch + 48);
    ++n;
  }
  return n;
}

// Value stored for count i = m + l, where the chunk's boundaries are a[3 + l] = P_{m+1+l}, a[0..2] = P_{m-2}, P_{m-1}, P_m, P_0 = 0:
// c_i = P_{i+1} - P_i, minus c_{i-2} when i > 2 (rleToString's delta rule, results.rle_encode).
__device__ __forceinline__ long long rle_value(const int* a, int l, long long m) {
  long long x = static_cast<long long>(a[3 + l]) - a[2 + l];
  if (m + l > 2) x -= static_cast<long long>(a[1 + l]) - a[l];
  return x;
}

// kWrite = false: out_len[k] = length of mask k's string (0 when not emitted).  kWrite = true: out_off[k] = sum of the earlier
// lengths, *out_total = all of them, and the string is written at chars + out_off[k] when it fits in capacity.
template <bool kWrite>
__global__ void __launch_bounds__(kRleThreads) mots_rle_kernel(const uint32_t* __restrict__ packed, int he, int we, int WY,
                                                                const int* __restrict__ emit, int K, long long* __restrict__ out_len,
                                                                long long* __restrict__ out_off, long long* __restrict__ out_total,
                                                                char* __restrict__ chars, long capacity) {
  extern __shared__ int spos[];
  __shared__ long long scan_ll[33];
  __shared__ int scan_i[33];
  pdl_wait();
  pdl_launch_dependents();
  const int k = blockIdx.x, t = threadIdx.x;
  long long row_off = 0;
  if (kWrite) {
    long long s = 0;
    for (int j = t; j < k; j += kRleThreads) s += out_len[j];
    block_exclusive_scan(s, scan_ll, row_off);
    if (t == 0) {
      out_off[k] = row_off;
      if (k == K - 1) *out_total = row_off + out_len[k];
    }
    if (!emit[k] || row_off + out_len[k] > capacity) return;
  } else if (!emit[k]) {
    if (t == 0) out_len[k] = 0;
    return;
  }
  const long row_words = static_cast<long>(we) * WY;
  const uint32_t* bits = packed + k * row_words;
  const int nwords = static_cast<int>(row_words), tail = he & 31;
  if (t < 3) spos[t] = 0;
  long long m = 0, nch = 0;  // boundaries and characters so far
  __syncthreads();
  for (int base = 0; base < nwords; base += kRleThreads) {
    const int w = base + t;
    uint32_t d = 0;
    int lin0 = 0;
    if (w < nwords) {
      const int x = w / WY, wy = w - x * WY;
      const uint32_t v = bits[w];
      uint32_t prev = 0;  // the pixel before this word in column-major order; 0 before the first, so a leading 1 gives count 0
      if (wy > 0) prev = bits[w - 1] >> 31;
      else if (x > 0) prev = (bits[w - 1] >> ((he - 1) & 31)) & 1u;
      const uint32_t valid = (wy == WY - 1 && tail) ? (1u << tail) - 1u : 0xffffffffu;
      d = (v ^ ((v << 1) | prev)) & valid;
      lin0 = x * he + wy * 32;
    }
    int nb;
    int e = block_exclusive_scan(static_cast<int>(__popc(d)), scan_i, nb);
    if (nb == 0) continue;
    while (d) {
      spos[3 + e++] = lin0 + __ffs(d) - 1;
      d &= d - 1;
    }
    __syncthreads();
    const int per = (nb + kRleThreads - 1) / kRleThreads;
    const int l0 = min(t * per, nb), l1 = min(l0 + per, nb);
    int n = 0;
    for (int l = l0; l < l1; ++l) n += rle_put(rle_value(spos, l, m), nullptr);
    int nc;
    const int ce = block_exclusive_scan(n, scan_i, nc);
    if (kWrite) {
      char* o = chars + row_off + nch + ce;
      for (int l = l0; l < l1; ++l) o += rle_put(rle_value(spos, l, m), o);
    }
    const int c0 = spos[nb], c1 = spos[nb + 1], c2 = spos[nb + 2];  // P_{m+nb-2}, P_{m+nb-1}, P_{m+nb}
    __syncthreads();
    if (t == 0) { spos[0] = c0; spos[1] = c1; spos[2] = c2; }
    m += nb;
    nch += nc;
    __syncthreads();
  }
  if (t == 0) {  // the last run ends at the end of the mask
    long long x = static_cast<long long>(he) * we - spos[2];
    if (m > 2) x -= static_cast<long long>(spos[1]) - spos[0];
    if (kWrite) rle_put(x, chars + row_off + nch);
    else out_len[k] = nch + rle_put(x, nullptr);
  }
}

// encoded size: the resized map (floor(Hin * sf) x floor(Win * sf), in double like F.interpolate) cropped to the frame
static bool mots_sizes(int Hin, int Win, int img_h, int img_w, double sf, int& he, int& we) {
  if (Hin < 1 || Win < 1 || img_h < 1 || img_w < 1 || !(sf > 0.0) || !std::isfinite(sf)) return false;
  he = static_cast<int>(std::min<double>(img_h, std::floor(Hin * sf)));
  we = static_cast<int>(std::min<double>(img_w, std::floor(Win * sf)));
  return he >= 1 && we >= 1 && static_cast<long>(he) * we <= INT_MAX;
}

}  // namespace uc

using namespace uc;

extern "C" long uc_mots_rle_workspace_bytes(int K, int Hin, int Win, int img_h, int img_w, double scale_factor) {
  int he, we;
  if (K < 1 || !mots_sizes(Hin, Win, img_h, img_w, scale_factor, he, we)) return 0;
  return static_cast<long>(K) * we * ((he + 31) / 32) * 4;
}

extern "C" int uc_mots_masks_rle(const float* masks, int n_max, int Hin, int Win, const int* rows, const int* emit, int K, int img_h,
                                 int img_w, float thres, double scale_factor, void* workspace, long workspace_bytes, long long* out_len,
                                 long long* out_off, long long* out_total, char* out_chars, long capacity, void* stream_v) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  if (!masks || !rows || !emit || !workspace || !out_len || !out_off || !out_total || !out_chars)
    return set_error(UC_EINVAL, "uc_mots_masks_rle: null pointer");
  if (n_max < 1 || K < 1 || K > n_max) return set_error(UC_EINVAL, "uc_mots_masks_rle: K = %d rows of %d masks (need 1 <= K <= n_max)", K, n_max);
  if (Hin < 1 || Win < 1 || img_h < 1 || img_w < 1)
    return set_error(UC_EINVAL, "uc_mots_masks_rle: non-positive sizes (%dx%d masks, %dx%d frame)", Hin, Win, img_h, img_w);
  if (!(scale_factor > 0.0) || !std::isfinite(scale_factor)) return set_error(UC_EINVAL, "uc_mots_masks_rle: scale_factor must be positive");
  int he, we;
  if (!mots_sizes(Hin, Win, img_h, img_w, scale_factor, he, we))
    return set_error(UC_EINVAL, "uc_mots_masks_rle: the resized %dx%d map at scale %g is empty or too large", Hin, Win, scale_factor);
  if (capacity < 1) return set_error(UC_EINVAL, "uc_mots_masks_rle: capacity must be positive");
  if (workspace_bytes < uc_mots_rle_workspace_bytes(K, Hin, Win, img_h, img_w, scale_factor))
    return set_error(UC_EINVAL, "uc_mots_masks_rle: workspace too small");
  static PerDeviceFlag attr_dev;
  bool& attr = attr_dev.get();
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(mots_rle_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRleSmem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(mots_rle_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRleSmem);
    if (e != cudaSuccess) return set_error(static_cast<int>(e), "uc_mots_masks_rle: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    attr = true;
  }
  const int WY = (he + 31) / 32;
  uint32_t* packed = static_cast<uint32_t*>(workspace);
  launch_pdl(mots_pack_kernel, dim3((we + 31) / 32, (WY + 7) / 8), dim3(32, 8), 0, stream, masks, n_max, Hin, Win, rows, emit, K, he, we, WY,
             thres, static_cast<float>(1.0 / scale_factor), packed);
  launch_pdl(mots_rle_kernel<false>, K, kRleThreads, kRleSmem, stream, packed, he, we, WY, emit, K, out_len, out_off, out_total, out_chars, capacity);
  launch_pdl(mots_rle_kernel<true>, K, kRleThreads, kRleSmem, stream, packed, he, we, WY, emit, K, out_len, out_off, out_total, out_chars, capacity);
  return check_launch("uc_mots_masks_rle");
}
