// Shared device/host helpers for libast_b200.so (sm_100a only).
#pragma once
#include <cstring>
#include <cstdlib>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>

#include "../../include/ast.h"

namespace ast {

// ---- error plumbing (no C++ exceptions cross the ABI; SURVEY 8b "Errors") ----
void set_error(const char* fmt, ...);
extern std::atomic<long long> g_launches;
inline void count_launch(int n = 1) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// ---- per-kernel-family accounting (ast_family_stats): launches + ALGORITHMIC flops / bytes computed from the launch
// geometry on the host.  bench.py divides these by the device time of the same family in the CUDA-graph replay; the
// tests use the launch counts to assert which kernel a case really ran on.
enum Family {
  FAM_CONV_TC = 0, FAM_CONV_PX, FAM_CONV_WS, FAM_CONV_HX, FAM_CONV_SIMT, FAM_WGRAD_TC, FAM_WGRAD_THIN, FAM_WGRAD_SIMT, FAM_GRAM_TC,
  FAM_GRAM_SIMT, FAM_IN_APPLY, FAM_IN_BWD, FAM_IN_STATS, FAM_POOL, FAM_MSE, FAM_POINTWISE, FAM_OPTIM, FAM_CONV_ST, FAM_COUNT
};
void count_work(int family, double flops, double bytes);
inline double esize(const ast_image* im) { return im->dtype == AST_F32 ? 4.0 : (im->dtype == AST_U8 ? 1.0 : 2.0); }
inline double img_bytes(const ast_image* im) { return im ? (double)im->n * im->h * im->w * im->c * esize(im) : 0.0; }
inline double conv_flops(const ast_image* in, const ast_image* out, const ast_gather_geom* g) {
  return 2.0 * in->n * g->mi * g->mj * g->ntaps * in->c * out->c;
}
// input pixels the launch covers (a phase of a strided op touches 1/so^2 of the output and all of its input window)
inline double conv_bytes(const ast_image* in, const ast_image* out, const ast_gather_geom* g, const ast_image* add = nullptr,
                         const ast_image* mask = nullptr) {
  double pix_in = (double)g->mi * g->mj * g->si * g->si;
  if (pix_in > (double)in->h * in->w) pix_in = (double)in->h * in->w;
  const double pix_out = (double)g->mi * g->mj;
  return in->n * (pix_in * in->c * esize(in) + pix_out * out->c * (esize(out) + (add ? esize(add) : 0) + (mask ? esize(mask) : 0)));
}

#define AST_CHECK_ARG(cond, ...)                    \
  do {                                              \
    if (!(cond)) {                                  \
      ast::set_error(__VA_ARGS__);                  \
      return -1;                                    \
    }                                               \
  } while (0)

#define AST_CUDA_LAUNCH_CHECK()                                             \
  do {                                                                      \
    cudaError_t e__ = cudaGetLastError();                                   \
    if (e__ != cudaSuccess) {                                               \
      ast::set_error("%s:%d launch failed: %s", __FILE__, __LINE__,         \
                     cudaGetErrorString(e__));                              \
      return (int)e__;                                                      \
    }                                                                       \
  } while (0)

// Every kernel of the library is launched through launch_k() (one place for launch attributes).  Programmatic dependent
// launch was measured slower on this path (early-scheduled successors take SM slots from multi-wave kernels:
// 13.86 vs 13.55 ms per step, profiles/r01_summary.md) and is not used.
template <typename... KP, typename... A>
inline cudaError_t launch_k(void (*kernel)(KP...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, A&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KP>(args)...);
}

// ---- device-side image view ----
struct Img {
  char* ptr;
  int dtype;
  int n, h, w, c;
  long long sn, sh, sw, sc;
};

inline Img to_img(const ast_image* a) {
  Img r;
  r.ptr = (char*)a->ptr; r.dtype = a->dtype; r.n = a->n; r.h = a->h; r.w = a->w; r.c = a->c;
  r.sn = a->sn; r.sh = a->sh; r.sw = a->sw; r.sc = a->sc;
  return r;
}
inline Img null_img() { Img r; r.ptr = nullptr; r.dtype = 0; r.n = r.h = r.w = r.c = 0; r.sn = r.sh = r.sw = r.sc = 0; return r; }
inline bool same_shape(const ast_image* a, const ast_image* b) {
  return a->n == b->n && a->h == b->h && a->w == b->w && a->c == b->c;
}

template <typename T> struct DT;
template <> struct DT<float> {
  static constexpr int id = AST_F32;
  __device__ static __forceinline__ float ld(const float* p) { return *p; }
  __device__ static __forceinline__ void st(float* p, float v) { *p = v; }
};
template <> struct DT<__nv_bfloat16> {
  static constexpr int id = AST_BF16;
  __device__ static __forceinline__ float ld(const __nv_bfloat16* p) { return __bfloat162float(*p); }
  __device__ static __forceinline__ void st(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
};

// AST_U8 (host-boundary images): loads widen exactly; stores follow numpy's `.clip(0, 255).astype('uint8')`
// (inference.py:116, train_cnn.py:112): clamp, then truncate toward zero.
// AST_F16 stores saturate (an fp32 value beyond +-65504 must not become inf)
__device__ __forceinline__ __half f2h_sat(float v) { return __float2half_rn(fminf(fmaxf(v, -65504.f), 65504.f)); }
// two values as one 32-bit word of 16-bit elements, a in the low half.  F16 is a COMPILE-TIME choice: callers test the
// element type once per chunk, never per element (a per-element test doubles the conversion instructions of the epilogue)
template <bool F16>
__device__ __forceinline__ unsigned pack2(float a, float b) {
  if (F16) { const __half2 h = __halves2half2(f2h_sat(a), f2h_sat(b)); return *reinterpret_cast<const unsigned*>(&h); }
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const unsigned*>(&h);
}
__device__ __forceinline__ unsigned pack2_16(int dtype, float a, float b) { return dtype == AST_F16 ? pack2<true>(a, b) : pack2<false>(a, b); }
__device__ __forceinline__ float ld_elem(const Img& im, long long off) {
  if (im.dtype == AST_F32) return ((const float*)im.ptr)[off];
  if (im.dtype == AST_U8) return (float)((const unsigned char*)im.ptr)[off];
  if (im.dtype == AST_BF16) return __bfloat162float(((const __nv_bfloat16*)im.ptr)[off]);
  return __half2float(((const __half*)im.ptr)[off]);
}
__device__ __forceinline__ void st_elem(const Img& im, long long off, float v) {
  if (im.dtype == AST_F32) ((float*)im.ptr)[off] = v;
  else if (im.dtype == AST_BF16) ((__nv_bfloat16*)im.ptr)[off] = __float2bfloat16_rn(v);
  else if (im.dtype == AST_F16) ((__half*)im.ptr)[off] = f2h_sat(v);
  else ((unsigned char*)im.ptr)[off] = (unsigned char)__float2uint_rz(fminf(fmaxf(v, 0.f), 255.f));
}
__device__ __forceinline__ long long img_off(const Img& im, int n, int y, int x, int c) {
  return (long long)n * im.sn + (long long)y * im.sh + (long long)x * im.sw + (long long)c * im.sc;
}
// nn.ReflectionPad2d index rule (no edge repeat): -1 -> 1, H -> H-2
__device__ __forceinline__ int reflect_idx(int i, int n) {
  if (i < 0) i = -i;
  if (i >= n) i = 2 * (n - 1) - i;
  return i;
}
// Adjoint of reflect padding by pad < H, W: besides the centre (i + pad, j + pad), the positions (r, c) of the
// (H+2pad) x (W+2pad) grid that reflect_idx maps onto interior pixel (i, j).  add(r, c) is called for each of them in a
// fixed order (rows: centre, top mirror, bottom mirror; columns likewise), so every caller sums in the same order.
template <typename F>
__device__ __forceinline__ void reflect_fold_border(int pad, int H, int W, int i, int j, F&& add) {
  const int r1 = (i >= 1 && i <= pad) ? pad - i : -1;
  const int r2 = (i <= H - 2 && i >= H - 1 - pad) ? pad + 2 * (H - 1) - i : -1;
  const int c1 = (j >= 1 && j <= pad) ? pad - j : -1;
  const int c2 = (j <= W - 2 && j >= W - 1 - pad) ? pad + 2 * (W - 1) - j : -1;
#pragma unroll
  for (int a_ = 0; a_ < 3; ++a_) {
    const int r = a_ == 0 ? i + pad : (a_ == 1 ? r1 : r2);
    if (r < 0) continue;
#pragma unroll
    for (int b_ = 0; b_ < 3; ++b_) {
      const int cc = b_ == 0 ? j + pad : (b_ == 1 ? c1 : c2);
      if (cc < 0 || (a_ == 0 && b_ == 0)) continue;
      add(r, cc);
    }
  }
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// 16-byte vector of elements (4 fp32 / 8 bf16) unpacked to floats
template <typename T> struct Vec16;
template <> struct Vec16<float> {
  static constexpr int N = 4;
  __device__ static __forceinline__ void load(const float* p, float* out) {
    float4 v = *reinterpret_cast<const float4*>(p);
    out[0] = v.x; out[1] = v.y; out[2] = v.z; out[3] = v.w;
  }
  __device__ static __forceinline__ void store(float* p, const float* in) {
    *reinterpret_cast<float4*>(p) = make_float4(in[0], in[1], in[2], in[3]);
  }
};
template <> struct Vec16<__nv_bfloat16> {
  static constexpr int N = 8;
  __device__ static __forceinline__ void load(const __nv_bfloat16* p, float* out) {
    uint4 v = *reinterpret_cast<const uint4*>(p);
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
    for (int i = 0; i < 4; ++i) { float2 f = __bfloat1622float2(h[i]); out[2 * i] = f.x; out[2 * i + 1] = f.y; }
  }
  __device__ static __forceinline__ void store(__nv_bfloat16* p, const float* in) {
    uint4 v;
    __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&v);
#pragma unroll
    for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(in[2 * i], in[2 * i + 1]);
    *reinterpret_cast<uint4*>(p) = v;
  }
};

// 4 consecutive channels (16 B fp32 / 8 B bf16); offsets must be multiples of 4 elements
__device__ __forceinline__ void ld4(const float* p, float* v) {
  const float4 f = *reinterpret_cast<const float4*>(p);
  v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w;
}
__device__ __forceinline__ void ld4(const __nv_bfloat16* p, float* v) {
  const uint2 u = *reinterpret_cast<const uint2*>(p);
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
  const float2 f0 = __bfloat1622float2(h[0]), f1 = __bfloat1622float2(h[1]);
  v[0] = f0.x; v[1] = f0.y; v[2] = f1.x; v[3] = f1.y;
}
__device__ __forceinline__ void st4(float* p, const float* v) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
}
__device__ __forceinline__ void st4(__nv_bfloat16* p, const float* v) {
  uint2 u;
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
  h[0] = __floats2bfloat162_rn(v[0], v[1]);
  h[1] = __floats2bfloat162_rn(v[2], v[3]);
  *reinterpret_cast<uint2*>(p) = u;
}
__device__ __forceinline__ void ld4(const __half* p, float* v) {
  const uint2 u = *reinterpret_cast<const uint2*>(p);
  const __half2* h = reinterpret_cast<const __half2*>(&u);
  const float2 f0 = __half22float2(h[0]), f1 = __half22float2(h[1]);
  v[0] = f0.x; v[1] = f0.y; v[2] = f1.x; v[3] = f1.y;
}
__device__ __forceinline__ void ld4_img(const Img& im, long long off, float* v) {
  if (im.dtype == AST_F32) ld4((const float*)im.ptr + off, v);
  else if (im.dtype == AST_BF16) ld4((const __nv_bfloat16*)im.ptr + off, v);
  else ld4((const __half*)im.ptr + off, v);
}
__device__ __forceinline__ void st4_img(const Img& im, long long off, const float* v) {
  if (im.dtype == AST_F32) st4((float*)im.ptr + off, v);
  else if (im.dtype == AST_BF16) st4((__nv_bfloat16*)im.ptr + off, v);
  else *reinterpret_cast<uint2*>((__half*)im.ptr + off) = make_uint2(pack2<true>(v[0], v[1]), pack2<true>(v[2], v[3]));
}

inline int num_sms() {
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (sms <= 0) sms = 148;
  }
  return sms;
}

}  // namespace ast
