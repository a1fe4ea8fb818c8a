// HBM-bound elementwise / reduction kernels of the path: max-pool (fwd, bwd fused with tap-gradient add and
// ReLU mask), MSE (loss + gradient seed), layout/dtype copies and the reflect-padding adjoint, feature accumulation,
// Gram (SIMT).
// Replaces aten::max_pool2d_with_indices(+backward), aten::threshold_backward, aten::mse_loss(+backward),
// aten::add_ / aten::add at train_cnn.py:54,239,300-301,307,323, aten::reflection_pad2d_backward at cnn.py:58.
#include "common.cuh"

namespace ast {

constexpr int NT = 256;

__device__ __forceinline__ unsigned pool_code(float a, float b, float c, float d) {
  int arg = 0; float m = a;
  if (b > m) { m = b; arg = 1; }
  if (c > m) { m = c; arg = 2; }
  if (d > m) { m = d; arg = 3; }
  return (unsigned)arg | ((a > 0.f) ? 4u : 0u) | ((b > 0.f) ? 8u : 0u) | ((c > 0.f) ? 16u : 0u) | ((d > 0.f) ? 32u : 0u);
}

__global__ void __launch_bounds__(NT) maxpool2_fwd_kernel(Img x, Img y, Img codes) {
  const int lanes = x.c / 4;
  const long long total = (long long)y.n * y.h * y.w * lanes;
  for (long long idx = blockIdx.x * (long long)NT + threadIdx.x; idx < total; idx += (long long)gridDim.x * NT) {
    const int c = (int)(idx % lanes) * 4;
    long long r = idx / lanes;
    const int j = (int)(r % y.w); r /= y.w;
    const int i = (int)(r % y.h);
    const int n = (int)(r / y.h);
    float m[4], v0[4], v1[4], v2[4], v3[4];
    ld4_img(x, img_off(x, n, 2 * i, 2 * j, c), v0);
    ld4_img(x, img_off(x, n, 2 * i, 2 * j + 1, c), v1);
    ld4_img(x, img_off(x, n, 2 * i + 1, 2 * j, c), v2);
    ld4_img(x, img_off(x, n, 2 * i + 1, 2 * j + 1, c), v3);
#pragma unroll
    for (int e = 0; e < 4; ++e) m[e] = fmaxf(fmaxf(v0[e], v1[e]), fmaxf(v2[e], v3[e]));
    st4_img(y, img_off(y, n, i, j, c), m);
    if (codes.ptr) {
      unsigned pk = 0;
#pragma unroll
      for (int e = 0; e < 4; ++e) pk |= pool_code(v0[e], v1[e], v2[e], v3[e]) << (8 * e);
      *reinterpret_cast<unsigned*>(codes.ptr + img_off(codes, n, i, j, c)) = pk;
    }
  }
}

// Backward of ReLU + MaxPool2d from the 1-byte window codes: 8 channels per thread (16-byte bf16 vectors).
//   gx[2i+dy, 2j+dx] = (gadd[2i+dy, 2j+dx] + (arg == 2dy+dx ? gy[i, j] : 0)) * bit(2dy+dx)
__global__ void __launch_bounds__(NT) maxpool2_bwd_codes_kernel(Img codes, Img gy, Img gadd, Img gx) {
  const int lanes = gx.c / 8;
  const long long total = (long long)gy.n * gy.h * gy.w * lanes;
  for (long long idx = blockIdx.x * (long long)NT + threadIdx.x; idx < total; idx += (long long)gridDim.x * NT) {
    const int c = (int)(idx % lanes) * 8;
    long long r = idx / lanes;
    const int j = (int)(r % gy.w); r /= gy.w;
    const int i = (int)(r % gy.h);
    const int n = (int)(r / gy.h);
    const uint2 cw = *reinterpret_cast<const uint2*>(codes.ptr + img_off(codes, n, i, j, c));
    float g[8];
    ld4_img(gy, img_off(gy, n, i, j, c), g); ld4_img(gy, img_off(gy, n, i, j, c + 4), g + 4);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int yy = 2 * i + (k >> 1), xx = 2 * j + (k & 1);
      float o[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      if (gadd.ptr) { ld4_img(gadd, img_off(gadd, n, yy, xx, c), o); ld4_img(gadd, img_off(gadd, n, yy, xx, c + 4), o + 4); }
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const unsigned code = ((e < 4 ? cw.x : cw.y) >> (8 * (e & 3))) & 0xffu;
        if ((int)(code & 3u) == k) o[e] += g[e];
        o[e] = (code >> (2 + k)) & 1u ? o[e] : 0.f;
      }
      st4_img(gx, img_off(gx, n, yy, xx, c), o); st4_img(gx, img_off(gx, n, yy, xx, c + 4), o + 4);
    }
  }
}

// one thread per 2x2 window (ceil-div grid so odd trailing rows/cols of x still get gadd*mask)
__global__ void __launch_bounds__(NT) maxpool2_bwd_kernel(Img x, Img gy, Img gadd, Img gx) {
  const int lanes = x.c / 4;
  const int wh = (x.h + 1) / 2, ww = (x.w + 1) / 2;
  const long long total = (long long)x.n * wh * ww * lanes;
  for (long long idx = blockIdx.x * (long long)NT + threadIdx.x; idx < total; idx += (long long)gridDim.x * NT) {
    const int c = (int)(idx % lanes) * 4;
    long long r = idx / lanes;
    const int j = (int)(r % ww); r /= ww;
    const int i = (int)(r % wh);
    const int n = (int)(r / wh);
    const bool pooled = i < gy.h && j < gy.w;   // window fully inside x (floor semantics of MaxPool2d)
    float xv[4][4], g[4] = {0.f, 0.f, 0.f, 0.f};
    int arg[4] = {0, 0, 0, 0};
    if (pooled) {
      ld4_img(gy, img_off(gy, n, i, j, c), g);
#pragma unroll
      for (int k = 0; k < 4; ++k) ld4_img(x, img_off(x, n, 2 * i + (k >> 1), 2 * j + (k & 1), c), xv[k]);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        float m = xv[0][e];
#pragma unroll
        for (int k = 1; k < 4; ++k)
          if (xv[k][e] > m) { m = xv[k][e]; arg[e] = k; }   // first maximum wins, like ATen
      }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int yy = 2 * i + (k >> 1), xx = 2 * j + (k & 1);
      if (yy >= x.h || xx >= x.w) continue;
      if (!pooled) ld4_img(x, img_off(x, n, yy, xx, c), xv[k]);
      float o[4] = {0.f, 0.f, 0.f, 0.f};
      if (gadd.ptr) ld4_img(gadd, img_off(gadd, n, yy, xx, c), o);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        if (pooled && arg[e] == k) o[e] += g[e];
        o[e] = xv[k][e] > 0.f ? o[e] : 0.f;
      }
      st4_img(gx, img_off(gx, n, yy, xx, c), o);
    }
  }
}

__global__ void __launch_bounds__(NT) mse_kernel(Img a, Img b, float* loss, float scale, Img grad, float gscale) {
  const long long total = (long long)a.n * a.h * a.w * a.c;
  float part = 0.f;
  for (long long idx = blockIdx.x * (long long)NT + threadIdx.x; idx < total; idx += (long long)gridDim.x * NT) {
    const int c = (int)(idx % a.c);
    long long r = idx / a.c;
    const int x = (int)(r % a.w); r /= a.w;
    const int y = (int)(r % a.h);
    const int n = (int)(r / a.h);
    const float d = ld_elem(a, img_off(a, n, y, x, c)) - ld_elem(b, img_off(b, n, y, x, c));
    part = fmaf(d, d, part);
    if (grad.ptr) st_elem(grad, img_off(grad, n, y, x, c), gscale * d);
  }
  __shared__ float red[NT / 32];
  part = warp_sum(part);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = part;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < NT / 32 ? red[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0 && loss) atomicAdd(loss, v * scale);
  }
}

// vectorised NHWC variant of the same thing (all images sc == 1, c % 4 == 0)
__global__ void __launch_bounds__(NT) mse_vec_kernel(Img a, Img b, float* loss, float scale, Img grad, float gscale) {
  const int lanes = a.c / 4;
  const long long total = (long long)a.n * a.h * a.w * lanes;
  float part = 0.f;
  for (long long idx = blockIdx.x * (long long)NT + threadIdx.x; idx < total; idx += (long long)gridDim.x * NT) {
    const int c = (int)(idx % lanes) * 4;
    long long r = idx / lanes;
    const int x = (int)(r % a.w); r /= a.w;
    const int y = (int)(r % a.h);
    const int n = (int)(r / a.h);
    float u[4], v[4];
    ld4_img(a, img_off(a, n, y, x, c), u);
    ld4_img(b, img_off(b, n, y, x, c), v);
#pragma unroll
    for (int e = 0; e < 4; ++e) { u[e] -= v[e]; part = fmaf(u[e], u[e], part); u[e] *= gscale; }
    if (grad.ptr) st4_img(grad, img_off(grad, n, y, x, c), u);
  }
  __shared__ float red[NT / 32];
  part = warp_sum(part);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = part;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < NT / 32 ? red[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0 && loss) atomicAdd(loss, v * scale);
  }
}

__global__ void __launch_bounds__(NT) copy_image_kernel(Img src, Img dst, const float* __restrict__ shift, int pad) {
  const long long total = (long long)dst.n * dst.h * dst.w * dst.c;
  // iterate in the destination's fastest-varying order for coalesced writes
  const bool chan_fast = dst.sc == 1;
  for (long long idx = blockIdx.x * (long long)NT + threadIdx.x; idx < total; idx += (long long)gridDim.x * NT) {
    int n, y, x, c;
    long long r = idx;
    if (chan_fast) { c = (int)(r % dst.c); r /= dst.c; x = (int)(r % dst.w); r /= dst.w; y = (int)(r % dst.h); n = (int)(r / dst.h); }
    else { x = (int)(r % dst.w); r /= dst.w; y = (int)(r % dst.h); r /= dst.h; c = (int)(r % dst.c); n = (int)(r / dst.c); }
    float v = 0.f;
    if (c < src.c) {
      const int i = reflect_idx(y - pad, src.h), j = reflect_idx(x - pad, src.w);
      v = ld_elem(src, img_off(src, n, i, j, c));
      if (shift) v += shift[c];
    }
    st_elem(dst, img_off(dst, n, y, x, c), v);
  }
}

// adjoint of copy_image_kernel's reflect padding: one thread per output element, in the output's fastest-varying order
__global__ void __launch_bounds__(NT) reflect_fold_kernel(Img gpad, Img add, Img out, int pad) {
  const long long total = (long long)out.n * out.h * out.w * out.c;
  const bool chan_fast = out.sc == 1;
  for (long long idx = blockIdx.x * (long long)NT + threadIdx.x; idx < total; idx += (long long)gridDim.x * NT) {
    int n, y, x, c;
    long long r = idx;
    if (chan_fast) { c = (int)(r % out.c); r /= out.c; x = (int)(r % out.w); r /= out.w; y = (int)(r % out.h); n = (int)(r / out.h); }
    else { x = (int)(r % out.w); r /= out.w; y = (int)(r % out.h); r /= out.h; c = (int)(r % out.c); n = (int)(r / out.c); }
    float v = ld_elem(gpad, img_off(gpad, n, y + pad, x + pad, c));
    reflect_fold_border(pad, out.h, out.w, y, x, [&](int yy, int xx) { v += ld_elem(gpad, img_off(gpad, n, yy, xx, c)); });
    if (add.ptr) v += ld_elem(add, img_off(add, n, y, x, c));
    st_elem(out, img_off(out, n, y, x, c), v);
  }
}

// acc += sum over the batch of x when acc holds ONE image (acc.n == 1), else acc[n] += x[n]
__global__ void __launch_bounds__(NT) accumulate_kernel(Img x, Img acc) {
  const int nsum = acc.n == 1 ? x.n : 1;
  const long long total = (long long)(acc.n == 1 ? 1 : x.n) * x.h * x.w * x.c;
  for (long long idx = blockIdx.x * (long long)NT + threadIdx.x; idx < total; idx += (long long)gridDim.x * NT) {
    const int c = (int)(idx % x.c);
    long long r = idx / x.c;
    const int xx = (int)(r % x.w); r /= x.w;
    const int y = (int)(r % x.h);
    const int n = (int)(r / x.h);
    float* p = (float*)acc.ptr + img_off(acc, n, y, xx, c);
    float s = *p;
    for (int k = 0; k < nsum; ++k) s += ld_elem(x, img_off(x, n + k, y, xx, c));
    *p = s;
  }
}

// vectorised NHWC variant (4 channels per thread)
__global__ void __launch_bounds__(NT) accumulate_vec_kernel(Img x, Img acc) {
  const int nsum = acc.n == 1 ? x.n : 1;
  const int lanes = x.c / 4;
  const long long total = (long long)(acc.n == 1 ? 1 : x.n) * x.h * x.w * lanes;
  for (long long idx = blockIdx.x * (long long)NT + threadIdx.x; idx < total; idx += (long long)gridDim.x * NT) {
    const int c = (int)(idx % lanes) * 4;
    long long r = idx / lanes;
    const int xx = (int)(r % x.w); r /= x.w;
    const int y = (int)(r % x.h);
    const int n = (int)(r / x.h);
    float s[4], v[4];
    const long long ao = img_off(acc, n, y, xx, c);
    ld4((const float*)acc.ptr + ao, s);
    for (int k = 0; k < nsum; ++k) {
      ld4_img(x, img_off(x, n + k, y, xx, c), v);
#pragma unroll
      for (int e = 0; e < 4; ++e) s[e] += v[e];
    }
    st4((float*)acc.ptr + ao, s);
  }
}

__global__ void __launch_bounds__(NT) mask_add_kernel(Img a, Img b, Img mask, Img out) {
  const long long total = (long long)a.n * a.h * a.w * a.c;
  for (long long idx = blockIdx.x * (long long)NT + threadIdx.x; idx < total; idx += (long long)gridDim.x * NT) {
    const int c = (int)(idx % a.c);
    long long r = idx / a.c;
    const int xx = (int)(r % a.w); r /= a.w;
    const int y = (int)(r % a.h);
    const int n = (int)(r / a.h);
    float v = ld_elem(a, img_off(a, n, y, xx, c));
    if (b.ptr) v += ld_elem(b, img_off(b, n, y, xx, c));
    if (mask.ptr) v = ld_elem(mask, img_off(mask, n, y, xx, c)) > 0.f ? v : 0.f;
    st_elem(out, img_off(out, n, y, xx, c), v);
  }
}

// 4 channels per thread (16 B fp32 / 8 B bf16 accesses); mixed dtypes allowed
__global__ void __launch_bounds__(NT) mask_add_vec_kernel(Img a, Img b, Img mask, Img out) {
  const int lanes = a.c / 4;
  const long long total = (long long)a.n * a.h * a.w * lanes;
  for (long long idx = blockIdx.x * (long long)NT + threadIdx.x; idx < total; idx += (long long)gridDim.x * NT) {
    const int c = (int)(idx % lanes) * 4;
    long long r = idx / lanes;
    const int xx = (int)(r % a.w); r /= a.w;
    const int y = (int)(r % a.h);
    const int n = (int)(r / a.h);
    float v[4], t[4];
    ld4_img(a, img_off(a, n, y, xx, c), v);
    if (b.ptr) {
      ld4_img(b, img_off(b, n, y, xx, c), t);
#pragma unroll
      for (int e = 0; e < 4; ++e) v[e] += t[e];
    }
    if (mask.ptr) {
      ld4_img(mask, img_off(mask, n, y, xx, c), t);
#pragma unroll
      for (int e = 0; e < 4; ++e) v[e] = t[e] > 0.f ? v[e] : 0.f;
    }
    st4_img(out, img_off(out, n, y, xx, c), v);
  }
}

static bool vec_ok(const ast_image* x) {
  return x->sc == 1 && x->c % 4 == 0 && x->sw % 4 == 0 && x->sh % 4 == 0 && x->sn % 4 == 0;
}
static int blocks_for(long long total) {
  long long b = (total + NT - 1) / NT;
  const long long cap = (long long)num_sms() * 16;
  return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}

int launch_wgrad_simt(const ast_image* x, const ast_image* gout, float* dw, const int32_t* tap_off,
                      int64_t s_co, int64_t s_ci, const ast_gather_geom* geom, int64_t dw_img_stride, float scale,
                      cudaStream_t s);  // gather_simt.cu
int gram_tc(const ast_image* x, float* g, float scale, const float* target, long long target_img_stride, double* loss,
            float loss_scale, float* dmat, float d_scale, int* counters, cudaStream_t s);  // contract_tc.cu

// strict-mode finish of ast_gram_mse after the FFMA Gram: loss += loss_scale * sum (G - S)^2 ; D = d_scale * (G - S)
__global__ void __launch_bounds__(NT) gram_finish_kernel(const float* __restrict__ g, const float* __restrict__ target,
                                                          long long target_img_stride, long long cc, long long total,
                                                          double* loss, float loss_scale, float* __restrict__ dmat, float d_scale) {
  float part = 0.f;
  for (long long idx = blockIdx.x * (long long)NT + threadIdx.x; idx < total; idx += (long long)gridDim.x * NT) {
    const long long img = idx / cc, r = idx - img * cc;
    const float d = g[idx] - target[img * target_img_stride + r];
    part = fmaf(d, d, part);
    if (dmat) dmat[idx] = d_scale * d;
  }
  __shared__ float red[NT / 32];
  part = warp_sum(part);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = part;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < NT / 32 ? red[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0 && loss) atomicAdd(loss, (double)v * (double)loss_scale);
  }
}

}  // namespace ast

using namespace ast;

static bool codes_ok(const ast_image* codes, const ast_image* pooled_like) {
  return codes->dtype == AST_U8 && same_shape(codes, pooled_like) && codes->sc == 1 && codes->c % 8 == 0 && codes->sw % 8 == 0 &&
         codes->sh % 8 == 0 && codes->sn % 8 == 0 && ((uintptr_t)codes->ptr & 7) == 0;
}

extern "C" int ast_maxpool2_fwd(const ast_image* x, const ast_image* y, const ast_image* codes, void* stream) {
  AST_CHECK_ARG(x && y, "ast_maxpool2_fwd: null argument");
  AST_CHECK_ARG(vec_ok(x) && vec_ok(y), "ast_maxpool2_fwd: needs NHWC, C %% 4 == 0");
  AST_CHECK_ARG(y->n == x->n && y->c == x->c && y->h == x->h / 2 && y->w == x->w / 2, "ast_maxpool2_fwd: y must be (h/2, w/2)");
  AST_CHECK_ARG(!codes || codes_ok(codes, y), "ast_maxpool2_fwd: codes must be uint8 NHWC [n, h/2, w/2, c], C %% 8 == 0");
  const long long total = (long long)y->n * y->h * y->w * (y->c / 4);
  if (total == 0) return 0;
  launch_k(maxpool2_fwd_kernel, blocks_for(total), NT, 0, (cudaStream_t)stream, to_img(x), to_img(y), codes ? to_img(codes) : null_img());
  count_launch();
  count_work(FAM_POOL, 0.0, img_bytes(x) + img_bytes(y));
  AST_CUDA_LAUNCH_CHECK();
  return 0;
}

extern "C" int ast_maxpool2_bwd(const ast_image* x, const ast_image* codes, const ast_image* gy, const ast_image* gadd,
                                const ast_image* gx, void* stream) {
  AST_CHECK_ARG((x || codes) && gy && gx, "ast_maxpool2_bwd: null argument");
  if (codes) {
    AST_CHECK_ARG(codes_ok(codes, gy), "ast_maxpool2_bwd: codes must be uint8 NHWC shaped like gy, C %% 8 == 0");
    AST_CHECK_ARG(gx->n == gy->n && gx->c == gy->c && gx->h == 2 * gy->h && gx->w == 2 * gy->w,
                  "ast_maxpool2_bwd: the code path needs even h, w (gx = 2 x gy)");
    AST_CHECK_ARG(vec_ok(gy) && vec_ok(gx) && (!gadd || (vec_ok(gadd) && same_shape(gadd, gx))), "ast_maxpool2_bwd: needs NHWC, C %% 4 == 0");
    const long long tot = (long long)gy->n * gy->h * gy->w * (gy->c / 8);
    if (tot == 0) return 0;
    launch_k(maxpool2_bwd_codes_kernel, blocks_for(tot), NT, 0, (cudaStream_t)stream, to_img(codes), to_img(gy),
             gadd ? to_img(gadd) : null_img(), to_img(gx));
    count_launch();
    count_work(FAM_POOL, 0.0, img_bytes(codes) + img_bytes(gy) + img_bytes(gadd) + img_bytes(gx));
    AST_CUDA_LAUNCH_CHECK();
    return 0;
  }
  AST_CHECK_ARG(vec_ok(x) && vec_ok(gy) && vec_ok(gx) && (!gadd || vec_ok(gadd)), "ast_maxpool2_bwd: needs NHWC, C %% 4 == 0");
  AST_CHECK_ARG(gy->n == x->n && gy->c == x->c && gy->h == x->h / 2 && gy->w == x->w / 2, "ast_maxpool2_bwd: gy must be (h/2, w/2)");
  AST_CHECK_ARG(same_shape(gx, x) && (!gadd || same_shape(gadd, x)), "ast_maxpool2_bwd: gx/gadd shape");
  const long long total = (long long)x->n * ((x->h + 1) / 2) * ((x->w + 1) / 2) * (x->c / 4);
  if (total == 0) return 0;
  launch_k(maxpool2_bwd_kernel, blocks_for(total), NT, 0, (cudaStream_t)stream, to_img(x), to_img(gy), gadd ? to_img(gadd) : null_img(), to_img(gx));
  count_launch();
  count_work(FAM_POOL, 0.0, img_bytes(x) + img_bytes(gy) + img_bytes(gadd) + img_bytes(gx));
  AST_CUDA_LAUNCH_CHECK();
  return 0;
}

extern "C" int ast_mse(const ast_image* a, const ast_image* b, float* loss, float scale, const ast_image* grad,
                       float gscale, void* stream) {
  AST_CHECK_ARG(a && b, "ast_mse: null argument");
  AST_CHECK_ARG(same_shape(a, b) && (!grad || same_shape(grad, a)), "ast_mse: shape mismatch");
  const long long total = (long long)a->n * a->h * a->w * a->c;
  if (total == 0) return 0;
  Img gi = grad ? to_img(grad) : null_img();
  if (vec_ok(a) && vec_ok(b) && (!grad || vec_ok(grad)))
    launch_k(mse_vec_kernel, blocks_for(total / 4), NT, 0, (cudaStream_t)stream, to_img(a), to_img(b), loss, scale, gi, gscale);
  else
    launch_k(mse_kernel, blocks_for(total), NT, 0, (cudaStream_t)stream, to_img(a), to_img(b), loss, scale, gi, gscale);
  count_launch();
  count_work(FAM_MSE, 0.0, img_bytes(a) + img_bytes(b) + img_bytes(grad));
  AST_CUDA_LAUNCH_CHECK();
  return 0;
}

extern "C" int ast_copy_image(const ast_image* src, const ast_image* dst, const float* shift, int32_t pad, void* stream) {
  AST_CHECK_ARG(src && dst, "ast_copy_image: null argument");
  AST_CHECK_ARG(dst->n == src->n && dst->h == src->h + 2 * pad && dst->w == src->w + 2 * pad && dst->c >= src->c,
                "ast_copy_image: dst must be (h+2p, w+2p, c>=src.c)");
  AST_CHECK_ARG(pad < src->h && pad < src->w, "ast_copy_image: pad too large");
  const long long total = (long long)dst->n * dst->h * dst->w * dst->c;
  if (total == 0) return 0;
  launch_k(copy_image_kernel, blocks_for(total), NT, 0, (cudaStream_t)stream, to_img(src), to_img(dst), shift, pad);
  count_launch();
  count_work(FAM_POINTWISE, 0.0, img_bytes(src) + img_bytes(dst));
  AST_CUDA_LAUNCH_CHECK();
  return 0;
}

static bool f32_or_bf16(const ast_image* x) { return x->dtype == AST_F32 || x->dtype == AST_BF16; }

extern "C" int ast_reflect_fold(const ast_image* gpad, const ast_image* add, const ast_image* out, int32_t pad, void* stream) {
  AST_CHECK_ARG(gpad && out, "ast_reflect_fold: null argument");
  AST_CHECK_ARG(f32_or_bf16(gpad) && f32_or_bf16(out) && (!add || f32_or_bf16(add)),
                "ast_reflect_fold: gpad, add and out must be fp32 or bf16");
  AST_CHECK_ARG(pad >= 0 && pad < out->h && pad < out->w, "ast_reflect_fold: pad must be >= 0 and < h, w");
  AST_CHECK_ARG(gpad->n == out->n && gpad->c == out->c && gpad->h == out->h + 2 * pad && gpad->w == out->w + 2 * pad,
                "ast_reflect_fold: gpad must be (n, h+2p, w+2p, c) of out");
  AST_CHECK_ARG(!add || same_shape(add, out), "ast_reflect_fold: add must be shaped like out");
  const long long total = (long long)out->n * out->h * out->w * out->c;
  if (total == 0) return 0;
  launch_k(reflect_fold_kernel, blocks_for(total), NT, 0, (cudaStream_t)stream, to_img(gpad), add ? to_img(add) : null_img(),
           to_img(out), pad);
  count_launch();
  count_work(FAM_POINTWISE, 0.0, img_bytes(gpad) + img_bytes(add) + img_bytes(out));
  AST_CUDA_LAUNCH_CHECK();
  return 0;
}

extern "C" int ast_accumulate(const ast_image* x, const ast_image* acc, void* stream) {
  AST_CHECK_ARG(x && acc, "ast_accumulate: null argument");
  AST_CHECK_ARG(acc->dtype == AST_F32 && acc->h == x->h && acc->w == x->w && acc->c == x->c && (acc->n == x->n || acc->n == 1),
                "ast_accumulate: acc must be fp32 of the same shape (or hold one image: batch sum)");
  const long long total = (long long)(acc->n == 1 ? 1 : x->n) * x->h * x->w * x->c;
  if (total == 0 || x->n == 0) return 0;
  if (vec_ok(x) && vec_ok(acc))
    launch_k(accumulate_vec_kernel, blocks_for(total / 4), NT, 0, (cudaStream_t)stream, to_img(x), to_img(acc));
  else
    launch_k(accumulate_kernel, blocks_for(total), NT, 0, (cudaStream_t)stream, to_img(x), to_img(acc));
  count_launch();
  count_work(FAM_POINTWISE, 0.0, img_bytes(x) + 2.0 * img_bytes(acc));
  AST_CUDA_LAUNCH_CHECK();
  return 0;
}

extern "C" int ast_mask_add(const ast_image* a, const ast_image* b, const ast_image* mask, const ast_image* out, void* stream) {
  AST_CHECK_ARG(a && out, "ast_mask_add: null argument");
  AST_CHECK_ARG(same_shape(a, out) && (!b || same_shape(b, a)) && (!mask || same_shape(mask, a)), "ast_mask_add: shape mismatch");
  const long long total = (long long)a->n * a->h * a->w * a->c;
  if (total == 0) return 0;
  if (vec_ok(a) && vec_ok(out) && (!b || vec_ok(b)) && (!mask || vec_ok(mask)))
    launch_k(mask_add_vec_kernel, blocks_for(total / 4), NT, 0, (cudaStream_t)stream, to_img(a), b ? to_img(b) : null_img(), mask ? to_img(mask) : null_img(), to_img(out));
  else
    launch_k(mask_add_kernel, blocks_for(total), NT, 0, (cudaStream_t)stream, to_img(a), b ? to_img(b) : null_img(), mask ? to_img(mask) : null_img(), to_img(out));
  count_launch();
  count_work(FAM_POINTWISE, 0.0, img_bytes(a) + img_bytes(b) + img_bytes(mask) + img_bytes(out));
  AST_CUDA_LAUNCH_CHECK();
  return 0;
}

extern "C" int ast_gram(const ast_image* x, float* g, float scale, int32_t flags, void* stream) {
  AST_CHECK_ARG(x && g, "ast_gram: null argument");
  cudaStream_t s = (cudaStream_t)stream;
  if (x->n == 0 || x->c == 0) return 0;
  if (flags & AST_CONV_TENSOR) return gram_tc(x, g, scale, nullptr, 0, nullptr, 0.f, nullptr, 0.f, nullptr, s);
  cudaMemsetAsync(g, 0, sizeof(float) * (size_t)x->n * x->c * x->c, s);
  ast_gather_geom geom;
  memset(&geom, 0, sizeof(geom));
  geom.mi = x->h; geom.mj = x->w; geom.si = 1; geom.so = 1; geom.ntaps = 1;
  return launch_wgrad_simt(x, x, g, nullptr, x->c, 1, &geom, (int64_t)x->c * x->c, scale, s);
}

extern "C" int ast_gram_mse(const ast_image* x, float* g, float scale, const float* target, int64_t target_img_stride,
                            double* loss, float loss_scale, float* d, float d_scale, int32_t* counters, int32_t flags,
                            void* stream) {
  AST_CHECK_ARG(x && g && target && counters, "ast_gram_mse: null argument");
  cudaStream_t s = (cudaStream_t)stream;
  if (x->n == 0 || x->c == 0) return 0;
  if (flags & AST_CONV_TENSOR)
    return gram_tc(x, g, scale, target, target_img_stride, loss, loss_scale, d, d_scale, counters, s);
  ast_gather_geom geom;
  memset(&geom, 0, sizeof(geom));
  geom.mi = x->h; geom.mj = x->w; geom.si = 1; geom.so = 1; geom.ntaps = 1;
  if (int rc = launch_wgrad_simt(x, x, g, nullptr, x->c, 1, &geom, (int64_t)x->c * x->c, scale, s)) return rc;
  const long long cc = (long long)x->c * x->c, total = cc * x->n;
  launch_k(gram_finish_kernel, blocks_for(total), NT, 0, s, (const float*)g, target, (long long)target_img_stride, cc, total,
           loss, loss_scale, d, d_scale);
  count_launch();
  count_work(FAM_MSE, 0.0, 12.0 * total);
  AST_CUDA_LAUNCH_CHECK();
  return 0;
}
