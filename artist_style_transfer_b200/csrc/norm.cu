// InstanceNorm kernels (HBM-bound, NHWC, 16-byte vector accesses).
// Replaces aten::instance_norm -> native_batch_norm, aten::relu, the residual aten::add and
// aten::reflection_pad2d at cnn.py:58,68,78,96-98,114,123 and their autograd backward.
//
// Statistics: the tensor-core convs accumulate them in their epilogue (in_finalize_kernel turns the sums into mean /
// rstd); the strict-mode FFMA convs do not, and in_stats_* computes them from the conv output instead.
//
// Apply and backward are staged through shared memory: a dedicated producer warp streams whole row segments (<= 16 KB
// per tensor) into a ring with cp.async.bulk (the 1-D TMA copy, completion on an mbarrier), so the bytes in flight (up to
// ~190 KB per SM) do not depend on registers; eight consumer warps read the staged rows with conflict-free 16-byte shared
// loads, do the math and write their results straight to global memory with coalesced 16-byte stores.  (Kernels that
// load the same 16-byte vectors from global memory into registers are latency bound at about 3 TB/s.)  Folded constants:
//   y  = A*x + D,   dx = A*g' + B*x + C,   g' = (fold_reflect(gpad) + gextra) * [A*x + D > 0]
// Requirements checked on the host, argument errors otherwise: one dtype (fp32 or bf16) for every tensor of a call, NHWC
// with pixel stride == C (dense rows), 16-byte aligned rows.
#include "tc_common.cuh"

namespace ast {

constexpr int NT = 256;

// ---------------------------------------------------------------- forward statistics
// Per-thread shifted sums -> (count, mean, M2); Chan merge inside the block and across blocks.
template <typename T>
__global__ void __launch_bounds__(NT)
in_stats_partial_kernel(Img x, float* __restrict__ ws, int nblk, int chunk) {
  constexpr int VEC = Vec16<T>::N;
  extern __shared__ float sm[];
  const int C = x.c, lanes = C / VEC, slots = NT / lanes;
  const int tid = threadIdx.x, lane = tid % lanes, slot = tid / lanes;
  const int n = blockIdx.y, blk = blockIdx.x;
  const int hw = x.h * x.w;
  const int pbeg = blk * chunk, pend = min(hw, pbeg + chunk);
  const T* base = (const T*)x.ptr + (long long)n * x.sn + lane * VEC;

  float k[VEC], s1[VEC], s2[VEC];
#pragma unroll
  for (int e = 0; e < VEC; ++e) { k[e] = 0.f; s1[e] = 0.f; s2[e] = 0.f; }
  int cnt = 0;
  if (slot < slots) {
    for (int p = pbeg + slot; p < pend; p += slots) {
      const int y = p / x.w, xx = p - y * x.w;
      float v[VEC];
      Vec16<T>::load(base + (long long)y * x.sh + (long long)xx * x.sw, v);
      if (cnt == 0) {
#pragma unroll
        for (int e = 0; e < VEC; ++e) k[e] = v[e];
      }
#pragma unroll
      for (int e = 0; e < VEC; ++e) { const float d = v[e] - k[e]; s1[e] += d; s2[e] = fmaf(d, d, s2[e]); }
      ++cnt;
    }
  }
  // smem: cntS[slots] | meanS[slots][C] | m2S[slots][C]
  float* cntS = sm;
  float* meanS = sm + NT;
  float* m2S = meanS + slots * C;
  if (slot < slots) {
    if (lane == 0) cntS[slot] = (float)cnt;
    const float inv = cnt > 0 ? 1.f / cnt : 0.f;
#pragma unroll
    for (int e = 0; e < VEC; ++e) {
      meanS[slot * C + lane * VEC + e] = k[e] + s1[e] * inv;
      m2S[slot * C + lane * VEC + e] = fmaxf(s2[e] - s1[e] * s1[e] * inv, 0.f);
    }
  }
  __syncthreads();
  for (int c = tid; c < C; c += NT) {
    float na = 0.f, ma = 0.f, qa = 0.f;
    for (int s = 0; s < slots; ++s) {
      const float nb = cntS[s];
      if (nb == 0.f) continue;
      const float mb = meanS[s * C + c], qb = m2S[s * C + c];
      const float nab = na + nb, d = mb - ma;
      ma += d * (nb / nab);
      qa += qb + d * d * (na * nb / nab);
      na = nab;
    }
    float* o = ws + ((long long)(n * nblk + blk) * C + c) * 3;
    o[0] = na; o[1] = ma; o[2] = qa;
  }
}

__global__ void in_stats_final_kernel(const float* __restrict__ ws, int nblk, int C, int hw, float eps,
                                      float* __restrict__ mean, float* __restrict__ rstd) {
  const int n = blockIdx.x;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float na = 0.f, ma = 0.f, qa = 0.f;
    for (int b = 0; b < nblk; ++b) {
      const float* o = ws + ((long long)(n * nblk + b) * C + c) * 3;
      const float nb = o[0];
      if (nb == 0.f) continue;
      const float d = o[1] - ma, nab = na + nb;
      ma += d * (nb / nab);
      qa += o[2] + d * d * (na * nb / nab);
      na = nab;
    }
    mean[n * C + c] = ma;
    rstd[n * C + c] = rsqrtf(qa / (float)hw + eps);
  }
}

__global__ void in_finalize_kernel(const double* __restrict__ sums, int total, double inv_hw, float eps,
                                   float* __restrict__ mean, float* __restrict__ rstd) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const double m = sums[2 * i] * inv_hw;
  const double var = fmax(sums[2 * i + 1] * inv_hw - m * m, 0.0);
  mean[i] = (float)m;
  rstd[i] = (float)(1.0 / sqrt(var + (double)eps));
}


// ================================================================ apply and backward: shared-memory staged
constexpr int NS_CONSUMER_WARPS = 8;
constexpr int NS_CONSUMERS = NS_CONSUMER_WARPS * 32;
constexpr int NS_THREADS = NS_CONSUMERS + 32;      // + one producer warp
constexpr int NS_SLAB_MAX = 16384;                 // bytes of one tensor's row segment
constexpr int NS_MAX_STAGES = 8;
constexpr int NS_SMEM_BUDGET = 100 * 1024;         // per block: two blocks per SM

struct Rows {            // dense-row tensor: element offset of pixel (n, i, j) = n*sn + i*sh + j*C
  char* ptr;
  long long sn;          // a batch may span more than 2^31 elements
  int sh;                // one image spans fewer (checked on the host)
};

struct NsShape {
  int C, H, W, pad;
  int nblk;              // blocks per image: block b owns rows [b*R/nblk, (b+1)*R/nblk) of the R iterated rows
  int seg, nseg;         // pixels per row segment (of the iterated row), segments per row
  int stages, slab_bytes;
};

template <typename T> struct NsVec;
template <> struct NsVec<float> {
  static constexpr int N = 4;
  __device__ static __forceinline__ void unpack(const uint4& r, float* v) {
    v[0] = __uint_as_float(r.x); v[1] = __uint_as_float(r.y); v[2] = __uint_as_float(r.z); v[3] = __uint_as_float(r.w);
  }
  __device__ static __forceinline__ uint4 pack(const float* v) {
    return make_uint4(__float_as_uint(v[0]), __float_as_uint(v[1]), __float_as_uint(v[2]), __float_as_uint(v[3]));
  }
};
template <> struct NsVec<__nv_bfloat16> {
  static constexpr int N = 8;
  __device__ static __forceinline__ void unpack(const uint4& r, float* v) {
    const unsigned w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) { v[2 * i] = __uint_as_float(w[i] << 16); v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u); }
  }
  __device__ static __forceinline__ uint4 pack(const float* v) {
    uint4 r;
    __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&r);
#pragma unroll
    for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
    return r;
  }
};

template <int VEC>
__device__ __forceinline__ void ns_ldc(const float* __restrict__ p, float* v) {
#pragma unroll
  for (int e = 0; e < VEC; e += 4) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(p + e));
    v[e] = t.x; v[e + 1] = t.y; v[e + 2] = t.z; v[e + 3] = t.w;
  }
}

__device__ __forceinline__ void bulk_load(unsigned dst, const void* src, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// first element of image n: the image offset is 64-bit, offsets inside the image (i * sh + j * C) stay 32-bit, so a
// pixel address is one 32-bit multiply-add plus one wide add onto this base
template <typename T>
__device__ __forceinline__ T* img_at(const Rows& t, int n) {
  return reinterpret_cast<T*>(t.ptr) + n * t.sn;
}

// Common prologue: barriers, then the block splits into the producer warp and the consumers.
__device__ __forceinline__ void ns_init(unsigned long long* full, unsigned long long* empty, int stages) {
  if (threadIdx.x == 0) {
    for (int s = 0; s < stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], NS_CONSUMER_WARPS); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();
}

// folded constants of channels c .. c+VEC-1 of image n: A = gamma * rstd, D = beta - A * mean (y = A*x + D)
template <int VEC>
__device__ __forceinline__ void ns_fold_ad(const float* __restrict__ gamma, const float* __restrict__ beta,
                                           const float* __restrict__ mean, const float* __restrict__ rstd, int n, int C,
                                           int c, float* A, float* D) {
  float mu[VEC];
  ns_ldc<VEC>(gamma + c, A); ns_ldc<VEC>(rstd + n * C + c, D); ns_ldc<VEC>(mean + n * C + c, mu);
#pragma unroll
  for (int e = 0; e < VEC; ++e) A[e] *= D[e];
  ns_ldc<VEC>(beta + c, D);
#pragma unroll
  for (int e = 0; e < VEC; ++e) D[e] -= A[e] * mu[e];
}

// x columns an output segment [oa, ob) of a reflect-padded row needs: [xa, xb)
__device__ __forceinline__ void apply_span(int oa, int ob, int pad, int W, int& xa, int& xb) {
  const int lo = oa - pad, hi = ob - 1 - pad;
  xa = max(lo, 0); xb = min(hi + 1, W);
  if (lo < 0) xb = max(xb, min(W, 1 - lo));
  if (hi >= W) xa = min(xa, max(0, 2 * (W - 1) - hi));
}

// ---------------------------------------------------------------- forward apply (+ReLU, +residual, reflect-pad write)
template <typename T>
__global__ void __launch_bounds__(NS_THREADS, 2)
in_apply_staged_kernel(Rows x, const float* __restrict__ mean, const float* __restrict__ rstd,
                       const float* __restrict__ gamma, const float* __restrict__ beta, Rows res, Rows out, NsShape sh,
                       int relu) {
  constexpr int VEC = NsVec<T>::N;
  extern __shared__ unsigned char smem_raw[];
  __shared__ __align__(8) unsigned long long full[NS_MAX_STAGES], empty[NS_MAX_STAGES];
  const unsigned buf = (smem_u32(smem_raw) + 127u) & ~127u;
  ns_init(full, empty, sh.stages);
  const int n = blockIdx.y, C = sh.C;
  const int OH = sh.H + 2 * sh.pad, OW = sh.W + 2 * sh.pad;
  const int rbeg = (int)((long long)blockIdx.x * OH / sh.nblk), rend = (int)((long long)(blockIdx.x + 1) * OH / sh.nblk);
  const int nunits = (rend - rbeg) * sh.nseg;
  const int nslabs = res.ptr ? 2 : 1;
  const int stage_bytes = nslabs * sh.slab_bytes;

  if (threadIdx.x >= NS_CONSUMERS) {
    if (threadIdx.x == NS_CONSUMERS) {
      for (int k = 0; k < nunits; ++k) {
        const int s = k % sh.stages;
        const unsigned ph = (unsigned)(k / sh.stages) & 1u;
        const int oy = rbeg + k / sh.nseg, sg = k % sh.nseg;
        const int i = reflect_idx(oy - sh.pad, sh.H);
        const int oa = sg * sh.seg, ob = min(OW, oa + sh.seg);
        int xa, xb;
        apply_span(oa, ob, sh.pad, sh.W, xa, xb);
        const unsigned bytes = (unsigned)((xb - xa) * C * (int)sizeof(T));
        mbar_wait(&empty[s], ph ^ 1u);
        mbar_expect_tx(&full[s], bytes * nslabs);
        bulk_load(buf + s * stage_bytes, img_at<T>(x, n) + (i * x.sh + xa * C), bytes, &full[s]);
        if (res.ptr) bulk_load(buf + s * stage_bytes + sh.slab_bytes, img_at<T>(res, n) + (i * res.sh + xa * C), bytes, &full[s]);
      }
    }
    return;
  }

  const int lanes = C / VEC, slots = NS_CONSUMERS / lanes;
  const int lane = threadIdx.x % lanes, slot = threadIdx.x / lanes;
  const int c = lane * VEC;
  float A[VEC], D[VEC];
  ns_fold_ad<VEC>(gamma, beta, mean, rstd, n, C, c, A, D);
  uint4* const oimg = reinterpret_cast<uint4*>(img_at<T>(out, n)) + lane;      // 16-byte units from here on
  for (int k = 0; k < nunits; ++k) {
    const int s = k % sh.stages;
    const unsigned ph = (unsigned)(k / sh.stages) & 1u;
    const int oy = rbeg + k / sh.nseg, sg = k % sh.nseg;
    const int oa = sg * sh.seg, ob = min(OW, oa + sh.seg);
    int xa, xb;
    apply_span(oa, ob, sh.pad, sh.W, xa, xb);
    const unsigned xs = buf + s * stage_bytes + (unsigned)(c * (int)sizeof(T));
    const int orow = oy * (out.sh / VEC);
    mbar_wait(&full[s], ph);
    for (int ox = oa + slot; ox < ob; ox += slots) {
      const int j = reflect_idx(ox - sh.pad, sh.W) - xa;
      float v[VEC];
      NsVec<T>::unpack(lds128(xs + (unsigned)(j * C * (int)sizeof(T))), v);
#pragma unroll
      for (int e = 0; e < VEC; ++e) v[e] = fmaf(A[e], v[e], D[e]);
      if (res.ptr) {
        float r[VEC];
        NsVec<T>::unpack(lds128(xs + sh.slab_bytes + (unsigned)(j * C * (int)sizeof(T))), r);
#pragma unroll
        for (int e = 0; e < VEC; ++e) v[e] += r[e];
      }
      if (relu) {
#pragma unroll
        for (int e = 0; e < VEC; ++e) v[e] = fmaxf(v[e], 0.f);
      }
      oimg[orow + ox * lanes] = NsVec<T>::pack(v);
    }
    __syncwarp();
    if ((threadIdx.x & 31) == 0) mbar_arrive(&empty[s]);
  }
}

// ---------------------------------------------------------------- backward
// mirrored positions of the padded gradient that fold onto (i, j): only evaluated on the border ring (global loads).
// gimg: channel c of pixel (0, 0) of this image of gpad, gsh: its row stride
template <typename T, int VEC>
__device__ __forceinline__ void ns_fold_border(const T* gimg, int gsh, int C, int pad, int H, int W, int i, int j, float* g) {
  reflect_fold_border(pad, H, W, i, j, [&](int r, int cc) {
    float t[VEC];
    NsVec<T>::unpack(__ldg(reinterpret_cast<const uint4*>(gimg + (r * gsh + cc * C))), t);
#pragma unroll
    for (int e = 0; e < VEC; ++e) g[e] += t[e];
  });
}

// producer of the backward: x row segment, the centre of the padded gradient row, the extra gradient, for this block's
// units at ring positions k0, k0+1, ..
template <typename T>
__device__ __forceinline__ void ns_bwd_produce(const Rows& x, const Rows& gpad, const Rows& gextra, const NsShape& sh, int n,
                                               int rbeg, int nunits, int k0, unsigned buf, int stage_bytes,
                                               unsigned long long* full, unsigned long long* empty) {
  const int C = sh.C;
  const int nslabs = 1 + (gpad.ptr ? 1 : 0) + (gextra.ptr ? 1 : 0);
  for (int k = 0; k < nunits; ++k) {
    const int s = (k0 + k) % sh.stages;
    const unsigned ph = (unsigned)((k0 + k) / sh.stages) & 1u;
    const int i = rbeg + k / sh.nseg, sg = k % sh.nseg;
    const int ja = sg * sh.seg, jb = min(sh.W, ja + sh.seg);
    const unsigned bytes = (unsigned)((jb - ja) * C * (int)sizeof(T));
    mbar_wait(&empty[s], ph ^ 1u);
    mbar_expect_tx(&full[s], bytes * nslabs);
    unsigned dst = buf + s * stage_bytes;
    bulk_load(dst, img_at<T>(x, n) + (i * x.sh + ja * C), bytes, &full[s]);
    dst += sh.slab_bytes;
    if (gpad.ptr) {
      bulk_load(dst, img_at<T>(gpad, n) + ((i + sh.pad) * gpad.sh + (ja + sh.pad) * C), bytes, &full[s]);
      dst += sh.slab_bytes;
    }
    if (gextra.ptr) bulk_load(dst, img_at<T>(gextra, n) + (i * gextra.sh + ja * C), bytes, &full[s]);
  }
}

// g' of pixel (i, j), whose staged x / gpad / gextra vectors start at shared addresses xs / gs / es; x is returned in xv
template <typename T, int VEC>
__device__ __forceinline__ void ns_gprime(unsigned xs, unsigned gs, unsigned es, const T* gimg, int gsh, bool has_gextra,
                                          const NsShape& sh, bool brow, int i, int j, const float* A, const float* D,
                                          int relu, float* xv, float* g) {
  NsVec<T>::unpack(lds128(xs), xv);
  if (gimg) {
    NsVec<T>::unpack(lds128(gs), g);
    if (sh.pad > 0 && (brow || j <= sh.pad || j >= sh.W - 1 - sh.pad))
      ns_fold_border<T, VEC>(gimg, gsh, sh.C, sh.pad, sh.H, sh.W, i, j, g);
  } else {
#pragma unroll
    for (int e = 0; e < VEC; ++e) g[e] = 0.f;
  }
  if (has_gextra) {
    float t[VEC];
    NsVec<T>::unpack(lds128(es), t);
#pragma unroll
    for (int e = 0; e < VEC; ++e) g[e] += t[e];
  }
#pragma unroll
  for (int e = 0; e < VEC; ++e)
    if (relu && !(fmaf(A[e], xv[e], D[e]) > 0.f)) g[e] = 0.f;   // same expression as the forward apply
}

enum NsMode { NS_STATS = 1, NS_APPLY = 2, NS_BOTH = 3 };

// Backward of pad o ReLU o (+residual) o InstanceNorm, by MODE:
//   NS_STATS  pass 1: s1[n,c] += sum g', s2[n,c] += sum g' * xhat
//   NS_APPLY  pass 2: dx = A*g' + B*x + C (and gtotal = g') from the finished s1 / s2
//   NS_BOTH   both passes in one cooperative launch.  Two launches read x and g' twice from HBM (7 physical passes for 5
//             algorithmic ones).  For layers whose x + g' fit in the 126 MB L2 this kernel runs the statistics pass, meets
//             the other blocks of the SAME image at a counter barrier (all blocks are co-resident: the grid is one wave,
//             launched cooperatively), and re-streams its own rows for the apply pass - which now hit L2.  The producer
//             warp does not wait at the barrier: it keeps prefetching the first apply units into the ring while the sums
//             settle.  `arrive`: n ints, zero on entry.
template <typename T, int MODE>
__global__ void __launch_bounds__(NS_THREADS, 2)
in_bwd_staged_kernel(Rows x, const float* __restrict__ mean, const float* __restrict__ rstd,
                     const float* __restrict__ gamma, const float* __restrict__ beta, Rows gpad, Rows gextra,
                     NsShape sh, int relu, float* __restrict__ s1, float* __restrict__ s2, int* __restrict__ arrive,
                     Rows dx, Rows gtotal) {
  constexpr int VEC = NsVec<T>::N;
  extern __shared__ unsigned char smem_raw[];
  __shared__ __align__(8) unsigned long long full[NS_MAX_STAGES], empty[NS_MAX_STAGES];
  const unsigned buf = (smem_u32(smem_raw) + 127u) & ~127u;
  ns_init(full, empty, sh.stages);
  const int n = blockIdx.y, C = sh.C;
  const int rbeg = (int)((long long)blockIdx.x * sh.H / sh.nblk), rend = (int)((long long)(blockIdx.x + 1) * sh.H / sh.nblk);
  const int nunits = (rend - rbeg) * sh.nseg;
  const int nslabs = 1 + (gpad.ptr ? 1 : 0) + (gextra.ptr ? 1 : 0);
  const int stage_bytes = nslabs * sh.slab_bytes;

  if (threadIdx.x >= NS_CONSUMERS) {
    if (threadIdx.x == NS_CONSUMERS) {      // NS_BOTH: the same unit sequence twice (ring positions simply continue)
      ns_bwd_produce<T>(x, gpad, gextra, sh, n, rbeg, nunits, 0, buf, stage_bytes, full, empty);
      if (MODE == NS_BOTH) ns_bwd_produce<T>(x, gpad, gextra, sh, n, rbeg, nunits, nunits, buf, stage_bytes, full, empty);
    }
    return;
  }
  const int lanes = C / VEC, slots = NS_CONSUMERS / lanes;
  const int lane = threadIdx.x % lanes, slot = threadIdx.x / lanes;
  const int c = lane * VEC;
  float A[VEC], D[VEC];
  ns_fold_ad<VEC>(gamma, beta, mean, rstd, n, C, c, A, D);
  const T* const gimg = gpad.ptr ? img_at<T>(gpad, n) + c : nullptr;

  // consumer side of unit k at ring position pos: f(j, x, g') for each of this thread's pixels, then the stage is freed
  auto consume = [&](int k, int pos, auto&& f) {
    const int s = pos % sh.stages;
    const unsigned ph = (unsigned)(pos / sh.stages) & 1u;
    const int i = rbeg + k / sh.nseg, sg = k % sh.nseg;
    const int ja = sg * sh.seg, jb = min(sh.W, ja + sh.seg);
    const bool brow = sh.pad > 0 && (i <= sh.pad || i >= sh.H - 1 - sh.pad);
    const unsigned xs = buf + s * stage_bytes + (unsigned)(c * (int)sizeof(T));
    const unsigned gs = xs + sh.slab_bytes;
    const unsigned es = xs + (gpad.ptr ? 2 : 1) * sh.slab_bytes;
    mbar_wait(&full[s], ph);
    for (int j = ja + slot; j < jb; j += slots) {
      const unsigned poff = (unsigned)((j - ja) * C * (int)sizeof(T));
      float xv[VEC], g[VEC];
      ns_gprime<T, VEC>(xs + poff, gs + poff, es + poff, gimg, gpad.sh, gextra.ptr != nullptr, sh, brow, i, j, A, D, relu,
                        xv, g);
      f(j, xv, g);
    }
    __syncwarp();
    if ((threadIdx.x & 31) == 0) mbar_arrive(&empty[s]);
  };

  if (MODE & NS_STATS) {
    float t1[VEC], t2[VEC];
#pragma unroll
    for (int e = 0; e < VEC; ++e) { t1[e] = 0.f; t2[e] = 0.f; }
    for (int k = 0; k < nunits; ++k)
      consume(k, k, [&](int, const float* xv, const float* g) {
#pragma unroll
        for (int e = 0; e < VEC; ++e) { t1[e] += g[e]; t2[e] = fmaf(g[e], xv[e], t2[e]); }
      });
    // block reduction.  NS_STATS: in the ring, once every consumer warp has consumed every stage.  NS_BOTH: in a scratch
    // area BEHIND the ring (the producer is already refilling the ring for pass 2).
    float* r1 = reinterpret_cast<float*>(smem_raw + (buf - smem_u32(smem_raw)) +
                                         (MODE == NS_BOTH ? (size_t)sh.stages * stage_bytes : 0));
    float* r2 = r1 + slots * C;
    if (MODE == NS_STATS) {
      __syncwarp();
      asm volatile("bar.sync 1, %0;" ::"n"(NS_CONSUMERS) : "memory");     // consumers only: all units consumed
    }
#pragma unroll
    for (int e = 0; e < VEC; ++e) { r1[slot * C + c + e] = t1[e]; r2[slot * C + c + e] = t2[e]; }
    asm volatile("bar.sync 1, %0;" ::"n"(NS_CONSUMERS) : "memory");
    for (int cc = threadIdx.x; cc < C; cc += NS_CONSUMERS) {
      float u1 = 0.f, u2 = 0.f;
      for (int q = 0; q < slots; ++q) { u1 += r1[q * C + cc]; u2 += r2[q * C + cc]; }
      atomicAdd(s1 + n * C + cc, u1);
      atomicAdd(s2 + n * C + cc, rstd[n * C + cc] * (u2 - mean[n * C + cc] * u1));
    }
    if (MODE == NS_BOTH) {
      // all blocks of image n have added their sums: release / acquire through the fence + counter
      __threadfence();
      asm volatile("bar.sync 1, %0;" ::"n"(NS_CONSUMERS) : "memory");
      if (threadIdx.x == 0) {
        atomicAdd(arrive + n, 1);
        const volatile int* cnt = arrive + n;
        for (unsigned spin = 0; *cnt < sh.nblk; ++spin)
          if (spin > (1u << 28)) __trap();            // bounded: a scheduling surprise traps instead of hanging the GPU
        __threadfence();
      }
      asm volatile("bar.sync 1, %0;" ::"n"(NS_CONSUMERS) : "memory");
    }
  }

  if (MODE & NS_APPLY) {
    // NS_BOTH: x and g' of this block's rows were just read, so pass 2 is served from L2
    const float inv_hw = 1.f / (float)(sh.H * sh.W);
    float B[VEC], Cc[VEC];
    {
      float mu[VEC], rs[VEC];
      ns_ldc<VEC>(rstd + n * C + c, rs); ns_ldc<VEC>(mean + n * C + c, mu);
#pragma unroll
      for (int e = 0; e < VEC; ++e) {
        const float S1 = __ldcg(s1 + n * C + c + e), S2 = __ldcg(s2 + n * C + c + e);   // NS_BOTH: written by this launch
        B[e] = -A[e] * rs[e] * S2 * inv_hw;
        Cc[e] = -A[e] * S1 * inv_hw - B[e] * mu[e];
      }
    }
    const int k0 = MODE == NS_BOTH ? nunits : 0;
    T* const dimg = img_at<T>(dx, n) + c;
    T* const timg = gtotal.ptr ? img_at<T>(gtotal, n) + c : nullptr;
    for (int k = 0; k < nunits; ++k) {
      const int i = rbeg + k / sh.nseg;
      const int drow = i * dx.sh, trow = i * gtotal.sh;
      consume(k, k0 + k, [&](int j, float* xv, const float* g) {
        if (timg) *reinterpret_cast<uint4*>(timg + (trow + j * C)) = NsVec<T>::pack(g);
#pragma unroll
        for (int e = 0; e < VEC; ++e) xv[e] = fmaf(A[e], g[e], fmaf(B[e], xv[e], Cc[e]));
        *reinterpret_cast<uint4*>(dimg + (drow + j * C)) = NsVec<T>::pack(xv);
      });
    }
  }
}

// ---------------------------------------------------------------- host side
static int stats_blocks(int n, int hw, int slots) {
  int nblk = (4 * num_sms() + n - 1) / n;
  const int maxb = (hw + slots * 4 - 1) / (slots * 4);
  if (nblk > maxb) nblk = maxb;
  if (nblk < 1) nblk = 1;
  return nblk;
}

static bool nhwc_ok(const ast_image* x, int vec) {
  return x->sc == 1 && x->c % vec == 0 && x->sw % vec == 0 && x->sh % vec == 0 && x->sn % vec == 0;
}

// dense rows the bulk copies take: pixel stride C, rows and images 16-byte aligned, one image < 2^31 elements
static bool rows_ok(const ast_image* im, int vec) {
  return im->sc == 1 && im->sw == im->c && im->c % vec == 0 && im->sh % vec == 0 && im->sn % vec == 0 && im->sh >= 0 &&
         im->sn >= 0 && ((uintptr_t)im->ptr & 15) == 0 && (long long)im->h * im->sh < (1ll << 31);
}
// The staged kernels take one dtype (fp32 or bf16) for every tensor of a call, dense rows, and a C the consumer mapping
// can split (C / VEC lanes must divide the consumer threads; a row segment holds at least 8 pixels).
static int staged_layout_check(const char* who, const ast_image* x, std::initializer_list<const ast_image*> tensors) {
  AST_CHECK_ARG(x->dtype == AST_F32 || x->dtype == AST_BF16, "%s: x must be fp32 or bf16 (dtype %d)", who, x->dtype);
  const int esz = x->dtype == AST_F32 ? 4 : 2, vec = 16 / esz;
  for (const ast_image* t : tensors) {
    if (!t) continue;
    AST_CHECK_ARG(t->dtype == x->dtype, "%s: every tensor must have the dtype of x (%d vs %d)", who, t->dtype, x->dtype);
    AST_CHECK_ARG(rows_ok(t, vec), "%s: needs NHWC with dense 16-byte aligned rows, < 2^31 elements per image (sc == 1, sw == c, C %% %d == 0; got "
                  "c=%d sw=%lld sc=%lld)", who, vec, t->c, (long long)t->sw, (long long)t->sc);
  }
  AST_CHECK_ARG(x->c > 0 && x->c * esz <= NS_SLAB_MAX / 8 && NS_CONSUMERS % (x->c / vec) == 0,
                "%s: C=%d is not supported", who, x->c);
  return 0;
}

static Rows to_rows(const ast_image* im) {
  Rows r;
  if (!im) { r.ptr = nullptr; r.sn = r.sh = 0; return r; }
  r.ptr = (char*)im->ptr; r.sn = im->sn; r.sh = (int)im->sh;
  return r;
}
// rows per block / segments / stages; false when the shape does not suit the staged kernels
static bool ns_plan(NsShape* sh, int n, int C, int H, int W, int pad, int rows_total, int width, int esz, int nslabs,
                    int slab_max = NS_SLAB_MAX, int budget = NS_SMEM_BUDGET) {
  sh->C = C; sh->H = H; sh->W = W; sh->pad = pad;
  const int seg_max = slab_max / (C * esz) - (width != W ? 2 * pad : 0);   // apply: the x span of a segment adds <= 2*pad
  if (seg_max < 4 * pad + 1) return false;
  sh->nseg = (width + seg_max - 1) / seg_max;
  sh->seg = (width + sh->nseg - 1) / sh->nseg;
  sh->nseg = (width + sh->seg - 1) / sh->seg;
  const int slab_px = sh->seg + (width != W ? 2 * pad : 0);
  sh->slab_bytes = (slab_px * C * esz + 127) / 128 * 128;
  sh->stages = budget / (nslabs * sh->slab_bytes);
  if (sh->stages > NS_MAX_STAGES) sh->stages = NS_MAX_STAGES;
  if (sh->stages < 2) return false;
  // as many blocks per image as fit one wave of 2 blocks per SM; rows are split proportionally (7/8 rows each at
  // H = 64, B = 32: 288 of the 296 block slots busy instead of 256 with a fixed 8 rows per block)
  int nb = (2 * num_sms()) / n;
  if (nb > rows_total) nb = rows_total;
  if (nb < 1) nb = 1;
  sh->nblk = nb;
  return true;
}

// Opts the kernel in to `smem` bytes of dynamic shared memory and launches it (cooperative: every block resident at once).
template <typename... KP, typename... A>
static int ns_launch(const char* who, int family, double bytes, void (*kernel)(KP...), dim3 grid, size_t smem,
                     bool cooperative, cudaStream_t s, A... args) {
  cudaError_t e = set_max_smem(kernel, smem);
  if (e == cudaSuccess && !cooperative) {
    e = launch_k(kernel, grid, NS_THREADS, smem, s, args...);
  } else if (e == cudaSuccess) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid; cfg.blockDim = dim3(NS_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeCooperative;
    attr.val.cooperative = 1;
    cfg.attrs = &attr; cfg.numAttrs = 1;
    e = cudaLaunchKernelEx(&cfg, kernel, static_cast<KP>(args)...);
  }
  if (e != cudaSuccess) { set_error("%s: launch failed: %s", who, cudaGetErrorString(e)); return (int)e; }
  count_launch();
  count_work(family, 0.0, bytes);
  AST_CUDA_LAUNCH_CHECK();
  return 0;
}

}  // namespace ast

using namespace ast;

extern "C" int64_t ast_instnorm_workspace_bytes(int32_t n, int32_t c) {
  return (int64_t)(4 * 148 * 2 + n) * c * 3 * sizeof(float);
}

extern "C" int ast_instnorm_stats(const ast_image* x, float* mean, float* rstd, float eps, void* workspace, void* stream) {
  AST_CHECK_ARG(x && mean && rstd && workspace, "ast_instnorm_stats: null argument");
  const int vec = x->dtype == AST_F32 ? 4 : 8;
  AST_CHECK_ARG(nhwc_ok(x, vec), "ast_instnorm_stats: needs NHWC with C %% %d == 0 (c=%d sc=%lld)", vec, x->c, (long long)x->sc);
  AST_CHECK_ARG(x->c / vec <= NT, "ast_instnorm_stats: C=%d too large", x->c);
  if (x->n == 0) return 0;
  const int lanes = x->c / vec, slots = NT / lanes, hw = x->h * x->w;
  const int nblk = stats_blocks(x->n, hw, slots);
  AST_CHECK_ARG((int64_t)x->n * nblk * x->c * 12 <= ast_instnorm_workspace_bytes(x->n, x->c), "ast_instnorm_stats: workspace");
  const int chunk = (hw + nblk - 1) / nblk;
  const size_t smem = (NT + 2 * slots * x->c) * sizeof(float);
  dim3 grid(nblk, x->n);
  cudaStream_t s = (cudaStream_t)stream;
  if (x->dtype == AST_F32) launch_k(in_stats_partial_kernel<float>, grid, NT, smem, s, to_img(x), (float*)workspace, nblk, chunk);
  else launch_k(in_stats_partial_kernel<__nv_bfloat16>, grid, NT, smem, s, to_img(x), (float*)workspace, nblk, chunk);
  launch_k(in_stats_final_kernel, x->n, 128, 0, s, (const float*)workspace, nblk, x->c, hw, eps, mean, rstd);
  count_launch(2);
  count_work(FAM_IN_STATS, 0.0, img_bytes(x));
  AST_CUDA_LAUNCH_CHECK();
  return 0;
}

extern "C" int ast_instnorm_finalize(const double* sums, int32_t n, int32_t c, int32_t hw, float eps, float* mean,
                                     float* rstd, void* stream) {
  AST_CHECK_ARG(sums && mean && rstd && hw > 0, "ast_instnorm_finalize: bad argument");
  const int total = n * c;
  if (total == 0) return 0;
  launch_k(in_finalize_kernel, (total + 255) / 256, 256, 0, (cudaStream_t)stream, sums, total, 1.0 / (double)hw, eps, mean, rstd);
  count_launch();
  count_work(FAM_IN_STATS, 0.0, 0.0);
  AST_CUDA_LAUNCH_CHECK();
  return 0;
}

extern "C" int ast_instnorm_apply(const ast_image* x, const float* mean, const float* rstd, const float* gamma,
                                  const float* beta, const ast_image* residual, const ast_image* out, int32_t pad,
                                  int32_t relu, void* stream) {
  AST_CHECK_ARG(x && mean && rstd && gamma && beta && out, "ast_instnorm_apply: null argument");
  if (int e = staged_layout_check("ast_instnorm_apply", x, {x, out, residual})) return e;
  AST_CHECK_ARG(out->n == x->n && out->c == x->c && out->h == x->h + 2 * pad && out->w == x->w + 2 * pad,
                "ast_instnorm_apply: out must be (h+2p, w+2p)");
  AST_CHECK_ARG(pad < x->h && pad < x->w, "ast_instnorm_apply: pad too large for reflection");
  AST_CHECK_ARG(!residual || same_shape(residual, x), "ast_instnorm_apply: residual shape");
  if (x->n == 0) return 0;
  const int esz = x->dtype == AST_F32 ? 4 : 2, nslabs = residual ? 2 : 1;
  NsShape sh;
  AST_CHECK_ARG(ns_plan(&sh, x->n, x->c, x->h, x->w, pad, out->h, out->w, esz, nslabs),
                "ast_instnorm_apply: C=%d, pad=%d cannot be staged", x->c, pad);
  return ns_launch("ast_instnorm_apply", FAM_IN_APPLY, img_bytes(x) + img_bytes(out) + img_bytes(residual),
                   x->dtype == AST_F32 ? in_apply_staged_kernel<float> : in_apply_staged_kernel<__nv_bfloat16>,
                   dim3(sh.nblk, x->n), (size_t)sh.stages * nslabs * sh.slab_bytes + 128, false, (cudaStream_t)stream,
                   to_rows(x), mean, rstd, gamma, beta, to_rows(residual), to_rows(out), sh, relu);
}

// (Measured and not kept: walking the batch in L2-sized image groups inside the single kernel so that the 256^2 x 32 and
// 128^2 x 64 layers qualify as well - 209 vs 164 us and 84 vs 84 us against two launches: the per-group barriers and the
// short per-block row ranges cost more than the second HBM read they save.)
extern "C" int ast_instnorm_bwd(const ast_image* x, const float* mean, const float* rstd, const float* gamma,
                                const float* beta, const ast_image* gpad, int32_t pad, const ast_image* gextra,
                                int32_t relu, float* s1, float* s2, int32_t* arrive, const ast_image* dx,
                                const ast_image* gtotal, void* stream) {
  AST_CHECK_ARG(x && mean && rstd && gamma && beta && s1 && s2 && arrive && dx, "ast_instnorm_bwd: null argument");
  AST_CHECK_ARG(relu == 0 || relu == 1, "ast_instnorm_bwd: relu must be 0 or 1 (got %d)", relu);
  if (int e = staged_layout_check("ast_instnorm_bwd", x, {x, gpad, gextra, dx, gtotal})) return e;
  AST_CHECK_ARG(!gpad || (gpad->n == x->n && gpad->c == x->c && gpad->h == x->h + 2 * pad && gpad->w == x->w + 2 * pad),
                "ast_instnorm_bwd: gpad must be (h+2p, w+2p)");
  AST_CHECK_ARG(!gextra || same_shape(gextra, x), "ast_instnorm_bwd: gextra shape");
  AST_CHECK_ARG(pad < x->h && pad < x->w, "ast_instnorm_bwd: pad too large");
  AST_CHECK_ARG(same_shape(dx, x), "ast_instnorm_bwd: dx shape");
  AST_CHECK_ARG(!gtotal || same_shape(gtotal, x), "ast_instnorm_bwd: gtotal shape");
  if (x->n == 0) return 0;
  const bool f32 = x->dtype == AST_F32;
  const int esz = f32 ? 4 : 2, vec = 16 / esz, nslabs = 1 + (gpad ? 1 : 0) + (gextra ? 1 : 0);
  const size_t scratch = 2 * (size_t)(NS_CONSUMERS / (x->c / vec)) * x->c * sizeof(float);   // block reduction
  // algorithmic traffic of the InstanceNorm backward (SURVEY 8d): read x and g' once, write dx (+ the skip gradient)
  const double bytes = 2.0 * img_bytes(x) + img_bytes(dx) + img_bytes(gtotal);
  cudaStream_t s = (cudaStream_t)stream;
  const Rows xr = to_rows(x), gp = to_rows(gpad), ge = to_rows(gextra), dxr = to_rows(dx), gt = to_rows(gtotal);
  NsShape sh;

  // One launch when x + g' survive in the 126 MB L2 next to the dx / skip-gradient writes and every block is resident
  // (the counter barrier needs them all).  The reduction scratch sits behind the ring (the producer refills the ring
  // during the barrier): the ring gets what is left of the per-block budget, with 8 KB slabs when three tensors are staged.
  const double resident = (double)nslabs * x->n * x->h * x->w * x->c * esz;      // bytes re-read by the second pass
  if (resident <= 104e6 &&
      ns_plan(&sh, x->n, x->c, x->h, x->w, pad, x->h, x->w, esz, nslabs, nslabs == 3 ? 8192 : NS_SLAB_MAX,
              NS_SMEM_BUDGET + 8192 - (int)scratch) &&
      (long long)sh.nblk * x->n <= 2ll * num_sms()) {
    const size_t smem = (size_t)sh.stages * nslabs * sh.slab_bytes + scratch + 128;
    if (smem <= 110 * 1024)
      return ns_launch("ast_instnorm_bwd", FAM_IN_BWD, bytes,
                       f32 ? in_bwd_staged_kernel<float, NS_BOTH> : in_bwd_staged_kernel<__nv_bfloat16, NS_BOTH>,
                       dim3(sh.nblk, x->n), smem, true, s, xr, mean, rstd, gamma, beta, gp, ge, sh, relu, s1, s2, arrive,
                       dxr, gt);
  }

  // Two launches: statistics, then apply.  The statistics kernel reduces in its ring.
  AST_CHECK_ARG(ns_plan(&sh, x->n, x->c, x->h, x->w, pad, x->h, x->w, esz, nslabs),
                "ast_instnorm_bwd: C=%d, pad=%d cannot be staged", x->c, pad);
  const size_t ring = (size_t)sh.stages * nslabs * sh.slab_bytes;
  if (int e = ns_launch("ast_instnorm_bwd", FAM_IN_BWD, 0.0,     // the apply launch books the algorithmic bytes
                        f32 ? in_bwd_staged_kernel<float, NS_STATS> : in_bwd_staged_kernel<__nv_bfloat16, NS_STATS>,
                        dim3(sh.nblk, x->n), (ring > scratch ? ring : scratch) + 128, false, s, xr, mean, rstd, gamma,
                        beta, gp, ge, sh, relu, s1, s2, arrive, dxr, gt))
    return e;
  return ns_launch("ast_instnorm_bwd", FAM_IN_BWD, bytes,
                   f32 ? in_bwd_staged_kernel<float, NS_APPLY> : in_bwd_staged_kernel<__nv_bfloat16, NS_APPLY>,
                   dim3(sh.nblk, x->n), ring + 128, false, s, xr, mean, rstd, gamma, beta, gp, ge, sh, relu, s1, s2,
                   arrive, dxr, gt);
}
