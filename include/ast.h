/*
 * ast.h - C ABI of libast_b200.so: the B200 (sm_100a) kernels behind the perceptual-loss
 * training step of edogariu/artist-style-transfer.
 *
 * Drop-in boundary (SURVEY.md 8b): the reference has no native code; the "FFI" it binds for this
 * path is the set of PyTorch library calls listed next to each entry point below.  Host code stays
 * Python/PyTorch (artist_style_transfer_b200/{cnn,train_cnn}.py mirror the reference modules) and
 * reaches these functions through ctypes with raw device pointers - no torch types cross the ABI.
 *
 * Conventions
 *   - every function returns 0 on success, <0 for an argument/shape/unsupported-config error
 *     (never a silent fallback), >0 for a cudaError_t / CUresult; ast_last_error() has the text.
 *   - the caller owns every buffer (inputs, outputs, workspaces) and keeps it alive until the work
 *     queued on `stream` has completed; the library never allocates device memory and keeps no
 *     pointers after return.  Launches are asynchronous on `stream`.
 *   - images are N x H x W x C views with explicit element strides (ast_image); the internal layout
 *     is NHWC (sc == 1), but NCHW tensors of the reference API are described with sc == H*W.
 */
#ifndef AST_B200_H
#define AST_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AST_ABI_VERSION 7

typedef enum {
  AST_F32 = 0, AST_BF16 = 1,
  AST_TF32 = 2, /* fp32 storage rounded to TF32; weight packing only */
  AST_U8 = 3,   /* uint8 images at the host boundary (dataset.py:97-108 / inference.py:110,116): ast_row_im2col input, ast_fold_rows output */
  AST_F16 = 4   /* IEEE half: the frozen VGG's non-tap activations and pooled tensors in fast mode.  10 mantissa bits = exactly
                   the precision a kind::tf32 MMA keeps of an fp32 operand, at half the bytes and twice the MMA rate
                   (kind::f16, fp32 accumulate).  Stores saturate at +-65504.  Tensor-core conv kernels, ast_maxpool2_fwd,
                   ast_row_im2col outputs and ReLU-mask operands only. */
} ast_dtype;

/* strided 4-D view; strides in ELEMENTS.  */
typedef struct {
  void*   ptr;
  int32_t dtype;          /* ast_dtype */
  int32_t n, h, w, c;
  int64_t sn, sh, sw, sc;
} ast_image;

#define AST_MAX_TAPS 81

/* A "gather" convolution: for every point (i,j) of an Mi x Mj iteration grid
 *   out[n, oy0 + so*i, ox0 + so*j, co] = epi( sum_t sum_ci  in[n, si*i + dy[t], si*j + dx[t], ci] * W[t][co][ci] )
 * Out-of-range input coordinates read 0 (or are mirrored when AST_CONV_REFLECT is set).
 * This single primitive expresses (tap tables are built by the host mirror, conv_geometry.py):
 *   nn.Conv2d stride 1/2 after nn.ReflectionPad2d      cnn.py:58,63,73-74   (si = stride)
 *   its data gradient (aten::convolution_backward)      train_cnn.py:333     (so = stride, 4 phases)
 *   nn.ConvTranspose2d k3 s2 p1 op1 and k1 s1           cnn.py:107-109,119   (so = 2, 4 sub-pixel phases)
 *   torchvision VGG16 Conv2d(3x3, pad 1) + ReLU         train_cnn.py:54,72-73
 *   the Gram backward  dF = (dG + dG^T) F / (CHW)       train_cnn.py:107,333 (1 tap, per-image weights)
 */
typedef struct {
  int32_t mi, mj;          /* iteration grid per image */
  int32_t si, so;          /* input / output coordinate multipliers */
  int32_t oy0, ox0;        /* output phase offset */
  int32_t ntaps;
  int32_t flags;           /* AST_CONV_* */
  int16_t dy[AST_MAX_TAPS];
  int16_t dx[AST_MAX_TAPS];
  int64_t w_img_stride;    /* elements between per-image weight sets, 0 = shared weights */
  double* stats;           /* optional fp64 [n][cout][2] (sum x, sum x^2 of the fp32 results, BEFORE bias/activation),
                              accumulated by the tensor-core epilogue: InstanceNorm statistics fused into the producing
                              conv (cnn.py:63,68).  Per-tile partial sums are fp32 (centred where a thread owns a channel),
                              the accumulation across the plane is fp64 so that var = E[x^2] - mean^2 survives |mean| >> std.
                              Zeroed by the caller; NULL = off; tensor-core launches only. */
  const ast_image* pooled; /* optional [n, mi/2, mj/2, cout]: nn.MaxPool2d(2, 2) of the epilogue result, written by the same
                              kernel (torchvision VGG16 features idx 4/9/16 after the conv+ReLU before them,
                              train_cnn.py:54,72-73).  Plain stride-1 launches (so = 1, no phase offset) of the
                              weight-stationary tensor-core kernel only, without add / mask, with an fp32 `out`; the
                              packed filter, two halo patches and a 32 KB pooling stage must fit in shared memory (64 -> 64
                              channels with 16-bit operands): any other request is an error.  With AST_CONV_POOL_ONLY the
                              full-resolution `out` is not written (no-grad content branch). */
  const ast_image* pool_codes; /* optional, with `pooled`: uint8 [n, mi/2, mj/2, cout], one byte per pooling window and channel
                              = everything the backward of ReLU + MaxPool2d needs from the forward activations:
                              bits 0-1 = arg max position k = 2*dy + dx (first maximum wins, like ATen), bits 2-5 = (x_k > 0)
                              for k = 0..3.  ast_maxpool2_bwd then reads 1 byte instead of four fp32 activations. */
} ast_gather_geom;

#define AST_CONV_RELU     1   /* epilogue max(v,0)                       (nn.ReLU, train_cnn.py VGG idx 1,3,...)   */
#define AST_CONV_REFLECT  2   /* mirror out-of-range input coordinates   (nn.ReflectionPad2d, cnn.py:58)          */
#define AST_CONV_POOL_ONLY 16  /* with geom.pooled: skip the store of the full-resolution output                      */
#define AST_CONV_TENSOR   4   /* request the tcgen05/TMA kernel; error if the shape is not supported              */
#define AST_CONV_ROUND_TF32 8 /* round the fp32 result to TF32 (cvt.rna) so a kind::tf32 consumer sees exact operands */

/* weights: packed [ntaps][cout][cin], same dtype as `in`.  bias: fp32[cout] or NULL.
 * in_shift: fp32[cin] added to in-range inputs before the product (VGG mean shift, train_cnn.py:300-301) or NULL.
 * add:  optional image added before the activation (tap-gradient accumulation in the VGG backward).
 * mask: optional image; out = (mask > 0) ? v : 0 after the activation (ReLU backward, threshold_backward). */
int ast_conv_gather(const ast_image* in, const void* weights, const float* bias, const float* in_shift,
                    const ast_image* add, const ast_image* mask, const ast_image* out,
                    const ast_gather_geom* geom, void* stream);

/* Weight gradient of the same gather convolution (aten::convolution_backward, filter part):
 *   dw[tap_off[t] + co*s_co + ci*s_ci] += sum_{n,i,j} gout[n, oy0+so*i, ox0+so*j, co] * x[n, si*i+dy[t], si*j+dx[t], ci]
 * dw is fp32 and must be zeroed (or hold a running sum) by the caller; accumulation uses fp32 atomics. */
int ast_wgrad_gather(const ast_image* x, const ast_image* gout, float* dw, const int32_t* tap_off,
                     int64_t s_co, int64_t s_ci, const ast_gather_geom* geom, void* stream);

/* BLOCK-STACKED gather convolution for thin outputs (32 or 64 output channels), tensor-core kernel only (conv_st.cu).
 *
 * A tcgen05 MMA has M = 128 rows.  With pixels as N and output channels as M, a 32-channel layer would leave 3/4 of the
 * tensor core idle; with pixels as M (conv_ws.cu) its N = 32 MMAs are bound by the A-operand fetch.  Here nblk = 128/cout
 * independent BLOCKS of outputs share every MMA: lane block g (cout consecutive TMEM lanes) accumulates
 *
 *   out[n, oy[g] + soy*i, ox[g] + sox*j, co] = epi( sum_v sum_ci in[n, sy*i + dy[v], j + dx[v], ci] * Ws[v][g*cout + co][ci] )
 *
 * over an mi x mj grid, all blocks reading the SAME input pixels through the `nvt` virtual taps (dy[v], dx[v]); rows of
 * Ws that belong to a (virtual tap, block) pair without a filter tap are zero.  Two uses (conv_geometry.py builds both):
 *   - the 4 (or 2) sub-pixel PHASES of a stride-2 ConvTranspose2d / of a stride-2 convolution's data gradient
 *     (cnn.py:107-109, train_cnn.py:333) as one launch: sy = 1, soy = sox = 2, (oy, ox)[g] = the phase, virtual taps = the
 *     union of the phases' input shifts (4 instead of 1+2+2+4 tap launches);
 *   - ROW-INTERLEAVED stride-1 convolutions (the vertical-tap forms of the 9x9 / 3x3 three-channel ends, cnn.py:32,39,
 *     train_cnn.py:54 conv1_1): block g owns output rows g, g+nblk, ..: sy = soy = nblk, sox = 1, oy[g] = g, virtual tap
 *     v = dy + g, so a k-tap layer costs k + nblk - 1 MMAs per nblk output rows instead of nblk * k.
 * Out-of-range inputs read 0; outputs outside `out` are skipped.  weights: [nvt][128][cin] in the dtype of `in`;
 * in->c * sizeof(elem) must be 64 or a multiple of 128 bytes; out->c == 128/nblk, channel-contiguous.
 * bias: fp32[cout] or NULL.  add / mask / flags (RELU, ROUND_TF32) as in ast_conv_gather.  stats: as ast_gather_geom.stats. */
#define AST_MAX_VTAPS 32
typedef struct {
  int32_t nblk;            /* 2 or 4 */
  int32_t mi, mj;          /* iteration grid per image */
  int32_t sy;              /* input rows per grid row */
  int32_t soy, sox;        /* output steps per grid row / column */
  int32_t oy[4], ox[4];    /* output origin of each block */
  int32_t nvt;
  int32_t ntaps;           /* filter taps summed over the blocks (non-zero [virtual tap][block] tiles): work accounting only */
  int32_t flags;           /* AST_CONV_RELU | AST_CONV_ROUND_TF32 */
  int16_t dy[AST_MAX_VTAPS];
  int16_t dx[AST_MAX_VTAPS];
  double* stats;
} ast_stacked_geom;
int ast_conv_stacked(const ast_image* in, const void* weights, const float* bias, const ast_image* add,
                     const ast_image* mask, const ast_image* out, const ast_stacked_geom* geom, void* stream);

/* Re-pack fp32 master weights into the [ntaps][a][b] operand layout of ast_conv_gather:
 *   dst[t][ia][ib] = src[tap_off[t] + ia*s_a + ib*s_b]      (dst dtype = ast_dtype) */
int ast_pack_weights(const float* src, const int32_t* tap_off, int32_t ntaps, int32_t a, int32_t b,
                     int64_t s_a, int64_t s_b, void* dst, int32_t dst_dtype, void* stream);

/* Same with a two-level inner index and zero padding (layouts of the 3-channel layers, see ast_row_im2col):
 *   dst[t][ia][ib] = (ia < a_valid && ib < b_valid) ? src[tap_off[t] + ia*s_a + (ib / b0)*s_b1 + (ib % b0)*s_b0] : 0 */
int ast_pack_weights_ex(const float* src, const int32_t* tap_off, int32_t ntaps, int32_t a, int32_t a_valid,
                        int32_t b, int32_t b_valid, int32_t b0, int64_t s_a, int64_t s_b1, int64_t s_b0,
                        void* dst, int32_t dst_dtype, void* stream);

/* "Row im2col" of a thin (3-channel) image so that its k x k convolution becomes a k-tap vertical convolution over
 * kw*C (zero-padded to out.c) channels that TMA / tcgen05 can consume:
 *   out[n, y, x, d*C + c] = src[n, Y(y - py), X(x + sign*d - px), c] (+ shift[c]),  d in [0, kw)
 * Out-of-range source coordinates are mirrored (reflect != 0: nn.ReflectionPad2d, cnn.py:58) or read as 0 (zero padding
 * of VGG conv1_1 applied AFTER the mean shift, train_cnn.py:300-301).  round_tf32 rounds fp32 outputs to TF32. */
int ast_row_im2col(const ast_image* src, const ast_image* out, const float* shift, int32_t kw, int32_t sign,
                   int32_t px, int32_t py, int32_t reflect, int32_t round_tf32, void* stream);

/* Finishes a thin-OUTPUT k x k convolution (cnn.py:39, the 32->3 9x9 layer) whose kw horizontal taps were computed as
 * kw*C output channels of a k-tap vertical ast_conv_gather:
 *   out[n, y, x, c] = bias[c] + sum_{d < kw} part[n, y, x + d, d*C + c]      (optional ReLU)
 * part: fp32 NHWC [n, h, w + kw - 1, >= kw*C] with dense rows; out: any dtype / strides (e.g. an NCHW view). */
int ast_fold_rows(const ast_image* part, const ast_image* out, const float* bias, int32_t kw, int32_t relu, void* stream);

/* nn.InstanceNorm2d(affine=True), eps 1e-5, biased variance (cnn.py:68,114).
 * stats: mean[n*c], rstd[n*c] (fp32).  workspace: ast_instnorm_workspace_bytes(). */
int64_t ast_instnorm_workspace_bytes(int32_t n, int32_t c);
int ast_instnorm_stats(const ast_image* x, float* mean, float* rstd, float eps, void* workspace, void* stream);
/* mean/rstd from the (sum x, sum x^2) pairs a conv epilogue accumulated (ast_gather_geom.stats): [n*c][2] -> [n*c]. */
int ast_instnorm_finalize(const double* sums, int32_t n, int32_t c, int32_t hw, float eps, float* mean, float* rstd,
                          void* stream);
/* y = gamma*(x-mean)*rstd + beta (+ residual) (ReLU if relu), written to the interior of `out`, which is an
 * (h+2*pad) x (w+2*pad) image whose border is filled by mirroring (the next layer's nn.ReflectionPad2d). */
int ast_instnorm_apply(const ast_image* x, const float* mean, const float* rstd, const float* gamma,
                       const float* beta, const ast_image* residual, const ast_image* out, int32_t pad,
                       int32_t relu, void* stream);
/* Backward of (ReflectionPad o ReLU o (+residual) o InstanceNorm).
 *   g'   = (fold_reflect(gpad, pad) + gextra) * (relu ? y>0 : 1)
 *   s1[n,c] = sum g' ; s2[n,c] = sum g'*xhat                       (pass 1)
 *   dx   = gamma*rstd*(g' - s1/HW - xhat*s2/HW) ; gtotal = g'      (pass 2)
 * gpad may be NULL (no padded consumer), gextra may be NULL, gtotal may be NULL.  relu: 0 or 1 (the forward applied ReLU).
 * s1, s2 (n*c floats) and arrive (n int32) must be ZERO on entry (one fill can serve every layer of a step).
 * When x + g' are small enough to stay in the 126 MB L2, ONE cooperative kernel runs the statistics pass, meets the other
 * blocks of the same image at a counter barrier (`arrive`) and re-reads its rows for the apply pass from L2 (5 HBM passes
 * instead of 7); otherwise the two passes run as two launches.  Same results either way. */
int ast_instnorm_bwd(const ast_image* x, const float* mean, const float* rstd, const float* gamma, const float* beta,
                     const ast_image* gpad, int32_t pad, const ast_image* gextra, int32_t relu, float* s1, float* s2,
                     int32_t* arrive, const ast_image* dx, const ast_image* gtotal, void* stream);

/* nn.MaxPool2d(2,2) of torchvision vgg16.features idx 4/9/16 and its backward fused with the tap-gradient add
 * and the ReLU mask of the producing layer:  gx = (route(gy) + gadd) * (x > 0). */
/* codes (optional, uint8 [n, h/2, w/2, c]): see ast_gather_geom.pool_codes - written by the forward, and accepted by the
 * backward INSTEAD of x (x may then be NULL; h and w must be even). */
int ast_maxpool2_fwd(const ast_image* x, const ast_image* y, const ast_image* codes, void* stream);
int ast_maxpool2_bwd(const ast_image* x, const ast_image* codes, const ast_image* gy, const ast_image* gadd,
                     const ast_image* gx, void* stream);

/* gram(), train_cnn.py:103-107:  G[n] = F[n] F[n]^T * scale, F = x viewed as (c, h*w).  G fp32 [n][c][c], zeroed here. */
int ast_gram(const ast_image* x, float* g, float scale, int32_t flags, void* stream);

/* The style term of one VGG tap in one call (train_cnn.py:321-325 with gram() :103-107; north_star: "fuse the 1/(CHW)
 * scale and the style-MSE reduction into the epilogue"):
 *   G[n]     = F[n] F[n]^T * scale                 (upper triangle on the tensor cores, mirrored by the finishing CTA)
 *   loss[0] += loss_scale * sum_{n,i,j} (G[n][i][j] - S[n][i][j])^2             (nn.MSELoss numerator)
 *   D[n]     = d_scale * (G[n] - S[n])             (optional; with d_scale = 4*w/(B*C^2*CHW) these are the per-image 1x1
 *                                                   weights of the Gram backward dF = D F, see ast_conv_gather)
 * target: S with `target_img_stride` elements between images (0 = one C x C target for the whole batch, which is what
 * train_cnn.py:187-190 builds by expanding one style image).  g ([n][c][c]) and counters
 * (AST_GRAM_COUNTERS_PER_IMAGE ints per image) must be ZERO on entry; loss is an fp64 accumulator shared by the taps of a
 * step (hundreds of small addends into a ~1e4 total: an fp32 accumulator loses 1e-5 of it).  flags: AST_CONV_TENSOR. */
#define AST_GRAM_COUNTERS_PER_IMAGE 16
int ast_gram_mse(const ast_image* x, float* g, float scale, const float* target, int64_t target_img_stride, double* loss,
                 float loss_scale, float* d, float d_scale, int32_t* counters, int32_t flags, void* stream);

/* nn.MSELoss pieces (train_cnn.py:249,307,323): loss[0] += scale * sum((a-b)^2) ; grad = gscale*(a-b) (optional).
 * a/b/grad are images of identical logical shape. */
int ast_mse(const ast_image* a, const ast_image* b, float* loss, float scale, const ast_image* grad,
            float gscale, void* stream);

/* dst = src converted/re-strided (NCHW fp32 <-> NHWC bf16/fp32), optional per-channel shift, reflect pad. */
int ast_copy_image(const ast_image* src, const ast_image* dst, const float* shift, int32_t pad, void* stream);
/* Adjoint of ast_copy_image's reflect padding (aten::reflection_pad2d_backward of cnn.py:58): the gradient of a layer's
 * input from the gradient of its reflection-padded copy,
 *   out[n,i,j,c] = sum over (y,x) of the (h+2p) x (w+2p) grid with R(y-p) = i, R(x-p) = j of gpad[n,y,x,c]  (+ add[n,i,j,c])
 * R = nn.ReflectionPad2d's index rule.  gpad: [n, h+2*pad, w+2*pad, c]; add: optional, shaped like out.  Each of gpad,
 * add and out is fp32 or bf16 with any strides (e.g. an NCHW out view).  0 <= pad < h, w; pad = 0 is a conversion (+ add). */
int ast_reflect_fold(const ast_image* gpad, const ast_image* add, const ast_image* out, int32_t pad, void* stream);
/* acc(fp32 image) += x   ('smartaverage' in-place feature sum, train_cnn.py:239).  With acc->n == 1 and x->n > 1 the batch
 * of x is summed into the one accumulator image (several paintings per VGG pass). */
int ast_accumulate(const ast_image* x, const ast_image* acc, void* stream);

/* out = (a + b) * (mask > 0)   (b may be NULL; nn.ReLU backward on an incoming tap gradient) */
int ast_mask_add(const ast_image* a, const ast_image* b, const ast_image* mask, const ast_image* out, void* stream);

/* ---- optimizer side (train_cnn.py:247-248,334,375: optim.Adam(lr 0.0024, weight_decay 1e-4) + StepLR), SURVEY 8f-1 ----
 * One table-driven launch applies L2 + Adam to every TransformerNet parameter tensor (addressed relative to one base
 * pointer, so the nn.Parameters stay where PyTorch allocated them) and refreshes the packed operand copies ([tap][cout][cin] bf16 / TF32 / fp32) the next step's convolutions read.
 * Gradients are read in the layout the filter-gradient kernels wrote them (tap-major scratch) through a per-tensor map,
 * so no permute / flatten pass is needed between backward, the NCCL all-reduce of the gradient arena and the update.
 *
 * Parameter element i of a tensor with logical shape dim = (A, B, U, V) decomposes as i = ((a*B + b)*U + u)*V + v;
 *   gradient  = grads[g_off + a*g_stride[0] + b*g_stride[1] + tap_table[g_tap + u*V + v]]
 *   pack k    = ((dtype*)((char*)pack_arena + pack[k].off))[a*stride[0] + b*stride[1] + tap_table[pack[k].tap + u*V + v]
 *                                                             + r*rep_stride],  r = 0 .. rep-1
 * (rep > 1: the row-interleaved stacked filters of ast_conv_stacked hold every tap once per lane block) */
typedef struct {
  int64_t off;            /* BYTES from the start of the pack arena */
  int64_t stride[2];      /* elements */
  int32_t tap;            /* first entry of this map in the tap table */
  int32_t dtype;          /* ast_dtype of the packed copy */
  int64_t rep_stride;     /* elements between the copies */
  int32_t rep;            /* copies of every element (>= 1) */
  int32_t reserved;
} ast_pack_map;
typedef struct {
  int64_t p_off;          /* first element relative to `params` (any fp32 tensors of one device: params = lowest address) */
  int64_t s_off;          /* first element in the exp_avg / exp_avg_sq arenas */
  int64_t numel;
  int32_t dim[4];
  int64_t g_off, g_stride[2];
  int32_t g_tap, n_pack;
  ast_pack_map pack[2];
} ast_param_desc;
typedef struct {          /* DEVICE-resident hyper-parameters and step state: graph replays read the current values */
  float lr, beta1, beta2, eps, weight_decay, grad_scale;
  float step, bias_c1, bias_c2;     /* step count, 1 - beta1^step, 1 - beta2^step: maintained by ast_adam_step */
} ast_adam_state;
/* descs / work / tap_table / state are DEVICE pointers.  work: n_work pairs (descriptor index, first element); every work
 * item covers ast_adam_work_item() consecutive elements of one tensor.  update = 0 only refreshes the packs (after
 * load_state_dict).  update = 1: state->step += 1 first (a one-thread kernel), then p, m, v and the packs are updated. */
int ast_adam_step(const ast_param_desc* descs, int32_t n_desc, const int32_t* work, int32_t n_work, float* params,
                  const float* grads, float* exp_avg, float* exp_avg_sq, void* pack_arena, const int64_t* tap_table,
                  ast_adam_state* state, int32_t update, void* stream);
int32_t ast_adam_work_item(void);

/* dst[dst_off + c] = sum_{r < rows} src[src_off + r*row_stride + c], c < cols, for n_desc descriptors (DEVICE array) in
 * one launch: dbeta / dgamma of all InstanceNorm layers from their per-(n, c) partial sums (aten::sum). */
typedef struct { int64_t src_off, dst_off, row_stride; int32_t rows, cols; } ast_reduce_desc;
int ast_batch_reduce(const float* src, float* dst, const ast_reduce_desc* descs, int32_t n_desc, int32_t max_cols,
                     void* stream);
/* out[c] += sum_{n,h,w} x[n,h,w,c]   (bias gradient of the last, norm-free conv layer, cnn.py:39; aten::sum) */
int ast_channel_sum(const ast_image* x, float* out, void* stream);

/* per-kernel-family accounting: launches and ALGORITHMIC flops / bytes of everything launched so far (bench.py divides
 * them by the family's device time; tests assert which kernel a case ran on).  Families: ast_family_name(0..count-1). */
int ast_family_count(void);
const char* ast_family_name(int family);
int ast_family_stats(int family, int64_t* launches, double* flops, double* bytes);
void ast_family_reset(void);

/* bitmask of the tensor-core kernels compiled into this build: 1 = tcgen05 gather conv, 2 = tcgen05 Gram/wgrad */
int ast_capabilities(void);
const char* ast_last_error(void);
int ast_abi_version(void);
/* number of kernel launches issued through this library by the calling process (bench.py gpu_launches) */
int64_t ast_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif
