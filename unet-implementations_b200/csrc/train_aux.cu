// The two steps either side of the hot path in the reference's trainer (SURVEY.md section 8f):
//  * the optimizer step -- torch.optim.SGD(momentum, nesterov=True, weight_decay) over the model's 90 parameter
//    tensors (Our_UNet/src/train.py:431-451) as ONE multi-tensor launch instead of ~5 foreach launches per step, and
//    torch.optim.Adam / AdamW (the autoencoder's, AE_pretrained/reconstruction/src/train.py:390-394) over the flat
//    buffers;
//  * the validation metric -- argmax over the 3 logits + per-class intersection / prediction / target counts over
//    the valid pixels (train.py:554-572, nine .item() host syncs per batch in the reference) as one pass with integer
//    counters (bit-exact) and no host sync.
#include "common.cuh"

namespace b200 {

constexpr int kSgdMaxTensors = 112;  // pointers travel in the kernel parameters (4 KB limit)
constexpr int kSgdThreads = 256, kSgdPerThread = 4;

struct SgdBatch {
  float* p[kSgdMaxTensors];
  const float* g[kSgdMaxTensors];
  float* buf[kSgdMaxTensors];
  int first_block[kSgdMaxTensors + 1];  // prefix sum of the blocks of each tensor
  int numel[kSgdMaxTensors];
  int count;
};

// Arithmetic mirrors torch's foreach SGD on CUDA operation by operation (each of its `a + alpha * b` kernels is one
// fused multiply-add; `buf.mul_(momentum)` and the following add are two roundings):
//   g1 = g + wd * p;  buf = first ? g1 : (buf * momentum) + g1;  g2 = g1 + momentum * buf;  p = p - lr * g2
__global__ void __launch_bounds__(kSgdThreads) sgd_nesterov_kernel(const __grid_constant__ SgdBatch B, float lr,
                                                                    float momentum, float wd, int nesterov,
                                                                    int first_step) {
  // which tensor owns this block: binary search in the prefix table
  int lo = 0, hi = B.count;
  const int b = blockIdx.x;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (B.first_block[mid] <= b) lo = mid; else hi = mid;
  }
  const int t = lo;
  const int n = B.numel[t];
  float* __restrict__ p = B.p[t];
  const float* __restrict__ g = B.g[t];
  float* __restrict__ buf = B.buf[t];
  const int base = (b - B.first_block[t]) * kSgdThreads * kSgdPerThread;
#pragma unroll
  for (int k = 0; k < kSgdPerThread; ++k) {
    const int i = base + k * kSgdThreads + threadIdx.x;
    if (i >= n) break;
    const float pv = p[i];
    float gv = g[i];
    if (wd != 0.f) gv = fmaf(wd, pv, gv);
    float upd = gv;
    if (momentum != 0.f) {
      const float bv = first_step ? gv : __fadd_rn(__fmul_rn(buf[i], momentum), gv);
      buf[i] = bv;
      upd = nesterov ? fmaf(momentum, bv, gv) : bv;
    }
    p[i] = fmaf(-lr, upd, pv);
  }
}

// ------------------------------------------------------------------------------------------------ flat optimizer step
// SURVEY.md 8f row 1 as written: ONE launch over the flat fp32 master / gradient / optimizer-state buffers that (i)
// applies the all-reduce epilogue scale to the gradient, (ii) updates master + state with an update rule (SgdRule:
// the SGD-Nesterov update of sgd_nesterov_kernel; AdamRule: torch's foreach Adam / AdamW; both bit-exact with torch
// for scale 1) and (iii) emits the bf16 operand packs the conv kernels consume -- [Cout][3][3][Cin] (fprop),
// [Cin][3][3][Cout] (dgrad) and the parity-stacked stride-2 dgrad pack -- so that no repack kernel runs between the
// optimizer and the next forward and the packs can never be stale.  The 3x3 weights of the tensor-core layers (99.9 %
// of the parameters) are processed in 32 x 32 x 9 tiles through shared memory so that the fp32 traffic AND the pack
// stores are coalesced; every other tensor (norm parameters, biases, the stem, 1x1 and padded heads) is walked element
// by element in storage order.
constexpr int kFlatThreads = 256, kFlatPerThread = 4;

// An update rule is built per block from the launch arguments and the block's tensor, and maps an element index of
// that tensor to its new master value (writing the optimizer state on the way); flat_step_kernel does the rest.
struct SgdRule {
  struct Args {
    float* master;
    const float* grad;
    float* mom;
    float lr, momentum, wd, grad_scale;
    int nesterov;
    const float* lr_dev;
  };
  float* __restrict__ p;
  const float* __restrict__ g;
  float* __restrict__ buf;
  float lr, momentum, wd, grad_scale;
  bool nesterov, first;
  __device__ __forceinline__ SgdRule(const Args& a, int, const b200unet_flat_tensor& D)
      : p(a.master + D.offset), g(a.grad + D.offset), buf(a.mom ? a.mom + D.offset : nullptr),
        // the learning rate as a device scalar (when given) keeps a CUDA graph of the whole training step valid across
        // LambdaLR updates (train.py:454-477): the host rewrites one float instead of re-capturing
        lr(a.lr_dev ? __ldg(a.lr_dev) : a.lr), momentum(a.momentum), wd(a.wd), grad_scale(a.grad_scale),
        nesterov(a.nesterov != 0), first((D.flags & 2) != 0) {}
  // torch's CUDA foreach SGD arithmetic, operation by operation
  __device__ __forceinline__ float operator()(int i) const {
    const float pv = p[i];
    float gv = __ldg(g + i);
    // every load before the first store: the compiler predicates the momentum path instead of branching around it,
    // and the loads of consecutive elements overlap
    const bool has_buf = momentum != 0.f;
    const float bo = has_buf && !first ? buf[i] : 0.f;
    if (grad_scale != 1.f) gv = __fmul_rn(gv, grad_scale);
    if (wd != 0.f) gv = fmaf(wd, pv, gv);
    float upd = gv;
    if (has_buf) {
      const float bv = first ? gv : __fadd_rn(__fmul_rn(bo, momentum), gv);
      buf[i] = bv;
      upd = nesterov ? fmaf(momentum, bv, gv) : bv;
    }
    const float pn = fmaf(-lr, upd, pv);
    p[i] = pn;
    return pn;
  }
};

// Adam / AdamW as torch 2.11's `_multi_tensor_adam` (torch/optim/adam.py, capturable=False) computes it on CUDA, one
// IEEE rounding per ATen kernel (the foreach kernels run in fp32 with their scalars rounded to fp32):
//   g = g * grad_scale                                  (only when grad_scale != 1)
//   L2:    g = fma(wd, p, g)                            _foreach_add(grads, params, alpha=wd)
//   AdamW: p = p * decay                                _foreach_mul_(params, 1 - lr * wd)
//   m = fma(w, g - m, m)                                _foreach_lerp_(exp_avgs, grads, 1 - beta1)  (ATen Lerp.h,
//                                                       |w| < 0.5; otherwise g - (g - m) * (1 - w))
//   v = fma(1 - beta2, g * g, v * beta2)                _foreach_mul_ + _foreach_addcmul_ (DeviceAddCmulCdiv.cuh)
//   d = sqrt(v) / bc2_sqrt + eps                        _foreach_sqrt, _foreach_div_, _foreach_add_
//   p = fma(step_size, m / d, p)                        _foreach_addcdiv_(params, exp_avgs, d, step_size)
// step_size, bc2_sqrt and decay are per tensor (each tensor has its own step count): adam_scalars_kernel writes them
// before this kernel runs.
struct AdamRule {
  struct Args {
    float* master;
    const float* grad;
    float* exp_avg;
    float* exp_avg_sq;
    const float4* scalars;  // per tensor: step_size, bc2_sqrt, decay (adam_scalars_kernel)
    float w1, w1c, beta2, c2, eps, wd, grad_scale;  // fp32 of 1 - beta1, 1 - w1, beta2, 1 - beta2, eps, weight_decay
    int decoupled;
  };
  float* __restrict__ p;
  const float* __restrict__ g;
  float* __restrict__ m;
  float* __restrict__ v;
  float step_size, bc2_sqrt, decay, w1, w1c, beta2, c2, eps, wd, grad_scale;
  bool decoupled;
  __device__ __forceinline__ AdamRule(const Args& a, int t, const b200unet_flat_tensor& D)
      : p(a.master + D.offset), g(a.grad + D.offset), m(a.exp_avg + D.offset), v(a.exp_avg_sq + D.offset),
        w1(a.w1), w1c(a.w1c), beta2(a.beta2), c2(a.c2), eps(a.eps), wd(a.wd), grad_scale(a.grad_scale),
        decoupled(a.decoupled != 0) {
    const float4 s = a.scalars[t];
    step_size = s.x;
    bc2_sqrt = s.y;
    decay = s.z;
  }
  __device__ __forceinline__ float operator()(int i) const {
    float pv = p[i];
    float gv = __ldg(g + i);
    const float mv = m[i], vv = v[i];
    if (grad_scale != 1.f) gv = __fmul_rn(gv, grad_scale);
    if (wd != 0.f) {
      if (decoupled) pv = __fmul_rn(pv, decay);
      else gv = fmaf(wd, pv, gv);
    }
    const float diff = __fsub_rn(gv, mv);
    const float mn = fabsf(w1) < 0.5f ? fmaf(w1, diff, mv) : fmaf(-diff, w1c, gv);
    const float gg = __fmul_rn(gv, gv);
    const float vb = __fmul_rn(vv, beta2);
    const float vn = c2 == 1.f ? fmaf(gv, gv, vb) : fmaf(c2, gg, vb);  // addcmul with value 1 is a single fma
    const float d = __fadd_rn(__fdiv_rn(__fsqrt_rn(vn), bc2_sqrt), eps);
    const float pn = fmaf(step_size, __fdiv_rn(mn, d), pv);
    m[i] = mn;
    v[i] = vn;
    p[i] = pn;
    return pn;
  }
};

template <class Rule>
__global__ void __launch_bounds__(kFlatThreads) flat_step_kernel(const b200unet_flat_tensor* __restrict__ T, int count,
                                                                  const __grid_constant__ typename Rule::Args A) {
  int lo = 0, hi = count;
  const int b = blockIdx.x;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(&T[mid].first_block) <= b) lo = mid; else hi = mid;
  }
  const b200unet_flat_tensor D = T[lo];
  if (!(D.flags & 1)) return;
  const Rule update(A, lo, D);
  __nv_bfloat16* wf = static_cast<__nv_bfloat16*>(D.wf);
  __nv_bfloat16* wdp = static_cast<__nv_bfloat16*>(D.wd);
  __nv_bfloat16* ws = static_cast<__nv_bfloat16*>(D.ws);
  const int kk = D.ksize * D.ksize;
  const int per_o = D.cin * kk;
  if (wf && kk == 9 && (D.cin & 31) == 0 && (D.cout & 31) == 0 && D.cin_pad == D.cin && D.cout_pad == D.cout) {
    // ---- 3x3 conv weights of the tensor-core path: TILES of 32 output x 32 input channels x 9 taps (9216 elements).
    // Walking a tensor in OIHW order made every bf16 pack store a lone 2-byte write (2-3 per parameter, 0.45 ms per
    // step for 0.5 GB of traffic); a tile is read as 32 runs of 288 contiguous floats (128-byte aligned), staged as
    // bf16 in shared memory, and written as 64-byte runs: 32 consecutive ci per (o, tap) into [Cout][3][3][Cin],
    // 32 consecutive o per (ci, tap) into [Cin][3][3][Cout] and the parity-stacked stride-2 pack.  The tensor owns
    // numel / 1024 = 9 x tiles blocks of the launch (the descriptor table's block count is unchanged): block j < tiles
    // takes tile j, the others have nothing to do.
    constexpr int kTileR = 288, kRowPad = 290;  // 145-word rows: the o-major read below is bank-conflict free
    __shared__ __nv_bfloat16 st[32 * kRowPad];
    const int ct_n = D.cin >> 5;
    const int tiles = (D.cout >> 5) * ct_n;
    const int j = b - D.first_block;
    if (j >= tiles) return;
    const int o0 = (j / ct_n) << 5, ci0 = (j - (j / ct_n) * ct_n) << 5;
    const int tile_base = o0 * per_o + ci0 * 9;
#pragma unroll 4
    for (int e = threadIdx.x; e < 32 * kTileR; e += kFlatThreads) {
      const int ol = e / kTileR, rl = e - ol * kTileR;
      st[ol * kRowPad + rl] = __float2bfloat16_rn(update(tile_base + ol * per_o + rl));
    }
    __syncthreads();
    for (int e = threadIdx.x; e < 32 * kTileR; e += kFlatThreads) {  // [o][tap][ci]: ci fastest
      const int cl = e & 31, tap = (e >> 5) % 9, ol = e / kTileR;
      wf[(static_cast<int64_t>(o0 + ol) * 9 + tap) * D.cin + ci0 + cl] = st[ol * kRowPad + cl * 9 + tap];
    }
    if (wdp || ws) {
      for (int e = threadIdx.x; e < 32 * kTileR; e += kFlatThreads) {  // [ci][tap][o]: o fastest
        const int ol = e & 31, tap = (e >> 5) % 9, cl = e / kTileR;
        const __nv_bfloat16 v = st[ol * kRowPad + cl * 9 + tap];
        const int ci = ci0 + cl, o = o0 + ol;
        if (wdp) wdp[(static_cast<int64_t>(ci) * 9 + tap) * D.cout + o] = v;
        if (ws) {
          const int kh = tap / 3, kw = tap - kh * 3;
          const int ph = kh == 1 ? 0 : 1, dh = kh == 0 ? 1 : 0;
          const int pw = kw == 1 ? 0 : 1, dw = kw == 0 ? 1 : 0;
          ws[((static_cast<int64_t>(ph * 2 + pw) * D.cin + ci) * 4 + (dh * 2 + dw)) * D.cout + o] = v;
        }
      }
    }
    return;
  }
  const int base = (b - D.first_block) * kFlatThreads * kFlatPerThread;
#pragma unroll
  for (int k = 0; k < kFlatPerThread; ++k) {
    const int i = base + k * kFlatThreads + threadIdx.x;
    if (i >= D.numel) break;
    const float pn = update(i);
    if (wf) {
      const int o = i / per_o;
      const int r = i - o * per_o;
      const int ci = r / kk;
      const int tap = (kk == 9) ? (r - ci * 9) : 4;  // a 1x1 weight is the centre tap of a zero 3x3 kernel
      const __nv_bfloat16 v = __float2bfloat16_rn(pn);
      wf[(static_cast<int64_t>(o) * 9 + tap) * D.cin_pad + ci] = v;
      if (wdp) wdp[(static_cast<int64_t>(ci) * 9 + tap) * D.cout_pad + o] = v;
      if (ws) {
        // parity-stacked stride-2 dgrad pack [4*Cin][4][Cout] (pack_s2_dgrad_weights_kernel): tap kh serves input-row
        // parity ph with shift dh:  kh = 1 -> (0, 0),  kh = 2 -> (1, 0),  kh = 0 -> (1, 1); same along w
        const int kh = tap / 3, kw = tap - kh * 3;
        const int ph = kh == 1 ? 0 : 1, dh = kh == 0 ? 1 : 0;
        const int pw = kw == 1 ? 0 : 1, dw = kw == 0 ? 1 : 0;
        ws[((static_cast<int64_t>(ph * 2 + pw) * D.cin + ci) * 4 + (dh * 2 + dw)) * D.cout + o] = v;
      }
    }
  }
}

// x * y in double-double arithmetic (hi + lo, |lo| <= ulp(hi) / 2)
__device__ __forceinline__ void dd_mul(double& xh, double& xl, double yh, double yl) {
  const double p = __dmul_rn(xh, yh);
  double e = fma(xh, yh, -p);
  e = fma(xh, yl, fma(xl, yh, e));
  xh = __dadd_rn(p, e);
  xl = __dsub_rn(e, __dsub_rn(xh, p));
}

// beta ** n for an integer n >= 1, correctly rounded to double like the libm pow behind Python's `beta ** step`:
// binary powering in double-double (relative error ~1e-30), rounded once at the end.  CUDA's pow() is within 2 ulp,
// which the cancellation in 1 - beta2 ** step (beta2 = 0.999) can carry into the fp32 scalars.
__device__ double pow_steps(double beta, unsigned n) {
  double rh = 1.0, rl = 0.0, bh = beta, bl = 0.0;
  while (true) {
    if (n & 1u) dd_mul(rh, rl, bh, bl);
    n >>= 1;
    if (!n) break;
    dd_mul(bh, bl, bh, bl);
  }
  return rh;
}

// The host-side half of torch's Adam step, on the device so that a CUDA graph replays it: advance the fp32 step count
// of every tensor that has a gradient (_foreach_add_(state_steps, 1)) and form its scalars in double exactly as
// adam.py does -- bc1 = 1 - beta1 ** step, step_size = (lr / bc1) * -1, bc2_sqrt = (1 - beta2 ** step) ** 0.5,
// decay = 1 - lr * weight_decay -- rounded to fp32 as ATen rounds a scalar list.  One block; the flat step kernel runs
// after it on the same stream.
__global__ void __launch_bounds__(128) adam_scalars_kernel(const b200unet_flat_tensor* __restrict__ T, int count,
                                                           float* __restrict__ steps, float4* __restrict__ scalars,
                                                           double lr_arg, const double* __restrict__ lr_dev,
                                                           double beta1, double beta2, double wd) {
  const double lr = lr_dev ? *lr_dev : lr_arg;
  for (int t = threadIdx.x; t < count; t += blockDim.x) {
    if (!(T[t].flags & 1)) continue;
    const float s = __fadd_rn(steps[t], 1.f);
    steps[t] = s;
    const unsigned n = static_cast<unsigned>(s);
    const double bc1 = __dsub_rn(1.0, pow_steps(beta1, n));
    const double bc2 = __dsub_rn(1.0, pow_steps(beta2, n));
    float4 o;
    o.x = __double2float_rn(-__ddiv_rn(lr, bc1));
    o.y = __double2float_rn(__dsqrt_rn(bc2));
    o.z = __double2float_rn(__dsub_rn(1.0, __dmul_rn(lr, wd)));
    o.w = 0.f;
    scalars[t] = o;
  }
}

// ------------------------------------------------------------------------------------------------ validation
constexpr int kEvalThreads = 256, kEvalPerThread = 8;

// counts[c][0] = #(pred == c & target == c & valid), [c][1] = #(pred == c & valid), [c][2] = #(target == c & valid)
__global__ void __launch_bounds__(kEvalThreads) argmax_counts_kernel(const float* __restrict__ logits,
                                                                      const int64_t* __restrict__ target,
                                                                      int ignore_index, int64_t* __restrict__ pred,
                                                                      unsigned long long* __restrict__ counts,
                                                                      int64_t HW) {
  __shared__ unsigned int sc[9];
  if (threadIdx.x < 9) sc[threadIdx.x] = 0;
  __syncthreads();
  const int n = blockIdx.y;
  const float* z = logits + static_cast<int64_t>(n) * 3 * HW;
  unsigned int c[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  const int64_t base = static_cast<int64_t>(blockIdx.x) * kEvalThreads * kEvalPerThread;
#pragma unroll
  for (int k = 0; k < kEvalPerThread; ++k) {
    const int64_t px = base + static_cast<int64_t>(k) * kEvalThreads + threadIdx.x;
    if (px >= HW) break;
    const float a0 = z[px], a1 = z[HW + px], a2 = z[2 * HW + px];
    // torch.argmax: first maximal index (ties -> lowest index); NaN is maximal, like torch
    int am = 0;
    float best = a0;
    if (a1 > best || (a1 != a1 && best == best)) { am = 1; best = a1; }
    if (a2 > best || (a2 != a2 && best == best)) { am = 2; best = a2; }
    if (pred) pred[static_cast<int64_t>(n) * HW + px] = am;
    const int64_t t = target[static_cast<int64_t>(n) * HW + px];
    if (t == ignore_index) continue;
    c[am * 3 + 1] += 1;
    if (t >= 0 && t < 3) {
      c[static_cast<int>(t) * 3 + 2] += 1;
      if (t == am) c[am * 3 + 0] += 1;
    }
  }
#pragma unroll
  for (int i = 0; i < 9; ++i) {
    unsigned int v = c[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(&sc[i], v);
  }
  __syncthreads();
  if (threadIdx.x < 9 && sc[threadIdx.x]) atomicAdd(&counts[threadIdx.x], static_cast<unsigned long long>(sc[threadIdx.x]));
}


// ------------------------------------------------------------------------------------------------ input pipeline
// PetSegmentationDataset.__getitem__ (Our_UNet/src/train.py:299-311) on the device: uint8 HWC image -> float / 255 ->
// (x - mean) / std -> fp32 NCHW, and uint8 mask -> clean-up (values > 2 other than 255 become 0) -> int64.  The batch
// crosses PCIe as uint8 (4 bytes per pixel instead of 20).  Same IEEE operations in the same order as the reference's
// torch CPU ops: bit-exact.
__global__ void __launch_bounds__(256) preprocess_u8_kernel(const uint8_t* __restrict__ img, const uint8_t* __restrict__ mask,
                                                             float* __restrict__ out, int64_t* __restrict__ mask_out,
                                                             float m0, float m1, float m2, float s0, float s1, float s2,
                                                             int64_t HW) {
  const int n = blockIdx.y;
  const int64_t px = static_cast<int64_t>(blockIdx.x) * 256 + threadIdx.x;
  if (px >= HW) return;
  if (img) {
    const uint8_t* p = img + (static_cast<int64_t>(n) * HW + px) * 3;
    float* o = out + static_cast<int64_t>(n) * 3 * HW + px;
    o[0] = __fdiv_rn(__fsub_rn(__fdiv_rn(static_cast<float>(p[0]), 255.f), m0), s0);
    o[HW] = __fdiv_rn(__fsub_rn(__fdiv_rn(static_cast<float>(p[1]), 255.f), m1), s1);
    o[2 * HW] = __fdiv_rn(__fsub_rn(__fdiv_rn(static_cast<float>(p[2]), 255.f), m2), s2);
  }
  if (mask) {
    const uint8_t v = mask[static_cast<int64_t>(n) * HW + px];
    mask_out[static_cast<int64_t>(n) * HW + px] = (v > 2 && v != 255) ? 0 : v;
  }
}


// uint8 HWC -> normalised bf16 NHWC zero-padded to 32 channels (the stem's operand): four pixels per thread (one
// 12-byte read, four 64-byte rows written).
__global__ void __launch_bounds__(256) preprocess_u8_nhwc32_kernel(const uint8_t* __restrict__ img, uint4* __restrict__ dst,
                                                                    float m0, float m1, float m2, float s0, float s1,
                                                                    float s2, int64_t total_px) {
  const int64_t px0 = (static_cast<int64_t>(blockIdx.x) * 256 + threadIdx.x) * 4;
  if (px0 >= total_px) return;
  uint8_t v[12];
  if (px0 + 4 <= total_px) {
    const uint32_t* q = reinterpret_cast<const uint32_t*>(img + px0 * 3);  // px0 % 4 == 0: 12-byte aligned groups
    const uint32_t w0 = __ldg(q), w1 = __ldg(q + 1), w2 = __ldg(q + 2);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      v[j] = (w0 >> (8 * j)) & 0xff;
      v[4 + j] = (w1 >> (8 * j)) & 0xff;
      v[8 + j] = (w2 >> (8 * j)) & 0xff;
    }
  } else {
#pragma unroll
    for (int j = 0; j < 12; ++j) v[j] = (px0 * 3 + j < total_px * 3) ? img[px0 * 3 + j] : 0;
  }
  const uint4 z = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (px0 + j >= total_px) break;
    const float r = __fdiv_rn(__fsub_rn(__fdiv_rn(static_cast<float>(v[3 * j + 0]), 255.f), m0), s0);
    const float g = __fdiv_rn(__fsub_rn(__fdiv_rn(static_cast<float>(v[3 * j + 1]), 255.f), m1), s1);
    const float b = __fdiv_rn(__fsub_rn(__fdiv_rn(static_cast<float>(v[3 * j + 2]), 255.f), m2), s2);
    const __nv_bfloat162 rg = __floats2bfloat162_rn(r, g);
    const __nv_bfloat162 b0 = __floats2bfloat162_rn(b, 0.f);
    uint4* o = dst + (px0 + j) * 4;
    o[0] = make_uint4(*reinterpret_cast<const uint32_t*>(&rg), *reinterpret_cast<const uint32_t*>(&b0), 0u, 0u);
    o[1] = z;
    o[2] = z;
    o[3] = z;
  }
}

}  // namespace b200

using namespace b200;

extern "C" int b200unet_sgd_max_tensors(void) { return kSgdMaxTensors; }

extern "C" int b200unet_sgd_nesterov_step(float* const* params, const float* const* grads, float* const* momentum_bufs,
                                          const int64_t* numels, int count, float lr, float momentum,
                                          float weight_decay, int nesterov, int first_step, void* stream) {
  B200_CHECK_ARG(params && grads && numels && count >= 0, "sgd_nesterov_step: null pointer");
  B200_CHECK_ARG(momentum == 0.f || momentum_bufs, "sgd_nesterov_step: momentum buffers required");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  for (int t0 = 0; t0 < count; t0 += kSgdMaxTensors) {
    SgdBatch B;
    B.count = count - t0 < kSgdMaxTensors ? count - t0 : kSgdMaxTensors;
    int blocks = 0;
    for (int i = 0; i < B.count; ++i) {
      const int64_t n = numels[t0 + i];
      B200_CHECK_ARG(n > 0 && n < (1ll << 31), "sgd_nesterov_step: tensor %d has %lld elements", t0 + i, (long long)n);
      B200_CHECK_ARG(params[t0 + i] && grads[t0 + i], "sgd_nesterov_step: tensor %d has a null pointer", t0 + i);
      B.p[i] = params[t0 + i];
      B.g[i] = grads[t0 + i];
      B.buf[i] = momentum_bufs ? momentum_bufs[t0 + i] : nullptr;
      B.numel[i] = static_cast<int>(n);
      B.first_block[i] = blocks;
      blocks += static_cast<int>(ceil_div64(n, kSgdThreads * kSgdPerThread));
    }
    B.first_block[B.count] = blocks;
    if (blocks == 0) continue;
    sgd_nesterov_kernel<<<blocks, kSgdThreads, 0, st>>>(B, lr, momentum, weight_decay, nesterov, first_step);
    B200_LAUNCH_CHECK("sgd_nesterov_kernel");
  }
  return 0;
}

extern "C" int b200unet_sgd_flat_block_elems(void) { return kFlatThreads * kFlatPerThread; }

extern "C" int b200unet_sgd_flat_step(const b200unet_flat_tensor* table_dev, int count, int total_blocks, float* master,
                                      const float* grad, float* momentum_buf, float lr, float momentum,
                                      float weight_decay, int nesterov, float grad_scale, const float* lr_dev,
                                      void* stream) {
  B200_CHECK_ARG(table_dev && master && grad && count > 0 && total_blocks > 0, "sgd_flat_step: null pointer or empty table");
  B200_CHECK_ARG(momentum == 0.f || momentum_buf, "sgd_flat_step: momentum buffer required");
  const SgdRule::Args a{master, grad, momentum_buf, lr, momentum, weight_decay, grad_scale, nesterov, lr_dev};
  flat_step_kernel<SgdRule><<<total_blocks, kFlatThreads, 0, static_cast<cudaStream_t>(stream)>>>(table_dev, count, a);
  B200_LAUNCH_CHECK("flat_step_kernel<SgdRule>");
  return 0;
}

extern "C" int b200unet_adam_flat_step(const b200unet_flat_tensor* table_dev, int count, int total_blocks, float* master,
                                       const float* grad, float* exp_avg, float* exp_avg_sq, float* steps,
                                       float* scalars_ws, double lr, const double* lr_dev, double beta1, double beta2,
                                       double eps, double weight_decay, int decoupled, float grad_scale, void* stream) {
  B200_CHECK_ARG(table_dev && master && grad && exp_avg && exp_avg_sq && steps && scalars_ws && count > 0 &&
                     total_blocks > 0, "adam_flat_step: null pointer or empty table");
  B200_CHECK_ARG((reinterpret_cast<uintptr_t>(scalars_ws) & 15) == 0, "adam_flat_step: scalars_ws must be 16-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  adam_scalars_kernel<<<1, 128, 0, st>>>(table_dev, count, steps, reinterpret_cast<float4*>(scalars_ws), lr, lr_dev,
                                          beta1, beta2, weight_decay);
  B200_LAUNCH_CHECK("adam_scalars_kernel");
  // the fp32 scalars of the foreach calls, rounded from the double the Python code computes
  const float w1 = static_cast<float>(1.0 - beta1);
  const AdamRule::Args a{master, grad, exp_avg, exp_avg_sq, reinterpret_cast<const float4*>(scalars_ws), w1, 1.f - w1,
                         static_cast<float>(beta2), static_cast<float>(1.0 - beta2), static_cast<float>(eps),
                         static_cast<float>(weight_decay), grad_scale, decoupled};
  flat_step_kernel<AdamRule><<<total_blocks, kFlatThreads, 0, st>>>(table_dev, count, a);
  B200_LAUNCH_CHECK("flat_step_kernel<AdamRule>");
  return 0;
}

extern "C" int b200unet_argmax_counts(const float* logits_nchw, const int64_t* target, int ignore_index,
                                      int64_t* pred_or_null, int64_t* counts9, int N, int64_t HW, void* stream) {
  B200_CHECK_ARG(logits_nchw && target && counts9, "argmax_counts: null pointer");
  B200_CHECK_ARG(N > 0 && N <= 65535 && HW > 0, "argmax_counts: bad sizes");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  B200_CUDA(cudaMemsetAsync(counts9, 0, 9 * sizeof(int64_t), st));
  const int blocks = static_cast<int>(ceil_div64(HW, kEvalThreads * kEvalPerThread));
  argmax_counts_kernel<<<dim3(blocks, N), kEvalThreads, 0, st>>>(logits_nchw, target, ignore_index, pred_or_null,
                                                                 reinterpret_cast<unsigned long long*>(counts9), HW);
  B200_LAUNCH_CHECK("argmax_counts_kernel");
  return 0;
}

extern "C" int b200unet_preprocess_u8(const void* image_u8_nhwc, const void* mask_u8, float* image_out_nchw,
                                      int64_t* mask_out, const float* mean3, const float* std3, int N, int64_t HW,
                                      void* stream) {
  B200_CHECK_ARG((image_u8_nhwc && image_out_nchw && mean3 && std3) || (mask_u8 && mask_out), "preprocess_u8: nothing to do");
  B200_CHECK_ARG(N > 0 && N <= 65535 && HW > 0, "preprocess_u8: bad sizes");
  const float m[3] = {mean3 ? mean3[0] : 0.f, mean3 ? mean3[1] : 0.f, mean3 ? mean3[2] : 0.f};
  const float sd[3] = {std3 ? std3[0] : 1.f, std3 ? std3[1] : 1.f, std3 ? std3[2] : 1.f};
  preprocess_u8_kernel<<<dim3((unsigned)ceil_div64(HW, 256), N), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const uint8_t*>(image_u8_nhwc), static_cast<const uint8_t*>(mask_u8), image_out_nchw, mask_out, m[0], m[1],
      m[2], sd[0], sd[1], sd[2], HW);
  B200_LAUNCH_CHECK("preprocess_u8_kernel");
  return 0;
}

extern "C" int b200unet_preprocess_u8_nhwc32(const void* image_u8_nhwc, void* dst_nhwc32, const float* mean3,
                                             const float* std3, int N, int64_t HW, void* stream) {
  B200_CHECK_ARG(image_u8_nhwc && dst_nhwc32 && mean3 && std3, "preprocess_u8_nhwc32: null pointer");
  B200_CHECK_ARG(N > 0 && HW > 0, "preprocess_u8_nhwc32: bad sizes");
  B200_CHECK_ARG((reinterpret_cast<uintptr_t>(image_u8_nhwc) & 3) == 0 && (reinterpret_cast<uintptr_t>(dst_nhwc32) & 15) == 0,
                 "preprocess_u8_nhwc32: source must be 4-byte and destination 16-byte aligned");
  const int64_t total = static_cast<int64_t>(N) * HW;
  preprocess_u8_nhwc32_kernel<<<(unsigned)ceil_div64(total, 1024), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const uint8_t*>(image_u8_nhwc), static_cast<uint4*>(dst_nhwc32), mean3[0], mean3[1], mean3[2], std3[0],
      std3[1], std3[2], total);
  B200_LAUNCH_CHECK("preprocess_u8_nhwc32_kernel");
  return 0;
}
