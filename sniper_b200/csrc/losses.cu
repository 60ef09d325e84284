// Loss layers of the SNIPER graph, forward + gradient in one pass, valid-count kept on the device.
//
// Replaces SoftmaxOutput (SNIPER-mxnet/src/operator/softmax_output-inl.h:108-132 fwd, :162-206
// multi_output bwd, :207-263 flat bwd; the reference copies the labels to the host every backward to
// count non-ignored entries, :184-195 / :243-253), smooth_l1 (mshadow_op.h:642-678) and MakeLoss as used by
// symbols/faster/resnet_mx_101_e2e.py:279-281, 310-319, 330-334.
#include "common.cuh"
#include <math.h>

namespace {

__global__ void count_valid_kernel(const float* __restrict__ label, long n, int ignore, int* __restrict__ out) {
  int c = 0;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x)
    c += ((int)label[i] != ignore);
  c = __reduce_add_sync(0xffffffffu, c);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, c);
}

// RPN 2-way softmax over (bg = channel a, fg = channel A+a) of NHWC scores [B,H,W,ld]; labels [B,A*H*W] in
// (a,h,w) order with -1 = ignore.  Writes prob (same layout as scores) and dscore = (p - onehot)*gs/valid.
__global__ void __launch_bounds__(256) rpn_softmax_kernel(const float* __restrict__ score, int ld,
                                                           const float* __restrict__ label, int B, int H, int W, int A,
                                                           float grad_scale, const int* __restrict__ valid_cnt,
                                                           float* __restrict__ prob, int ldp,
                                                           float* __restrict__ dscore, int ldg,
                                                           float* __restrict__ loss_sum) {
  const long total = (long)B * H * W * A;
  const int HW = H * W;
  float norm = 1.0f;
  if (valid_cnt) {
    const int v = *valid_cnt;
    norm = grad_scale / (float)(v == 0 ? 1 : v);
  }
  float lsum = 0.f;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int a = (int)(i % A);
    const long pix = i / A;  // b*HW + hw
    const int b = (int)(pix / HW), hw = (int)(pix - (long)b * HW);
    const float s0 = score[pix * ld + a], s1 = score[pix * ld + A + a];
    const float m = fmaxf(s0, s1);
    const float e0 = expf(s0 - m), e1 = expf(s1 - m);
    const float inv = 1.0f / (e0 + e1);
    const float p0 = e0 * inv, p1 = e1 * inv;
    prob[pix * ldp + a] = p0;
    prob[pix * ldp + A + a] = p1;
    if (dscore) {
      const int l = (int)label[(long)b * A * HW + (long)a * HW + hw];
      float g0 = 0.f, g1 = 0.f;
      if (l != -1) {
        g0 = (p0 - (l == 0 ? 1.f : 0.f)) * norm;
        g1 = (p1 - (l == 1 ? 1.f : 0.f)) * norm;
        lsum -= logf(fmaxf(l == 1 ? p1 : p0, 1e-14f));
      }
      dscore[pix * ldg + a] = g0;
      dscore[pix * ldg + A + a] = g1;
    }
  }
  if (loss_sum) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) lsum += __shfl_xor_sync(0xffffffffu, lsum, off);
    if ((threadIdx.x & 31) == 0 && lsum != 0.f) atomicAdd(loss_sum, lsum);
  }
}

__device__ __forceinline__ float smooth_l1(float d) { return fabsf(d) < 1.f ? 0.5f * d * d : fabsf(d) - 0.5f; }
__device__ __forceinline__ float smooth_l1_grad(float d) { return fabsf(d) < 1.f ? d : (d > 0.f ? 1.f : -1.f); }

// RPN box loss: pred NHWC [B,H,W,ld] channel 4a+j; target/weight NCHW [B,4A,H,W] (the iterator's layout)
__global__ void __launch_bounds__(256) rpn_smooth_l1_kernel(const float* __restrict__ pred, int ld,
                                                             const float* __restrict__ target,
                                                             const float* __restrict__ weight, int B, int H, int W,
                                                             int C4, float grad_scale, float* __restrict__ dpred,
                                                             int ldg, float* __restrict__ loss_sum) {
  const long total = (long)B * H * W * C4;
  const int HW = H * W;
  float lsum = 0.f;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C4);
    const long pix = i / C4;
    const int b = (int)(pix / HW), hw = (int)(pix - (long)b * HW);
    const long t = ((long)b * C4 + c) * HW + hw;
    const float w = weight[t];
    const float d = pred[pix * ld + c] - target[t];
    dpred[pix * ldg + c] = w * smooth_l1_grad(d) * grad_scale;
    lsum += w * smooth_l1(d);
  }
  if (loss_sum) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) lsum += __shfl_xor_sync(0xffffffffu, lsum, off);
    if ((threadIdx.x & 31) == 0 && lsum != 0.f) atomicAdd(loss_sum, lsum);
  }
}

// flat softmax + CE gradient, one warp per row of [N,K] (K <= 1024)
__global__ void __launch_bounds__(256) softmax_ce_kernel(const float* __restrict__ logits, int ld,
                                                          const float* __restrict__ label, int N, int K, int ignore,
                                                          float grad_scale, const int* __restrict__ valid_cnt,
                                                          float* __restrict__ prob, int ldp, float* __restrict__ grad,
                                                          int ldg, float* __restrict__ loss_sum) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= N) return;
  float norm = grad_scale;
  if (valid_cnt) {
    const int v = *valid_cnt;
    norm = grad_scale / (float)(v == 0 ? 1 : v);
  }
  const float* row = logits + (long)warp * ld;
  float m = -INFINITY;
  for (int k = lane; k < K; k += 32) m = fmaxf(m, row[k]);
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, off));
  float s = 0.f;
  for (int k = lane; k < K; k += 32) s += expf(row[k] - m);
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
  const float inv = 1.0f / s;
  const int l = (int)label[warp];
  for (int k = lane; k < K; k += 32) {
    const float p = expf(row[k] - m) * inv;
    if (prob) prob[(long)warp * ldp + k] = p;
    if (grad) grad[(long)warp * ldg + k] = l == ignore ? 0.f : (p - (k == l ? 1.f : 0.f)) * norm;
    if (loss_sum && k == l && l != ignore) atomicAdd(loss_sum, -logf(fmaxf(p, 1e-14f)));
  }
}

// R-CNN box loss on [N,C]: grad = weight * smooth_l1'(pred - target) * grad_scale
__global__ void __launch_bounds__(256) smooth_l1_kernel(const float* __restrict__ pred, int ld,
                                                         const float* __restrict__ target,
                                                         const float* __restrict__ weight, long N, int C,
                                                         float grad_scale, float* __restrict__ grad, int ldg,
                                                         float* __restrict__ loss_sum) {
  const long total = N * C;
  float lsum = 0.f;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const long r = i / C;
    const int c = (int)(i - r * C);
    const float w = weight[i];
    const float d = pred[r * ld + c] - target[i];
    grad[r * ldg + c] = w * smooth_l1_grad(d) * grad_scale;
    lsum += w * smooth_l1(d);
  }
  if (loss_sum) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) lsum += __shfl_xor_sync(0xffffffffu, lsum, off);
    if ((threadIdx.x & 31) == 0 && lsum != 0.f) atomicAdd(loss_sum, lsum);
  }
}

// AutoFocus FocusPixel head (resnet_mx_101_e2e.py:264-267, 313-315): conv_new_out (1x1, C = 256 -> 2) + SoftmaxOutput(
// multi_output, normalization='valid', use_ignore, ignore_label=-1) + the whole backward of that layer, in one pass over
// x3 = conv_new_3_relu [M, 256].  One warp per row: lane l holds channels [4l, 4l+4) and [128+4l, 128+4l+4) of the row
// and of both weight rows (registers); the two logits are warp all-reductions (xor butterfly: every lane ends with the
// same bits).  Softmax / gradient / loss arithmetic is rpn_softmax_kernel's.  dx3 = (x3 > 0) * (dz0 * W0 + dz1 * W1)
// folds conv_new_3's ReLU backward; dW / db are per-warp register partials, summed over the block in shared memory and
// added with one float atomic per element and block.  FP32 FMA throughout (no tensor-core contraction).
constexpr int kFocusC = 256;
constexpr int kFocusTPB = 256;

__global__ void __launch_bounds__(kFocusTPB) focus_head_kernel(const float* __restrict__ x3, long M,
                                                               const float* __restrict__ w, const float* __restrict__ bias,
                                                               const float* __restrict__ label, float grad_scale,
                                                               const int* __restrict__ valid_cnt, float* __restrict__ prob,
                                                               float* __restrict__ dx3, float* __restrict__ dw,
                                                               float* __restrict__ db, float* __restrict__ stats) {
  __shared__ float red[kFocusTPB / 32][2 * kFocusC];
  __shared__ float red_b[kFocusTPB / 32][2];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int c0 = 4 * lane, c1 = 128 + 4 * lane;
  float w0[8], w1[8];
  {
    const float4 a = *reinterpret_cast<const float4*>(w + c0), b = *reinterpret_cast<const float4*>(w + c1);
    const float4 c = *reinterpret_cast<const float4*>(w + kFocusC + c0), d = *reinterpret_cast<const float4*>(w + kFocusC + c1);
    w0[0] = a.x; w0[1] = a.y; w0[2] = a.z; w0[3] = a.w; w0[4] = b.x; w0[5] = b.y; w0[6] = b.z; w0[7] = b.w;
    w1[0] = c.x; w1[1] = c.y; w1[2] = c.z; w1[3] = c.w; w1[4] = d.x; w1[5] = d.y; w1[6] = d.z; w1[7] = d.w;
  }
  const float b0 = bias[0], b1 = bias[1];
  const int v = *valid_cnt;
  const float norm = grad_scale / (float)(v == 0 ? 1 : v);
  float g0[8], g1[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) g0[j] = g1[j] = 0.f;
  float gb0 = 0.f, gb1 = 0.f, lsum = 0.f, ncor = 0.f;
  const long nwarps = (long)gridDim.x * (kFocusTPB / 32);
  for (long r = (long)blockIdx.x * (kFocusTPB / 32) + wib; r < M; r += nwarps) {
    const float* xr = x3 + r * kFocusC;
    const float4 xa = __ldg(reinterpret_cast<const float4*>(xr + c0)), xb = __ldg(reinterpret_cast<const float4*>(xr + c1));
    const float x[8] = {xa.x, xa.y, xa.z, xa.w, xb.x, xb.y, xb.z, xb.w};
    float z0 = 0.f, z1 = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      z0 = fmaf(x[j], w0[j], z0);
      z1 = fmaf(x[j], w1[j], z1);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      z0 += __shfl_xor_sync(0xffffffffu, z0, off);
      z1 += __shfl_xor_sync(0xffffffffu, z1, off);
    }
    z0 += b0;
    z1 += b1;
    const float m = fmaxf(z0, z1);
    const float e0 = expf(z0 - m), e1 = expf(z1 - m);
    const float inv = 1.0f / (e0 + e1);
    const float p0 = e0 * inv, p1 = e1 * inv;
    const int l = (int)label[r];
    float d0 = 0.f, d1 = 0.f;
    if (l != -1) {
      d0 = (p0 - (l == 0 ? 1.f : 0.f)) * norm;
      d1 = (p1 - (l == 1 ? 1.f : 0.f)) * norm;
      lsum -= logf(fmaxf(l == 1 ? p1 : p0, 1e-14f));
      ncor += ((p1 > p0 ? 1 : 0) == l) ? 1.f : 0.f;        // argmax_channel: the first maximum on a tie
      gb0 += d0;
      gb1 += d1;
    }
    if (lane == 0) *reinterpret_cast<float2*>(prob + 2 * r) = make_float2(p0, p1);
    float y[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      y[j] = x[j] > 0.f ? fmaf(d1, w1[j], d0 * w0[j]) : 0.f;
      g0[j] = fmaf(d0, x[j], g0[j]);
      g1[j] = fmaf(d1, x[j], g1[j]);
    }
    float* dr = dx3 + r * kFocusC;
    *reinterpret_cast<float4*>(dr + c0) = make_float4(y[0], y[1], y[2], y[3]);
    *reinterpret_cast<float4*>(dr + c1) = make_float4(y[4], y[5], y[6], y[7]);
  }
  // block reduction of the weight / bias gradient partials, then one atomic per element
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    red[wib][c0 + j] = g0[j];
    red[wib][c1 + j] = g0[4 + j];
    red[wib][kFocusC + c0 + j] = g1[j];
    red[wib][kFocusC + c1 + j] = g1[4 + j];
  }
  if (lane == 0) {
    red_b[wib][0] = gb0;
    red_b[wib][1] = gb1;
    if (lsum != 0.f) atomicAdd(stats, lsum);
    if (ncor != 0.f) atomicAdd(stats + 1, ncor);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * kFocusC; i += kFocusTPB) {
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < kFocusTPB / 32; ++k) s += red[k][i];
    if (s != 0.f) atomicAdd(dw + i, s);
  }
  if (threadIdx.x < 2) {
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < kFocusTPB / 32; ++k) s += red_b[k][threadIdx.x];
    if (s != 0.f) atomicAdd(db + threadIdx.x, s);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(stats + 2, (float)v);
}

int lgrid(long n) {
  long g = (n + 255) / 256;
  const long cap = (long)sn::kNumSMs * 8;
  return (int)(g > cap ? cap : (g < 1 ? 1 : g));
}

}  // namespace

extern "C" {

// out_count must be zeroed by the caller (device int)
int sniper_count_valid(const float* label, long n, int ignore_label, int* out_count, void* stream) {
  count_valid_kernel<<<lgrid(n), 256, 0, (cudaStream_t)stream>>>(label, n, ignore_label, out_count);
  SN_LAUNCH_CHECK();
  return 0;
}

int sniper_rpn_softmax_loss(const float* score, int ld, const float* label, int B, int H, int W, int A,
                            float grad_scale, const int* valid_cnt, float* prob, int ldp, float* dscore, int ldg,
                            float* loss_sum, void* stream) {
  rpn_softmax_kernel<<<lgrid((long)B * H * W * A), 256, 0, (cudaStream_t)stream>>>(
      score, ld, label, B, H, W, A, grad_scale, valid_cnt, prob, ldp, dscore, ldg, loss_sum);
  SN_LAUNCH_CHECK();
  return 0;
}

int sniper_rpn_smooth_l1_loss(const float* pred, int ld, const float* target, const float* weight, int B, int H, int W,
                              int C4, float grad_scale, float* dpred, int ldg, float* loss_sum, void* stream) {
  rpn_smooth_l1_kernel<<<lgrid((long)B * H * W * C4), 256, 0, (cudaStream_t)stream>>>(
      pred, ld, target, weight, B, H, W, C4, grad_scale, dpred, ldg, loss_sum);
  SN_LAUNCH_CHECK();
  return 0;
}

int sniper_softmax_ce(const float* logits, int ld, const float* label, int N, int K, int ignore_label,
                      float grad_scale, const int* valid_cnt, float* prob, int ldp, float* grad, int ldg,
                      float* loss_sum, void* stream) {
  SN_CHECK(K <= 4096, "softmax_ce: K too large");
  softmax_ce_kernel<<<sn::div_up((long)N * 32, 256), 256, 0, (cudaStream_t)stream>>>(
      logits, ld, label, N, K, ignore_label, grad_scale, valid_cnt, prob, ldp, grad, ldg, loss_sum);
  SN_LAUNCH_CHECK();
  return 0;
}

int sniper_smooth_l1_loss(const float* pred, int ld, const float* target, const float* weight, long N, int C,
                          float grad_scale, float* grad, int ldg, float* loss_sum, void* stream) {
  smooth_l1_kernel<<<lgrid(N * C), 256, 0, (cudaStream_t)stream>>>(pred, ld, target, weight, N, C, grad_scale, grad,
                                                                 ldg, loss_sum);
  SN_LAUNCH_CHECK();
  return 0;
}

// x3: [M, C] fp32 rows (C = 256, contiguous); w: [>=2, C] fp32 (rows 0 and 1 = the two classes), bias: [>=2]; label: [M]
// in {-1, 0, 1} (-1 = ignore); valid_cnt: device int (number of labels != -1, sniper_count_valid).  Writes prob [M, 2] and
// dx3 [M, C]; ACCUMULATES dw rows 0..1 (+= dz^T x3), db[0..1] (+= sum dz) and stats[0] += sum of -log p(label),
// stats[1] += #correct (argmax == label), stats[2] += valid count.  Rows of w / dw beyond 1 are neither read nor written.
int sniper_focus_head(const float* x3, long M, int C, const float* w, const float* bias, const float* label,
                      float grad_scale, const int* valid_cnt, float* prob, float* dx3, float* dw, float* db, float* stats,
                      void* stream) {
  SN_CHECK(C == kFocusC, "focus_head: C must be %d", kFocusC);
  SN_CHECK(M > 0, "focus_head: empty input");
  SN_CHECK(((uintptr_t)x3 | (uintptr_t)w | (uintptr_t)dx3) % 16 == 0 && (uintptr_t)prob % 8 == 0,
           "focus_head: misaligned operand");
  long g = (M + 4 * (kFocusTPB / 32) - 1) / (4 * (kFocusTPB / 32));      // >= 4 rows per warp
  const long cap = (long)sn::kNumSMs * 4;
  focus_head_kernel<<<(int)(g > cap ? cap : g), kFocusTPB, 0, (cudaStream_t)stream>>>(
      x3, M, w, bias, label, grad_scale, valid_cnt, prob, dx3, dw, db, stats);
  SN_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
