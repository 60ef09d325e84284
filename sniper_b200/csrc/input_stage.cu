// GPU input stage of the SNIPER training iterator: decoded uint8 image crops -> the network's `data` tensor, and the
// random fg / bg subsampling of the RPN labels.
//
// Replaces, per chip, the body of `im_worker.worker` (lib/data_utils/data_workers.py:80-121: horizontal flip, crop,
// cv2.resize(fx = fy = scale, INTER_LINEAR), zero padding to crop_size x crop_size, BGR -> RGB with the per-channel
// PIXEL_MEANS subtracted) and the `npr.choice` subsampling of `anchor_worker.worker` (:326-338) that in the reference
// run on host worker processes (Pool(64) + pickling per batch).  The host now only slices the source rectangle of each
// chip out of the decoded image (uint8, 1/4 of the fp32 bytes, before up-scaling) into one pinned staging buffer.
//
// Resize arithmetic = OpenCV's 8-bit INTER_LINEAR path as documented in imgproc/resize.cpp (this image has no OpenCV to
// compare against: parity with cv2 is UNPINNED; tests compare with exact bilinear interpolation to <= 1 grey level):
//   dsize = (cvRound(w * fx), cvRound(h * fy)), source coordinate sx = (dx + 0.5) / fx - 0.5, x0 = floor(sx),
//   clamped taps, coefficients quantised to 1/2048 (cvRound), horizontal pass in int32, vertical pass
//   ((b0 * (S0 >> 4)) >> 16) + ((b1 * (S1 >> 4)) >> 16) + 2) >> 2.
#include "common.cuh"
#include <math.h>

namespace {

struct ChipDesc {          // one row of the chip table (host-filled, int64 x 8)
  long long src_off;       // byte offset of the chip's source rectangle in the staging buffer (BGR, HWC, uint8)
  long long src_h, src_w;  // rows / columns of that rectangle
  long long dst_h, dst_w;  // size after the resize = cvRound(src * scale)
  long long flipped;       // 1: the rectangle was cut from the UNflipped image and must be mirrored horizontally
  long long scale_bits;    // the float64 scale, bit pattern
  long long pad;
};

__device__ __forceinline__ int cv_round(double v) { return (int)rint(v); }   // cvRound: round half to even

// one tap pair along one axis: index of the first tap (clamped) and the two 11-bit coefficients
__device__ __forceinline__ void taps(int d, double inv_scale, int n_src, int& i0, int& i1, int& c0, int& c1) {
  double s = (d + 0.5) * inv_scale - 0.5;
  int i = (int)floor(s);
  float f = (float)(s - i);
  if (i < 0) { i = 0; f = 0.f; }
  if (i >= n_src - 1) { i = n_src - 1; f = 0.f; }
  i0 = i;
  i1 = min(i + 1, n_src - 1);
  c0 = (int)rintf((1.f - f) * 2048.f);
  c1 = (int)rintf(f * 2048.f);
}

// data[b, j, y, x] (fp32 NCHW, SH x SW) = resized(chip b)[y, x, 2 - j] - mean[2 - j] inside the resized extent, 0 outside
__global__ void __launch_bounds__(256) chip_input_kernel(const uint8_t* __restrict__ src, const ChipDesc* __restrict__ tab,
                                                         const float* __restrict__ means_bgr, float* __restrict__ data,
                                                         int B, int SH, int SW) {
  const long total = (long)B * SH * SW;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int x = (int)(i % SW);
    const int y = (int)((i / SW) % SH);
    const int b = (int)(i / ((long)SH * SW));
    const ChipDesc d = tab[b];
    float out[3] = {0.f, 0.f, 0.f};
    if (y < d.dst_h && x < d.dst_w && d.src_h > 0 && d.src_w > 0) {
      const double inv = 1.0 / __longlong_as_double(d.scale_bits);
      int y0, y1, b0, b1, x0, x1, a0, a1;
      taps(y, inv, (int)d.src_h, y0, y1, b0, b1);
      taps(x, inv, (int)d.src_w, x0, x1, a0, a1);
      if (d.flipped) {               // the resize runs on the flipped crop: mirror the source columns
        x0 = (int)d.src_w - 1 - x0;
        x1 = (int)d.src_w - 1 - x1;
      }
      const uint8_t* base = src + d.src_off;
      const long rs = d.src_w * 3;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const int s00 = base[y0 * rs + x0 * 3 + c], s01 = base[y0 * rs + x1 * 3 + c];
        const int s10 = base[y1 * rs + x0 * 3 + c], s11 = base[y1 * rs + x1 * 3 + c];
        const int r0 = s00 * a0 + s01 * a1, r1 = s10 * a0 + s11 * a1;        // horizontal pass, scaled by 2^11
        const int v = (((b0 * (r0 >> 4)) >> 16) + ((b1 * (r1 >> 4)) >> 16) + 2) >> 2;
        out[c] = (float)min(max(v, 0), 255);
      }
    }
    const bool inside = (y < d.dst_h && x < d.dst_w);
#pragma unroll
    for (int j = 0; j < 3; ++j)     // output channel j = BGR channel 2 - j, mean-subtracted; padding stays 0
      data[(((long)b * 3 + j) * SH + y) * SW + x] = inside ? out[2 - j] - means_bgr[2 - j] : 0.f;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Random subsampling of RPN labels: per chip keep at most num_fg labels == 1 and batch_size - #fg labels == 0; the rest
// become -1 (anchor_worker.worker :326-338).  One CTA per chip.  The subset is chosen by a counter-based hash of
// (seed, chip, anchor): the (n - keep) SMALLEST keys of a class are disabled; the threshold key is found by a 4-pass
// byte-wise radix select (shared-memory histograms).
__device__ __forceinline__ uint32_t mix32(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t h = a * 0x9E3779B1u ^ (b + 0x7F4A7C15u) * 0x85EBCA77u ^ (c + 0x165667B1u) * 0xC2B2AE3Du;
  h ^= h >> 16; h *= 0x7FEB352Du; h ^= h >> 15; h *= 0x846CA68Bu; h ^= h >> 16;
  return h;
}

constexpr int kSubTPB = 1024;

// returns (threshold key, how many keys equal to the threshold must also be taken); k >= 1 keys to take of class `cls`
__device__ void radix_select(const float* lab, int n, float cls, uint32_t seed, uint32_t chip, int k, uint32_t& thr,
                             int& take_eq, int* hist /*[256]*/, int* sh /*[2]*/) {
  uint32_t prefix = 0, mask = 0;
  int remaining = k;
  for (int pass = 3; pass >= 0; --pass) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x)
      if (lab[i] == cls) {
        const uint32_t key = mix32(seed, chip, (uint32_t)i);
        if ((key & mask) == prefix) atomicAdd(&hist[(key >> (8 * pass)) & 255u], 1);
      }
    __syncthreads();
    if (threadIdx.x == 0) {
      int acc = 0, bsel = 255;
      for (int bkt = 0; bkt < 256; ++bkt) {
        if (acc + hist[bkt] >= remaining) { bsel = bkt; break; }
        acc += hist[bkt];
      }
      sh[0] = bsel;
      sh[1] = remaining - acc;
    }
    __syncthreads();
    prefix |= (uint32_t)sh[0] << (8 * pass);
    mask |= 255u << (8 * pass);
    remaining = sh[1];
    __syncthreads();
  }
  thr = prefix;
  take_eq = remaining;
}

__global__ void __launch_bounds__(kSubTPB) anchor_subsample_kernel(float* __restrict__ label, float* __restrict__ bbox_target,
                                                                    float* __restrict__ bbox_weight, int n, int A,
                                                                    int HW, int num_fg, int batch_size, uint32_t seed) {
  __shared__ int hist[256];
  __shared__ int sh[2];
  __shared__ int cnt[2];
  __shared__ int eq_taken;
  const int b = blockIdx.x;
  float* lab = label + (long)b * n;
  for (int cls = 1; cls >= 0; --cls) {
    if (threadIdx.x < 2) cnt[threadIdx.x] = 0;
    if (threadIdx.x == 0) eq_taken = 0;
    __syncthreads();
    int local = 0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) local += (lab[i] == (float)cls);
    atomicAdd(&cnt[0], local);
    if (cls == 0) {
      int l1 = 0;
      for (int i = threadIdx.x; i < n; i += blockDim.x) l1 += (lab[i] == 1.0f);
      atomicAdd(&cnt[1], l1);
    }
    __syncthreads();
    const int have = cnt[0];
    const int keep = cls == 1 ? num_fg : batch_size - cnt[1];
    __syncthreads();
    if (have <= keep) continue;            // block-uniform
    const int drop = have - keep;
    uint32_t thr;
    int take_eq;
    radix_select(lab, n, (float)cls, seed + (uint32_t)cls * 0x51ED27u, (uint32_t)b, drop, thr, take_eq, hist, sh);
    // keys below the threshold go; of the keys EQUAL to it (a 32-bit collision exactly at the threshold: probability
    // ~n / 2^32) the first take_eq to arrive go
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const float l = lab[i];
      bool kill = false;
      if (l == (float)cls) {
        const uint32_t key = mix32(seed + (uint32_t)cls * 0x51ED27u, (uint32_t)b, (uint32_t)i);
        if (key < thr) kill = true;
        else if (key == thr) kill = atomicAdd(&eq_taken, 1) < take_eq;
      }
      if (kill) {
        lab[i] = -1.0f;
        if (cls == 1) {                    // a disabled positive loses its regression weight and target
          const int a = i / HW, hw = i - a * HW;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const long o = ((long)b * 4 * A + 4 * a + j) * HW + hw;
            bbox_weight[o] = 0.f;
            bbox_target[o] = 0.f;
          }
        }
      }
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------------------------
// AutoFocus FocusPixel labels: `gen_mask` of anchor_worker.worker (lib/data_utils/data_workers.py:165-192) on device.  A
// box of side s = sqrt((x2-x1)*(y2-y1)) (no +1) is flagged 1 when DC_LOW < s < SMALL, -1 when SMALL <= s < DC_HIGH or
// s <= DC_LOW, and writes nothing when s >= DC_HIGH; it covers the cells [int(x1/stride), min(ceil(x2/stride)+1, W)) x
// (the same in y) -- one cell past the ceiling, as the reference's loop runs.  Boxes are scanned in the chip's GT order and
// the last writer wins, so a cell keeps the flag of the last box that covers it with a non-zero flag; uncovered cells are
// 0.  The coordinates are integers (rounded, clipped), so the product is exact in double and the correctly rounded sqrt
// decides every threshold the way numpy does.
// One CTA per chip: the per-box work (side, flag, cell rectangle) is done once per box into shared memory, 256 boxes at a
// time; then each thread scans that chunk in order for the cells it owns, whose labels live in shared memory.
constexpr int kFocusBoxes = 256;

__global__ void __launch_bounds__(kFocusBoxes) focus_label_kernel(const float* __restrict__ boxes,
                                                                  const int* __restrict__ offsets, int H, int W, int stride,
                                                                  double dc_low, double small, double dc_high,
                                                                  float* __restrict__ out) {
  extern __shared__ float lab[];                    // [H*W]
  __shared__ int4 rect[kFocusBoxes];                // cell rectangle [x1, x2) x [y1, y2); empty when the box writes nothing
  __shared__ float flag[kFocusBoxes];
  const int b = blockIdx.x, HW = H * W;
  for (int c = threadIdx.x; c < HW; c += blockDim.x) lab[c] = 0.f;
  const int k0 = offsets[b], k1 = offsets[b + 1];
  for (int base = k0; base < k1; base += kFocusBoxes) {
    __syncthreads();
    const int k = base + (int)threadIdx.x;
    if (k < k1) {
      const double x1 = boxes[4 * (long)k], y1 = boxes[4 * (long)k + 1];
      const double x2 = boxes[4 * (long)k + 2], y2 = boxes[4 * (long)k + 3];
      const double area = sqrt((x2 - x1) * (y2 - y1));
      float f = 0.f;
      if (area > dc_low && area < small) f = 1.f;
      else if ((area >= small && area < dc_high) || area <= dc_low) f = -1.f;
      int4 r = make_int4((int)(x1 / stride), min((int)ceil(x2 / stride) + 1, W), (int)(y1 / stride),
                         min((int)ceil(y2 / stride) + 1, H));
      if (f == 0.f) r.y = r.x;                         // writes nothing
      rect[threadIdx.x] = r;
      flag[threadIdx.x] = f;
    }
    __syncthreads();
    const int n = min(kFocusBoxes, k1 - base);
    for (int c = threadIdx.x; c < HW; c += blockDim.x) {
      const int y = c / W, x = c - (c / W) * W;
      float v = lab[c];
      for (int j = 0; j < n; ++j) {
        const int4 r = rect[j];
        if (x >= r.x && x < r.y && y >= r.z && y < r.w) v = flag[j];
      }
      lab[c] = v;
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < HW; c += blockDim.x) out[(long)b * HW + c] = lab[c];
}

}  // namespace

extern "C" {

// src: device copy of the host staging buffer (uint8 BGR HWC rectangles back to back); table: device int64[B][8] =
// {src_off, src_h, src_w, dst_h, dst_w, flipped, bits of the float64 scale, 0}; means_bgr: device float[3]
// (cfg.network.PIXEL_MEANS order); data: [B,3,S,S] fp32, fully written.
int sniper_chip_input_hw(const void* src, const void* table, const float* means_bgr, float* data, int B, int SH, int SW,
                         void* stream);

int sniper_chip_input(const void* src, const void* table, const float* means_bgr, float* data, int B, int S,
                      void* stream) {
  return sniper_chip_input_hw(src, table, means_bgr, data, B, S, S, stream);
}

// The same with a rectangular canvas [B,3,SH,SW]: the test iterator pads a batch of chips to the largest resized chip
// (MNIteratorTestAutoFocus._get_batch, im_worker.worker_autofocus lib/data_utils/data_workers.py:51-78).
int sniper_chip_input_hw(const void* src, const void* table, const float* means_bgr, float* data, int B, int SH, int SW,
                         void* stream) {
  SN_CHECK(B > 0 && SH > 0 && SW > 0, "chip_input: empty batch");
  const long total = (long)B * SH * SW;
  long g = (total + 255) / 256;
  const long cap = (long)sn::kNumSMs * 16;
  chip_input_kernel<<<(int)(g > cap ? cap : g), 256, 0, (cudaStream_t)stream>>>(
      static_cast<const uint8_t*>(src), static_cast<const ChipDesc*>(table), means_bgr, data, B, SH, SW);
  SN_LAUNCH_CHECK();
  return 0;
}

// label [B, A*H*W] in (a,h,w) order, bbox_target / bbox_weight [B,4A,H,W] (as sniper_anchor_target writes them), in
// place.  Keeps <= num_fg positives and <= batch_size - #positives negatives per chip, chosen by hash(seed, chip, anchor).
int sniper_anchor_subsample(float* label, float* bbox_target, float* bbox_weight, int B, int A, int H, int W, int num_fg,
                            int batch_size, unsigned seed, void* stream) {
  SN_CHECK(B > 0 && num_fg >= 0 && batch_size >= num_fg, "anchor_subsample: bad sizes");
  anchor_subsample_kernel<<<B, kSubTPB, 0, (cudaStream_t)stream>>>(label, bbox_target, bbox_weight, A * H * W, A, H * W,
                                                                  num_fg, batch_size, seed);
  SN_LAUNCH_CHECK();
  return 0;
}

// boxes: [N,4] fp32 (x1, y1, x2, y2) of every chip's GT after shift / scale / round / clip, chip-major, unfiltered;
// offsets: int32 [B+1], chip b owns rows [offsets[b], offsets[b+1]); out: scale_label [B, H*W] in {-1, 0, 1}, fully written.
int sniper_focus_label(const float* boxes, const int* offsets, int B, int H, int W, int stride, double dc_low,
                       double small_thresh, double dc_high, float* out, void* stream) {
  SN_CHECK(B > 0 && H > 0 && W > 0 && stride > 0, "focus_label: bad sizes");
  SN_CHECK((long)H * W * 4 <= 48 * 1024, "focus_label: label map of %d x %d cells does not fit in shared memory", H, W);
  focus_label_kernel<<<B, kFocusBoxes, (size_t)H * W * sizeof(float), (cudaStream_t)stream>>>(
      boxes, offsets, H, W, stride, dc_low, small_thresh, dc_high, out);
  SN_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
