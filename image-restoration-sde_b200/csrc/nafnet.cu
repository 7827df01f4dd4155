// Kernels specific to ConditionalNAFNet / NAFBlock (Refusion's score network):
// codes/config/deraining/models/modules/DenoisingNAFNet_arch.py:15-188.
// All are HBM-bound NHWC kernels (fp32 math; float or bf16 storage).
#include <math.h>

#include "nafnet.cuh"

namespace irsde {

// =============================================================================================
// depthwise 3x3 (pad 1, bias) over 2c channels fused with SimpleGate and the SCA pooling partials
//   gate[b,p,ch] = dw(x)[ch] * dw(x)[ch + c]                   (DenoisingNAFNet_arch.py:65-66)
//   partial[b][chunk][ch] = sum over the chunk's pixels of gate (AdaptiveAvgPool2d numerator, :29-30)
// block = 64 channels x 4 pixel lanes, chunk = 64 pixels of one image - 16 for images of <= 1024 pixels, where 64-pixel
// chunks leave a handful of blocks each walking 16 pixels x 9 taps serially (30 us for 512 KB of data at c=512,
// 16x16) - (deterministic reduction order, fixed by the image shape)
// =============================================================================================
static inline int dw_pix(int N) { return N <= 1024 ? 16 : 64; }

template <typename T>
__global__ void __launch_bounds__(256) dwgate_kernel(const T* __restrict__ x, int x_pitch, const float* __restrict__ w,
                                                     const float* __restrict__ bias, T* __restrict__ gate, int g_pitch,
                                                     float* __restrict__ partial, int H, int W, int c, int nchunks,
                                                     int DW_PIX) {
  PDL_ENTRY();
  __shared__ float red[4][64];
  const int cl = threadIdx.x & 63, pl = threadIdx.x >> 6;
  const int ch = blockIdx.x * 64 + cl;
  const int chunk = blockIdx.y, b = blockIdx.z;
  const int N = H * W;
  float acc_sum = 0.f;
  if (ch < c) {
    float w1[9], w2[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) { w1[k] = w[ch * 9 + k]; w2[k] = w[(ch + c) * 9 + k]; }
    const float b1 = bias[ch], b2 = bias[ch + c];
    for (int i = pl; i < DW_PIX; i += 4) {
      const int p = chunk * DW_PIX + i;
      if (p >= N) break;
      const int h = p / W, wq = p - h * W;
      float a1 = b1, a2 = b2;
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        const int hh = h + r - 1;
        if (hh < 0 || hh >= H) continue;
#pragma unroll
        for (int s = 0; s < 3; ++s) {
          const int ww = wq + s - 1;
          if (ww < 0 || ww >= W) continue;
          const T* row = x + (((long long)b * H + hh) * W + ww) * x_pitch;
          a1 = fmaf(w1[r * 3 + s], to_f(row[ch]), a1);
          a2 = fmaf(w2[r * 3 + s], to_f(row[ch + c]), a2);
        }
      }
      const float gv = a1 * a2;
      const T gq = from_f<T>(gv);
      gate[((long long)b * N + p) * g_pitch + ch] = gq;
      acc_sum += to_f(gq);  // pool the stored (rounded) value: what conv3 will actually read
    }
  }
  red[pl][cl] = acc_sum;
  __syncthreads();
  if (pl == 0 && ch < c)
    partial[((long long)b * nchunks + chunk) * c + ch] = (red[0][cl] + red[1][cl]) + (red[2][cl] + red[3][cl]);
}

// mean over pixels -> 1x1 conv (c x c mat-vec + bias): sca[b][o]            (DenoisingNAFNet_arch.py:29-33)
// grid (ceil(c/8), B): every block re-derives the c means (c*nchunks floats, L2 resident) and its 8 warps each own
// one output row, so the c x c weight matrix is streamed by c/8 SMs instead of one.
template <typename T>
__global__ void __launch_bounds__(256) sca_kernel(const float* __restrict__ partial, const float* __restrict__ w,
                                                  const float* __restrict__ bias, float* __restrict__ sca, int c, int nchunks,
                                                  int N, T* __restrict__ g, int g_pitch) {
  PDL_ENTRY();
  extern __shared__ float mean_s[];
  __shared__ float row_s[8];
  const int b = blockIdx.y;
  for (int ch = threadIdx.x; ch < c; ch += blockDim.x) {
    float s = 0.f;
    for (int k = 0; k < nchunks; ++k) s += partial[((long long)b * nchunks + k) * c + ch];
    mean_s[ch] = s / (float)N;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int o = blockIdx.x * 8 + warp;
  if (o < c) {
    float s = 0.f;
    for (int k = lane; k < c; k += 32) s += w[(long long)o * c + k] * mean_s[k];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
    if (lane == 0) { s += bias[o]; sca[(long long)b * c + o] = s; row_s[warp] = s; }
  }
  if (g == nullptr) return;
  // small images: scale this block's 8 channels of the gate tensor in place (the "x * self.sca(x)" of :67)
  __syncthreads();
  const int nch = min(8, c - blockIdx.x * 8);
  for (int p = threadIdx.x; p < N; p += blockDim.x) {
    T* e = g + ((long long)b * N + p) * g_pitch + blockIdx.x * 8;
    for (int j = 0; j < nch; ++j) e[j] = from_f<T>(to_f(e[j]) * row_s[j]);
  }
}

// x[b,p,ch] *= sca[b][ch]   (in place; the "x * self.sca(x)" of :67)
template <typename T>
__global__ void scale_channels_kernel(T* __restrict__ x, int pitch, const float* __restrict__ sca, long long npix, int N, int c) {
  PDL_ENTRY();
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long total = npix * c;
  if (idx >= total) return;
  const int ch = idx % c;
  const long long p = idx / c;
  const int b = (int)(p / N);
  T* e = x + p * pitch + ch;
  *e = from_f<T>(to_f(*e) * sca[(long long)b * c + ch]);
}

// SimpleGate on a [.., 2c] tensor -> [.., c]                                   (:9-12)
// cam != null: the lens network's per-image FFN modulation follows the gate
//   g = (a*b) * (cam_scale[img][ch] + 1) + cam_shift[img][ch]      (latent-bokeh/.../DenoisingNAFNet_arch.py:82-83)
// in fp32 with the reference's separate roundings (mul, then add), stored once as T.
template <typename T>
__global__ void simple_gate_kernel(const T* __restrict__ x, int x_pitch, T* __restrict__ out, int o_pitch, long long npix, int c,
                                   CamMod cm) {
  PDL_ENTRY();
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long total = npix * c;
  if (idx >= total) return;
  const int ch = idx % c;
  const long long p = idx / c;
  float v = to_f(x[p * x_pitch + ch]) * to_f(x[p * x_pitch + ch + c]);
  if (cm.cam) {
    const float* r = cm.cam + (long long)(p / cm.pix_per_img) * cm.img_stride * cm.S + cm.off;
    v = __fadd_rn(__fmul_rn(v, __fadd_rn(r[ch], 1.f)), r[c + ch]);
  }
  out[p * o_pitch + ch] = from_f<T>(v);
}

// 16-byte vector loads/stores of the same modulated gate: grid (pixel groups, 1, image), block (channel vectors, pixels);
// needs c % VEC == 0 (VEC = 16 bytes of T) and 16-byte aligned views.  No per-element index arithmetic.
template <typename T>
struct alignas(16) Vec16 {
  static constexpr int N = 16 / sizeof(T);
  T v[N];
};
template <typename T>
__global__ void __launch_bounds__(256) simple_gate_cam_vec_kernel(const T* __restrict__ x, int x_pitch, T* __restrict__ out,
                                                                  int o_pitch, int N, int c, CamMod cm) {
  PDL_ENTRY();
  constexpr int VEC = Vec16<T>::N;
  const int pix = blockIdx.x * blockDim.y + threadIdx.y;
  if (pix >= N) return;
  const long long p = (long long)blockIdx.z * N + pix;
  const float* r = cm.cam + (long long)blockIdx.z * cm.img_stride * cm.S + cm.off;
  const T* xa = x + p * x_pitch;
  T* o = out + p * o_pitch;
  for (int j = threadIdx.x * VEC; j < c; j += blockDim.x * VEC) {
    const Vec16<T> a = *reinterpret_cast<const Vec16<T>*>(xa + j);
    const Vec16<T> b = *reinterpret_cast<const Vec16<T>*>(xa + c + j);
    Vec16<T> g;
#pragma unroll
    for (int e = 0; e < VEC; ++e) {
      const float v = to_f(a.v[e]) * to_f(b.v[e]);
      g.v[e] = from_f<T>(__fadd_rn(__fmul_rn(v, __fadd_rn(r[j + e], 1.f)), r[c + j + e]));
    }
    *reinterpret_cast<Vec16<T>*>(o + j) = g;
  }
}

// PixelShuffle(2) of a [B,h,w,4q] tensor + skip add -> [B,2h,2w,q]              (:132-137,172-174)
//   out[b, 2h+i, 2w+j, cq] = in[b, h, w, cq*4 + i*2 + j] + skip[b, 2h+i, 2w+j, cq]
template <typename T>
__global__ void pixel_shuffle_add_kernel(const T* __restrict__ in, int in_pitch, const T* __restrict__ skip, int s_pitch,
                                         T* __restrict__ out, int o_pitch, int B, int h, int w, int q) {
  PDL_ENTRY();
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long total = (long long)B * h * w * q;
  if (idx >= total) return;
  const int cq = idx % q;
  long long p = idx / q;
  const int ww = p % w;
  const int hh = (p / w) % h;
  const int b = p / ((long long)w * h);
  const T* src = in + p * in_pitch + cq * 4;
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const long long op = ((long long)b * 2 * h + 2 * hh + i) * (2 * w) + 2 * ww + j;
      out[op * o_pitch + cq] = from_f<T>(to_f(src[i * 2 + j]) + to_f(skip[op * s_pitch + cq]));
    }
}

template <typename T>
__global__ void add_kernel(const T* __restrict__ a, int a_pitch, const T* __restrict__ b, int b_pitch, T* __restrict__ out,
                           int o_pitch, long long npix, int c) {
  PDL_ENTRY();
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long total = npix * c;
  if (idx >= total) return;
  const int ch = idx % c;
  const long long p = idx / c;
  out[p * o_pitch + ch] = from_f<T>(to_f(a[p * a_pitch + ch]) + to_f(b[p * b_pitch + ch]));
}

// ---- launchers -------------------------------------------------------------------------------------
int dwgate_chunks(int H, int W) { return (H * W + dw_pix(H * W) - 1) / dw_pix(H * W); }

template <typename T>
void launch_dwgate(const T* x, int x_pitch, const float* w, const float* bias, T* gate, int g_pitch, float* partial, int B,
                   int H, int W, int c, cudaStream_t st) {
  const int nchunks = dwgate_chunks(H, W);
  pdl_launch(dwgate_kernel<T>, dim3((c + 63) / 64, nchunks, B), 256, 0, st, x, x_pitch, w, bias, gate, g_pitch, partial, H, W, c, nchunks,
             dw_pix(H * W));
}
template void launch_dwgate<float>(const float*, int, const float*, const float*, float*, int, float*, int, int, int, int, cudaStream_t);
template void launch_dwgate<bf16>(const bf16*, int, const float*, const float*, bf16*, int, float*, int, int, int, int, cudaStream_t);

template <typename T>
void launch_scale_channels(T* x, int pitch, const float* sca, int B, int N, int c, cudaStream_t st);

// sca[b][:] and g *= sca in place.  N <= 1024 pixels: one launch does both; larger images use a second, fully
// parallel pass (8 channels per block would not cover the pixels fast enough).
template <typename T>
void launch_sca_scale(const float* partial, const float* w, const float* bias, float* sca, T* g, int g_pitch, int B, int c,
                      int nchunks, int N, int* launches, cudaStream_t st) {
  const bool fused = N <= 1024;
  pdl_launch(sca_kernel<T>, dim3((c + 7) / 8, B), 256, c * sizeof(float), st, partial, w, bias, sca, c, nchunks, N, fused ? g : (T*)nullptr, g_pitch);
  *launches = 1;
  if (!fused) { launch_scale_channels<T>(g, g_pitch, sca, B, N, c, st); *launches = 2; }
}
template void launch_sca_scale<float>(const float*, const float*, const float*, float*, float*, int, int, int, int, int, int*, cudaStream_t);
template void launch_sca_scale<bf16>(const float*, const float*, const float*, float*, bf16*, int, int, int, int, int, int*, cudaStream_t);

template <typename T>
void launch_scale_channels(T* x, int pitch, const float* sca, int B, int N, int c, cudaStream_t st) {
  long long total = (long long)B * N * c;
  pdl_launch(scale_channels_kernel<T>, (unsigned)((total + 255) / 256), 256, 0, st, x, pitch, sca, (long long)B * N, N, c);
}
template void launch_scale_channels<float>(float*, int, const float*, int, int, int, cudaStream_t);
template void launch_scale_channels<bf16>(bf16*, int, const float*, int, int, int, cudaStream_t);

template <typename T>
void launch_simple_gate(const T* x, int x_pitch, T* out, int o_pitch, long long npix, int c, cudaStream_t st) {
  CamMod none;
  memset(&none, 0, sizeof none);
  long long total = npix * c;
  pdl_launch(simple_gate_kernel<T>, (unsigned)((total + 255) / 256), 256, 0, st, x, x_pitch, out, o_pitch, npix, c, none);
}
template void launch_simple_gate<float>(const float*, int, float*, int, long long, int, cudaStream_t);
template void launch_simple_gate<bf16>(const bf16*, int, bf16*, int, long long, int, cudaStream_t);

template <typename T>
void launch_simple_gate(const T* x, int x_pitch, T* out, int o_pitch, long long npix, int c, cudaStream_t st, const CamMod& cam,
                        int B) {
  constexpr int VEC = Vec16<T>::N;
  const bool aligned = ((uintptr_t)x % 16 == 0) && ((uintptr_t)out % 16 == 0) && x_pitch % VEC == 0 && o_pitch % VEC == 0;
  if (cam.cam && c % VEC == 0 && aligned) {
    const int cv = c / VEC, bx = cv < 256 ? cv : 256, by = 256 / bx;
    const int N = (int)(npix / B);
    pdl_launch(simple_gate_cam_vec_kernel<T>, dim3((N + by - 1) / by, 1, B), dim3(bx, by), 0, st, x, x_pitch, out, o_pitch, N, c,
               cam);
    return;
  }
  long long total = npix * c;
  pdl_launch(simple_gate_kernel<T>, (unsigned)((total + 255) / 256), 256, 0, st, x, x_pitch, out, o_pitch, npix, c, cam);
}
template void launch_simple_gate<float>(const float*, int, float*, int, long long, int, cudaStream_t, const CamMod&, int);
template void launch_simple_gate<bf16>(const bf16*, int, bf16*, int, long long, int, cudaStream_t, const CamMod&, int);

template <typename T>
void launch_pixel_shuffle_add(const T* in, int in_pitch, const T* skip, int s_pitch, T* out, int o_pitch, int B, int h, int w, int q,
                              cudaStream_t st) {
  long long total = (long long)B * h * w * q;
  pdl_launch(pixel_shuffle_add_kernel<T>, (unsigned)((total + 255) / 256), 256, 0, st, in, in_pitch, skip, s_pitch, out, o_pitch, B, h, w, q);
}
template void launch_pixel_shuffle_add<float>(const float*, int, const float*, int, float*, int, int, int, int, int, cudaStream_t);
template void launch_pixel_shuffle_add<bf16>(const bf16*, int, const bf16*, int, bf16*, int, int, int, int, int, cudaStream_t);

template <typename T>
void launch_add(const T* a, int a_pitch, const T* b, int b_pitch, T* out, int o_pitch, long long npix, int c, cudaStream_t st) {
  long long total = npix * c;
  pdl_launch(add_kernel<T>, (unsigned)((total + 255) / 256), 256, 0, st, a, a_pitch, b, b_pitch, out, o_pitch, npix, c);
}
template void launch_add<float>(const float*, int, const float*, int, float*, int, long long, int, cudaStream_t);
template void launch_add<bf16>(const bf16*, int, const bf16*, int, bf16*, int, long long, int, cudaStream_t);

// =============================================================================================
// NAFNet timestep embedding: SinusoidalPosEmb(w) -> Linear(w, 8w) -> SimpleGate -> Linear(4w, 4w) = t;
// every NAFBlock: SimpleGate(t) -> Linear(2w, 4c) -> (shift_att, scale_att, shift_ffn, scale_ffn)
// (DenoisingNAFNet_arch.py:18-20,51-54,96-101).  Stores SimpleGate(t) [2w] per row for time_table_kernel.
// A row holds k scalars: the embedding is [sin, cos] of each, concatenated in order (k*w inputs to the first Linear).
// k = 3 is the lens network's camera embedding cat(SinusoidalPosEmb(w)(src_lens, tgt_lens, disparity)) -> cam_mlp
// (latent-bokeh/models/modules/DenoisingNAFNet_arch.py:109-114,171-173); k = 1 is the time path.
// =============================================================================================
__global__ void naf_time_mlp_kernel(const float* __restrict__ times, int k, int width, const float* __restrict__ w1,
                                    const float* __restrict__ b1, const float* __restrict__ w2, const float* __restrict__ b2,
                                    float* __restrict__ tgate) {
  extern __shared__ float sm[];
  const int td = width * 4, half = width / 2, kw = k * width;
  float* emb = sm;            // [k*w]
  float* h1 = sm + kw;        // [8w]
  float* tt = h1 + 2 * td;    // [4w]
  const int row = blockIdx.x;
  const float e = logf(10000.0f) / (float)(half - 1);
  for (int j = 0; j < k; ++j) {
    const float t = times[row * k + j];
    for (int i = threadIdx.x; i < half; i += blockDim.x) {
      const float a = t * expf((float)i * -e);
      emb[j * width + i] = sinf(a);
      emb[j * width + half + i] = cosf(a);
    }
  }
  __syncthreads();
  for (int o = threadIdx.x; o < 2 * td; o += blockDim.x) {
    float s = 0.f;
    for (int q = 0; q < kw; ++q) s += w1[o * kw + q] * emb[q];
    h1[o] = s + b1[o];
  }
  __syncthreads();
  for (int o = threadIdx.x; o < td; o += blockDim.x) {
    float s = 0.f;
    for (int q = 0; q < td; ++q) s += w2[o * td + q] * (h1[q] * h1[q + td]);
    tt[o] = s + b2[o];
  }
  __syncthreads();
  for (int o = threadIdx.x; o < td / 2; o += blockDim.x) tgate[(long long)row * (td / 2) + o] = tt[o] * tt[o + td / 2];
}

void launch_naf_time_gate_k(const float* times, int rows, int k, int width, const float* w1, const float* b1, const float* w2,
                            const float* b2, float* tgate, cudaStream_t st) {
  const int td = width * 4;
  naf_time_mlp_kernel<<<rows, 256, (k * width + 2 * td + td) * sizeof(float), st>>>(times, k, width, w1, b1, w2, b2, tgate);
}
void launch_naf_time_gate(const float* times, int rows, int width, const float* w1, const float* b1, const float* w2,
                          const float* b2, float* tgate, cudaStream_t st) {
  launch_naf_time_gate_k(times, rows, 1, width, w1, b1, w2, b2, tgate, st);
}

}  // namespace irsde
