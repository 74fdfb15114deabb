// Sampler tail: the SD-VAE DECODE path the reference runs on every batch of sampled latents (sample.py:275
// `images = vae.decode(z)`; autoencoder.py:306-453: post_quant_conv, conv_in, ResnetBlocks with GroupNorm(32)+swish,
// one single-head AttnBlock, nearest-2x Upsample + conv, norm_out + conv_out), and the ENCODE path in front of training
// (extract_latent.py:77 `encode_moments`; autoencoder.py:212-303,431-434: conv_in on the 3-channel image, ResnetBlocks,
// stride-2 Downsample convolutions with (0,1,0,1) padding, the AttnBlock, norm_out + conv_out, quant_conv).
//
// Layout: activations are pixel-major ("NHWC") fp32 row matrices [B*H*W, C], so every convolution is a GEMM on the
// tcgen05 kernel of gemm_tcgen05.cu: a 3x3 convolution reads an im2col operand A[(b,y,x), (ky,kx,c)] (bf16) that ONE
// kernel builds with the GroupNorm affine, the swish and the nearest-2x upsample of the source fused in (the normalised
// tensor is never materialised), weights are pre-flattened to [C_out, (ky,kx,c)]; bias and the residual add ride in the
// GEMM epilogue.  The kernels here are the HBM-bound glue: statistics, im2col, row softmax, layout conversion.
#include <math.h>

#include "common.cuh"
#include "../../include/maskdit_b200.h"

namespace mdt {

static inline cudaStream_t VS(void* s) { return static_cast<cudaStream_t>(s); }
static inline int vae_status() { return cudaGetLastError() == cudaSuccess ? MDT_OK : MDT_ERR_CUDA; }

// z [B,Cz,h,w] f32 (NCHW, the sampler's latent) -> out [B*h*w, Cz] f32 = post_quant_conv(z / scale_factor)
// (FrozenAutoencoderKL.decode, autoencoder.py:449-451; a 1x1 convolution over <= 8 channels)
__global__ void vae_post_quant_kernel(const float* __restrict__ z, const float* __restrict__ W,
                                      const float* __restrict__ bias, float inv_sf, float* __restrict__ out, int B,
                                      int C, int P) {
  const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;  // (b, pixel)
  if (i >= static_cast<long long>(B) * P) return;
  const int b = static_cast<int>(i / P), p = static_cast<int>(i % P);
  float v[8];
  for (int c = 0; c < C; ++c) v[c] = inv_sf * z[(static_cast<long long>(b) * C + c) * P + p];
  for (int o = 0; o < C; ++o) {
    float acc = bias[o];
    for (int c = 0; c < C; ++c) acc = fmaf(W[o * C + c], v[c], acc);
    out[i * C + o] = acc;
  }
}

// GroupNorm(32) statistics of x [B, P, C] f32, DETERMINISTIC (no atomics: with bf16 GEMM operands downstream, 1e-7
// order noise in a mean flips bf16 roundings and shows up as 4e-3 run-to-run differences in the decoded image, measured):
//   pass 1: block (b, chunk of kGnPix pixels) -> partial[b][chunk][g] = (sum, sum of squares) fp32, fixed-order tree
//   pass 2: sums[b][g] = fixed-order fp64 sum of the partials.
// Thread = 4 channels of one pixel lane; block = C/4 x (256 / (C/4)) threads: always 8 threads per group.
constexpr int kGnPix = 256;
__global__ void __launch_bounds__(256)
vae_gn_partial_kernel(const float* __restrict__ x, float* __restrict__ partial, int P, int C) {
  __shared__ float s_part[256][2];
  const int tx = threadIdx.x, ty = threadIdx.y, b = blockIdx.y;
  const int p0 = blockIdx.x * kGnPix;
  float s = 0.f, ss = 0.f;
  for (int p = p0 + ty; p < min(P, p0 + kGnPix); p += blockDim.y) {
    const float4 v = *reinterpret_cast<const float4*>(x + (static_cast<long long>(b) * P + p) * C + 4 * tx);
    s += (v.x + v.y) + (v.z + v.w);
    ss += (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
  }
  // slot = (group, member): the 8 threads of a group occupy 8 consecutive slots
  const int tpg = (C / 32) / 4;                       // threads per group along x (1, 2 or 4)
  const int g = tx / tpg, member = ty * tpg + (tx - g * tpg);
  s_part[g * 8 + member][0] = s;
  s_part[g * 8 + member][1] = ss;
  __syncthreads();
  const int tid = ty * blockDim.x + tx;
  if (tid < 64) {
    const int gg = tid >> 1, w = tid & 1;
    float acc = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) acc += s_part[gg * 8 + k][w];
    partial[((static_cast<long long>(b) * gridDim.x + blockIdx.x) * 32 + gg) * 2 + w] = acc;
  }
}
__global__ void vae_gn_finish_kernel(const float* __restrict__ partial, double* __restrict__ sums, int nchunk) {
  const int b = blockIdx.x, t = threadIdx.x;  // 64 threads: (group, which)
  double acc = 0.0;
  for (int k = 0; k < nchunk; ++k) acc += static_cast<double>(partial[(static_cast<long long>(b) * nchunk + k) * 64 + t]);
  sums[static_cast<long long>(b) * 64 + t] = acc;
}

// im2col with the producer fused in:  A[(b, y, x), (ky, kx, c)] = f(src[b, (y+ky-pad)/up, (x+kx-pad)/up, c])  (0 outside)
//   f = identity | GroupNorm affine (sums / gamma / beta given) | GroupNorm affine then swish (silu != 0)
//   ks = 3 (pad 1) or 1 (pad 0);  up = 1 or 2 (nearest upsample of the source, Upsample.forward autoencoder.py:49-53)
//   src [B, H/up, W/up, C] f32  ->  A [B*H*W, Kp] bf16,  Kp >= ks*ks*C (extra columns zero)
// Downsample mode (down != 0; ks = 3, up = 1, f = identity): the output grid is H/2 x W/2 and
//   A[(b, y, x), (ky, kx, c)] = src[b, 2y+ky, 2x+kx, c], zero where 2y+ky >= H or 2x+kx >= W
//   = F.pad(x, (0,1,0,1)) then the 3x3 stride-2 convolution of Downsample.forward (autoencoder.py:56-75).
// Thread = 4 channels; blockDim = (C/4, 256/(C/4)) (C = 4: 1 x 256); each y-lane walks output pixels.
__global__ void __launch_bounds__(256)
vae_im2col_kernel(const float* __restrict__ src, const double* __restrict__ sums, const float* __restrict__ gamma,
                  const float* __restrict__ beta, int silu_on, int ks, int up, int down, __nv_bfloat16* __restrict__ A,
                  int B, int H, int W, int C, int Kp, float eps) {
  const int tx = threadIdx.x, c = 4 * tx;
  const int Hs = H / up, Ws = W / up;                  // source dims (H, W: the source dims in downsample mode)
  const int Ho = down ? H / 2 : H, Wo = down ? W / 2 : W;
  const int stride = down ? 2 : 1;
  const long long npix = static_cast<long long>(B) * Ho * Wo;
  const int pad = down ? 0 : ks / 2, taps = ks * ks;
  float4 ga = make_float4(1.f, 1.f, 1.f, 1.f), be = make_float4(0.f, 0.f, 0.f, 0.f);
  if (sums) {
    ga = *reinterpret_cast<const float4*>(gamma + c);
    be = *reinterpret_cast<const float4*>(beta + c);
  }
  const int cg = C / 32 > 0 ? C / 32 : 1;
  const double cnt = static_cast<double>(Hs) * Ws * cg;
  for (long long pix = blockIdx.x * static_cast<long long>(blockDim.y) + threadIdx.y; pix < npix;
       pix += static_cast<long long>(gridDim.x) * blockDim.y) {
    const int b = static_cast<int>(pix / (static_cast<long long>(Ho) * Wo));
    const int yx = static_cast<int>(pix - static_cast<long long>(b) * Ho * Wo);
    const int y = yx / Wo, x = yx - y * Wo;
    float mean = 0.f, rstd = 1.f;
    if (sums) {
      const int g = c / cg;
      const double s = sums[(static_cast<long long>(b) * 32 + g) * 2], q = sums[(static_cast<long long>(b) * 32 + g) * 2 + 1];
      const double m = s / cnt;
      mean = static_cast<float>(m);
      rstd = rsqrtf(static_cast<float>(q / cnt - m * m) + eps);
    }
    __nv_bfloat16* arow = A + pix * Kp;
    for (int t = 0; t < taps; ++t) {
      const int ky = t / ks, kx = t - ky * ks;
      const int sy = stride * y + ky - pad, sx = stride * x + kx - pad;
      uint2 o = make_uint2(0u, 0u);
      if (sy >= 0 && sy < H && sx >= 0 && sx < W) {
        const float4 v = *reinterpret_cast<const float4*>(
            src + ((static_cast<long long>(b) * Hs + sy / up) * Ws + sx / up) * C + c);
        float4 r = v;
        if (sums) {
          r.x = fmaf((v.x - mean) * rstd, ga.x, be.x), r.y = fmaf((v.y - mean) * rstd, ga.y, be.y);
          r.z = fmaf((v.z - mean) * rstd, ga.z, be.z), r.w = fmaf((v.w - mean) * rstd, ga.w, be.w);
        }
        if (silu_on) r = make_float4(silu(r.x), silu(r.y), silu(r.z), silu(r.w));
        o = make_uint2(pack_bf16(r.x, r.y), pack_bf16(r.z, r.w));
      }
      *reinterpret_cast<uint2*>(arow + t * C + c) = o;
    }
    if (tx == 0)
      for (int k = taps * C; k < Kp; ++k) arow[k] = __float2bfloat16_rn(0.f);
  }
}

// x [B,3,H,W] f32 NCHW (the normalised image batch) -> out [B*H*W, 4] f32 pixel-major rows, channel 3 = 0, so that
// conv_in (autoencoder.py:230-234) is the im2col GEMM with C = 4.  flip != 0 reads x mirrored along W (the xflip pass
// of extract_latent.py:85, `img.flip(dims=[-1])`).
__global__ void vae_image_to_rows_kernel(const float* __restrict__ x, float* __restrict__ out, int B, int H, int W,
                                         int flip) {
  const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;  // (b, y, x)
  const long long P = static_cast<long long>(H) * W;
  if (i >= B * P) return;
  const int b = static_cast<int>(i / P), yx = static_cast<int>(i - b * P);
  const int y = yx / W, xx = yx - y * W;
  const long long s = static_cast<long long>(b) * 3 * P + static_cast<long long>(y) * W + (flip ? W - 1 - xx : xx);
  *reinterpret_cast<float4*>(out + 4 * i) = make_float4(x[s], x[s + P], x[s + 2 * P], 0.f);
}

// rows [B*P, ldx] f32 (encoder conv_out, first C columns valid) -> moments [B,C,P] f32 NCHW = quant_conv (1x1, C -> C)
// (FrozenAutoencoderKL.encode_moments, autoencoder.py:431-434); C <= 8
__global__ void vae_quant_out_kernel(const float* __restrict__ rows, int ldx, const float* __restrict__ Wq,
                                     const float* __restrict__ bias, float* __restrict__ moments, int B, int C, int P) {
  const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;  // (b, pixel)
  if (i >= static_cast<long long>(B) * P) return;
  const int b = static_cast<int>(i / P), p = static_cast<int>(i % P);
  float v[8];
  for (int c = 0; c < C; ++c) v[c] = rows[i * ldx + c];
  for (int o = 0; o < C; ++o) {
    float acc = bias[o];
    for (int c = 0; c < C; ++c) acc = fmaf(Wq[o * C + c], v[c], acc);
    moments[(static_cast<long long>(b) * C + o) * P + p] = acc;
  }
}

// P[r, :cols] = softmax(scale * S[r, :cols]) as bf16, P[r, cols:ld] = 0; S and P have row stride ld >= cols; one
// warp per row (AttnBlock, autoencoder.py:186-187)
__global__ void __launch_bounds__(256)
vae_softmax_rows_kernel(const float* __restrict__ S, float scale, __nv_bfloat16* __restrict__ P, int rows, int cols,
                        int ld) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* s = S + static_cast<long long>(row) * ld;
  float mx = -INFINITY;
  for (int j = lane; j < cols; j += 32) mx = fmaxf(mx, s[j]);
  mx = warp_max(mx);
  float sum = 0.f;
  for (int j = lane; j < cols; j += 32) sum += __expf(scale * (s[j] - mx));
  const float inv = 1.f / warp_sum(sum);
  __nv_bfloat16* p = P + static_cast<long long>(row) * ld;
  for (int j = lane; j < cols; j += 32) p[j] = __float2bfloat16_rn(__expf(scale * (s[j] - mx)) * inv);
  for (int j = cols + lane; j < ld; j += 32) p[j] = __float2bfloat16_rn(0.f);
}

// x [B, P, ldx] f32 (first C columns valid) -> out [B, C, P] f32 (the [B,3,H,W] image the reference's decode returns)
__global__ void vae_rows_to_nchw_kernel(const float* __restrict__ x, float* __restrict__ out, int B, int P, int C,
                                        int ldx) {
  const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (i >= static_cast<long long>(B) * C * P) return;
  const int p = static_cast<int>(i % P), c = static_cast<int>((i / P) % C), b = static_cast<int>(i / (static_cast<long long>(P) * C));
  out[i] = x[(static_cast<long long>(b) * P + p) * ldx + c];
}

}  // namespace mdt

using namespace mdt;

extern "C" {

int mdt_vae_post_quant(const float* z, const float* W, const float* bias, float scale_factor, float* out, int B,
                       int C, int P, void* stream) {
  if (!z || !W || !bias || !out || B <= 0 || C <= 0 || C > 8 || P <= 0 || scale_factor == 0.f) return MDT_ERR_ARG;
  const long long n = static_cast<long long>(B) * P;
  vae_post_quant_kernel<<<static_cast<int>((n + 255) / 256), 256, 0, VS(stream)>>>(z, W, bias, 1.f / scale_factor, out,
                                                                                  B, C, P);
  return vae_status();
}

int mdt_vae_gn_stats(const float* x, double* sums, float* scratch, int B, int P, int C, void* stream) {
  if (!x || !sums || !scratch || B <= 0 || P <= 0 || C % 128 || C > 512) return MDT_ERR_ARG;  // 4..16 channels / group
  if (reinterpret_cast<uintptr_t>(x) & 15) return MDT_ERR_ARG;
  const int nchunk = (P + kGnPix - 1) / kGnPix;
  dim3 block(C / 4, 256 / (C / 4)), grid(nchunk, B);
  vae_gn_partial_kernel<<<grid, block, 0, VS(stream)>>>(x, scratch, P, C);
  vae_gn_finish_kernel<<<B, 64, 0, VS(stream)>>>(scratch, sums, nchunk);
  return vae_status();
}

int mdt_vae_im2col(const float* src, const double* sums, const float* gamma, const float* beta, int silu, int ks,
                   int up, void* A_bf16, int B, int H, int W, int C, int Kp, void* stream) {
  if (!src || !A_bf16 || B <= 0 || H <= 0 || W <= 0 || C % 4 || C > 1024 || (ks != 1 && ks != 3) ||
      (up != 1 && up != 2) || H % up || W % up || Kp < ks * ks * C || Kp % 8)
    return MDT_ERR_ARG;
  if (sums && (!gamma || !beta || C % 128)) return MDT_ERR_ARG;
  if ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(A_bf16)) & 15) return MDT_ERR_ARG;
  const int tx = C / 4, ty = tx >= 256 ? 1 : 256 / tx;
  const long long npix = static_cast<long long>(B) * H * W;
  long long blocks = (npix + ty - 1) / ty;
  if (blocks > 148 * 16) blocks = 148 * 16;
  vae_im2col_kernel<<<static_cast<int>(blocks), dim3(tx, ty), 0, VS(stream)>>>(
      src, sums, gamma, beta, silu, ks, up, 0, static_cast<__nv_bfloat16*>(A_bf16), B, H, W, C, Kp, 1e-6f);
  return vae_status();
}

int mdt_vae_im2col_down(const float* src, void* A_bf16, int B, int H, int W, int C, int Kp, void* stream) {
  if (!src || !A_bf16 || B <= 0 || H <= 0 || W <= 0 || H % 2 || W % 2 || C % 4 || C > 1024 || Kp < 9 * C || Kp % 8)
    return MDT_ERR_ARG;
  if ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(A_bf16)) & 15) return MDT_ERR_ARG;
  const int tx = C / 4, ty = tx >= 256 ? 1 : 256 / tx;
  const long long npix = static_cast<long long>(B) * (H / 2) * (W / 2);
  long long blocks = (npix + ty - 1) / ty;
  if (blocks > 148 * 16) blocks = 148 * 16;
  vae_im2col_kernel<<<static_cast<int>(blocks), dim3(tx, ty), 0, VS(stream)>>>(
      src, nullptr, nullptr, nullptr, 0, 3, 1, 1, static_cast<__nv_bfloat16*>(A_bf16), B, H, W, C, Kp, 1e-6f);
  return vae_status();
}

int mdt_vae_image_to_rows(const float* x, float* out, int B, int H, int W, int flip, void* stream) {
  if (!x || !out || B <= 0 || H <= 0 || W <= 0) return MDT_ERR_ARG;
  if (reinterpret_cast<uintptr_t>(out) & 15) return MDT_ERR_ARG;
  const long long n = static_cast<long long>(B) * H * W;
  vae_image_to_rows_kernel<<<static_cast<int>((n + 255) / 256), 256, 0, VS(stream)>>>(x, out, B, H, W, flip);
  return vae_status();
}

int mdt_vae_quant_out(const float* rows, int ldx, const float* W, const float* bias, float* moments, int B, int C,
                      int P, void* stream) {
  if (!rows || !W || !bias || !moments || B <= 0 || C <= 0 || C > 8 || P <= 0 || ldx < C) return MDT_ERR_ARG;
  const long long n = static_cast<long long>(B) * P;
  vae_quant_out_kernel<<<static_cast<int>((n + 255) / 256), 256, 0, VS(stream)>>>(rows, ldx, W, bias, moments, B, C,
                                                                                 P);
  return vae_status();
}

int mdt_vae_softmax_rows(const float* S, float scale, void* P_bf16, int rows, int cols, void* stream) {
  if (!S || !P_bf16 || rows <= 0 || cols <= 0) return MDT_ERR_ARG;
  vae_softmax_rows_kernel<<<(rows + 7) / 8, 256, 0, VS(stream)>>>(S, scale, static_cast<__nv_bfloat16*>(P_bf16), rows,
                                                                  cols, cols);
  return vae_status();
}

int mdt_vae_softmax_rows_ld(const float* S, float scale, void* P_bf16, int rows, int cols, int ld, void* stream) {
  if (!S || !P_bf16 || rows <= 0 || cols <= 0 || ld < cols) return MDT_ERR_ARG;
  vae_softmax_rows_kernel<<<(rows + 7) / 8, 256, 0, VS(stream)>>>(S, scale, static_cast<__nv_bfloat16*>(P_bf16), rows,
                                                                  cols, ld);
  return vae_status();
}

int mdt_vae_rows_to_nchw(const float* x, float* out, int B, int P, int C, int ldx, void* stream) {
  if (!x || !out || B <= 0 || P <= 0 || C <= 0 || ldx < C) return MDT_ERR_ARG;
  const long long n = static_cast<long long>(B) * C * P;
  vae_rows_to_nchw_kernel<<<static_cast<int>((n + 255) / 256), 256, 0, VS(stream)>>>(x, out, B, P, C, ldx);
  return vae_status();
}

}  // extern "C"
