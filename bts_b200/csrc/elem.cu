// Streaming NHWC kernels that replace the ATen/cuDNN glue of the BTS decoder and encoder transitions (reference
// pytorch/bts.py:69-80 upconv, :154-182 decoder BatchNorms, :199-260 the nine torch.cat, torchvision transitions),
// sm_100a, HBM-bound.  All tensors are fp32 NHWC with an explicit pixel stride, so a channel slice of a wider slab is
// read or written in place (concat = one vectorised slice copy per input instead of CatArrayBatchedCopy).
//
//   bts_bn_apply       out = x*scale + shift [ReLU | ReLU6]            BatchNorm apply (train or folded eval stats)
//   bts_bn_add         out = x*scale + shift + res                     MobileNetV2 inverted-residual tail
//   bts_elu_bwd        out = gy * (y > 0 ? 1 : y + 1)                  ELU'(a) expressed through the saved OUTPUT y
//   bts_upsample2_sum  out[b,y,x,c] = sum of the 2x2 block of g        backward of the nearest x2 up-sample folded into
//                      [* (x > 0) when relu_src != null]               upconv's im2col map (+ the ReLU in front of upconv5)
//   bts_copy_channels  dst[:, c] (=|+=) src[:, c]                      concat / concat-backward slice traffic
//   bts_avgpool2 / _bwd  2x2 stride-2 average pool (DenseNet transitions) and its backward
// Each thread moves 16 bytes; a warp covers 512 contiguous bytes of a pixel row group -> fully coalesced 128-bit
// transactions whenever C % 4 == 0 and the strides / bases are 16-byte aligned (scalar tail path otherwise).
#include <cmath>

#include "common.cuh"

namespace {

constexpr int TPB = 256;

__host__ inline int stream_grid(long long items) {
    long long grid = (items + TPB - 1) / TPB;
    const long long cap = (long long)bts_num_sms() * 16;
    if (grid > cap) grid = cap;
    if (grid < 1) grid = 1;
    return (int)grid;
}

__device__ __forceinline__ bool al16(const void *p) { return (((uintptr_t)p) & 15u) == 0; }

// RELU6 (host flag relu == 2): clamp(., 0, 6) instead of the ReLU; a separate instantiation leaves the relu 0 / 1 code as is
template <bool RELU6>
__global__ void __launch_bounds__(TPB) bn_apply_kernel(const float *__restrict__ x, long long xs, long long M, int C,
                                                       const float *__restrict__ scale, const float *__restrict__ shift,
                                                       int relu, float *__restrict__ out, long long os) {
    const int cq = (C + 3) >> 2;
    const long long total = M * cq;
    const bool vec = ((C & 3) == 0) && ((xs & 3) == 0) && ((os & 3) == 0) && al16(x) && al16(out) && al16(scale) && al16(shift);
    for (long long idx = (long long)blockIdx.x * TPB + threadIdx.x; idx < total; idx += (long long)gridDim.x * TPB) {
        const long long m = idx / cq;
        const int c = (int)(idx - m * cq) * 4;
        if (vec) {
            const float4 q = __ldg(reinterpret_cast<const float4 *>(x + m * xs + c));
            const float4 s = __ldg(reinterpret_cast<const float4 *>(scale + c));
            const float4 h = __ldg(reinterpret_cast<const float4 *>(shift + c));
            float4 r = make_float4(fmaf(q.x, s.x, h.x), fmaf(q.y, s.y, h.y), fmaf(q.z, s.z, h.z), fmaf(q.w, s.w, h.w));
            if (RELU6) {
                r.x = fminf(fmaxf(r.x, 0.f), 6.f); r.y = fminf(fmaxf(r.y, 0.f), 6.f);
                r.z = fminf(fmaxf(r.z, 0.f), 6.f); r.w = fminf(fmaxf(r.w, 0.f), 6.f);
            } else if (relu) { r.x = fmaxf(r.x, 0.f); r.y = fmaxf(r.y, 0.f); r.z = fmaxf(r.z, 0.f); r.w = fmaxf(r.w, 0.f); }
            *reinterpret_cast<float4 *>(out + m * os + c) = r;
        } else {
            for (int e = 0; e < 4 && c + e < C; ++e) {
                float r = fmaf(x[m * xs + c + e], scale[c + e], shift[c + e]);
                if (RELU6) r = fminf(fmaxf(r, 0.f), 6.f);
                else if (relu) r = fmaxf(r, 0.f);
                out[m * os + c + e] = r;
            }
        }
    }
}

__global__ void __launch_bounds__(TPB) elu_bwd_kernel(const float *__restrict__ gy, long long gs, const float *__restrict__ y,
                                                      long long ys, long long M, int C, float *__restrict__ out, long long os) {
    const int cq = (C + 3) >> 2;
    const long long total = M * cq;
    const bool vec = ((C & 3) == 0) && ((gs & 3) == 0) && ((ys & 3) == 0) && ((os & 3) == 0) && al16(gy) && al16(y) && al16(out);
    for (long long idx = (long long)blockIdx.x * TPB + threadIdx.x; idx < total; idx += (long long)gridDim.x * TPB) {
        const long long m = idx / cq;
        const int c = (int)(idx - m * cq) * 4;
        if (vec) {
            const float4 g = __ldg(reinterpret_cast<const float4 *>(gy + m * gs + c));
            const float4 v = __ldg(reinterpret_cast<const float4 *>(y + m * ys + c));
            float4 r;
            r.x = v.x > 0.f ? g.x : g.x * (v.x + 1.f);
            r.y = v.y > 0.f ? g.y : g.y * (v.y + 1.f);
            r.z = v.z > 0.f ? g.z : g.z * (v.z + 1.f);
            r.w = v.w > 0.f ? g.w : g.w * (v.w + 1.f);
            *reinterpret_cast<float4 *>(out + m * os + c) = r;
        } else {
            for (int e = 0; e < 4 && c + e < C; ++e) {
                const float g = gy[m * gs + c + e], v = y[m * ys + c + e];
                out[m * os + c + e] = v > 0.f ? g : g * (v + 1.f);
            }
        }
    }
}

// g: (B, 2H, 2W, C) pixel stride gs;  out: (B, H, W, C) pixel stride os;  relu_src: (B, H, W, C) stride rs or null
__global__ void __launch_bounds__(TPB) upsample2_sum_kernel(const float *__restrict__ g, long long gs, int B, int H, int W, int C,
                                                            const float *__restrict__ relu_src, long long rs,
                                                            float *__restrict__ out, long long os) {
    const int cq = (C + 3) >> 2;
    const long long M = (long long)B * H * W;
    const long long total = M * cq;
    const bool vec = ((C & 3) == 0) && ((gs & 3) == 0) && ((os & 3) == 0) && al16(g) && al16(out) &&
                     (!relu_src || (((rs & 3) == 0) && al16(relu_src)));
    for (long long idx = (long long)blockIdx.x * TPB + threadIdx.x; idx < total; idx += (long long)gridDim.x * TPB) {
        const long long m = idx / cq;
        const int c = (int)(idx - m * cq) * 4;
        const int x = (int)(m % W);
        const long long q = m / W;
        const int y = (int)(q % H);
        const long long b = q / H;
        const long long p00 = ((b * 2 * H + 2 * y) * 2 * W + 2 * x);
        const long long p10 = p00 + 2 * W;
        if (vec) {
            const float4 a = __ldg(reinterpret_cast<const float4 *>(g + p00 * gs + c));
            const float4 bq = __ldg(reinterpret_cast<const float4 *>(g + (p00 + 1) * gs + c));
            const float4 cc = __ldg(reinterpret_cast<const float4 *>(g + p10 * gs + c));
            const float4 d = __ldg(reinterpret_cast<const float4 *>(g + (p10 + 1) * gs + c));
            float4 r = make_float4((a.x + bq.x) + (cc.x + d.x), (a.y + bq.y) + (cc.y + d.y), (a.z + bq.z) + (cc.z + d.z),
                                   (a.w + bq.w) + (cc.w + d.w));
            if (relu_src) {
                const float4 s = __ldg(reinterpret_cast<const float4 *>(relu_src + m * rs + c));
                r.x = s.x > 0.f ? r.x : 0.f; r.y = s.y > 0.f ? r.y : 0.f; r.z = s.z > 0.f ? r.z : 0.f; r.w = s.w > 0.f ? r.w : 0.f;
            }
            *reinterpret_cast<float4 *>(out + m * os + c) = r;
        } else {
            for (int e = 0; e < 4 && c + e < C; ++e) {
                float r = (g[p00 * gs + c + e] + g[(p00 + 1) * gs + c + e]) + (g[p10 * gs + c + e] + g[(p10 + 1) * gs + c + e]);
                if (relu_src && !(relu_src[m * rs + c + e] > 0.f)) r = 0.f;
                out[m * os + c + e] = r;
            }
        }
    }
}

__global__ void __launch_bounds__(TPB) copy_channels_kernel(const float *__restrict__ src, long long ss, long long M, int C,
                                                            float *__restrict__ dst, long long ds, int accumulate) {
    const int cq = (C + 3) >> 2;
    const long long total = M * cq;
    const bool vec = ((C & 3) == 0) && ((ss & 3) == 0) && ((ds & 3) == 0) && al16(src) && al16(dst);
    for (long long idx = (long long)blockIdx.x * TPB + threadIdx.x; idx < total; idx += (long long)gridDim.x * TPB) {
        const long long m = idx / cq;
        const int c = (int)(idx - m * cq) * 4;
        if (vec) {
            float4 v = __ldg(reinterpret_cast<const float4 *>(src + m * ss + c));
            float4 *d = reinterpret_cast<float4 *>(dst + m * ds + c);
            if (accumulate) { const float4 o = *d; v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w; }
            *d = v;
        } else {
            for (int e = 0; e < 4 && c + e < C; ++e) {
                const float v = src[m * ss + c + e];
                if (accumulate) dst[m * ds + c + e] += v; else dst[m * ds + c + e] = v;
            }
        }
    }
}

// zero the channels [c0, c1) of an NHWC slab (the 16-byte alignment padding of concat3 / concat2)
__global__ void __launch_bounds__(TPB) zero_channels_kernel(float *__restrict__ dst, long long ds, long long M, int c0, int c1) {
    const int n = c1 - c0;
    const long long total = M * n;
    for (long long idx = (long long)blockIdx.x * TPB + threadIdx.x; idx < total; idx += (long long)gridDim.x * TPB) {
        const long long m = idx / n;
        dst[m * ds + c0 + (int)(idx - m * n)] = 0.f;
    }
}

// x: (B, 2Ho, 2Wo, C) -> out (B, Ho, Wo, C) = mean of the 2x2 block     (fwd);   bwd: gx = g[b, y/2, x/2, c] / 4
template <bool BWD>
__global__ void __launch_bounds__(TPB) avgpool2_kernel(const float *__restrict__ in, long long is, int B, int Ho, int Wo, int C,
                                                       float *__restrict__ out, long long os) {
    const int cq = (C + 3) >> 2;
    const long long M = BWD ? (long long)B * 4 * Ho * Wo : (long long)B * Ho * Wo;   // output pixels of this pass
    const long long total = M * cq;
    const bool vec = ((C & 3) == 0) && ((is & 3) == 0) && ((os & 3) == 0) && al16(in) && al16(out);
    for (long long idx = (long long)blockIdx.x * TPB + threadIdx.x; idx < total; idx += (long long)gridDim.x * TPB) {
        const long long m = idx / cq;
        const int c = (int)(idx - m * cq) * 4;
        if (!BWD) {
            const int x = (int)(m % Wo);
            const long long q = m / Wo;
            const int y = (int)(q % Ho);
            const long long b = q / Ho;
            const long long p00 = (b * 2 * Ho + 2 * y) * 2 * Wo + 2 * x, p10 = p00 + 2 * Wo;
            if (vec) {
                const float4 a = __ldg(reinterpret_cast<const float4 *>(in + p00 * is + c));
                const float4 bq = __ldg(reinterpret_cast<const float4 *>(in + (p00 + 1) * is + c));
                const float4 cc = __ldg(reinterpret_cast<const float4 *>(in + p10 * is + c));
                const float4 d = __ldg(reinterpret_cast<const float4 *>(in + (p10 + 1) * is + c));
                *reinterpret_cast<float4 *>(out + m * os + c) =
                    make_float4(((a.x + bq.x) + (cc.x + d.x)) * 0.25f, ((a.y + bq.y) + (cc.y + d.y)) * 0.25f,
                                ((a.z + bq.z) + (cc.z + d.z)) * 0.25f, ((a.w + bq.w) + (cc.w + d.w)) * 0.25f);
            } else {
                for (int e = 0; e < 4 && c + e < C; ++e)
                    out[m * os + c + e] = ((in[p00 * is + c + e] + in[(p00 + 1) * is + c + e]) +
                                           (in[p10 * is + c + e] + in[(p10 + 1) * is + c + e])) * 0.25f;
            }
        } else {
            const int x = (int)(m % (2 * Wo));
            const long long q = m / (2 * Wo);
            const int y = (int)(q % (2 * Ho));
            const long long b = q / (2 * Ho);
            const long long ps = (b * Ho + (y >> 1)) * Wo + (x >> 1);
            if (vec) {
                const float4 a = __ldg(reinterpret_cast<const float4 *>(in + ps * is + c));
                *reinterpret_cast<float4 *>(out + m * os + c) = make_float4(a.x * 0.25f, a.y * 0.25f, a.z * 0.25f, a.w * 0.25f);
            } else {
                for (int e = 0; e < 4 && c + e < C; ++e) out[m * os + c + e] = in[ps * is + c + e] * 0.25f;
            }
        }
    }
}

// ResNet / ResNeXt bottleneck tail (torchvision Bottleneck.forward: out = relu(bn3(conv3) + identity)):
//   out = max(x*scale + shift + res, 0);   RELU = false: out = x*scale + shift + res (MobileNetV2 InvertedResidual:
//   x + bn3(conv3), no activation)
template <bool RELU>
__global__ void __launch_bounds__(TPB) bn_add_relu_kernel(const float *__restrict__ x, long long xs, long long M, int C,
                                                          const float *__restrict__ scale, const float *__restrict__ shift,
                                                          const float *__restrict__ res, long long rs,
                                                          float *__restrict__ out, long long os) {
    const int cq = (C + 3) >> 2;
    const long long total = M * cq;
    const bool vec = ((C & 3) == 0) && ((xs & 3) == 0) && ((os & 3) == 0) && ((rs & 3) == 0) && al16(x) && al16(out) && al16(res) &&
                     al16(scale) && al16(shift);
    for (long long idx = (long long)blockIdx.x * TPB + threadIdx.x; idx < total; idx += (long long)gridDim.x * TPB) {
        const long long m = idx / cq;
        const int c = (int)(idx - m * cq) * 4;
        if (vec) {
            const float4 q = __ldg(reinterpret_cast<const float4 *>(x + m * xs + c));
            const float4 r0 = __ldg(reinterpret_cast<const float4 *>(res + m * rs + c));
            const float4 s = __ldg(reinterpret_cast<const float4 *>(scale + c));
            const float4 h = __ldg(reinterpret_cast<const float4 *>(shift + c));
            float4 r = make_float4(fmaf(q.x, s.x, h.x) + r0.x, fmaf(q.y, s.y, h.y) + r0.y, fmaf(q.z, s.z, h.z) + r0.z,
                                   fmaf(q.w, s.w, h.w) + r0.w);
            if (RELU) { r.x = fmaxf(r.x, 0.f); r.y = fmaxf(r.y, 0.f); r.z = fmaxf(r.z, 0.f); r.w = fmaxf(r.w, 0.f); }
            *reinterpret_cast<float4 *>(out + m * os + c) = r;
        } else {
            for (int e = 0; e < 4 && c + e < C; ++e) {
                const float r = fmaf(x[m * xs + c + e], scale[c + e], shift[c + e]) + res[m * rs + c + e];
                out[m * os + c + e] = RELU ? fmaxf(r, 0.f) : r;
            }
        }
    }
}

// out = gy * (y > 0): backward of a ReLU expressed through its saved OUTPUT
__global__ void __launch_bounds__(TPB) relu_bwd_kernel(const float *__restrict__ gy, long long gs, const float *__restrict__ y,
                                                       long long ys, long long M, int C, float *__restrict__ out, long long os) {
    const int cq = (C + 3) >> 2;
    const long long total = M * cq;
    const bool vec = ((C & 3) == 0) && ((gs & 3) == 0) && ((ys & 3) == 0) && ((os & 3) == 0) && al16(gy) && al16(y) && al16(out);
    for (long long idx = (long long)blockIdx.x * TPB + threadIdx.x; idx < total; idx += (long long)gridDim.x * TPB) {
        const long long m = idx / cq;
        const int c = (int)(idx - m * cq) * 4;
        if (vec) {
            const float4 g = __ldg(reinterpret_cast<const float4 *>(gy + m * gs + c));
            const float4 v = __ldg(reinterpret_cast<const float4 *>(y + m * ys + c));
            *reinterpret_cast<float4 *>(out + m * os + c) =
                make_float4(v.x > 0.f ? g.x : 0.f, v.y > 0.f ? g.y : 0.f, v.z > 0.f ? g.z : 0.f, v.w > 0.f ? g.w : 0.f);
        } else {
            for (int e = 0; e < 4 && c + e < C; ++e) out[m * os + c + e] = y[m * ys + c + e] > 0.f ? gy[m * gs + c + e] : 0.f;
        }
    }
}

// 3x3 / stride 2 / pad 1 max-pool of the encoder stems (torchvision densenet `pool0`, resnet `maxpool`), NHWC.
// Forward also records which of the 9 window positions won (first maximum in row-major scan order, NaN propagates --
// the tie rule of at::max_pool2d) so the backward is a deterministic gather: each input pixel looks at the <= 4 windows
// that contain it.
__global__ void __launch_bounds__(TPB) maxpool3s2_fwd_kernel(const float *__restrict__ x, long long xs, int B, int H, int W, int C,
                                                             int Ho, int Wo, float *__restrict__ out, long long os,
                                                             unsigned char *__restrict__ arg) {
    const long long total = (long long)B * Ho * Wo * C;
    for (long long idx = (long long)blockIdx.x * TPB + threadIdx.x; idx < total; idx += (long long)gridDim.x * TPB) {
        const int c = (int)(idx % C);
        long long t = idx / C;
        const int ox = (int)(t % Wo);
        t /= Wo;
        const int oy = (int)(t % Ho);
        const int b = (int)(t / Ho);
        float best = -INFINITY;
        int bi = 0;
        bool first = true;
#pragma unroll
        for (int ky = 0; ky < 3; ++ky)
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) {
                const int y = 2 * oy - 1 + ky, xx = 2 * ox - 1 + kx;
                if ((unsigned)y < (unsigned)H && (unsigned)xx < (unsigned)W) {
                    const float v = __ldg(x + (((long long)b * H + y) * W + xx) * xs + c);
                    if (first) { bi = ky * 3 + kx; first = false; }       // at::max_pool2d: index starts at the first valid tap
                    if (v > best || v != v) { best = v; bi = ky * 3 + kx; }   // strict >: the first maximum wins; NaN propagates
                }
            }
        out[(((long long)b * Ho + oy) * Wo + ox) * os + c] = best;
        arg[idx] = (unsigned char)bi;
    }
}

__global__ void __launch_bounds__(TPB) maxpool3s2_bwd_kernel(const float *__restrict__ g, long long gs,
                                                             const unsigned char *__restrict__ arg, int B, int H, int W, int C,
                                                             int Ho, int Wo, float *__restrict__ gx, long long gxs) {
    const long long total = (long long)B * H * W * C;
    for (long long idx = (long long)blockIdx.x * TPB + threadIdx.x; idx < total; idx += (long long)gridDim.x * TPB) {
        const int c = (int)(idx % C);
        long long t = idx / C;
        const int xx = (int)(t % W);
        t /= W;
        const int y = (int)(t % H);
        const int b = (int)(t / H);
        float acc = 0.f;
        // windows (oy, ox) with 2*oy - 1 <= y <= 2*oy + 1
        for (int oy = y >> 1; oy <= ((y + 1) >> 1); ++oy) {
            if (oy >= Ho) continue;
            const int ky = y - (2 * oy - 1);
            for (int ox = xx >> 1; ox <= ((xx + 1) >> 1); ++ox) {
                if (ox >= Wo) continue;
                const int kx = xx - (2 * ox - 1);
                const long long o = (((long long)b * Ho + oy) * Wo + ox);
                if (arg[o * C + c] == ky * 3 + kx) acc += __ldg(g + o * gs + c);
            }
        }
        gx[(((long long)b * H + y) * W + xx) * gxs + c] = acc;
    }
}

}  // namespace

extern "C" int bts_bn_apply(const float *x, long long x_pixel_stride, long long M, int C, const float *scale,
                            const float *shift, int relu, float *out, long long out_pixel_stride, void *stream) {
    if (!x || !scale || !shift || !out || M < 1 || C < 1) return BTS_EINVAL;
    if (relu == 2)
        bn_apply_kernel<true><<<stream_grid(M * ((C + 3) / 4)), TPB, 0, (cudaStream_t)stream>>>(x, x_pixel_stride, M, C, scale,
                                                                                             shift, relu, out, out_pixel_stride);
    else
        bn_apply_kernel<false><<<stream_grid(M * ((C + 3) / 4)), TPB, 0, (cudaStream_t)stream>>>(x, x_pixel_stride, M, C, scale,
                                                                                              shift, relu, out, out_pixel_stride);
    BTS_LAUNCH_CHECK();
    return 0;
}

extern "C" int bts_elu_bwd(const float *gy, long long gy_pixel_stride, const float *y, long long y_pixel_stride, long long M,
                           int C, float *out, long long out_pixel_stride, void *stream) {
    if (!gy || !y || !out || M < 1 || C < 1) return BTS_EINVAL;
    elu_bwd_kernel<<<stream_grid(M * ((C + 3) / 4)), TPB, 0, (cudaStream_t)stream>>>(gy, gy_pixel_stride, y, y_pixel_stride, M,
                                                                                      C, out, out_pixel_stride);
    BTS_LAUNCH_CHECK();
    return 0;
}

extern "C" int bts_upsample2_sum(const float *g, long long g_pixel_stride, int B, int H, int W, int C, const float *relu_src,
                                 long long relu_pixel_stride, float *out, long long out_pixel_stride, void *stream) {
    if (!g || !out || B < 1 || H < 1 || W < 1 || C < 1) return BTS_EINVAL;
    upsample2_sum_kernel<<<stream_grid((long long)B * H * W * ((C + 3) / 4)), TPB, 0, (cudaStream_t)stream>>>(
        g, g_pixel_stride, B, H, W, C, relu_src, relu_pixel_stride, out, out_pixel_stride);
    BTS_LAUNCH_CHECK();
    return 0;
}

extern "C" int bts_copy_channels(const float *src, long long src_pixel_stride, long long M, int C, float *dst,
                                 long long dst_pixel_stride, int accumulate, void *stream) {
    if (!src || !dst || M < 1 || C < 1) return BTS_EINVAL;
    copy_channels_kernel<<<stream_grid(M * ((C + 3) / 4)), TPB, 0, (cudaStream_t)stream>>>(src, src_pixel_stride, M, C, dst,
                                                                                            dst_pixel_stride, accumulate);
    BTS_LAUNCH_CHECK();
    return 0;
}

extern "C" int bts_zero_channels(float *dst, long long dst_pixel_stride, long long M, int c0, int c1, void *stream) {
    if (!dst || M < 1 || c0 < 0 || c1 <= c0) return BTS_EINVAL;
    zero_channels_kernel<<<stream_grid(M * (c1 - c0)), TPB, 0, (cudaStream_t)stream>>>(dst, dst_pixel_stride, M, c0, c1);
    BTS_LAUNCH_CHECK();
    return 0;
}

extern "C" int bts_avgpool2_fwd(const float *x, long long x_pixel_stride, int B, int Hout, int Wout, int C, float *out,
                                long long out_pixel_stride, void *stream) {
    if (!x || !out || B < 1 || Hout < 1 || Wout < 1 || C < 1) return BTS_EINVAL;
    avgpool2_kernel<false><<<stream_grid((long long)B * Hout * Wout * ((C + 3) / 4)), TPB, 0, (cudaStream_t)stream>>>(
        x, x_pixel_stride, B, Hout, Wout, C, out, out_pixel_stride);
    BTS_LAUNCH_CHECK();
    return 0;
}

extern "C" int bts_avgpool2_bwd(const float *g, long long g_pixel_stride, int B, int Hout, int Wout, int C, float *gx,
                                long long gx_pixel_stride, void *stream) {
    if (!g || !gx || B < 1 || Hout < 1 || Wout < 1 || C < 1) return BTS_EINVAL;
    avgpool2_kernel<true><<<stream_grid((long long)B * 4 * Hout * Wout * ((C + 3) / 4)), TPB, 0, (cudaStream_t)stream>>>(
        g, g_pixel_stride, B, Hout, Wout, C, gx, gx_pixel_stride);
    BTS_LAUNCH_CHECK();
    return 0;
}

extern "C" int bts_bn_add_relu(const float *x, long long x_pixel_stride, long long M, int C, const float *scale,
                               const float *shift, const float *res, long long res_pixel_stride, float *out,
                               long long out_pixel_stride, void *stream) {
    if (!x || !scale || !shift || !res || !out || M < 1 || C < 1) return BTS_EINVAL;
    bn_add_relu_kernel<true><<<stream_grid(M * ((C + 3) / 4)), TPB, 0, (cudaStream_t)stream>>>(
        x, x_pixel_stride, M, C, scale, shift, res, res_pixel_stride, out, out_pixel_stride);
    BTS_LAUNCH_CHECK();
    return 0;
}

extern "C" int bts_bn_add(const float *x, long long x_pixel_stride, long long M, int C, const float *scale, const float *shift,
                          const float *res, long long res_pixel_stride, float *out, long long out_pixel_stride, void *stream) {
    if (!x || !scale || !shift || !res || !out || M < 1 || C < 1) return BTS_EINVAL;
    bn_add_relu_kernel<false><<<stream_grid(M * ((C + 3) / 4)), TPB, 0, (cudaStream_t)stream>>>(
        x, x_pixel_stride, M, C, scale, shift, res, res_pixel_stride, out, out_pixel_stride);
    BTS_LAUNCH_CHECK();
    return 0;
}

extern "C" int bts_relu_bwd(const float *gy, long long gy_pixel_stride, const float *y, long long y_pixel_stride, long long M,
                            int C, float *out, long long out_pixel_stride, void *stream) {
    if (!gy || !y || !out || M < 1 || C < 1) return BTS_EINVAL;
    relu_bwd_kernel<<<stream_grid(M * ((C + 3) / 4)), TPB, 0, (cudaStream_t)stream>>>(gy, gy_pixel_stride, y, y_pixel_stride, M,
                                                                                       C, out, out_pixel_stride);
    BTS_LAUNCH_CHECK();
    return 0;
}

extern "C" int bts_maxpool3s2_fwd(const float *x, long long x_pixel_stride, int B, int H, int W, int C, float *out,
                                  long long out_pixel_stride, unsigned char *argmax, void *stream) {
    if (!x || !out || !argmax || B < 1 || H < 1 || W < 1 || C < 1) return BTS_EINVAL;
    const int Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1;
    maxpool3s2_fwd_kernel<<<stream_grid((long long)B * Ho * Wo * C), TPB, 0, (cudaStream_t)stream>>>(
        x, x_pixel_stride, B, H, W, C, Ho, Wo, out, out_pixel_stride, argmax);
    BTS_LAUNCH_CHECK();
    return 0;
}

extern "C" int bts_maxpool3s2_bwd(const float *g, long long g_pixel_stride, const unsigned char *argmax, int B, int H, int W,
                                  int C, float *gx, long long gx_pixel_stride, void *stream) {
    if (!g || !gx || !argmax || B < 1 || H < 1 || W < 1 || C < 1) return BTS_EINVAL;
    const int Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1;
    maxpool3s2_bwd_kernel<<<stream_grid((long long)B * H * W * C), TPB, 0, (cudaStream_t)stream>>>(
        g, g_pixel_stride, argmax, B, H, W, C, Ho, Wo, gx, gx_pixel_stride);
    BTS_LAUNCH_CHECK();
    return 0;
}
