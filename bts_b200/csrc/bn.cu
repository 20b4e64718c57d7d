// Train-mode BatchNorm pieces for the fused BN -> ReLU -> conv chains (DenseNet dense layers `norm1/relu1/conv1/norm2/
// relu2/conv2`, torchvision densenet.py; decoder BNs pytorch/bts.py:154-182), sm_100a, HBM-bound.
//
// The normalisation itself never runs as a kernel: it is folded into the consumer conv's A-operand prologue
// (conv_tc.cu, PRE = affine + ReLU) as y = x*scale + shift with scale = gamma*invstd, shift = beta - mean*scale.
// What remains are per-channel reductions over the NHWC activation (channel = fastest index -> lanes own channels,
// fully coalesced) and one elementwise backward pass:
//   bts_bn_stats      : sum, sum of squares per channel (fp32 per-thread strips, fp64 cross-block accumulation)
//   bts_bn_finalize   : mean / biased var -> scale, shift, invstd; running-stat update with momentum (unbiased var)
//   bts_bn_relu_bwd_reduce : S1 = sum g*[y>0], S2 = sum g*[y>0]*xhat            (y = x*scale+shift, xhat = (x-mean)*invstd)
//   bts_bn_relu_bwd_apply  : dx = scale * ( g*[y>0] - S1/N - xhat*S2/N ), written or ACCUMULATED into a (slice of a)
//                            gradient slab -- the concat fan-out of a dense block sums into one buffer, no add kernels.
// All tensors are NHWC with an explicit pixel stride, so channel slices of wider slabs work in place.
#include "common.cuh"

namespace {

// Column reductions over NHWC: a 256-thread block covers up to 256 channels (64 channel quads) x `rows` pixels; with
// fewer channels the spare threads take extra pixel rows.  Four independent 16-byte loads per tensor are in flight per
// thread; the row groups of a block are combined in shared memory, then ONE fp64 atomic per channel per block.
// `relu`: 0 none, 1 ReLU (mask y > 0); RELU6 (host flag relu == 2) replaces that mask by 0 < y < 6, strict: torch's
// hardtanh_backward of an in-place ReLU6.  A separate instantiation, so the relu 0 / 1 code is unchanged by it.
// MODE 0: forward statistics; 1: backward sums; 2: backward sums AND out += [y>0]*scale*g in the same pass (the part of dx
// that does not depend on the sums -- the k1*x + k0 remainder is deferred, see bts_bn_relu_bwd_fused).
template <int MODE, bool RELU6 = false>
__global__ void __launch_bounds__(256) bn_reduce_kernel(const float *__restrict__ x, long long xs, const float *__restrict__ g,
                                                        long long gs, long long M, int C, int rows,
                                                        const float *__restrict__ scale, const float *__restrict__ shift,
                                                        const float *__restrict__ mean, const float *__restrict__ invstd,
                                                        double *__restrict__ acc0, double *__restrict__ acc1, int relu,
                                                        float *out, long long os) {
    constexpr bool BWD = MODE != 0;
    constexpr bool ACC = MODE == 2;
    __shared__ float red[2][256 * 4];
    const int cchunk = min(256, C - (int)blockIdx.y * 256);
    const int tpc = (cchunk + 3) >> 2;                 // threads per pixel row
    const int rp = 256 / tpc;                          // pixel rows processed concurrently
    const int tq = (int)threadIdx.x % tpc, rsub = (int)threadIdx.x / tpc;
    const bool active = rsub < rp;
    const int c = blockIdx.y * 256 + tq * 4;
    float a0[4] = {0.f, 0.f, 0.f, 0.f}, a1[4] = {0.f, 0.f, 0.f, 0.f};
    if (active) {
        const long long m0 = (long long)blockIdx.x * rows + rsub;
        long long m1 = (long long)(blockIdx.x + 1) * rows;
        if (m1 > M) m1 = M;
        float sc[4], sh[4], mu[4], is[4];
        if (BWD) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int ce = c + e < C ? c + e : C - 1;
                sc[e] = scale[ce]; sh[e] = shift[ce]; mu[e] = mean[ce]; is[e] = invstd[ce];
            }
        }
        const bool vec = (c + 3 < C) && ((xs & 3) == 0) && ((((uintptr_t)x) & 15) == 0) &&
                         (!BWD || (((gs & 3) == 0) && ((((uintptr_t)g) & 15) == 0))) &&
                         (!ACC || (((os & 3) == 0) && ((((uintptr_t)out) & 15) == 0)));
        auto accum = [&](const float (&xv)[4], const float (&gv)[4], float (&ov)[4]) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                if (!BWD) {
                    a0[e] += xv[e];
                    a1[e] = fmaf(xv[e], xv[e], a1[e]);
                } else {
                    const float y = fmaf(xv[e], sc[e], sh[e]);
                    const float gm = (RELU6 ? (y > 0.f && y < 6.f) : (!relu || y > 0.f)) ? gv[e] : 0.f;
                    a0[e] += gm;
                    a1[e] = fmaf(gm, (xv[e] - mu[e]) * is[e], a1[e]);
                    if (ACC) ov[e] = fmaf(sc[e], gm, ov[e]);
                }
            }
        };
        if (vec) {
            long long m = m0;
            for (; m + 3LL * rp < m1; m += 4LL * rp) {
                float4 q[4], r[4], o[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) q[u] = __ldg(reinterpret_cast<const float4 *>(x + (m + (long long)u * rp) * xs + c));
                if (BWD) {
#pragma unroll
                    for (int u = 0; u < 4; ++u) r[u] = __ldg(reinterpret_cast<const float4 *>(g + (m + (long long)u * rp) * gs + c));
                }
                if (ACC) {
#pragma unroll
                    for (int u = 0; u < 4; ++u) o[u] = *reinterpret_cast<const float4 *>(out + (m + (long long)u * rp) * os + c);
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const float xv[4] = {q[u].x, q[u].y, q[u].z, q[u].w};
                    const float gv[4] = {BWD ? r[u].x : 0.f, BWD ? r[u].y : 0.f, BWD ? r[u].z : 0.f, BWD ? r[u].w : 0.f};
                    float ov[4] = {ACC ? o[u].x : 0.f, ACC ? o[u].y : 0.f, ACC ? o[u].z : 0.f, ACC ? o[u].w : 0.f};
                    accum(xv, gv, ov);
                    if (ACC)
                        *reinterpret_cast<float4 *>(out + (m + (long long)u * rp) * os + c) = make_float4(ov[0], ov[1], ov[2], ov[3]);
                }
            }
            for (; m < m1; m += rp) {
                const float4 q = __ldg(reinterpret_cast<const float4 *>(x + m * xs + c));
                float4 r = make_float4(0.f, 0.f, 0.f, 0.f), o = make_float4(0.f, 0.f, 0.f, 0.f);
                if (BWD) r = __ldg(reinterpret_cast<const float4 *>(g + m * gs + c));
                if (ACC) o = *reinterpret_cast<const float4 *>(out + m * os + c);
                const float xv[4] = {q.x, q.y, q.z, q.w};
                const float gv[4] = {r.x, r.y, r.z, r.w};
                float ov[4] = {o.x, o.y, o.z, o.w};
                accum(xv, gv, ov);
                if (ACC) *reinterpret_cast<float4 *>(out + m * os + c) = make_float4(ov[0], ov[1], ov[2], ov[3]);
            }
        } else {
            for (long long m = m0; m < m1; m += rp) {
                float xv[4], gv[4], ov[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    xv[e] = c + e < C ? __ldg(x + m * xs + c + e) : 0.f;
                    gv[e] = (BWD && c + e < C) ? __ldg(g + m * gs + c + e) : 0.f;
                    ov[e] = (ACC && c + e < C) ? out[m * os + c + e] : 0.f;
                }
                accum(xv, gv, ov);
                if (ACC) {
#pragma unroll
                    for (int e = 0; e < 4; ++e)
                        if (c + e < C) out[m * os + c + e] = ov[e];
                }
            }
        }
    }
    // combine the rp row groups: red[k][rsub*tpc*4 + tq*4 + e]
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        red[0][threadIdx.x * 4 + e] = a0[e];
        red[1][threadIdx.x * 4 + e] = a1[e];
    }
    __syncthreads();
    if (rsub == 0 && (int)threadIdx.x < tpc) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            if (c + e < C) {
                double s0 = 0.0, s1 = 0.0;
                for (int r2 = 0; r2 < rp; ++r2) {
                    s0 += (double)red[0][(r2 * tpc + tq) * 4 + e];
                    s1 += (double)red[1][(r2 * tpc + tq) * 4 + e];
                }
                atomicAdd(acc0 + c + e, s0);
                atomicAdd(acc1 + c + e, s1);
            }
        }
    }
}

// per-channel backward coefficients in fp32 (fp64 stays out of the streaming pass):
//   dx = [y>0]*scale*g + k1*x + k0,   k1 = -scale*invstd*S2/N,   k0 = -scale*S1/N - k1*mean
__global__ void bn_bwd_coef_kernel(const double *__restrict__ S1, const double *__restrict__ S2, long long N, int C,
                                   const float *__restrict__ scale, const float *__restrict__ mean,
                                   const float *__restrict__ invstd, float *__restrict__ coef) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const double s = scale[c];
    const double k1 = -s * (double)invstd[c] * S2[c] / (double)N;
    const double k0 = -s * S1[c] / (double)N - k1 * (double)mean[c];
    coef[c] = (float)k0;
    coef[C + c] = (float)k1;
}

// deferred form: the (k0, k1) of every BatchNorm that reads channel c of a concat slab add up (dx is linear in them)
__global__ void bn_bwd_coef_accum_kernel(const double *__restrict__ S1, const double *__restrict__ S2, long long N, int C,
                                         const float *__restrict__ scale, const float *__restrict__ mean,
                                         const float *__restrict__ invstd, double *__restrict__ K0, double *__restrict__ K1) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const double s = scale[c];
    const double k1 = -s * (double)invstd[c] * S2[c] / (double)N;
    K1[c] += k1;
    K0[c] += -s * S1[c] / (double)N - k1 * (double)mean[c];
}

// out[m, c] += K1[c]*x[m, c] + K0[c]
__global__ void __launch_bounds__(256) bn_bwd_correct_kernel(const float *__restrict__ x, long long xs, long long M, int C,
                                                             const double *__restrict__ K0, const double *__restrict__ K1,
                                                             float *__restrict__ out, long long os) {
    const int cq = (C + 3) >> 2;
    const long long total = M * cq;
    const bool vec = ((xs & 3) == 0) && ((os & 3) == 0) && ((((uintptr_t)x) & 15) == 0) && ((((uintptr_t)out) & 15) == 0) &&
                     ((C & 3) == 0);
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long m = idx / cq;
        const int c = (int)(idx - m * cq) * 4;
        if (vec) {
            const float4 q = __ldg(reinterpret_cast<const float4 *>(x + m * xs + c));
            float4 o = *reinterpret_cast<const float4 *>(out + m * os + c);
            o.x += fmaf(q.x, (float)K1[c], (float)K0[c]);
            o.y += fmaf(q.y, (float)K1[c + 1], (float)K0[c + 1]);
            o.z += fmaf(q.z, (float)K1[c + 2], (float)K0[c + 2]);
            o.w += fmaf(q.w, (float)K1[c + 3], (float)K0[c + 3]);
            *reinterpret_cast<float4 *>(out + m * os + c) = o;
        } else {
#pragma unroll
            for (int e = 0; e < 4; ++e)
                if (c + e < C) out[m * os + c + e] += fmaf(x[m * xs + c + e], (float)K1[c + e], (float)K0[c + e]);
        }
    }
}

__global__ void bn_finalize_kernel(const double *__restrict__ sum, const double *__restrict__ sumsq, long long N, int C,
                                   const float *__restrict__ gamma, const float *__restrict__ beta, float eps,
                                   float momentum, float *__restrict__ running_mean, float *__restrict__ running_var,
                                   float *__restrict__ scale, float *__restrict__ shift, float *__restrict__ mean,
                                   float *__restrict__ invstd, long long *__restrict__ num_batches_tracked) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c == 0 && num_batches_tracked) *num_batches_tracked += 1;     // nn.BatchNorm2d.num_batches_tracked += 1
    if (c >= C) return;
    const double m = sum[c] / (double)N;
    double var = sumsq[c] / (double)N - m * m;     // biased, used for normalisation
    if (var < 0.0) var = 0.0;
    const float is = (float)(1.0 / sqrt(var + (double)eps));
    const float gm = gamma ? gamma[c] : 1.f, bt = beta ? beta[c] : 0.f;
    const float s = gm * is;
    scale[c] = s;
    shift[c] = bt - (float)m * s;
    mean[c] = (float)m;
    invstd[c] = is;
    if (running_mean) {   // nn.BatchNorm2d: running = (1-mom)*running + mom*stat, unbiased variance
        const double unb = N > 1 ? var * (double)N / (double)(N - 1) : var;
        running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * (float)m;
        running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unb;
    }
}

// eval mode / frozen statistics: scale, shift straight from the running buffers
__global__ void bn_fold_kernel(int C, const float *__restrict__ gamma, const float *__restrict__ beta, float eps,
                               const float *__restrict__ running_mean, const float *__restrict__ running_var,
                               float *__restrict__ scale, float *__restrict__ shift, float *__restrict__ mean,
                               float *__restrict__ invstd) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const float is = 1.0f / sqrtf(running_var[c] + eps);
    const float s = (gamma ? gamma[c] : 1.f) * is;
    scale[c] = s;
    shift[c] = (beta ? beta[c] : 0.f) - running_mean[c] * s;
    mean[c] = running_mean[c];
    invstd[c] = is;
}

// dx = [y>0]*scale*g + k1*x + k0  (train; coef = (k0,k1) from bn_bwd_coef_kernel)   or   [y>0]*scale*g  (coef == null);
// RELU6: the mask is [0 < y < 6]
template <bool RELU6>
__global__ void __launch_bounds__(256) bn_relu_bwd_apply_kernel(const float *__restrict__ x, long long xs,
                                                                const float *__restrict__ g, long long gs, long long M,
                                                                int C, const float *__restrict__ scale,
                                                                const float *__restrict__ shift, const float *__restrict__ coef,
                                                                float *__restrict__ out, long long os, int accumulate,
                                                                int relu) {
    const int cq = (C + 3) >> 2;
    const long long total = M * cq;
    const bool vec = ((xs & 3) == 0) && ((gs & 3) == 0) && ((os & 3) == 0) && ((((uintptr_t)x) & 15) == 0) &&
                     ((((uintptr_t)g) & 15) == 0) && ((((uintptr_t)out) & 15) == 0) && ((C & 3) == 0);
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long m = idx / cq;
        const int c = (int)(idx - m * cq) * 4;
        float xv[4], gv[4], ov[4] = {0.f, 0.f, 0.f, 0.f}, sc[4], sh[4], k0[4] = {0.f, 0.f, 0.f, 0.f}, k1[4] = {0.f, 0.f, 0.f, 0.f};
        if (vec) {
            const float4 q = __ldg(reinterpret_cast<const float4 *>(x + m * xs + c));
            const float4 r = __ldg(reinterpret_cast<const float4 *>(g + m * gs + c));
            const float4 s4 = __ldg(reinterpret_cast<const float4 *>(scale + c));
            const float4 h4 = __ldg(reinterpret_cast<const float4 *>(shift + c));
            xv[0] = q.x; xv[1] = q.y; xv[2] = q.z; xv[3] = q.w;
            gv[0] = r.x; gv[1] = r.y; gv[2] = r.z; gv[3] = r.w;
            sc[0] = s4.x; sc[1] = s4.y; sc[2] = s4.z; sc[3] = s4.w;
            sh[0] = h4.x; sh[1] = h4.y; sh[2] = h4.z; sh[3] = h4.w;
            if (coef) {
                const float4 a4 = __ldg(reinterpret_cast<const float4 *>(coef + c));
                const float4 b4 = __ldg(reinterpret_cast<const float4 *>(coef + C + c));
                k0[0] = a4.x; k0[1] = a4.y; k0[2] = a4.z; k0[3] = a4.w;
                k1[0] = b4.x; k1[1] = b4.y; k1[2] = b4.z; k1[3] = b4.w;
            }
            if (accumulate) {
                const float4 o = *reinterpret_cast<const float4 *>(out + m * os + c);
                ov[0] = o.x; ov[1] = o.y; ov[2] = o.z; ov[3] = o.w;
            }
        } else {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const bool ok = c + e < C;
                const int ce = ok ? c + e : C - 1;
                xv[e] = ok ? x[m * xs + c + e] : 0.f;
                gv[e] = ok ? g[m * gs + c + e] : 0.f;
                ov[e] = (ok && accumulate) ? out[m * os + c + e] : 0.f;
                sc[e] = scale[ce]; sh[e] = shift[ce];
                if (coef) { k0[e] = coef[ce]; k1[e] = coef[C + ce]; }
            }
        }
        float r[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float y = fmaf(xv[e], sc[e], sh[e]);
            float d = (RELU6 ? (y > 0.f && y < 6.f) : (!relu || y > 0.f)) ? sc[e] * gv[e] : 0.f;
            d += fmaf(xv[e], k1[e], k0[e]);
            r[e] = ov[e] + d;
        }
        if (vec) {
            *reinterpret_cast<float4 *>(out + m * os + c) = make_float4(r[0], r[1], r[2], r[3]);
        } else {
#pragma unroll
            for (int e = 0; e < 4; ++e)
                if (c + e < C) out[m * os + c + e] = r[e];
        }
    }
}

int reduce_rows(long long M, int cgroups) {
    // enough blocks for ~8 per SM, at least 32 rows each
    long long want = (long long)bts_num_sms() * 8 / cgroups;
    if (want < 1) want = 1;
    long long rows = (M + want - 1) / want;
    if (rows < 32) rows = 32;
    if (rows > 4096) rows = 4096;
    return (int)rows;
}

}  // namespace

extern "C" int bts_bn_stats(const float *x, long long x_pixel_stride, long long M, int C, double *sum, double *sumsq,
                            void *stream) {
    if (!x || !sum || !sumsq || M < 1 || C < 1) return BTS_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e;
    if (sumsq == sum + C) {
        if ((e = cudaMemsetAsync(sum, 0, sizeof(double) * 2 * C, st)) != cudaSuccess) return (int)e;
    } else {
        if ((e = cudaMemsetAsync(sum, 0, sizeof(double) * C, st)) != cudaSuccess) return (int)e;
        if ((e = cudaMemsetAsync(sumsq, 0, sizeof(double) * C, st)) != cudaSuccess) return (int)e;
    }
    const int cg = (C + 255) / 256;
    const int rows = reduce_rows(M, cg);
    dim3 grid((unsigned)((M + rows - 1) / rows), (unsigned)cg);
    bn_reduce_kernel<0><<<grid, 256, 0, st>>>(x, x_pixel_stride, nullptr, 0, M, C, rows, nullptr, nullptr, nullptr, nullptr,
                                              sum, sumsq, 0, nullptr, 0);
    BTS_LAUNCH_CHECK();
    return 0;
}

extern "C" int bts_bn_finalize(const double *sum, const double *sumsq, long long N, int C, const float *gamma,
                               const float *beta, float eps, float momentum, float *running_mean, float *running_var,
                               float *scale, float *shift, float *mean, float *invstd, void *stream) {
    if (!sum || !sumsq || !scale || !shift || !mean || !invstd || N < 1 || C < 1) return BTS_EINVAL;
    bn_finalize_kernel<<<(C + 127) / 128, 128, 0, (cudaStream_t)stream>>>(sum, sumsq, N, C, gamma, beta, eps, momentum,
                                                                          running_mean, running_var, scale, shift, mean, invstd,
                                                                          nullptr);
    BTS_LAUNCH_CHECK();
    return 0;
}

// the same, also incrementing the module's int64 `num_batches_tracked` buffer in the same launch
extern "C" int bts_bn_finalize_track(const double *sum, const double *sumsq, long long N, int C, const float *gamma,
                                     const float *beta, float eps, float momentum, float *running_mean, float *running_var,
                                     long long *num_batches_tracked, float *scale, float *shift, float *mean, float *invstd,
                                     void *stream) {
    if (!sum || !sumsq || !scale || !shift || !mean || !invstd || N < 1 || C < 1) return BTS_EINVAL;
    bn_finalize_kernel<<<(C + 127) / 128, 128, 0, (cudaStream_t)stream>>>(sum, sumsq, N, C, gamma, beta, eps, momentum,
                                                                          running_mean, running_var, scale, shift, mean, invstd,
                                                                          num_batches_tracked);
    BTS_LAUNCH_CHECK();
    return 0;
}

extern "C" int bts_bn_fold(int C, const float *gamma, const float *beta, float eps, const float *running_mean,
                           const float *running_var, float *scale, float *shift, float *mean, float *invstd, void *stream) {
    if (!running_mean || !running_var || !scale || !shift || !mean || !invstd || C < 1) return BTS_EINVAL;
    bn_fold_kernel<<<(C + 127) / 128, 128, 0, (cudaStream_t)stream>>>(C, gamma, beta, eps, running_mean, running_var, scale,
                                                                      shift, mean, invstd);
    BTS_LAUNCH_CHECK();
    return 0;
}

extern "C" int bts_bn_bwd_reduce(const float *x, long long x_pixel_stride, const float *g, long long g_pixel_stride,
                                 long long M, int C, const float *scale, const float *shift, const float *mean,
                                 const float *invstd, int relu, double *S1, double *S2, float *coef, void *stream) {
    if (!x || !g || !scale || !shift || !mean || !invstd || !S1 || !S2 || !coef || M < 1 || C < 1) return BTS_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e;
    if (S2 == S1 + C) {                         // the usual [2, C] tensor: one memset
        if ((e = cudaMemsetAsync(S1, 0, sizeof(double) * 2 * C, st)) != cudaSuccess) return (int)e;
    } else {
        if ((e = cudaMemsetAsync(S1, 0, sizeof(double) * C, st)) != cudaSuccess) return (int)e;
        if ((e = cudaMemsetAsync(S2, 0, sizeof(double) * C, st)) != cudaSuccess) return (int)e;
    }
    const int cg = (C + 255) / 256;
    const int rows = reduce_rows(M, cg);
    dim3 grid((unsigned)((M + rows - 1) / rows), (unsigned)cg);
    if (relu == 2)
        bn_reduce_kernel<1, true><<<grid, 256, 0, st>>>(x, x_pixel_stride, g, g_pixel_stride, M, C, rows, scale, shift, mean,
                                                        invstd, S1, S2, relu, nullptr, 0);
    else
        bn_reduce_kernel<1><<<grid, 256, 0, st>>>(x, x_pixel_stride, g, g_pixel_stride, M, C, rows, scale, shift, mean, invstd,
                                                  S1, S2, relu, nullptr, 0);
    BTS_LAUNCH_CHECK();
    bn_bwd_coef_kernel<<<(C + 127) / 128, 128, 0, st>>>(S1, S2, M, C, scale, mean, invstd, coef);
    BTS_LAUNCH_CHECK();
    return 0;
}

// One-pass BatchNorm(+ReLU) backward into a concat gradient slab.  dx = [y>0]*scale*g + k1*x + k0 splits into a part that
// needs no reduction -- accumulated into `out` by the same pass that reduces S1, S2 -- and the per-channel affine remainder,
// which is linear in (k0, k1): K0/K1 (fp64, one entry per slab channel) collect it over every BatchNorm that reads the
// channel, and bts_bn_bwd_correct applies the total once, just before the channel's gradient is consumed.  One streaming
// pass over (x, g, out) per layer instead of reduce + apply.  K0 == NULL: frozen statistics (no remainder).
extern "C" int bts_bn_relu_bwd_fused(const float *x, long long x_pixel_stride, const float *g, long long g_pixel_stride,
                                     long long M, int C, const float *scale, const float *shift, const float *mean,
                                     const float *invstd, double *S1, double *S2, float *out, long long out_pixel_stride,
                                     double *K0, double *K1, void *stream) {
    if (!x || !g || !scale || !shift || !mean || !invstd || !S1 || !S2 || !out || M < 1 || C < 1) return BTS_EINVAL;
    if ((K0 == nullptr) != (K1 == nullptr)) return BTS_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e;
    if (S2 == S1 + C) {                         // the usual [2, C] tensor: one memset
        if ((e = cudaMemsetAsync(S1, 0, sizeof(double) * 2 * C, st)) != cudaSuccess) return (int)e;
    } else {
        if ((e = cudaMemsetAsync(S1, 0, sizeof(double) * C, st)) != cudaSuccess) return (int)e;
        if ((e = cudaMemsetAsync(S2, 0, sizeof(double) * C, st)) != cudaSuccess) return (int)e;
    }
    const int cg = (C + 255) / 256;
    const int rows = reduce_rows(M, cg);
    dim3 grid((unsigned)((M + rows - 1) / rows), (unsigned)cg);
    bn_reduce_kernel<2><<<grid, 256, 0, st>>>(x, x_pixel_stride, g, g_pixel_stride, M, C, rows, scale, shift, mean, invstd,
                                              S1, S2, 1, out, out_pixel_stride);
    BTS_LAUNCH_CHECK();
    if (K0) {
        bn_bwd_coef_accum_kernel<<<(C + 127) / 128, 128, 0, st>>>(S1, S2, M, C, scale, mean, invstd, K0, K1);
        BTS_LAUNCH_CHECK();
    }
    return 0;
}

extern "C" int bts_bn_bwd_correct(const float *x, long long x_pixel_stride, long long M, int C, const double *K0,
                                  const double *K1, float *out, long long out_pixel_stride, void *stream) {
    if (!x || !K0 || !K1 || !out || M < 1 || C < 1) return BTS_EINVAL;
    const long long total = M * ((C + 3) / 4);
    long long grid = (total + 255) / 256;
    const long long cap = (long long)bts_num_sms() * 16;
    if (grid > cap) grid = cap;
    bn_bwd_correct_kernel<<<(int)grid, 256, 0, (cudaStream_t)stream>>>(x, x_pixel_stride, M, C, K0, K1, out, out_pixel_stride);
    BTS_LAUNCH_CHECK();
    return 0;
}

// (k0, k1) coefficients of the backward apply pass from already-reduced sums (the reduction fused into a dgrad epilogue,
// bts_conv_fwd_bnbwd)
extern "C" int bts_bn_bwd_coef(const double *S1, const double *S2, long long M, int C, const float *scale, const float *mean,
                               const float *invstd, float *coef, void *stream) {
    if (!S1 || !S2 || !scale || !mean || !invstd || !coef || M < 1 || C < 1) return BTS_EINVAL;
    bn_bwd_coef_kernel<<<(C + 127) / 128, 128, 0, (cudaStream_t)stream>>>(S1, S2, M, C, scale, mean, invstd, coef);
    BTS_LAUNCH_CHECK();
    return 0;
}

extern "C" int bts_bn_relu_bwd_reduce(const float *x, long long x_pixel_stride, const float *g, long long g_pixel_stride,
                                      long long M, int C, const float *scale, const float *shift, const float *mean,
                                      const float *invstd, double *S1, double *S2, float *coef, void *stream) {
    return bts_bn_bwd_reduce(x, x_pixel_stride, g, g_pixel_stride, M, C, scale, shift, mean, invstd, 1, S1, S2, coef, stream);
}

extern "C" int bts_bn_bwd_apply(const float *x, long long x_pixel_stride, const float *g, long long g_pixel_stride,
                                long long M, int C, const float *scale, const float *shift, const float *coef, int relu,
                                float *out, long long out_pixel_stride, int accumulate, void *stream) {
    if (!x || !g || !scale || !shift || !out || M < 1 || C < 1) return BTS_EINVAL;
    const long long total = M * ((C + 3) / 4);
    long long grid = (total + 255) / 256;
    const long long cap = (long long)bts_num_sms() * 16;
    if (grid > cap) grid = cap;
    if (relu == 2)
        bn_relu_bwd_apply_kernel<true><<<(int)grid, 256, 0, (cudaStream_t)stream>>>(
            x, x_pixel_stride, g, g_pixel_stride, M, C, scale, shift, coef, out, out_pixel_stride, accumulate, relu);
    else
        bn_relu_bwd_apply_kernel<false><<<(int)grid, 256, 0, (cudaStream_t)stream>>>(
            x, x_pixel_stride, g, g_pixel_stride, M, C, scale, shift, coef, out, out_pixel_stride, accumulate, relu);
    BTS_LAUNCH_CHECK();
    return 0;
}

extern "C" int bts_bn_relu_bwd_apply(const float *x, long long x_pixel_stride, const float *g, long long g_pixel_stride,
                                     long long M, int C, const float *scale, const float *shift, const float *coef,
                                     float *out, long long out_pixel_stride, int accumulate, void *stream) {
    return bts_bn_bwd_apply(x, x_pixel_stride, g, g_pixel_stride, M, C, scale, shift, coef, 1, out, out_pixel_stride,
                            accumulate, stream);
}
