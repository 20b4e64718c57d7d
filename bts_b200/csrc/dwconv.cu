// Depthwise 3x3 convolution (padding 1, stride 1 or 2) of the MobileNetV2 inverted residuals (torchvision
// mobilenetv2.py, the `mobilenetv2_bts` encoder of reference pytorch/bts.py:298-300), fp32 NHWC, CUDA cores, HBM-bound.
//
// A depthwise conv has one input channel per output channel: no GEMM, 9 multiply-adds per output element, so these are
// streaming kernels.  Layout: lanes own float4 channel quads (a 256-thread block covers up to 256 channels; with fewer
// channels the spare threads take further rows), so a warp reads 512 contiguous bytes of a pixel row.  Each thread walks a
// run of RUN output columns and keeps the 3x3 window of its quad and the 36 weights in registers: per output column it
// loads one (stride 1) or two (stride 2) new input columns of the three rows; the row overlap between the threads of
// neighbouring output rows is served by L1 / L2.
//   fwd  : y = dw(act_in(x)), act_in(x) = clamp(x*scale + shift, 0, 6) when a prologue is given (the expand layer's
//          BN + ReLU6; out-of-bounds taps contribute 0, i.e. the padding applies to the ACTIVATED tensor).
//          Epilogue: none | per-block fp32 column sums (sum y, sum y^2) -> fp64 partials + a fixed-order second pass
//          (train-mode BatchNorm statistics, deterministic) | clamp(y*s + t, 0, 6) (the following eval-mode BN + ReLU6).
//   dgrad: gather form, each input pixel sums the taps that reach it (stride 1: the forward with flipped taps; stride 2:
//          only the taps of matching parity).  No atomics.
//   wgrad: dW[c,t] = sum_p g[p,c] * act_in(x)[p*stride + off_t, c]: 36 fp32 accumulators per thread, block partials in
//          fp64, then the same fixed-order second pass -- bit-reproducible from run to run.
// The weights are read from the (C,1,3,3) parameter on every call (no packed copy that could go stale after an update).
#include "common.cuh"

namespace {

constexpr int TPB = 256;
constexpr int RUN = 8;

struct Lanes {
    int c, rsub, rp;
    bool active;
};

// thread -> (channel quad, row group) for the channel chunk blockIdx.y (C % 4 == 0)
__device__ __forceinline__ Lanes lanes(int C) {
    const int tpc = min(256, C - (int)blockIdx.y * 256) >> 2;
    Lanes l;
    l.rp = TPB / tpc;
    l.rsub = (int)threadIdx.x / tpc;
    l.c = (int)blockIdx.y * 256 + ((int)threadIdx.x % tpc) * 4;
    l.active = l.rsub < l.rp;
    return l;
}

__device__ __forceinline__ float4 ld4(const float *p) { return __ldg(reinterpret_cast<const float4 *>(p)); }
__device__ __forceinline__ float relu6(float v) { return fminf(fmaxf(v, 0.f), 6.f); }
__device__ __forceinline__ float4 affine_relu6(float4 v, float4 s, float4 h) {
    return make_float4(relu6(fmaf(v.x, s.x, h.x)), relu6(fmaf(v.y, s.y, h.y)), relu6(fmaf(v.z, s.z, h.z)),
                       relu6(fmaf(v.w, s.w, h.w)));
}
__device__ __forceinline__ void fma4(float4 &acc, float4 a, float4 b) {
    acc.x = fmaf(a.x, b.x, acc.x); acc.y = fmaf(a.y, b.y, acc.y); acc.z = fmaf(a.z, b.z, acc.z); acc.w = fmaf(a.w, b.w, acc.w);
}
__device__ __forceinline__ float4 ld_vec(const float *p, int c) {
    return make_float4(__ldg(p + c), __ldg(p + c + 1), __ldg(p + c + 2), __ldg(p + c + 3));
}

// the 36 weights of channels c..c+3 (tap-major float4s); FLIP reverses the taps (stride-1 dgrad = correlation with them)
template <bool FLIP>
__device__ __forceinline__ void load_taps(const float *__restrict__ w, int c, float4 (&wt)[9]) {
#pragma unroll
    for (int k = 0; k < 9; ++k) {
        const int t = FLIP ? 8 - k : k;
        wt[k] = make_float4(__ldg(w + c * 9 + t), __ldg(w + (c + 1) * 9 + t), __ldg(w + (c + 2) * 9 + t),
                            __ldg(w + (c + 3) * 9 + t));
    }
}

// work items = (image, row, run of RUN columns); block x takes a contiguous range, its row groups stride through it
struct Items {
    long long i0, i1;
    int nruns, rows;
};
__device__ __forceinline__ Items items_of(int B, int rows, int cols) {
    Items r;
    r.nruns = (cols + RUN - 1) / RUN;
    r.rows = rows;
    const long long n = (long long)B * rows * r.nruns;
    const long long per = (n + gridDim.x - 1) / gridDim.x;
    r.i0 = (long long)blockIdx.x * per;
    r.i1 = min(n, r.i0 + per);
    return r;
}

// The input window of output row `oy`: three input rows (oy*S - 1 .. oy*S + 1), out-of-bounds taps are zero.
template <int S, bool PRE>
struct Window {
    const float *row[3];
    bool ok[3];
    int W;
    long long xs;
    float4 sc, sh;
    __device__ __forceinline__ float4 load(int r, int ix) const {
        if (!ok[r] || ix < 0 || ix >= W) return make_float4(0.f, 0.f, 0.f, 0.f);
        const float4 v = ld4(row[r] + (long long)ix * xs);
        return PRE ? affine_relu6(v, sc, sh) : v;
    }
};

template <int S, bool PRE>
__device__ __forceinline__ Window<S, PRE> window_at(const float *x, long long xs, int H, int W, long long b, int oy, int c,
                                                   float4 sc, float4 sh) {
    Window<S, PRE> win;
    win.W = W;
    win.xs = xs;
    win.sc = sc;
    win.sh = sh;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const int iy = oy * S - 1 + r;
        win.ok[r] = iy >= 0 && iy < H;
        win.row[r] = x + ((b * H + (win.ok[r] ? iy : 0)) * (long long)W) * xs + c;
    }
    return win;
}

// Forward (and, with FLIP and S == 1, the stride-1 dgrad); minimum 1 block/SM lets the window + taps stay in registers.  EPI 0: y; 1: y + statistics partials; 2: clamp(y*qs + qh, 0, 6)
template <int S, bool PRE, int EPI, bool FLIP>
__global__ void __launch_bounds__(TPB, 1) dw_fwd_kernel(const float *__restrict__ x, long long xs, int B, int H, int W,
                                                        int C, int Ho, int Wo, const float *__restrict__ w,
                                                        const float *__restrict__ ps, const float *__restrict__ ph,
                                                        const float *__restrict__ qs, const float *__restrict__ qh,
                                                        float *__restrict__ y, long long ys, double *__restrict__ part) {
    const Lanes l = lanes(C);
    float4 s1 = make_float4(0.f, 0.f, 0.f, 0.f), s2 = s1;
    if (l.active) {
        float4 wt[9];
        load_taps<FLIP>(w, l.c, wt);
        const float4 sc = PRE ? ld_vec(ps, l.c) : s1, sh = PRE ? ld_vec(ph, l.c) : s1;
        const float4 osc = EPI == 2 ? ld_vec(qs, l.c) : s1, osh = EPI == 2 ? ld_vec(qh, l.c) : s1;
        const Items it = items_of(B, Ho, Wo);
        for (long long i = it.i0 + l.rsub; i < it.i1; i += l.rp) {
            const int run = (int)(i % it.nruns);
            const long long q = i / it.nruns;
            const int oy = (int)(q % Ho);
            const long long b = q / Ho;
            const Window<S, PRE> win = window_at<S, PRE>(x, xs, H, W, b, oy, l.c, sc, sh);
            const int ox0 = run * RUN;
            float4 cur[3][3];
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                cur[r][0] = win.load(r, ox0 * S - 1);
                if (S == 1) cur[r][1] = win.load(r, ox0);
            }
            float *yrow = y + ((b * Ho + oy) * (long long)Wo) * ys + l.c;
#pragma unroll
            for (int j = 0; j < RUN; ++j) {
                const int ox = ox0 + j;
                if (ox >= Wo) break;
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    if (S == 2) cur[r][1] = win.load(r, ox * 2);
                    cur[r][2] = win.load(r, ox * S + 1);
                }
                float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int r = 0; r < 3; ++r)
#pragma unroll
                    for (int k = 0; k < 3; ++k) fma4(acc, cur[r][k], wt[r * 3 + k]);
                if (EPI == 1) {
                    s1.x += acc.x; s1.y += acc.y; s1.z += acc.z; s1.w += acc.w;
                    s2.x = fmaf(acc.x, acc.x, s2.x); s2.y = fmaf(acc.y, acc.y, s2.y);
                    s2.z = fmaf(acc.z, acc.z, s2.z); s2.w = fmaf(acc.w, acc.w, s2.w);
                }
                if (EPI == 2) acc = affine_relu6(acc, osc, osh);
                *reinterpret_cast<float4 *>(yrow + (long long)ox * ys) = acc;
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    if (S == 1) { cur[r][0] = cur[r][1]; cur[r][1] = cur[r][2]; }
                    else cur[r][0] = cur[r][2];
                }
            }
        }
    }
    if (EPI == 1) {
        // combine the row groups of the block in a fixed order, one fp64 partial per (block, channel)
        __shared__ float red[2][TPB * 4];
        const float a0[4] = {s1.x, s1.y, s1.z, s1.w}, a1[4] = {s2.x, s2.y, s2.z, s2.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            red[0][threadIdx.x * 4 + e] = a0[e];
            red[1][threadIdx.x * 4 + e] = a1[e];
        }
        __syncthreads();
        const int tpc = min(256, C - (int)blockIdx.y * 256) >> 2;
        for (int o = threadIdx.x; o < 2 * tpc * 4; o += TPB) {
            const int k = o / (tpc * 4), ce = o % (tpc * 4);
            double s = 0.0;
            for (int r = 0; r < l.rp; ++r) s += (double)red[k][r * tpc * 4 + ce];
            part[((long long)blockIdx.x * 2 + k) * C + blockIdx.y * 256 + ce] = s;
        }
    }
}

// stride-2 dgrad: gx[iy, ix] = sum over the taps (ky, kx) with iy + 1 - ky and ix + 1 - kx even of g[oy, ox] * w[ky, kx]
__global__ void __launch_bounds__(TPB) dw_dgrad_s2_kernel(const float *__restrict__ g, long long gs, int B, int H, int W, int C,
                                                          int Ho, int Wo, const float *__restrict__ w,
                                                          float *__restrict__ gx, long long gxs) {
    const Lanes l = lanes(C);
    if (!l.active) return;
    float4 wt[9];
    load_taps<false>(w, l.c, wt);
    const Items it = items_of(B, H, W);
    for (long long i = it.i0 + l.rsub; i < it.i1; i += l.rp) {
        const int run = (int)(i % it.nruns);
        const long long q = i / it.nruns;
        const int iy = (int)(q % H);
        const long long b = q / H;
        float *orow = gx + ((b * H + iy) * (long long)W) * gxs + l.c;
#pragma unroll
        for (int j = 0; j < RUN; ++j) {
            const int ix = run * RUN + j;
            if (ix >= W) break;
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int ky = 0; ky < 3; ++ky) {
                const int ty = iy + 1 - ky;
                if ((ty & 1) || ty < 0 || (ty >> 1) >= Ho) continue;
                const float *grow = g + ((b * Ho + (ty >> 1)) * (long long)Wo) * gs + l.c;
#pragma unroll
                for (int kx = 0; kx < 3; ++kx) {
                    const int tx = ix + 1 - kx;
                    if ((tx & 1) || tx < 0 || (tx >> 1) >= Wo) continue;
                    fma4(acc, ld4(grow + (long long)(tx >> 1) * gs), wt[ky * 3 + kx]);
                }
            }
            *reinterpret_cast<float4 *>(orow + (long long)ix * gxs) = acc;
        }
    }
}

// wgrad partials: part[block][tap][c] = sum over the block's output pixels of g * act_in(x) at that tap
template <int S, bool PRE>
__global__ void __launch_bounds__(TPB) dw_wgrad_kernel(const float *__restrict__ x, long long xs, int B, int H, int W, int C,
                                                       int Ho, int Wo, const float *__restrict__ ps,
                                                       const float *__restrict__ ph, const float *__restrict__ g,
                                                       long long gs, double *__restrict__ part) {
    __shared__ float red[TPB * 36];
    const Lanes l = lanes(C);
    float4 acc[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) acc[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (l.active) {
        const float4 z = acc[0];
        const float4 sc = PRE ? ld_vec(ps, l.c) : z, sh = PRE ? ld_vec(ph, l.c) : z;
        const Items it = items_of(B, Ho, Wo);
        for (long long i = it.i0 + l.rsub; i < it.i1; i += l.rp) {
            const int run = (int)(i % it.nruns);
            const long long q = i / it.nruns;
            const int oy = (int)(q % Ho);
            const long long b = q / Ho;
            const Window<S, PRE> win = window_at<S, PRE>(x, xs, H, W, b, oy, l.c, sc, sh);
            const int ox0 = run * RUN;
            float4 cur[3][3];
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                cur[r][0] = win.load(r, ox0 * S - 1);
                if (S == 1) cur[r][1] = win.load(r, ox0);
            }
            const float *grow = g + ((b * Ho + oy) * (long long)Wo) * gs + l.c;
#pragma unroll
            for (int j = 0; j < RUN; ++j) {
                const int ox = ox0 + j;
                if (ox >= Wo) break;
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    if (S == 2) cur[r][1] = win.load(r, ox * 2);
                    cur[r][2] = win.load(r, ox * S + 1);
                }
                const float4 gv = ld4(grow + (long long)ox * gs);
#pragma unroll
                for (int r = 0; r < 3; ++r)
#pragma unroll
                    for (int k = 0; k < 3; ++k) fma4(acc[r * 3 + k], cur[r][k], gv);
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    if (S == 1) { cur[r][0] = cur[r][1]; cur[r][1] = cur[r][2]; }
                    else cur[r][0] = cur[r][2];
                }
            }
        }
    }
#pragma unroll
    for (int k = 0; k < 9; ++k) {
        red[threadIdx.x * 36 + k * 4 + 0] = acc[k].x;
        red[threadIdx.x * 36 + k * 4 + 1] = acc[k].y;
        red[threadIdx.x * 36 + k * 4 + 2] = acc[k].z;
        red[threadIdx.x * 36 + k * 4 + 3] = acc[k].w;
    }
    __syncthreads();
    const int tpc = min(256, C - (int)blockIdx.y * 256) >> 2;
    for (int o = threadIdx.x; o < 9 * tpc * 4; o += TPB) {
        const int k = o / (tpc * 4), ce = o % (tpc * 4), tq = ce >> 2, e = ce & 3;
        double s = 0.0;
        for (int r = 0; r < l.rp; ++r) s += (double)red[(r * tpc + tq) * 36 + k * 4 + e];
        part[((long long)blockIdx.x * 9 + k) * C + blockIdx.y * 256 + ce] = s;
    }
}

// second pass: out[k][c] = sum over blocks of part[block][k][c] -> fp64 sums or the fp32 weight gradient.  One warp per
// entry: lane l sums blocks l, l+32, ... in order, then a fixed shuffle tree -- the same order on every run.
__global__ void __launch_bounds__(256) dw_part_reduce_kernel(const double *__restrict__ part, int nblk, int K, int C,
                                                             double *__restrict__ sums, float *__restrict__ dw, long long s0,
                                                             long long s2, long long s3) {
    const int o = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (o >= K * C) return;
    double s = 0.0;
    for (int b = lane; b < nblk; b += 32) s += part[(long long)b * K * C + o];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
    if (lane) return;
    if (sums) {
        sums[o] = s;
    } else {
        const int k = o / C, c = o % C;
        dw[c * s0 + (k / 3) * s2 + (k % 3) * s3] = (float)s;
    }
}

// blocks along the pixel dimension: `per_sm` per SM over the channel chunks, at most one item per row group
int dw_blocks(int B, int rows, int cols, int C, int per_sm) {
    const int cg = (C + 255) / 256;
    const int rp = TPB / (min(C, 256) / 4);
    const long long items = (long long)B * rows * ((cols + RUN - 1) / RUN);
    long long n = (long long)bts_num_sms() * per_sm / cg;
    const long long cap = (items + rp - 1) / rp;
    if (n > cap) n = cap;
    if (n < 1) n = 1;
    return (int)n;
}

constexpr int FWD_PER_SM = 8;
constexpr int WGRAD_PER_SM = 4;

bool dw_shape_ok(int B, int H, int W, int C, int stride) {
    return B >= 1 && H >= 1 && W >= 1 && C >= 4 && (C & 3) == 0 && (stride == 1 || stride == 2);
}
bool vec_ok(const void *p, long long s) { return p && bts_aligned16(p) && (s & 3) == 0; }

template <int S, bool PRE, int EPI, bool FLIP>
void launch_fwd(dim3 grid, cudaStream_t st, const float *x, long long xs, int B, int H, int W, int C, int Ho, int Wo,
                const float *w, const float *ps, const float *ph, const float *qs, const float *qh, float *y, long long ys,
                double *part) {
    dw_fwd_kernel<S, PRE, EPI, FLIP><<<grid, TPB, 0, st>>>(x, xs, B, H, W, C, Ho, Wo, w, ps, ph, qs, qh, y, ys, part);
}

template <int S>
void launch_fwd_s(dim3 grid, cudaStream_t st, bool pre, int epi, const float *x, long long xs, int B, int H, int W, int C,
                  int Ho, int Wo, const float *w, const float *ps, const float *ph, const float *qs, const float *qh, float *y,
                  long long ys, double *part) {
#define BTS_DW_FWD(P, E) launch_fwd<S, P, E, false>(grid, st, x, xs, B, H, W, C, Ho, Wo, w, ps, ph, qs, qh, y, ys, part)
    if (pre) {
        if (epi == 0) BTS_DW_FWD(true, 0); else if (epi == 1) BTS_DW_FWD(true, 1); else BTS_DW_FWD(true, 2);
    } else {
        if (epi == 0) BTS_DW_FWD(false, 0); else if (epi == 1) BTS_DW_FWD(false, 1); else BTS_DW_FWD(false, 2);
    }
#undef BTS_DW_FWD
}

}  // namespace

extern "C" long long bts_dw_partials(int B, int Hout, int Wout, int C, int wgrad) {
    if (B < 1 || Hout < 1 || Wout < 1 || C < 4 || (C & 3)) return -1;
    return (long long)dw_blocks(B, Hout, Wout, C, wgrad ? WGRAD_PER_SM : FWD_PER_SM) * (wgrad ? 9 : 2) * C;
}

extern "C" int bts_dw_fwd(const float *x, long long x_pixel_stride, int B, int H, int W, int C, int stride, const float *w,
                          const float *pre_scale, const float *pre_shift, const float *post_scale, const float *post_shift,
                          float *y, long long y_pixel_stride, double *partials, double *sums, void *stream) {
    if (!x || !w || !y || !dw_shape_ok(B, H, W, C, stride)) return BTS_EINVAL;
    if ((pre_scale == nullptr) != (pre_shift == nullptr) || (post_scale == nullptr) != (post_shift == nullptr) ||
        (partials == nullptr) != (sums == nullptr) || (post_scale && sums))
        return BTS_EINVAL;
    if (!vec_ok(x, x_pixel_stride) || !vec_ok(y, y_pixel_stride)) return BTS_EALIGN;
    const int Ho = (H - 1) / stride + 1, Wo = (W - 1) / stride + 1;
    const int epi = sums ? 1 : (post_scale ? 2 : 0);
    const dim3 grid(dw_blocks(B, Ho, Wo, C, FWD_PER_SM), (C + 255) / 256);
    cudaStream_t st = (cudaStream_t)stream;
    if (stride == 1)
        launch_fwd_s<1>(grid, st, pre_scale != nullptr, epi, x, x_pixel_stride, B, H, W, C, Ho, Wo, w, pre_scale, pre_shift,
                        post_scale, post_shift, y, y_pixel_stride, partials);
    else
        launch_fwd_s<2>(grid, st, pre_scale != nullptr, epi, x, x_pixel_stride, B, H, W, C, Ho, Wo, w, pre_scale, pre_shift,
                        post_scale, post_shift, y, y_pixel_stride, partials);
    BTS_LAUNCH_CHECK();
    if (sums) {
        dw_part_reduce_kernel<<<(2 * C + 7) / 8, 256, 0, st>>>(partials, (int)grid.x, 2, C, sums, nullptr, 0, 0, 0);
        BTS_LAUNCH_CHECK();
    }
    return 0;
}

extern "C" int bts_dw_dgrad(const float *g, long long g_pixel_stride, int B, int H, int W, int C, int stride, const float *w,
                            float *gx, long long gx_pixel_stride, void *stream) {
    if (!g || !w || !gx || !dw_shape_ok(B, H, W, C, stride)) return BTS_EINVAL;
    if (!vec_ok(g, g_pixel_stride) || !vec_ok(gx, gx_pixel_stride)) return BTS_EALIGN;
    const int Ho = (H - 1) / stride + 1, Wo = (W - 1) / stride + 1;
    const dim3 grid(dw_blocks(B, H, W, C, FWD_PER_SM), (C + 255) / 256);
    cudaStream_t st = (cudaStream_t)stream;
    if (stride == 1)   // gx = correlation of g with the flipped taps: the forward kernel over the same geometry
        dw_fwd_kernel<1, false, 0, true><<<grid, TPB, 0, st>>>(g, g_pixel_stride, B, H, W, C, H, W, w, nullptr, nullptr,
                                                               nullptr, nullptr, gx, gx_pixel_stride, nullptr);
    else
        dw_dgrad_s2_kernel<<<grid, TPB, 0, st>>>(g, g_pixel_stride, B, H, W, C, Ho, Wo, w, gx, gx_pixel_stride);
    BTS_LAUNCH_CHECK();
    return 0;
}

extern "C" int bts_dw_wgrad(const float *x, long long x_pixel_stride, int B, int H, int W, int C, int stride,
                            const float *pre_scale, const float *pre_shift, const float *g, long long g_pixel_stride,
                            double *partials, float *dw, long long s_c, long long s_kh, long long s_kw, void *stream) {
    if (!x || !g || !partials || !dw || !dw_shape_ok(B, H, W, C, stride)) return BTS_EINVAL;
    if ((pre_scale == nullptr) != (pre_shift == nullptr)) return BTS_EINVAL;
    if (!vec_ok(x, x_pixel_stride) || !vec_ok(g, g_pixel_stride)) return BTS_EALIGN;
    const int Ho = (H - 1) / stride + 1, Wo = (W - 1) / stride + 1;
    const dim3 grid(dw_blocks(B, Ho, Wo, C, WGRAD_PER_SM), (C + 255) / 256);
    cudaStream_t st = (cudaStream_t)stream;
    const bool pre = pre_scale != nullptr;
#define BTS_DW_WG(S, P) \
    dw_wgrad_kernel<S, P><<<grid, TPB, 0, st>>>(x, x_pixel_stride, B, H, W, C, Ho, Wo, pre_scale, pre_shift, g, g_pixel_stride, partials)
    if (stride == 1) { if (pre) BTS_DW_WG(1, true); else BTS_DW_WG(1, false); }
    else { if (pre) BTS_DW_WG(2, true); else BTS_DW_WG(2, false); }
#undef BTS_DW_WG
    BTS_LAUNCH_CHECK();
    dw_part_reduce_kernel<<<(9 * C + 7) / 8, 256, 0, st>>>(partials, (int)grid.x, 9, C, nullptr, dw, s_c, s_kh, s_kw);
    BTS_LAUNCH_CHECK();
    return 0;
}
