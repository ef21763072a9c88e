// Q-learning update path of the bi-head pointer model for sm_100a (include/ofb_train.h):
// Trainer.replay's targets and model.fit = one Adam step on mse(output1) + mse(output2) with BatchNormalization in
// training mode (reference: agents/qlearnIA_V2.py:123-190 model, :237-287 replay / fit; Keras defaults of SURVEY.md
// Appendix B).  fp32 NHWC activations, fp64 accumulation of every sum over the batch.  The batch is tiny (8 samples,
// 3.7 GFLOP per step), so these are plain CUDA-core kernels: one thread per output element, weights in shared memory.
#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <string.h>
#include "../../include/ofb.h"
#include "../../include/ofb_train.h"

void ofb_set_error(const char *fmt, ...);
#define TR_CHECK(expr)                                                                    \
    do {                                                                                  \
        cudaError_t e__ = (expr);                                                         \
        if (e__ != cudaSuccess) {                                                         \
            ofb_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
            return OFB_E_CUDA;                                                            \
        }                                                                                 \
    } while (0)

#define IMG 400
#define MAP_WORDS 5000

// ---------------------------------------------------------------------------------------------- parameter table
struct Ref { int off, n; };
struct ConvP { Ref k, b, g, be, m, v; int cin, cout, bn; };
struct DenseP { Ref k, b; int fin, fout; };
struct Table {
    ConvP conv[4], up[4];
    DenseP d1, d2, o1, ud;
    int total;
};

static Table make_table() {
    Table t;
    int off = 0;
    auto take = [&](int n) { Ref r = {off, n}; off += n; return r; };
    auto conv = [&](ConvP &c, int cin, int cout, int bn) {
        c.cin = cin; c.cout = cout; c.bn = bn;
        c.k = take(9 * cin * cout); c.b = take(cout);
        if (bn) { c.g = take(cout); c.be = take(cout); c.m = take(cout); c.v = take(cout); }
        else c.g = c.be = c.m = c.v = Ref{0, 0};
    };
    auto dense = [&](DenseP &d, int fin, int fout) { d.fin = fin; d.fout = fout; d.k = take(fin * fout); d.b = take(fout); };
    const int tc[4][2] = {{2, 8}, {8, 8}, {8, 8}, {8, 8}}, uc[4][2] = {{1, 2}, {2, 4}, {4, 8}, {8, 1}};
    for (int i = 0; i < 4; i++) conv(t.conv[i], tc[i][0], tc[i][1], 1);
    dense(t.d1, 5008, 100); dense(t.d2, 100, 50); dense(t.o1, 50, 2); dense(t.ud, 100, 625);
    for (int i = 0; i < 4; i++) conv(t.up[i], uc[i][0], uc[i][1], i < 3);
    t.total = off;
    return t;
}

struct ofb_trainer {
    ofb_train_config cfg;
    Table tab;
    int device;
    int64_t steps;
    float *params, *grads, *adam_m, *adam_v;     // [total]
    uint8_t *trainable;                          // [total]: 0 for the BN moving statistics
    // activations (max_batch samples)
    float *x0;                                   // [B,400,400,2]
    float *y[4], *p[4];                          // conv output (pre-BN) [B,H,W,8], pooled [B,H/2,W/2,8]
    float *cat, *h1, *d2, *act, *u0;             // [B,5008] [B,100] [B,50] [B,2] [B,625]
    float *a[4], *yu[4];                         // upsampled input [B,h,w,cin], conv output (pre-BN) [B,h,w,cout]; yu[3] = ptr
    float *bn_mean, *bn_var;                     // [7][8] batch statistics (trunk 0-3, up 4-6)
    double *sums;                                // [7][2][8] scratch: per-channel sums (forward: x, x^2; backward: dz, dz * xhat)
    double *loss_acc;                            // [2]
    float *g0, *g1;                              // [B,400,400,8] gradient ping-pong
    float *gu, *dh1, *dd2, *dact, *dcat;         // [B,625] [B,100] [B,50] [B,2] [B,5008]
    // the buffers every entry point uses: the handle's own (fs = bs = sums, la = loss_acc, gr = grads) or, after
    // ofb_trainer_set_exchange, the caller's exchange buffers (forward sums, loss accumulators, backward sums, gradients)
    double *fs, *la, *bs;
    float *gr;
    ofb_reduce_fn reducer;
    void *reducer_ctx;
};

// ---------------------------------------------------------------------------------------------- small helpers
__device__ __forceinline__ double warp_sum(double v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
// block-wide sums of up to 16 doubles per thread -> atomicAdd to dst (blockDim.x <= 1024)
template <int NV>
__device__ __forceinline__ void block_accumulate(const double (&v)[NV], double *dst, int n_valid) {
    __shared__ double red[32][NV];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int j = 0; j < NV; j++) {
        const double s = warp_sum(v[j]);
        if (lane == 0) red[warp][j] = s;
    }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
        for (int j = 0; j < NV; j++) {
            double s = lane < nw ? red[lane][j] : 0.0;
            s = warp_sum(s);
            if (lane == 0 && j < n_valid) atomicAdd(&dst[j], s);
        }
    }
    __syncthreads();
}

// N consecutive floats of one pixel: 16-byte accesses when the channel count allows (pixels are N * 4-byte aligned)
template <int N>
__device__ __forceinline__ void load_vec(const float *__restrict__ p, float (&v)[N]) {
    if constexpr (N % 4 == 0) {
#pragma unroll
        for (int j = 0; j < N / 4; j++) {
            const float4 t = reinterpret_cast<const float4 *>(p)[j];
            v[4 * j] = t.x; v[4 * j + 1] = t.y; v[4 * j + 2] = t.z; v[4 * j + 3] = t.w;
        }
    } else if constexpr (N == 2) {
        const float2 t = *reinterpret_cast<const float2 *>(p);
        v[0] = t.x; v[1] = t.y;
    } else {
#pragma unroll
        for (int j = 0; j < N; j++) v[j] = p[j];
    }
}
template <int N>
__device__ __forceinline__ void store_vec(float *__restrict__ p, const float (&v)[N]) {
    if constexpr (N % 4 == 0) {
#pragma unroll
        for (int j = 0; j < N / 4; j++) reinterpret_cast<float4 *>(p)[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
    } else if constexpr (N == 2) {
        *reinterpret_cast<float2 *>(p) = make_float2(v[0], v[1]);
    } else {
#pragma unroll
        for (int j = 0; j < N; j++) p[j] = v[j];
    }
}

// ---------------------------------------------------------------------------------------------- forward kernels
__global__ void k_tr_unpack(const uint32_t *__restrict__ bits, float *__restrict__ x0, long long n_px_total) {
    // x0[b, y, x, c] = bit (y*400 + x) of bits[b, c]
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_px_total; i += (long long)gridDim.x * blockDim.x) {
        const long long b = i / (IMG * IMG);
        const int px = (int)(i % (IMG * IMG));
        const uint32_t s = bits[(b * 2 + 0) * MAP_WORDS + (px >> 5)] >> (px & 31), l = bits[(b * 2 + 1) * MAP_WORDS + (px >> 5)] >> (px & 31);
        reinterpret_cast<float2 *>(x0)[i] = make_float2((float)(s & 1u), (float)(l & 1u));
    }
}

// Conv2D 3x3 'same' + bias, NHWC, kernel HWIO.  One thread per output pixel, all COUT channels.
template <int CIN, int COUT>
__global__ void k_tr_conv_fwd(const float *__restrict__ x, const float *__restrict__ w, const float *__restrict__ bias,
                              float *__restrict__ y, int B, int H, int W) {
    __shared__ float ws[9 * CIN * COUT + COUT];
    for (int i = threadIdx.x; i < 9 * CIN * COUT; i += blockDim.x) ws[i] = w[i];
    for (int i = threadIdx.x; i < COUT; i += blockDim.x) ws[9 * CIN * COUT + i] = bias[i];
    __syncthreads();
    const long long n = (long long)B * H * W;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int xx = (int)(i % W), yy = (int)((i / W) % H);
        const long long b = i / ((long long)W * H);
        float acc[COUT], xv[9][CIN];
#pragma unroll
        for (int co = 0; co < COUT; co++) acc[co] = ws[9 * CIN * COUT + co];
        // all nine taps are loaded (zeros outside the image) before the first multiply, so their latencies overlap
#pragma unroll
        for (int ky = 0; ky < 3; ky++) {
#pragma unroll
            for (int kx = 0; kx < 3; kx++) {
                const int sy = yy + ky - 1, sx = xx + kx - 1;
                if (sy >= 0 && sy < H && sx >= 0 && sx < W) load_vec<CIN>(x + ((b * H + sy) * W + sx) * CIN, xv[ky * 3 + kx]);
                else {
#pragma unroll
                    for (int ci = 0; ci < CIN; ci++) xv[ky * 3 + kx][ci] = 0.0f;
                }
            }
        }
#pragma unroll
        for (int tp = 0; tp < 9; tp++) {
#pragma unroll
            for (int ci = 0; ci < CIN; ci++) {
#pragma unroll
                for (int co = 0; co < COUT; co++) acc[co] = fmaf(xv[tp][ci], ws[(tp * CIN + ci) * COUT + co], acc[co]);
            }
        }
        store_vec<COUT>(y + i * COUT, acc);
    }
}

// per-channel sum and sum of squares of y [n_px, C] -> sums[0..C) , sums[8..8+C)
__global__ void k_tr_chan_sums(const float *__restrict__ y, long long n_px, int C, double *__restrict__ sums) {
    double v[16];
#pragma unroll
    for (int j = 0; j < 16; j++) v[j] = 0.0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_px; i += (long long)gridDim.x * blockDim.x) {
#pragma unroll
        for (int c = 0; c < 8; c++) {                    // fixed trip count: the accumulators stay in registers
            if (c < C) {
                const double t = (double)y[i * C + c];
                v[c] += t;
                v[8 + c] += t * t;
            }
        }
    }
    block_accumulate<16>(v, sums, 16);
}
// batch mean / biased variance from the sums; moving averages updated (BatchNormalization in training mode)
__global__ void k_tr_bn_finalize(const double *__restrict__ sums, long long n_px, int C, float *__restrict__ mean, float *__restrict__ var,
                                 float *__restrict__ mov_mean, float *__restrict__ mov_var, float momentum, int unbiased, int update) {
    const int c = threadIdx.x;
    if (c >= C) return;
    const double m = sums[c] / (double)n_px;
    double v = sums[8 + c] / (double)n_px - m * m;
    if (v < 0.0) v = 0.0;
    mean[c] = (float)m;
    var[c] = (float)v;
    if (update) {
        const double vu = unbiased && n_px > 1 ? v * (double)n_px / (double)(n_px - 1) : v;
        mov_mean[c] = mov_mean[c] * momentum + (float)m * (1.0f - momentum);
        mov_var[c] = mov_var[c] * momentum + (float)vu * (1.0f - momentum);
    }
}

__device__ __forceinline__ float bn_relu(float y, float mean, float rstd, float gamma, float beta) {
    return fmaxf(fmaf((y - mean) * rstd, gamma, beta), 0.0f);
}
// index (0..3, row-major in the window) of the first maximum of relu(bn(.)) over a 2x2 window, and that maximum
__device__ __forceinline__ int pool_argmax(const float *__restrict__ y, long long base, int W, int C, int c, float mean, float rstd,
                                           float gamma, float beta, float &zmax) {
    const float z0 = bn_relu(y[base + c], mean, rstd, gamma, beta), z1 = bn_relu(y[base + C + c], mean, rstd, gamma, beta);
    const float z2 = bn_relu(y[base + (long long)W * C + c], mean, rstd, gamma, beta);
    const float z3 = bn_relu(y[base + (long long)W * C + C + c], mean, rstd, gamma, beta);
    int k = 0;
    zmax = z0;
    if (z1 > zmax) { zmax = z1; k = 1; }
    if (z2 > zmax) { zmax = z2; k = 2; }
    if (z3 > zmax) { zmax = z3; k = 3; }
    return k;
}

// p[b, yo, xo, c] = max over the 2x2 window of relu(bn(y));  out may be strided per sample (the flatten -> concat slot)
__global__ void k_tr_bn_relu_pool(const float *__restrict__ y, const float *__restrict__ mean, const float *__restrict__ var,
                                  const float *__restrict__ gamma, const float *__restrict__ beta, float eps, float *__restrict__ p,
                                  int B, int H, int W, int C) {
    const int Ho = H / 2, Wo = W / 2;
    const long long n = (long long)B * Ho * Wo * C;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(i % C), xo = (int)((i / C) % Wo), yo = (int)((i / ((long long)C * Wo)) % Ho);
        const long long b = i / ((long long)C * Wo * Ho);
        const long long base = ((b * H + 2 * yo) * W + 2 * xo) * C;
        float zmax;
        pool_argmax(y, base, W, C, c, mean[c], rsqrtf(var[c] + eps), gamma[c], beta[c], zmax);
        p[i] = zmax;
    }
}

// The 2 x 2 source pixels and weights of output pixel (Y, X) of a bilinear x2 (TF2 half-pixel centres, edge clamp):
// Y = 2i: rows i-1 (1/4), i (3/4);  Y = 2i+1: rows i (3/4), i+1 (1/4); clamped to the image
struct UpTap { int ia, ib, ja, jb; float wy, wx; };
__device__ __forceinline__ UpTap up_tap(int Y, int X, int h, int w) {
    UpTap t;
    t.ia = (Y & 1) ? (Y >> 1) : max((Y >> 1) - 1, 0);
    t.ib = (Y & 1) ? min((Y >> 1) + 1, h - 1) : (Y >> 1);
    t.wy = (Y & 1) ? 0.75f : 0.25f;
    t.ja = (X & 1) ? (X >> 1) : max((X >> 1) - 1, 0);
    t.jb = (X & 1) ? min((X >> 1) + 1, w - 1) : (X >> 1);
    t.wx = (X & 1) ? 0.75f : 0.25f;
    return t;
}
// a[b, Y, X, :] = bilinear x2 of relu(bn(src)) (or of src itself when mean == NULL); one thread per output pixel
template <int C>
__global__ void k_tr_upsample(const float *__restrict__ src, const float *__restrict__ mean, const float *__restrict__ var,
                              const float *__restrict__ gamma, const float *__restrict__ beta, float eps, float *__restrict__ a,
                              int B, int h, int w) {
    const int H = 2 * h, W = 2 * w;
    const long long n = (long long)B * H * W;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int X = (int)(i % W), Y = (int)((i / W) % H);
        const long long b = i / ((long long)W * H);
        const UpTap t = up_tap(Y, X, h, w);
        float v00[C], v01[C], v10[C], v11[C], o[C];
        load_vec<C>(src + ((b * h + t.ia) * w + t.ja) * C, v00);
        load_vec<C>(src + ((b * h + t.ia) * w + t.jb) * C, v01);
        load_vec<C>(src + ((b * h + t.ib) * w + t.ja) * C, v10);
        load_vec<C>(src + ((b * h + t.ib) * w + t.jb) * C, v11);
#pragma unroll
        for (int c = 0; c < C; c++) {
            float p00 = v00[c], p01 = v01[c], p10 = v10[c], p11 = v11[c];
            if (mean) {
                const float m = mean[c], r = rsqrtf(var[c] + eps), g = gamma[c], be = beta[c];
                p00 = bn_relu(p00, m, r, g, be); p01 = bn_relu(p01, m, r, g, be);
                p10 = bn_relu(p10, m, r, g, be); p11 = bn_relu(p11, m, r, g, be);
            }
            const float top = p00 * t.wx + p01 * (1.0f - t.wx), bot = p10 * t.wx + p11 * (1.0f - t.wx);
            o[c] = top * t.wy + bot * (1.0f - t.wy);
        }
        store_vec<C>(a + i * C, o);
    }
}

// y[b, o] = act(sum_i x[b, i] * W[i, o] + bias[o]);  one thread per (b, o).  Like every element-wise kernel here it strides
// over the grid: blocks_for caps the grid, so a thread may own several elements at large B.
__global__ void k_tr_dense_fwd(const float *__restrict__ x, const float *__restrict__ W, const float *__restrict__ bias,
                               float *__restrict__ y, int B, int fin, int fout, int relu) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < (long long)B * fout; i += (long long)gridDim.x * blockDim.x) {
        const int b = (int)(i / fout), o = (int)(i % fout);
        float acc = bias[o];
        const float *xp = x + (long long)b * fin;
        for (int k = 0; k < fin; k++) acc = fmaf(xp[k], W[(long long)k * fout + o], acc);
        y[i] = relu ? fmaxf(acc, 0.0f) : acc;
    }
}
// the same for a long reduction (dense1: 5008 inputs): grid (slices, B), thread o sums its slice of k and adds it to y, which
// k_tr_bias_fill initialised with the bias; k_tr_relu applies the activation afterwards
__global__ void k_tr_dense_fwd_splitk(const float *__restrict__ x, const float *__restrict__ W, float *__restrict__ y, int fin, int fout) {
    const int o = threadIdx.x, b = blockIdx.y;
    const int per = (fin + gridDim.x - 1) / gridDim.x, k0 = blockIdx.x * per, k1 = min(fin, k0 + per);
    if (o >= fout) return;
    const float *xp = x + (long long)b * fin;
    float acc = 0.0f;
    for (int k = k0; k < k1; k++) acc = fmaf(xp[k], W[(long long)k * fout + o], acc);
    atomicAdd(&y[b * fout + o], acc);
}
__global__ void k_tr_bias_fill(const float *__restrict__ bias, float *__restrict__ y, int B, int fout) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < (long long)B * fout; i += (long long)gridDim.x * blockDim.x)
        y[i] = bias[i % fout];
}
__global__ void k_tr_relu(float *__restrict__ y, int n) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        y[i] = fmaxf(y[i], 0.0f);
}
__global__ void k_tr_set_vec(const float *__restrict__ vec, float *__restrict__ cat, int B) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < (long long)B * 8; i += (long long)gridDim.x * blockDim.x)
        cat[(i / 8) * 5008 + (i % 8)] = vec[i];
}
// the 25x25x8 pooled map of sample b lands in cat[b, 8:5008] (Flatten on NHWC, vector first: qlearnIA_V2.py:150-154)
__global__ void k_tr_flat_to_cat(const float *__restrict__ p4, float *__restrict__ cat, int B) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < (long long)B * 5000; i += (long long)gridDim.x * blockDim.x)
        cat[(i / 5000) * 5008 + 8 + (i % 5000)] = p4[i];
}

// ---------------------------------------------------------------------------------------------- backward kernels
// dpred = 2 (pred - target) / n_norm, loss_acc += sum (pred - target)^2 over the n local elements (n_norm: the elements of
// the global batch; n for a single fit)
__global__ void k_tr_mse(const float *__restrict__ pred, const float *__restrict__ target, long long n, long long n_norm,
                         float *__restrict__ dpred, double *__restrict__ loss_acc) {
    double v[1] = {0.0};
    const float scale = 2.0f / (float)n_norm;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float d = pred[i] - target[i];
        dpred[i] = d * scale;
        v[0] += (double)d * (double)d;
    }
    block_accumulate<1>(v, loss_acc, 1);
}
// the same with per-sample weights w[b] over `per` elements each: dpred = 2 w_b (pred - target) / n,
// loss_acc += sum w_b (pred - target)^2  (so loss_acc / n = (1/B) sum_b w_b mse_b)
__global__ void k_tr_mse_weighted(const float *__restrict__ pred, const float *__restrict__ target, long long n, long long n_norm,
                                  long long per, const float *__restrict__ w, float *__restrict__ dpred, double *__restrict__ loss_acc) {
    double v[1] = {0.0};
    const float scale = 2.0f / (float)n_norm;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float d = pred[i] - target[i], wb = w[i / per];
        dpred[i] = (d * scale) * wb;
        v[0] += (double)wb * ((double)d * (double)d);
    }
    block_accumulate<1>(v, loss_acc, 1);
}
__global__ void k_tr_loss_out(const double *__restrict__ loss_acc, long long n_act, long long n_ptr, float *__restrict__ out) {
    const double la = loss_acc[0] / (double)n_act, lp = loss_acc[1] / (double)n_ptr;
    out[0] = (float)(la + lp); out[1] = (float)la; out[2] = (float)lp;
}

// dx[b, y, x, ci] = sum_{ky,kx,co} dy[b, y+1-ky, x+1-kx, co] * w[ky][kx][ci][co]
template <int CIN, int COUT>
__global__ void k_tr_conv_bwd_data(const float *__restrict__ dy, const float *__restrict__ w, float *__restrict__ dx, int B, int H,
                                   int W) {
    __shared__ float ws[9 * CIN * COUT];
    for (int i = threadIdx.x; i < 9 * CIN * COUT; i += blockDim.x) ws[i] = w[i];
    __syncthreads();
    const long long n = (long long)B * H * W;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int xx = (int)(i % W), yy = (int)((i / W) % H);
        const long long b = i / ((long long)W * H);
        float acc[CIN], gv[9][COUT];
#pragma unroll
        for (int ci = 0; ci < CIN; ci++) acc[ci] = 0.0f;
#pragma unroll
        for (int ky = 0; ky < 3; ky++) {
#pragma unroll
            for (int kx = 0; kx < 3; kx++) {
                const int oy = yy + 1 - ky, ox = xx + 1 - kx;
                if (oy >= 0 && oy < H && ox >= 0 && ox < W) load_vec<COUT>(dy + ((b * H + oy) * W + ox) * COUT, gv[ky * 3 + kx]);
                else {
#pragma unroll
                    for (int co = 0; co < COUT; co++) gv[ky * 3 + kx][co] = 0.0f;
                }
            }
        }
#pragma unroll
        for (int tp = 0; tp < 9; tp++) {
#pragma unroll
            for (int co = 0; co < COUT; co++) {
#pragma unroll
                for (int ci = 0; ci < CIN; ci++) acc[ci] = fmaf(gv[tp][co], ws[(tp * CIN + ci) * COUT + co], acc[ci]);
            }
        }
        store_vec<CIN>(dx + i * CIN, acc);
    }
}

// dw[ky][kx][ci][co] += sum_{b,y,x} x[b, y+ky-1, x+kx-1, ci] * dy[b, y, x, co];  db[co] += sum dy.
// One thread per weight; a block walks row segments of TW pixels staged in shared memory and adds its partial sums once.
// One thread per weight x pixel group; a block walks whole image rows staged in (dynamic) shared memory -- the three input
// rows a 3x3 stencil needs plus the row of output gradients -- and adds its partial sums once at the end.
template <int CIN, int COUT>
struct BwdW {
    static constexpr int NW = 9 * CIN * COUT;
    static constexpr int PG = NW >= 288 ? 1 : (576 / NW > 16 ? 16 : 576 / NW);      // pixel groups sharing a row
    static constexpr int NT0 = NW * PG < 64 ? 64 : NW * PG;
    static constexpr int NT = NT0 < 32 * COUT ? 32 * COUT : (NT0 + 31) / 32 * 32;       // whole warps, one per bias channel at least
};
template <int CIN, int COUT>
__global__ void __launch_bounds__(BwdW<CIN, COUT>::NT)
k_tr_conv_bwd_weight(const float *__restrict__ x, const float *__restrict__ dy, float *__restrict__ dw, float *__restrict__ db, int B,
                     int H, int W) {
    constexpr int NW = BwdW<CIN, COUT>::NW, PG = BwdW<CIN, COUT>::PG;
    extern __shared__ __align__(16) float tr_smem[];
    float *xs = tr_smem;                                 // [3][W + 2][CIN]
    float *dys = tr_smem + 3 * (W + 2) * CIN;            // [W][COUT]
    const int t = threadIdx.x;
    const int wi = t % NW, pg = t / NW;                 // weight index, pixel group (threads beyond NW * PG only help staging)
    const int co = wi % COUT, ci = (wi / COUT) % CIN, kx = (wi / (COUT * CIN)) % 3, ky = wi / (COUT * CIN * 3);
    const long long rows = (long long)B * H;
    double acc = 0.0, accb = 0.0;
    for (long long row = blockIdx.x; row < rows; row += gridDim.x) {
        const int yy = (int)(row % H);
        const long long b = row / H;
        __syncthreads();
        // stage the three input rows (zero halo pixel on either side, zero rows outside the image) and the gradient row in
        // 16 / 8 / 4-byte chunks, several loads in flight per thread
        constexpr int CHX = (CIN % 4 == 0) ? 4 : ((CIN % 2 == 0) ? 2 : 1), CHY = (COUT % 4 == 0) ? 4 : ((COUT % 2 == 0) ? 2 : 1);
#pragma unroll
        for (int r = 0; r < 3; r++) {
            const int sy = yy + r - 1;
            float *dst = xs + (r * (W + 2) + 1) * CIN;
            const float *src = x + ((b * H + sy) * W) * CIN;
            const bool inside = sy >= 0 && sy < H;
#pragma unroll 4
            for (int q = t; q < W * CIN / CHX; q += blockDim.x) {
                float v[CHX];
                if (inside) load_vec<CHX>(src + q * CHX, v);
                else {
#pragma unroll
                    for (int e = 0; e < CHX; e++) v[e] = 0.0f;
                }
                store_vec<CHX>(dst + q * CHX, v);
            }
            if (t < CIN) { xs[r * (W + 2) * CIN + t] = 0.0f; xs[(r * (W + 2) + W + 1) * CIN + t] = 0.0f; }
        }
        {
            const float *src = dy + (b * H + yy) * (long long)W * COUT;
#pragma unroll 4
            for (int q = t; q < W * COUT / CHY; q += blockDim.x) {
                float v[CHY];
                load_vec<CHY>(src + q * CHY, v);
                store_vec<CHY>(dys + q * CHY, v);
            }
        }
        __syncthreads();
        if (pg < PG) {
            float s0 = 0.0f, s1 = 0.0f;                  // two chains: the sum over a 400-pixel row stays short in fp32
            const float *xr = xs + (ky * (W + 2) + kx) * CIN + ci;
            int px = pg;
            for (; px + PG < W; px += 2 * PG) {
                s0 = fmaf(xr[px * CIN], dys[px * COUT + co], s0);
                s1 = fmaf(xr[(px + PG) * CIN], dys[(px + PG) * COUT + co], s1);
            }
            if (px < W) s0 = fmaf(xr[px * CIN], dys[px * COUT + co], s0);
            acc += (double)s0 + (double)s1;
        }
        if ((t >> 5) < COUT) {                           // warp co sums channel co of the row, lane-strided
            const int cb = t >> 5;
            float s = 0.0f;
            for (int px = t & 31; px < W; px += 32) s += dys[px * COUT + cb];
            accb += (double)s;
        }
    }
    if (pg < PG) atomicAdd(&dw[wi], (float)acc);
    if ((t >> 5) < COUT) {
        accb = warp_sum(accb);
        if ((t & 31) == 0) atomicAdd(&db[t >> 5], (float)accb);
    }
}

// BatchNormalization + ReLU + MaxPool backward, pass 1: s1 = sum dz, s2 = sum dz * xhat over the layer, where dz is the
// pooled gradient routed to the window's first maximum if that maximum is positive.  sums[0..C) = s1, sums[8..8+C) = s2.
__global__ void k_tr_bnpool_bwd_reduce(const float *__restrict__ y, const float *__restrict__ mean, const float *__restrict__ var,
                                       const float *__restrict__ gamma, const float *__restrict__ beta, float eps,
                                       const float *__restrict__ dp, long long dp_stride, int B, int H, int W, int C,
                                       double *__restrict__ sums) {
    const int Ho = H / 2, Wo = W / 2;
    const long long n = (long long)B * Ho * Wo;
    double v[16];
#pragma unroll
    for (int j = 0; j < 16; j++) v[j] = 0.0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int xo = (int)(i % Wo), yo = (int)((i / Wo) % Ho);
        const long long b = i / ((long long)Wo * Ho);
        const long long base = ((b * H + 2 * yo) * W + 2 * xo) * C;
#pragma unroll
        for (int c = 0; c < 8; c++) {
            if (c >= C) continue;
            const float m = mean[c], r = rsqrtf(var[c] + eps);
            float zmax;
            const int k = pool_argmax(y, base, W, C, c, m, r, gamma[c], beta[c], zmax);
            if (zmax > 0.0f) {
                const float g = dp[b * dp_stride + ((long long)yo * Wo + xo) * C + c];
                const float xhat = (y[base + ((k >> 1) * (long long)W + (k & 1)) * C + c] - m) * r;
                v[c] += (double)g;
                v[8 + c] += (double)g * (double)xhat;
            }
        }
    }
    block_accumulate<16>(v, sums, 16);
}
// pass 2: dy[b, y, x, c] = gamma * rstd * (dz - s1 / N - xhat * s2 / N), N = n_norm (the global batch's pixels; B * H * W for
// a single fit).  One thread per 2x2 window and all 8 channels (the trunk's convolutions all have 8): the window's 4 pixels
// are read and written as float4 pairs.
__global__ void k_tr_bnpool_bwd_apply(const float *__restrict__ y, const float *__restrict__ mean, const float *__restrict__ var,
                                      const float *__restrict__ gamma, const float *__restrict__ beta, float eps,
                                      const float *__restrict__ dp, long long dp_stride, const double *__restrict__ sums,
                                      float *__restrict__ dy, int B, int H, int W, long long n_norm) {
    constexpr int C = 8;
    __shared__ float cm[C], cr[C], cg[C], cb[C], c1[C], c2[C];
    const double inv_n = 1.0 / (double)n_norm;
    if (threadIdx.x < C) {
        const int c = threadIdx.x;
        cm[c] = mean[c]; cr[c] = rsqrtf(var[c] + eps); cg[c] = gamma[c]; cb[c] = beta[c];
        c1[c] = (float)(sums[c] * inv_n); c2[c] = (float)(sums[8 + c] * inv_n);
    }
    __syncthreads();
    const int Ho = H / 2, Wo = W / 2;
    const long long n = (long long)B * Ho * Wo;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int xo = (int)(i % Wo), yo = (int)((i / Wo) % Ho);
        const long long b = i / ((long long)Wo * Ho);
        const long long base = ((b * H + 2 * yo) * W + 2 * xo) * C;
        const long long off[4] = {base, base + C, base + (long long)W * C, base + (long long)W * C + C};
        float v[4][C], g[C];
#pragma unroll
        for (int q = 0; q < 4; q++) load_vec<C>(y + off[q], v[q]);
        load_vec<C>(dp + b * dp_stride + ((long long)yo * Wo + xo) * C, g);
#pragma unroll
        for (int c = 0; c < C; c++) {
            const float m = cm[c], r = cr[c], ga = cg[c], be = cb[c];
            float zmax = bn_relu(v[0][c], m, r, ga, be);
            int k = 0;
#pragma unroll
            for (int q = 1; q < 4; q++) {                // first maximum in window order, like pool_argmax
                const float z = bn_relu(v[q][c], m, r, ga, be);
                if (z > zmax) { zmax = z; k = q; }
            }
            const float dz = zmax > 0.0f ? g[c] : 0.0f;
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const float xhat = (v[q][c] - m) * r;
                v[q][c] = ga * r * ((q == k ? dz : 0.0f) - c1[c] - xhat * c2[c]);
            }
        }
#pragma unroll
        for (int q = 0; q < 4; q++) store_vec<C>(dy + off[q], v[q]);
    }
}
// BatchNormalization + ReLU backward (no pooling; the pointer head), in place on dz [n_px, C]
__global__ void k_tr_bn_bwd_reduce(const float *__restrict__ y, const float *__restrict__ mean, const float *__restrict__ var,
                                   const float *__restrict__ gamma, const float *__restrict__ beta, float eps,
                                   const float *__restrict__ dz, long long n_px, int C, double *__restrict__ sums) {
    double v[16];
#pragma unroll
    for (int j = 0; j < 16; j++) v[j] = 0.0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_px; i += (long long)gridDim.x * blockDim.x) {
#pragma unroll
        for (int c = 0; c < 8; c++) {
            if (c >= C) continue;
            const float m = mean[c], r = rsqrtf(var[c] + eps);
            const float xhat = (y[i * C + c] - m) * r;
            if (fmaf(xhat, gamma[c], beta[c]) > 0.0f) {
                const float g = dz[i * C + c];
                v[c] += (double)g;
                v[8 + c] += (double)g * (double)xhat;
            }
        }
    }
    block_accumulate<16>(v, sums, 16);
}
__global__ void k_tr_bn_bwd_apply(const float *__restrict__ y, const float *__restrict__ mean, const float *__restrict__ var,
                                  const float *__restrict__ gamma, const float *__restrict__ beta, float eps, float *__restrict__ dz,
                                  const double *__restrict__ sums, long long n_px, int C, long long n_norm) {
    const double inv_n = 1.0 / (double)n_norm;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_px * C; i += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(i % C);
        const float m = mean[c], r = rsqrtf(var[c] + eps);
        const float xhat = (y[i] - m) * r;
        const float g = fmaf(xhat, gamma[c], beta[c]) > 0.0f ? dz[i] : 0.0f;
        dz[i] = gamma[c] * r * (g - (float)(sums[c] * inv_n) - xhat * (float)(sums[8 + c] * inv_n));
    }
}
// dgamma = s2, dbeta = s1
__global__ void k_tr_bn_param_grads(const double *__restrict__ sums, int C, float *__restrict__ dgamma, float *__restrict__ dbeta) {
    const int c = threadIdx.x;
    if (c < C) { dgamma[c] = (float)sums[8 + c]; dbeta[c] = (float)sums[c]; }
}

// transpose of k_tr_upsample's stencil as a gather: source row i feeds output rows 2i-1 (1/4), 2i (3/4), 2i+1 (3/4),
// 2i+2 (1/4); at the edges the clamped tap folds its 1/4 onto the edge row (2i resp. 2i+1).  One thread per source pixel.
__device__ __forceinline__ void up_bwd_w(int i, int h, float (&wt)[4]) {
    wt[0] = i > 0 ? 0.25f : 0.0f;
    wt[1] = i == 0 ? 1.0f : 0.75f;
    wt[2] = i == h - 1 ? 1.0f : 0.75f;
    wt[3] = i < h - 1 ? 0.25f : 0.0f;
}
template <int C>
__global__ void k_tr_upsample_bwd(const float *__restrict__ da, float *__restrict__ dsrc, int B, int h, int w) {
    const int H = 2 * h, W = 2 * w;
    const long long n = (long long)B * h * w;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += (long long)gridDim.x * blockDim.x) {
        const int j = (int)(idx % w), i = (int)((idx / w) % h);
        const long long b = idx / ((long long)w * h);
        float wr[4], wc[4], acc[C];
        up_bwd_w(i, h, wr);
        up_bwd_w(j, w, wc);
#pragma unroll
        for (int c = 0; c < C; c++) acc[c] = 0.0f;
#pragma unroll
        for (int a = 0; a < 4; a++) {
            const int Y = 2 * i - 1 + a;
            if (wr[a] == 0.0f) continue;
#pragma unroll
            for (int e = 0; e < 4; e++) {
                const int X = 2 * j - 1 + e;
                if (wc[e] == 0.0f) continue;
                float g[C];
                load_vec<C>(da + ((b * H + Y) * W + X) * C, g);
                const float wgt = wr[a] * wc[e];
#pragma unroll
                for (int c = 0; c < C; c++) acc[c] = fmaf(g[c], wgt, acc[c]);
            }
        }
        store_vec<C>(dsrc + idx * C, acc);
    }
}

// dW[i, o] = sum_b x[b, i] * dy[b, o];  db[o] = sum_b dy[b, o]
__global__ void k_tr_dense_bwd_w(const float *__restrict__ x, const float *__restrict__ dy, float *__restrict__ dW, float *__restrict__ db,
                                 int B, int fin, int fout) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < (long long)fin * fout) {
        const int k = (int)(i / fout), o = (int)(i % fout);
        float s = 0.0f;
        for (int b = 0; b < B; b++) s = fmaf(x[(long long)b * fin + k], dy[b * fout + o], s);
        dW[i] = s;
    }
    if (i < fout) {
        float s = 0.0f;
        for (int b = 0; b < B; b++) s += dy[b * fout + (int)i];
        db[i] = s;
    }
}
// dx[b, i] (+)= sum_o dy[b, o] * W[i, o]
__global__ void k_tr_dense_bwd_x(const float *__restrict__ dy, const float *__restrict__ W, float *__restrict__ dx, int B, int fin,
                                 int fout, int accumulate) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < (long long)B * fin; i += (long long)gridDim.x * blockDim.x) {
        const int b = (int)(i / fin), k = (int)(i % fin);
        float s = 0.0f;
        for (int o = 0; o < fout; o++) s = fmaf(dy[b * fout + o], W[(long long)k * fout + o], s);
        dx[i] = accumulate ? dx[i] + s : s;
    }
}
// g[i] = (a[i] > 0) ? g[i] : 0     (ReLU backward through the stored activation)
__global__ void k_tr_relu_mask(const float *__restrict__ a, float *__restrict__ g, long long n) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        if (!(a[i] > 0.0f)) g[i] = 0.0f;
}

// Keras Adam: m = b1 m + (1 - b1) g; v = b2 v + (1 - b2) g^2; p -= lr_t m / (sqrt(v) + eps)
__global__ void k_tr_adam(float *__restrict__ p, const float *__restrict__ g, float *__restrict__ m, float *__restrict__ v,
                          const uint8_t *__restrict__ trainable, int n, float lr_t, float b1, float b2, float eps) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !trainable[i]) return;
    const float gi = g[i];
    const float mi = b1 * m[i] + (1.0f - b1) * gi, vi = b2 * v[i] + (1.0f - b2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    p[i] -= lr_t * mi / (sqrtf(vi) + eps);
}

__global__ void k_tr_td_targets(const float *__restrict__ act_obs, const float *__restrict__ ptr_obs, const float *__restrict__ act_next,
                                const float *__restrict__ ptr_next, const int32_t *__restrict__ iaction, const int32_t *__restrict__ pointer,
                                const float *__restrict__ reward, const uint8_t *__restrict__ done, float gamma,
                                const float *__restrict__ discount, float *__restrict__ t_act, float *__restrict__ t_ptr) {
    // one block per sample: max over the next pointer map, copy of the obs predictions, the two overwritten entries.
    // discount [B] (n-step returns) replaces the scalar gamma when it is not NULL.
    const long long b = blockIdx.x;
    const int n = IMG * IMG;
    __shared__ float red[32];
    float mx = -INFINITY;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        mx = fmaxf(mx, ptr_next[b * n + i]);
        if (t_ptr != ptr_obs) t_ptr[b * n + i] = ptr_obs[b * n + i];
    }
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int wv = 1; wv < (int)((blockDim.x + 31) >> 5); wv++) mx = fmaxf(mx, red[wv]);
        const float keep = done[b] ? 0.0f : 1.0f, r = reward[b];
        const float g = discount ? discount[b] : gamma;
        const float a0 = act_obs[b * 2], a1 = act_obs[b * 2 + 1];
        const float ma = fmaxf(act_next[b * 2], act_next[b * 2 + 1]);
        t_act[b * 2] = a0;
        t_act[b * 2 + 1] = a1;
        t_act[b * 2 + iaction[b]] = __fadd_rn(r, __fmul_rn(__fmul_rn(g, ma), keep));      // no fma: same roundings as the host oracle
        // ptr_target[ipointer] with ipointer = (x, y) indexes the [row, col] map as [x][y]   (qlearnIA_V2.py:280)
        t_ptr[b * n + (long long)pointer[b * 2] * IMG + pointer[b * 2 + 1]] = __fadd_rn(r, __fmul_rn(__fmul_rn(g, mx), keep));
    }
}

// target - prediction at the two entries k_tr_td_targets overwrites, each target by k_tr_td_targets' own fp32 expression (the
// maximum is order-independent), so td = t_target - prediction exactly.  One block per sample.
__global__ void k_tr_td_errors(const float *__restrict__ act_obs, const float *__restrict__ ptr_obs, const float *__restrict__ act_next,
                               const float *__restrict__ ptr_next, const int32_t *__restrict__ iaction, const int32_t *__restrict__ pointer,
                               const float *__restrict__ reward, const uint8_t *__restrict__ done, float gamma,
                               const float *__restrict__ discount, float *__restrict__ td_act, float *__restrict__ td_ptr) {
    const long long b = blockIdx.x;
    const int n = IMG * IMG;
    __shared__ float red[32];
    float mx = -INFINITY;
    for (int i = threadIdx.x; i < n; i += blockDim.x) mx = fmaxf(mx, ptr_next[b * n + i]);
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int wv = 1; wv < (int)((blockDim.x + 31) >> 5); wv++) mx = fmaxf(mx, red[wv]);
        const float keep = done[b] ? 0.0f : 1.0f, r = reward[b];
        const float g = discount ? discount[b] : gamma;
        const float ma = fmaxf(act_next[b * 2], act_next[b * 2 + 1]);
        const float ta = __fadd_rn(r, __fmul_rn(__fmul_rn(g, ma), keep));
        const float tp = __fadd_rn(r, __fmul_rn(__fmul_rn(g, mx), keep));
        td_act[b] = __fsub_rn(ta, act_obs[b * 2 + iaction[b]]);
        td_ptr[b] = __fsub_rn(tp, ptr_obs[b * n + (long long)pointer[b * 2] * IMG + pointer[b * 2 + 1]]);
    }
}

// Double DQN targets (ofb_trainer_td_targets_double): one cluster of DD_CTAS blocks per sample.  Block r of the cluster scans
// the float4 slice [r, r + 1) * DD_SLICE of the online next map for its (value, first index) maximum -- NaN never compares
// greater or equal, so it is never chosen -- and, out of place, copies the same slice of ptr_obs to t_ptr.  After a cluster
// barrier rank 0 combines the partials over DSMEM (the comparator is a total order on (value, -index), so the result does not
// depend on the order), reads the target network's two selected entries and writes the overwritten entries (after the barrier:
// the other blocks' copy may cover them) and the TD errors.  No atomics, no global scratch.
#define DD_CTAS 8
#define DD_THREADS 512
#define DD_SLICE (IMG * IMG / 4 / DD_CTAS)      // 5000 float4 per block
#define DD_NONE 0x7fffffff

__device__ __forceinline__ void dd_take(float v, int i, float &bv, int &bi) {
    if (v > bv || (v == bv && i < bi)) { bv = v; bi = i; }
}

__global__ void __cluster_dims__(DD_CTAS, 1, 1) __launch_bounds__(DD_THREADS, 2)
k_tr_td_targets_double(const float *act_obs, const float *ptr_obs, const float *__restrict__ act_on,
                       const float *__restrict__ ptr_on, const float *__restrict__ act_tg, const float *__restrict__ ptr_tg,
                       const int32_t *__restrict__ iaction, const int32_t *__restrict__ pointer, const float *__restrict__ reward,
                       const uint8_t *__restrict__ done, float gamma, const float *__restrict__ discount, float *t_act, float *t_ptr,
                       float *__restrict__ td_act, float *__restrict__ td_ptr) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    const unsigned rank = cluster.block_rank();
    const long long b = blockIdx.x / DD_CTAS;
    const long long n = IMG * IMG;
    const float4 *on4 = reinterpret_cast<const float4 *>(ptr_on + b * n);
    const float4 *src4 = reinterpret_cast<const float4 *>(ptr_obs + b * n);
    float4 *dst4 = reinterpret_cast<float4 *>(t_ptr + b * n);
    const bool copy = t_ptr != ptr_obs;
    const int lo = rank * DD_SLICE, hi = lo + DD_SLICE;
    __shared__ float red_v[DD_THREADS / 32];
    __shared__ int red_i[DD_THREADS / 32];
    __shared__ float part_v;
    __shared__ int part_i;

    float bv = -INFINITY;
    int bi = DD_NONE;
    for (int base = lo + threadIdx.x; base < hi; base += 4 * DD_THREADS) {
        float4 v[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int i = base + k * DD_THREADS;
            if (i < hi) v[k] = __ldcs(on4 + i);
        }
        if (copy) {
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const int i = base + k * DD_THREADS;
                if (i < hi) __stcs(dst4 + i, __ldcs(src4 + i));
            }
        }
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int i = base + k * DD_THREADS;
            if (i < hi) {
                dd_take(v[k].x, 4 * i, bv, bi);
                dd_take(v[k].y, 4 * i + 1, bv, bi);
                dd_take(v[k].z, 4 * i + 2, bv, bi);
                dd_take(v[k].w, 4 * i + 3, bv, bi);
            }
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        dd_take(ov, oi, bv, bi);
    }
    if ((threadIdx.x & 31) == 0) { red_v[threadIdx.x >> 5] = bv; red_i[threadIdx.x >> 5] = bi; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < DD_THREADS / 32; w++) dd_take(red_v[w], red_i[w], bv, bi);
        part_v = bv;
        part_i = bi;
    }
    cluster.sync();                       // partials visible cluster-wide; every block's copy of t_ptr is done
    if (rank == 0 && threadIdx.x == 0) {
        bv = -INFINITY;
        bi = DD_NONE;
        for (unsigned r = 0; r < DD_CTAS; r++) {
            const float v = *cluster.map_shared_rank(&part_v, r);
            const int i = *cluster.map_shared_rank(&part_i, r);
            dd_take(v, i, bv, bi);
        }
        const int p_star = bi == DD_NONE ? 0 : bi;        // a map without a non-NaN value selects index 0
        const float keep = done[b] ? 0.0f : 1.0f, r = reward[b];
        const float g = discount ? discount[b] : gamma;
        const int a_star = act_on[b * 2 + 1] > act_on[b * 2] ? 1 : 0;    // ties to 0, as the decode
        const float ta = __fadd_rn(r, __fmul_rn(__fmul_rn(g, act_tg[b * 2 + a_star]), keep));
        const float tp = __fadd_rn(r, __fmul_rn(__fmul_rn(g, ptr_tg[b * n + p_star]), keep));
        const int ia = iaction[b];
        const long long e = (long long)pointer[b * 2] * IMG + pointer[b * 2 + 1];     // [x][y], as k_tr_td_targets
        const float a0 = act_obs[b * 2], a1 = act_obs[b * 2 + 1], pa = ia ? a1 : a0, pp = ptr_obs[b * n + e];
        if (td_act) {
            td_act[b] = __fsub_rn(ta, pa);
            td_ptr[b] = __fsub_rn(tp, pp);
        }
        t_act[b * 2] = a0;
        t_act[b * 2 + 1] = a1;
        t_act[b * 2 + ia] = ta;
        t_ptr[b * n + e] = tp;
    }
    cluster.sync();                       // keep every block's shared partial alive until rank 0 has read it
}

// ---------------------------------------------------------------------------------------------- host side
static inline unsigned blocks_for(long long n, int threads, long long cap = 148 * 16) {
    long long b = (n + threads - 1) / threads;
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    return (unsigned)b;
}

extern "C" void ofb_train_default_config(ofb_train_config *c) {
    if (!c) return;
    memset(c, 0, sizeof(*c));
    c->lr = 1e-4f; c->beta1 = 0.9f; c->beta2 = 0.999f; c->adam_eps = 1e-7f;
    c->bn_momentum = 0.99f; c->bn_eps = 1e-3f; c->bn_unbiased_moving_var = 0; c->max_batch = 8;
}

template <typename T>
static cudaError_t dev_alloc(T **p, size_t n) { return cudaMalloc((void **)p, n * sizeof(T)); }

extern "C" int ofb_trainer_destroy(ofb_trainer *t) {
    if (!t) return OFB_OK;
    cudaSetDevice(t->device);
    void *ptrs[] = {t->params, t->grads, t->adam_m, t->adam_v, t->trainable, t->x0, t->y[0], t->y[1], t->y[2], t->y[3], t->p[0], t->p[1],
                    t->p[2], t->p[3], t->cat, t->h1, t->d2, t->act, t->u0, t->a[0], t->a[1], t->a[2], t->a[3], t->yu[0], t->yu[1],
                    t->yu[2], t->yu[3], t->bn_mean, t->bn_var, t->sums, t->loss_acc, t->g0, t->g1, t->gu, t->dh1, t->dd2, t->dact,
                    t->dcat};
    for (void *p : ptrs) if (p) cudaFree(p);
    delete t;
    return OFB_OK;
}

extern "C" int ofb_trainer_create(const float *w_host, int64_t n_params, const ofb_train_config *cfg, int device, ofb_trainer **out) {
    if (!w_host || !out) { ofb_set_error("ofb_trainer_create: null argument"); return OFB_E_ARG; }
    Table tab = make_table();
    if (n_params != tab.total || tab.total != OFB_TRAIN_N_PARAMS) {
        ofb_set_error("ofb_trainer_create: expected %d weights in Keras layer order, got %lld", tab.total, (long long)n_params);
        return OFB_E_ARG;
    }
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0 || device < 0 || device >= n_dev) {
        ofb_set_error("ofb_trainer_create: no CUDA device %d (there is no CPU fallback)", device);
        return OFB_E_CUDA;
    }
    TR_CHECK(cudaSetDevice(device));
    ofb_trainer *t = new ofb_trainer();
    memset(t, 0, sizeof(*t));
    if (cfg) t->cfg = *cfg; else ofb_train_default_config(&t->cfg);
    if (t->cfg.max_batch <= 0) t->cfg.max_batch = 8;
    t->tab = tab;
    t->device = device;
    const size_t B = (size_t)t->cfg.max_batch, N = (size_t)tab.total;
    const int Hs[4] = {400, 200, 100, 50}, hs[4] = {50, 100, 200, 400}, ucin[4] = {1, 2, 4, 8}, ucout[4] = {2, 4, 8, 1};
    cudaError_t e = cudaSuccess;
    auto A = [&](cudaError_t r) { if (e == cudaSuccess) e = r; };
    A(dev_alloc(&t->params, N)); A(dev_alloc(&t->grads, N)); A(dev_alloc(&t->adam_m, N)); A(dev_alloc(&t->adam_v, N));
    A(dev_alloc(&t->trainable, N));
    A(dev_alloc(&t->x0, B * IMG * IMG * 2));
    for (int i = 0; i < 4; i++) {
        A(dev_alloc(&t->y[i], B * Hs[i] * Hs[i] * 8));
        A(dev_alloc(&t->p[i], B * (Hs[i] / 2) * (Hs[i] / 2) * 8));
        A(dev_alloc(&t->a[i], B * hs[i] * hs[i] * ucin[i]));
        A(dev_alloc(&t->yu[i], B * hs[i] * hs[i] * ucout[i]));
    }
    A(dev_alloc(&t->cat, B * 5008)); A(dev_alloc(&t->h1, B * 100)); A(dev_alloc(&t->d2, B * 50)); A(dev_alloc(&t->act, B * 2));
    A(dev_alloc(&t->u0, B * 625));
    A(dev_alloc(&t->bn_mean, 7 * 8)); A(dev_alloc(&t->bn_var, 7 * 8)); A(dev_alloc(&t->sums, 7 * 16)); A(dev_alloc(&t->loss_acc, 2));
    A(dev_alloc(&t->g0, B * IMG * IMG * 8)); A(dev_alloc(&t->g1, B * IMG * IMG * 8));
    A(dev_alloc(&t->gu, B * 625)); A(dev_alloc(&t->dh1, B * 100)); A(dev_alloc(&t->dd2, B * 50)); A(dev_alloc(&t->dact, B * 2));
    A(dev_alloc(&t->dcat, B * 5008));
    if (e != cudaSuccess) {
        ofb_set_error("ofb_trainer_create: cudaMalloc failed: %s", cudaGetErrorString(e));
        ofb_trainer_destroy(t);
        return OFB_E_NOMEM;
    }
    uint8_t *mask = new uint8_t[N];
    memset(mask, 1, N);
    auto frozen = [&](const Ref &r) { for (int i = 0; i < r.n; i++) mask[r.off + i] = 0; };
    for (int i = 0; i < 4; i++) {
        frozen(tab.conv[i].m); frozen(tab.conv[i].v);
        if (tab.up[i].bn) { frozen(tab.up[i].m); frozen(tab.up[i].v); }
    }
    e = cudaMemcpy(t->params, w_host, N * sizeof(float), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(t->trainable, mask, N, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemset(t->adam_m, 0, N * sizeof(float));
    if (e == cudaSuccess) e = cudaMemset(t->adam_v, 0, N * sizeof(float));
    if (e == cudaSuccess) e = cudaMemset(t->grads, 0, N * sizeof(float));
    delete[] mask;
    if (e != cudaSuccess) {
        ofb_set_error("ofb_trainer_create: upload failed: %s", cudaGetErrorString(e));
        ofb_trainer_destroy(t);
        return OFB_E_CUDA;
    }
    t->fs = t->bs = t->sums;
    t->la = t->loss_acc;
    t->gr = t->grads;
    *out = t;
    return OFB_OK;
}

template <int CIN, int COUT>
static void conv_fwd(const float *x, const float *w, const float *b, float *y, int B, int H, int W, cudaStream_t st) {
    k_tr_conv_fwd<CIN, COUT><<<blocks_for((long long)B * H * W, 256), 256, 0, st>>>(x, w, b, y, B, H, W);
}
template <int CIN, int COUT>
static void conv_bwd(const float *x, const float *dy, const float *w, float *dw, float *db, float *dx, int B, int H, int W, cudaStream_t st) {
    constexpr int NT = BwdW<CIN, COUT>::NT;
    const long long rows = (long long)B * H;
    const size_t smem = (size_t)(3 * (W + 2) * CIN + W * COUT) * sizeof(float);      // <= 40.2 KB (upconv4: 8 -> 1 at W = 400)
    k_tr_conv_bwd_weight<CIN, COUT><<<(unsigned)(rows < 148 * 4 ? rows : 148 * 4), NT, smem, st>>>(x, dy, dw, db, B, H, W);
    if (dx) k_tr_conv_bwd_data<CIN, COUT><<<blocks_for((long long)B * H * W, 256), 256, 0, st>>>(dy, w, dx, B, H, W);
}

// The reducer's call for one stage of a sharded fit (no-op for a local fit).
static int reduce_stage(ofb_trainer *t, int shard, int stage, cudaStream_t st) {
    if (!shard || !t->reducer) return OFB_OK;
    const int r = t->reducer(t->reducer_ctx, stage, (void *)st);
    if (r != 0) {
        ofb_set_error("ofb_trainer_fit_shard: the reducer failed at stage %d (returned %d); the trainer's state is undefined",
                      stage, r);
        return OFB_E_STATE;
    }
    return OFB_OK;
}

// training-mode forward on the B local samples; update_moving: BatchNormalization's moving averages follow the batch
// statistics.  Bn: the samples the statistics are over (B for a local forward); shard: the forward of a sharded fit, whose
// per-layer sums the reducer sums over the ranks (stage FWD_BN + layer) before they are consumed.
static int forward_train(ofb_trainer *t, const uint32_t *maps, const float *vec, int B, int Bn, int shard, int update_moving,
                         cudaStream_t st) {
    const Table &T = t->tab;
    float *P = t->params;
    const float eps = t->cfg.bn_eps;
    int rc;
    TR_CHECK(cudaMemsetAsync(t->fs, 0, 7 * 16 * sizeof(double), st));
    k_tr_unpack<<<blocks_for((long long)B * IMG * IMG, 256), 256, 0, st>>>(maps, t->x0, (long long)B * IMG * IMG);
    const int Hs[4] = {400, 200, 100, 50};
    for (int i = 0; i < 4; i++) {
        const ConvP &c = T.conv[i];
        const float *in = i == 0 ? t->x0 : t->p[i - 1];
        const int H = Hs[i];
        if (i == 0) conv_fwd<2, 8>(in, P + c.k.off, P + c.b.off, t->y[i], B, H, H, st);
        else conv_fwd<8, 8>(in, P + c.k.off, P + c.b.off, t->y[i], B, H, H, st);
        const long long npx = (long long)B * H * H;
        k_tr_chan_sums<<<blocks_for(npx, 256, 148 * 4), 256, 0, st>>>(t->y[i], npx, 8, t->fs + i * 16);
        if ((rc = reduce_stage(t, shard, OFB_STAGE_FWD_BN + i, st)) != OFB_OK) return rc;
        k_tr_bn_finalize<<<1, 32, 0, st>>>(t->fs + i * 16, (long long)Bn * H * H, 8, t->bn_mean + i * 8, t->bn_var + i * 8, P + c.m.off,
                                         P + c.v.off, t->cfg.bn_momentum, t->cfg.bn_unbiased_moving_var, update_moving);
        k_tr_bn_relu_pool<<<blocks_for(npx * 2, 256), 256, 0, st>>>(t->y[i], t->bn_mean + i * 8, t->bn_var + i * 8, P + c.g.off,
                                                                    P + c.be.off, eps, t->p[i], B, H, H, 8);
    }
    k_tr_set_vec<<<blocks_for(B * 8, 64), 64, 0, st>>>(vec, t->cat, B);
    k_tr_flat_to_cat<<<blocks_for((long long)B * 5000, 256), 256, 0, st>>>(t->p[3], t->cat, B);
    k_tr_bias_fill<<<blocks_for(B * 100, 128), 128, 0, st>>>(P + T.d1.b.off, t->h1, B, 100);
    k_tr_dense_fwd_splitk<<<dim3(40, B), 128, 0, st>>>(t->cat, P + T.d1.k.off, t->h1, 5008, 100);
    k_tr_relu<<<blocks_for(B * 100, 128), 128, 0, st>>>(t->h1, B * 100);
    k_tr_dense_fwd<<<blocks_for(B * 50, 64), 64, 0, st>>>(t->h1, P + T.d2.k.off, P + T.d2.b.off, t->d2, B, 100, 50, 1);
    k_tr_dense_fwd<<<blocks_for(B * 2, 64), 64, 0, st>>>(t->d2, P + T.o1.k.off, P + T.o1.b.off, t->act, B, 50, 2, 0);
    k_tr_dense_fwd<<<blocks_for(B * 625, 128), 128, 0, st>>>(t->h1, P + T.ud.k.off, P + T.ud.b.off, t->u0, B, 100, 625, 1);
    const int hs[4] = {25, 50, 100, 200}, cin[4] = {1, 2, 4, 8};
    for (int j = 0; j < 4; j++) {
        const ConvP &c = T.up[j];
        const int h = hs[j], H = 2 * h;
        // input of stage j: u0 (already activated) or relu(bn(yu[j-1]))
        {
            const float *src = j == 0 ? t->u0 : t->yu[j - 1];
            const float *mean = j == 0 ? nullptr : t->bn_mean + (4 + j - 1) * 8, *var = j == 0 ? nullptr : t->bn_var + (4 + j - 1) * 8;
            const float *ga = j == 0 ? nullptr : P + T.up[j - 1].g.off, *be = j == 0 ? nullptr : P + T.up[j - 1].be.off;
            const unsigned nb = blocks_for((long long)B * H * H, 256);
            if (cin[j] == 1) k_tr_upsample<1><<<nb, 256, 0, st>>>(src, mean, var, ga, be, eps, t->a[j], B, h, h);
            else if (cin[j] == 2) k_tr_upsample<2><<<nb, 256, 0, st>>>(src, mean, var, ga, be, eps, t->a[j], B, h, h);
            else if (cin[j] == 4) k_tr_upsample<4><<<nb, 256, 0, st>>>(src, mean, var, ga, be, eps, t->a[j], B, h, h);
            else k_tr_upsample<8><<<nb, 256, 0, st>>>(src, mean, var, ga, be, eps, t->a[j], B, h, h);
        }
        if (j == 0) conv_fwd<1, 2>(t->a[j], P + c.k.off, P + c.b.off, t->yu[j], B, H, H, st);
        else if (j == 1) conv_fwd<2, 4>(t->a[j], P + c.k.off, P + c.b.off, t->yu[j], B, H, H, st);
        else if (j == 2) conv_fwd<4, 8>(t->a[j], P + c.k.off, P + c.b.off, t->yu[j], B, H, H, st);
        else conv_fwd<8, 1>(t->a[j], P + c.k.off, P + c.b.off, t->yu[j], B, H, H, st);
        if (c.bn) {
            const long long npx = (long long)B * H * H;
            k_tr_chan_sums<<<blocks_for(npx, 256, 148 * 4), 256, 0, st>>>(t->yu[j], npx, c.cout, t->fs + (4 + j) * 16);
            if ((rc = reduce_stage(t, shard, OFB_STAGE_FWD_BN + 4 + j, st)) != OFB_OK) return rc;
            k_tr_bn_finalize<<<1, 32, 0, st>>>(t->fs + (4 + j) * 16, (long long)Bn * H * H, c.cout, t->bn_mean + (4 + j) * 8,
                                             t->bn_var + (4 + j) * 8, P + c.m.off, P + c.v.off, t->cfg.bn_momentum,
                                             t->cfg.bn_unbiased_moving_var, update_moving);
        }
    }
    TR_CHECK(cudaGetLastError());
    return OFB_OK;
}

static int check_batch(ofb_trainer *t, int B, const char *who) {
    if (!t) { ofb_set_error("%s: null handle", who); return OFB_E_ARG; }
    if (B < 1 || B > t->cfg.max_batch) {
        ofb_set_error("%s: batch %d outside 1..max_batch=%d", who, B, t->cfg.max_batch);
        return OFB_E_ARG;
    }
    TR_CHECK(cudaSetDevice(t->device));
    return OFB_OK;
}

extern "C" int ofb_trainer_forward(ofb_trainer *t, const uint32_t *maps, const float *vec, int B, float *act_dev, float *ptr_dev,
                                   void *stream) {
    int rc = check_batch(t, B, "ofb_trainer_forward");
    if (rc != OFB_OK) return rc;
    if (!maps || !vec) { ofb_set_error("ofb_trainer_forward: null input"); return OFB_E_ARG; }
    TR_CHECK(cudaSetDevice(t->device));
    cudaStream_t st = (cudaStream_t)stream;
    rc = forward_train(t, maps, vec, B, B, 0, 0, st);
    if (rc != OFB_OK) return rc;
    if (act_dev) TR_CHECK(cudaMemcpyAsync(act_dev, t->act, (size_t)B * 2 * sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (ptr_dev) TR_CHECK(cudaMemcpyAsync(ptr_dev, t->yu[3], (size_t)B * IMG * IMG * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return OFB_OK;
}

// one Adam step on the B local samples of a batch of Bn; sample_weight == NULL: today's unweighted loss, with the kernels of
// ofb_trainer_fit unchanged.  shard: a sharded fit (ofb_trainer_fit_shard): the reducer sums every accumulated slice over
// the ranks before it is consumed, and each BN layer's gamma / beta gradients are taken from the local backward sums.
static int fit_impl(ofb_trainer *t, const uint32_t *maps, const float *vec, const float *target_act, const float *target_ptr,
                    const float *sample_weight, int B, int Bn, int shard, float *loss_dev, void *stream) {
    int rc;
    TR_CHECK(cudaSetDevice(t->device));
    cudaStream_t st = (cudaStream_t)stream;
    const Table &T = t->tab;
    float *P = t->params, *G = t->gr;
    const float eps = t->cfg.bn_eps;
    rc = forward_train(t, maps, vec, B, Bn, shard, 1, st);
    if (rc != OFB_OK) return rc;
    TR_CHECK(cudaMemsetAsync(G, 0, (size_t)T.total * sizeof(float), st));
    TR_CHECK(cudaMemsetAsync(t->bs, 0, 7 * 16 * sizeof(double), st));
    TR_CHECK(cudaMemsetAsync(t->la, 0, 2 * sizeof(double), st));

    // ---- losses: mse(output1) + mse(output2), each a mean over all of its elements (of the global batch)
    const long long n_act = (long long)B * 2, n_ptr = (long long)B * IMG * IMG;
    const long long N_act = (long long)Bn * 2, N_ptr = (long long)Bn * IMG * IMG;
    if (!sample_weight) {
        k_tr_mse<<<1, 64, 0, st>>>(t->act, target_act, n_act, N_act, t->dact, t->la);
        k_tr_mse<<<blocks_for(n_ptr, 256, 148 * 4), 256, 0, st>>>(t->yu[3], target_ptr, n_ptr, N_ptr, t->g0, t->la + 1);
    } else {
        k_tr_mse_weighted<<<1, 64, 0, st>>>(t->act, target_act, n_act, N_act, 2, sample_weight, t->dact, t->la);
        k_tr_mse_weighted<<<blocks_for(n_ptr, 256, 148 * 4), 256, 0, st>>>(t->yu[3], target_ptr, n_ptr, N_ptr, IMG * IMG, sample_weight,
                                                                          t->g0, t->la + 1);
    }
    if ((rc = reduce_stage(t, shard, OFB_STAGE_LOSS, st)) != OFB_OK) return rc;
    if (loss_dev) k_tr_loss_out<<<1, 1, 0, st>>>(t->la, N_act, N_ptr, loss_dev);

    // ---- pointer head, top down.  g0 holds the gradient w.r.t. the stage's conv output, g1 w.r.t. its (upsampled) input.
    const int hs[4] = {25, 50, 100, 200}, cin[4] = {1, 2, 4, 8};
    for (int j = 3; j >= 0; j--) {
        const ConvP &c = T.up[j];
        const int h = hs[j], H = 2 * h;
        const long long npx = (long long)B * H * H;
        if (c.bn) {       // g0 = d relu(bn(yu[j])) -> d yu[j]
            double *s = t->bs + (4 + j) * 16;
            const float *mean = t->bn_mean + (4 + j) * 8, *var = t->bn_var + (4 + j) * 8;
            k_tr_bn_bwd_reduce<<<blocks_for(npx, 256, 148 * 4), 256, 0, st>>>(t->yu[j], mean, var, P + c.g.off, P + c.be.off, eps, t->g0, npx,
                                                                              c.cout, s);
            if (shard) {  // local gamma / beta gradients, before the sums become global
                k_tr_bn_param_grads<<<1, 32, 0, st>>>(s, c.cout, G + c.g.off, G + c.be.off);
                if ((rc = reduce_stage(t, shard, OFB_STAGE_BWD_BN + 4 + j, st)) != OFB_OK) return rc;
            }
            k_tr_bn_bwd_apply<<<blocks_for(npx * c.cout, 256), 256, 0, st>>>(t->yu[j], mean, var, P + c.g.off, P + c.be.off, eps, t->g0, s,
                                                                             npx, c.cout, (long long)Bn * H * H);
            if (!shard) k_tr_bn_param_grads<<<1, 32, 0, st>>>(s, c.cout, G + c.g.off, G + c.be.off);
        }
        if (j == 3) conv_bwd<8, 1>(t->a[j], t->g0, P + c.k.off, G + c.k.off, G + c.b.off, t->g1, B, H, H, st);
        else if (j == 2) conv_bwd<4, 8>(t->a[j], t->g0, P + c.k.off, G + c.k.off, G + c.b.off, t->g1, B, H, H, st);
        else if (j == 1) conv_bwd<2, 4>(t->a[j], t->g0, P + c.k.off, G + c.k.off, G + c.b.off, t->g1, B, H, H, st);
        else conv_bwd<1, 2>(t->a[j], t->g0, P + c.k.off, G + c.k.off, G + c.b.off, t->g1, B, H, H, st);
        // g1 = d a[j] [B,H,H,cin] -> gradient w.r.t. the stage input [B,h,h,cin] (for j = 0: u0 [B,625])
        float *dst = j == 0 ? t->gu : t->g0;
        const unsigned nb = blocks_for((long long)B * h * h, 128);
        if (cin[j] == 1) k_tr_upsample_bwd<1><<<nb, 128, 0, st>>>(t->g1, dst, B, h, h);
        else if (cin[j] == 2) k_tr_upsample_bwd<2><<<nb, 128, 0, st>>>(t->g1, dst, B, h, h);
        else if (cin[j] == 4) k_tr_upsample_bwd<4><<<nb, 128, 0, st>>>(t->g1, dst, B, h, h);
        else k_tr_upsample_bwd<8><<<nb, 128, 0, st>>>(t->g1, dst, B, h, h);
    }
    // ---- dense part
    k_tr_relu_mask<<<blocks_for((long long)B * 625, 128), 128, 0, st>>>(t->u0, t->gu, (long long)B * 625);
    k_tr_dense_bwd_w<<<blocks_for(100 * 625, 128), 128, 0, st>>>(t->h1, t->gu, G + T.ud.k.off, G + T.ud.b.off, B, 100, 625);
    k_tr_dense_bwd_x<<<blocks_for(B * 100, 64), 64, 0, st>>>(t->gu, P + T.ud.k.off, t->dh1, B, 100, 625, 0);
    k_tr_dense_bwd_w<<<blocks_for(50 * 2, 64), 64, 0, st>>>(t->d2, t->dact, G + T.o1.k.off, G + T.o1.b.off, B, 50, 2);
    k_tr_dense_bwd_x<<<blocks_for(B * 50, 64), 64, 0, st>>>(t->dact, P + T.o1.k.off, t->dd2, B, 50, 2, 0);
    k_tr_relu_mask<<<blocks_for(B * 50, 64), 64, 0, st>>>(t->d2, t->dd2, (long long)B * 50);
    k_tr_dense_bwd_w<<<blocks_for(100 * 50, 128), 128, 0, st>>>(t->h1, t->dd2, G + T.d2.k.off, G + T.d2.b.off, B, 100, 50);
    k_tr_dense_bwd_x<<<blocks_for(B * 100, 64), 64, 0, st>>>(t->dd2, P + T.d2.k.off, t->dh1, B, 100, 50, 1);
    k_tr_relu_mask<<<blocks_for(B * 100, 64), 64, 0, st>>>(t->h1, t->dh1, (long long)B * 100);
    k_tr_dense_bwd_w<<<blocks_for((long long)5008 * 100, 256), 256, 0, st>>>(t->cat, t->dh1, G + T.d1.k.off, G + T.d1.b.off, B, 5008, 100);
    k_tr_dense_bwd_x<<<blocks_for((long long)B * 5008, 128), 128, 0, st>>>(t->dh1, P + T.d1.k.off, t->dcat, B, 5008, 100, 0);
    // ---- trunk, top down: dp = gradient w.r.t. the pooled output (conv4: the flat slice of dcat)
    const int Hs[4] = {400, 200, 100, 50};
    const float *dp = t->dcat + 8;
    long long dp_stride = 5008;
    for (int i = 3; i >= 0; i--) {
        const ConvP &c = T.conv[i];
        const int H = Hs[i];
        const long long npx = (long long)B * H * H;
        double *s = t->bs + i * 16;
        const float *mean = t->bn_mean + i * 8, *var = t->bn_var + i * 8;
        k_tr_bnpool_bwd_reduce<<<blocks_for(npx / 4, 256, 148 * 4), 256, 0, st>>>(t->y[i], mean, var, P + c.g.off, P + c.be.off, eps, dp,
                                                                                  dp_stride, B, H, H, 8, s);
        if (shard) {
            k_tr_bn_param_grads<<<1, 32, 0, st>>>(s, 8, G + c.g.off, G + c.be.off);
            if ((rc = reduce_stage(t, shard, OFB_STAGE_BWD_BN + i, st)) != OFB_OK) return rc;
        }
        k_tr_bnpool_bwd_apply<<<blocks_for(npx / 4, 128), 128, 0, st>>>(t->y[i], mean, var, P + c.g.off, P + c.be.off, eps, dp, dp_stride, s,
                                                                        t->g1, B, H, H, (long long)Bn * H * H);
        if (!shard) k_tr_bn_param_grads<<<1, 32, 0, st>>>(s, 8, G + c.g.off, G + c.be.off);
        if (i == 0) conv_bwd<2, 8>(t->x0, t->g1, P + c.k.off, G + c.k.off, G + c.b.off, nullptr, B, H, H, st);
        else conv_bwd<8, 8>(t->p[i - 1], t->g1, P + c.k.off, G + c.k.off, G + c.b.off, t->g0, B, H, H, st);
        dp = t->g0;                                      // d p[i-1]: [B, H, H, 8] = the pooled output of layer i - 1
        dp_stride = (long long)H * H * 8;
    }
    // ---- Adam, on the gradients of the global batch
    if ((rc = reduce_stage(t, shard, OFB_STAGE_GRADS, st)) != OFB_OK) return rc;
    t->steps += 1;
    const double b1 = t->cfg.beta1, b2 = t->cfg.beta2;
    const float lr_t = (float)((double)t->cfg.lr * sqrt(1.0 - pow(b2, (double)t->steps)) / (1.0 - pow(b1, (double)t->steps)));
    k_tr_adam<<<blocks_for(T.total, 256, 1 << 20), 256, 0, st>>>(P, G, t->adam_m, t->adam_v, t->trainable, T.total, lr_t, t->cfg.beta1,
                                                                  t->cfg.beta2, t->cfg.adam_eps);
    TR_CHECK(cudaGetLastError());
    return OFB_OK;
}

extern "C" int ofb_trainer_fit(ofb_trainer *t, const uint32_t *maps, const float *vec, const float *target_act, const float *target_ptr,
                               int B, float *loss_dev, void *stream) {
    int rc = check_batch(t, B, "ofb_trainer_fit");
    if (rc != OFB_OK) return rc;
    if (!maps || !vec || !target_act || !target_ptr) { ofb_set_error("ofb_trainer_fit: null argument"); return OFB_E_ARG; }
    return fit_impl(t, maps, vec, target_act, target_ptr, nullptr, B, B, 0, loss_dev, stream);
}

extern "C" int ofb_trainer_fit_weighted(ofb_trainer *t, const uint32_t *maps, const float *vec, const float *target_act,
                                        const float *target_ptr, const float *sample_weight, int B, float *loss_dev, void *stream) {
    int rc = check_batch(t, B, "ofb_trainer_fit_weighted");
    if (rc != OFB_OK) return rc;
    if (!maps || !vec || !target_act || !target_ptr || !sample_weight) {
        ofb_set_error("ofb_trainer_fit_weighted: null argument");
        return OFB_E_ARG;
    }
    return fit_impl(t, maps, vec, target_act, target_ptr, sample_weight, B, B, 0, loss_dev, stream);
}

extern "C" int ofb_trainer_fit_shard(ofb_trainer *t, const uint32_t *maps, const float *vec, const float *target_act,
                                     const float *target_ptr, const float *sample_weight, int B, int Bn, float *loss_dev, void *stream) {
    int rc = check_batch(t, B, "ofb_trainer_fit_shard");
    if (rc != OFB_OK) return rc;
    if (!maps || !vec || !target_act || !target_ptr) { ofb_set_error("ofb_trainer_fit_shard: null argument"); return OFB_E_ARG; }
    if (Bn < B) {
        ofb_set_error("ofb_trainer_fit_shard: batch_global %d is smaller than batch_local %d", Bn, B);
        return OFB_E_ARG;
    }
    if (Bn != B && !t->reducer) {
        ofb_set_error("ofb_trainer_fit_shard: batch_global %d != batch_local %d needs a reducer (ofb_trainer_set_reducer)", Bn, B);
        return OFB_E_ARG;
    }
    if (t->reducer && t->fs == t->sums) {
        ofb_set_error("ofb_trainer_fit_shard: a reducer needs exchange buffers (ofb_trainer_set_exchange)");
        return OFB_E_ARG;
    }
    return fit_impl(t, maps, vec, target_act, target_ptr, sample_weight, B, Bn, 1, loss_dev, stream);
}

extern "C" int ofb_trainer_set_exchange(ofb_trainer *t, double *stats_dev, float *grads_dev) {
    if (!t) { ofb_set_error("ofb_trainer_set_exchange: null handle"); return OFB_E_ARG; }
    if (!stats_dev != !grads_dev) {
        ofb_set_error("ofb_trainer_set_exchange: stats_dev and grads_dev are both given or both NULL");
        return OFB_E_ARG;
    }
    if (!stats_dev && t->reducer) {
        ofb_set_error("ofb_trainer_set_exchange: remove the reducer before the exchange buffers");
        return OFB_E_ARG;
    }
    if (stats_dev) {
        t->fs = stats_dev + OFB_TRAIN_STATS_FWD;
        t->la = stats_dev + OFB_TRAIN_STATS_LOSS;
        t->bs = stats_dev + OFB_TRAIN_STATS_BWD;
        t->gr = grads_dev;
    } else {
        t->fs = t->bs = t->sums;
        t->la = t->loss_acc;
        t->gr = t->grads;
    }
    return OFB_OK;
}

extern "C" int ofb_trainer_set_reducer(ofb_trainer *t, ofb_reduce_fn fn, void *ctx) {
    if (!t) { ofb_set_error("ofb_trainer_set_reducer: null handle"); return OFB_E_ARG; }
    if (fn && t->fs == t->sums) {
        ofb_set_error("ofb_trainer_set_reducer: a reducer needs exchange buffers (ofb_trainer_set_exchange)");
        return OFB_E_ARG;
    }
    t->reducer = fn;
    t->reducer_ctx = fn ? ctx : nullptr;
    return OFB_OK;
}

static int td_errors_impl(const float *act_obs, const float *ptr_obs, const float *act_next, const float *ptr_next,
                          const int32_t *iaction, const int32_t *pointer, const float *reward, const uint8_t *done, float gamma,
                          const float *discount, int B, float *td_act, float *td_ptr, void *stream, const char *who) {
    if (!act_obs || !ptr_obs || !act_next || !ptr_next || !iaction || !pointer || !reward || !done || !td_act || !td_ptr || B < 1) {
        ofb_set_error("%s: bad argument", who);
        return OFB_E_ARG;
    }
    k_tr_td_errors<<<B, 256, 0, (cudaStream_t)stream>>>(act_obs, ptr_obs, act_next, ptr_next, iaction, pointer, reward, done, gamma,
                                                        discount, td_act, td_ptr);
    TR_CHECK(cudaGetLastError());
    return OFB_OK;
}

static int td_targets_impl(const float *act_obs, const float *ptr_obs, const float *act_next, const float *ptr_next,
                           const int32_t *iaction, const int32_t *pointer, const float *reward, const uint8_t *done, float gamma,
                           const float *discount, int B, float *t_act, float *t_ptr, void *stream, const char *who) {
    if (!act_obs || !ptr_obs || !act_next || !ptr_next || !iaction || !pointer || !reward || !done || !t_act || !t_ptr || B < 1) {
        ofb_set_error("%s: bad argument", who);
        return OFB_E_ARG;
    }
    k_tr_td_targets<<<B, 256, 0, (cudaStream_t)stream>>>(act_obs, ptr_obs, act_next, ptr_next, iaction, pointer, reward, done, gamma,
                                                         discount, t_act, t_ptr);
    TR_CHECK(cudaGetLastError());
    return OFB_OK;
}

extern "C" int ofb_trainer_td_errors(const float *act_obs, const float *ptr_obs, const float *act_next, const float *ptr_next,
                                     const int32_t *iaction, const int32_t *pointer, const float *reward, const uint8_t *done, float gamma,
                                     int B, float *td_act, float *td_ptr, void *stream) {
    return td_errors_impl(act_obs, ptr_obs, act_next, ptr_next, iaction, pointer, reward, done, gamma, nullptr, B, td_act, td_ptr,
                          stream, "ofb_trainer_td_errors");
}

extern "C" int ofb_trainer_td_targets(const float *act_obs, const float *ptr_obs, const float *act_next, const float *ptr_next,
                                      const int32_t *iaction, const int32_t *pointer, const float *reward, const uint8_t *done, float gamma,
                                      int B, float *t_act, float *t_ptr, void *stream) {
    return td_targets_impl(act_obs, ptr_obs, act_next, ptr_next, iaction, pointer, reward, done, gamma, nullptr, B, t_act, t_ptr,
                           stream, "ofb_trainer_td_targets");
}

extern "C" int ofb_trainer_td_errors_discounted(const float *act_obs, const float *ptr_obs, const float *act_next,
                                                const float *ptr_next, const int32_t *iaction, const int32_t *pointer,
                                                const float *reward, const uint8_t *done, const float *discount, int B, float *td_act,
                                                float *td_ptr, void *stream) {
    if (!discount) { ofb_set_error("ofb_trainer_td_errors_discounted: null discount"); return OFB_E_ARG; }
    return td_errors_impl(act_obs, ptr_obs, act_next, ptr_next, iaction, pointer, reward, done, 0.0f, discount, B, td_act, td_ptr,
                          stream, "ofb_trainer_td_errors_discounted");
}

extern "C" int ofb_trainer_td_targets_discounted(const float *act_obs, const float *ptr_obs, const float *act_next,
                                                 const float *ptr_next, const int32_t *iaction, const int32_t *pointer,
                                                 const float *reward, const uint8_t *done, const float *discount, int B, float *t_act,
                                                 float *t_ptr, void *stream) {
    if (!discount) { ofb_set_error("ofb_trainer_td_targets_discounted: null discount"); return OFB_E_ARG; }
    return td_targets_impl(act_obs, ptr_obs, act_next, ptr_next, iaction, pointer, reward, done, 0.0f, discount, B, t_act, t_ptr,
                           stream, "ofb_trainer_td_targets_discounted");
}

extern "C" int ofb_trainer_td_targets_double(const float *act_obs, const float *ptr_obs, const float *act_next_online,
                                             const float *ptr_next_online, const float *act_next_target,
                                             const float *ptr_next_target, const int32_t *iaction, const int32_t *pointer,
                                             const float *reward, const uint8_t *done, float gamma, const float *discount, int B,
                                             float *t_act, float *t_ptr, float *td_act, float *td_ptr, void *stream) {
    if (!act_obs || !ptr_obs || !act_next_online || !ptr_next_online || !act_next_target || !ptr_next_target || !iaction ||
        !pointer || !reward || !done || !t_act || !t_ptr || B < 1) {
        ofb_set_error("ofb_trainer_td_targets_double: bad argument");
        return OFB_E_ARG;
    }
    if (!td_act != !td_ptr) {
        ofb_set_error("ofb_trainer_td_targets_double: td_act and td_ptr are both given or both NULL");
        return OFB_E_ARG;
    }
    if (((uintptr_t)ptr_obs | (uintptr_t)ptr_next_online | (uintptr_t)t_ptr) & 15) {
        ofb_set_error("ofb_trainer_td_targets_double: ptr_obs, ptr_next_online and target_ptr must be 16-byte aligned");
        return OFB_E_ARG;
    }
    k_tr_td_targets_double<<<(unsigned)B * DD_CTAS, DD_THREADS, 0, (cudaStream_t)stream>>>(
        act_obs, ptr_obs, act_next_online, ptr_next_online, act_next_target, ptr_next_target, iaction, pointer, reward, done, gamma,
        discount, t_act, t_ptr, td_act, td_ptr);
    TR_CHECK(cudaGetLastError());
    return OFB_OK;
}

static int copy_out(ofb_trainer *t, const float *src, float *dst_host, void *stream, const char *who) {
    if (!t || !dst_host) { ofb_set_error("%s: null argument", who); return OFB_E_ARG; }
    TR_CHECK(cudaSetDevice(t->device));
    TR_CHECK(cudaStreamSynchronize((cudaStream_t)stream));
    TR_CHECK(cudaMemcpy(dst_host, src, (size_t)t->tab.total * sizeof(float), cudaMemcpyDeviceToHost));
    return OFB_OK;
}
extern "C" int ofb_trainer_get_weights(ofb_trainer *t, float *out_host, void *stream) {
    return copy_out(t, t ? t->params : nullptr, out_host, stream, "ofb_trainer_get_weights");
}
extern "C" int ofb_trainer_get_grads(ofb_trainer *t, float *out_host, void *stream) {
    return copy_out(t, t ? t->gr : nullptr, out_host, stream, "ofb_trainer_get_grads");
}
extern "C" int64_t ofb_trainer_steps(const ofb_trainer *t) { return t ? t->steps : -1; }
