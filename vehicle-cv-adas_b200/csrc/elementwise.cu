// elementwise.cu -- HBM-bound glue kernels on the padded-NHWC fp16 layout (16-byte vector accesses,
// one thread per 8 channels, grids sized in waves of the 148 SMs by the launch helpers).
// These are the non-GEMM graph nodes that ONNXRuntime/TensorRT execute inside the opaque model
// behind coreEngine.py:150-157/184-186: strided-conv patch gather (feeds the GEMM), MaxPool
// (SPPF 5x5 s1, ResNet 3x3 s2), nearest Upsample x2 (+Concat by writing a channel slice),
// LayerNorm (UFLDv2 fc_norm, exportLib/ultrafastLaneV2/model_culane.py:34) and the NCHW fp32
// input binding -> NHWC fp16 conversion.
#include "common.h"

namespace adas {

static inline int grid_for(long long work, int threads) {
    long long b = (work + threads - 1) / threads;
    if (b < 1) b = 1;
    return (int)b;
}

// ---- im2col for strided / large-kernel / thin-channel convs ------------------------------------
// out row = (b, yo+1, xo+1) in the padded output grid, k = (ky*kw + kx)*Cin + c. Cin % 4 == 0.
// One thread moves 4 channels (8 bytes) of one tap.
__global__ void im2col_kernel(const __half* __restrict__ in, int in_ld, int in_coff, int B, int H, int W, int Cin,
                              int kh, int kw, int stride, int pad, int Ho, int Wo, __half* __restrict__ out, int Kpad) {
    const int c4 = Cin >> 2;
    const long long per_row = (long long)kh * kw * c4;
    const long long total = (long long)B * Ho * Wo * per_row;
    const int Hp = H + 2, Wp = W + 2, Hop = Ho + 2, Wop = Wo + 2;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int cg = (int)(i % c4);
        long long t = i / c4;
        const int kx = (int)(t % kw); t /= kw;
        const int ky = (int)(t % kh); t /= kh;
        const int xo = (int)(t % Wo); t /= Wo;
        const int yo = (int)(t % Ho);
        const int b = (int)(t / Ho);
        const int yi = yo * stride - pad + ky;
        const int xi = xo * stride - pad + kx;
        uint2 v = make_uint2(0u, 0u);
        if (yi >= 0 && yi < H && xi >= 0 && xi < W) {
            const size_t r = ((size_t)b * Hp + (yi + 1)) * Wp + (xi + 1);
            v = *reinterpret_cast<const uint2*>(in + r * in_ld + in_coff + cg * 4);
        }
        const size_t orow = ((size_t)b * Hop + (yo + 1)) * Wop + (xo + 1);
        *reinterpret_cast<uint2*>(out + orow * Kpad + ((ky * kw + kx) * Cin + cg * 4)) = v;
    }
}

// 16-byte variant (Cin % 8 == 0): one thread moves 8 channels of one tap; consecutive threads cover consecutive
// 16-byte chunks of the output row, so both the gather reads (Cin*2-byte runs) and the writes are full sectors.
__global__ void im2col8_kernel(const __half* __restrict__ in, int in_ld, int in_coff, int B, int H, int W, int Cin,
                               int kh, int kw, int stride, int pad, int Ho, int Wo, __half* __restrict__ out, int Kpad) {
    const int c8 = Cin >> 3;
    const int per_px = kh * kw * c8;
    const long long total = (long long)B * Ho * Wo * per_px;
    const int Hp = H + 2, Wp = W + 2, Hop = Ho + 2, Wop = Wo + 2;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int r = (int)(i % per_px);
        long long t = i / per_px;
        const int cg = r % c8;
        const int tap = r / c8;
        const int kx = tap % kw, ky = tap / kw;
        const int xo = (int)(t % Wo); t /= Wo;
        const int yo = (int)(t % Ho);
        const int b = (int)(t / Ho);
        const int yi = yo * stride - pad + ky;
        const int xi = xo * stride - pad + kx;
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (yi >= 0 && yi < H && xi >= 0 && xi < W) {
            const size_t rr = ((size_t)b * Hp + (yi + 1)) * Wp + (xi + 1);
            v = *reinterpret_cast<const uint4*>(in + rr * in_ld + in_coff + cg * 8);
        }
        const size_t orow = ((size_t)b * Hop + (yo + 1)) * Wop + (xo + 1);
        *reinterpret_cast<uint4*>(out + orow * Kpad + (tap * Cin + cg * 8)) = v;
    }
}

int launch_im2col(const __half* in, int in_ld, int in_coff, int B, int H, int W, int Cin, int kh, int kw, int stride,
                  int pad, int Ho, int Wo, __half* out, int Kpad, cudaStream_t st) {
    ADAS_CHECK(Cin % 4 == 0 && in_ld % 4 == 0 && in_coff % 4 == 0 && Kpad % 4 == 0, "im2col: channel alignment");
    if (Cin % 8 == 0 && in_ld % 8 == 0 && in_coff % 8 == 0 && Kpad % 8 == 0) {
        const long long total8 = (long long)B * Ho * Wo * kh * kw * (Cin / 8);
        int blocks8 = grid_for(total8, 256);
        if (blocks8 > 148 * 16) blocks8 = 148 * 16;
        im2col8_kernel<<<blocks8, 256, 0, st>>>(in, in_ld, in_coff, B, H, W, Cin, kh, kw, stride, pad, Ho, Wo, out, Kpad);
        count_launch();
        ADAS_CUDA(cudaGetLastError());
        return 0;
    }
    const long long total = (long long)B * Ho * Wo * kh * kw * (Cin / 4);
    int blocks = grid_for(total, 256);
    if (blocks > 148 * 32) blocks = 148 * 32;
    im2col_kernel<<<blocks, 256, 0, st>>>(in, in_ld, in_coff, B, H, W, Cin, kh, kw, stride, pad, Ho, Wo, out, Kpad);
    count_launch();
    ADAS_CUDA(cudaGetLastError());
    return 0;
}

// ---- max pooling (window positions outside the image are ignored, like torch's -inf padding) ----
__device__ __forceinline__ uint4 hmax8(uint4 a, uint4 b) {
    uint4 r;
    const __half2* x = reinterpret_cast<const __half2*>(&a);
    const __half2* y = reinterpret_cast<const __half2*>(&b);
    __half2* z = reinterpret_cast<__half2*>(&r);
#pragma unroll
    for (int j = 0; j < 4; ++j) z[j] = __hmax2(x[j], y[j]);
    return r;
}

__global__ void maxpool_kernel(const __half* __restrict__ in, int in_ld, int B, int H, int W, int C, int k, int s, int p,
                               __half* __restrict__ out, int out_ld, int Ho, int Wo) {
    const int c8 = C >> 3;
    const long long total = (long long)B * Ho * Wo * c8;
    const int Hp = H + 2, Wp = W + 2, Hop = Ho + 2, Wop = Wo + 2;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int cg = (int)(i % c8);
        long long t = i / c8;
        const int xo = (int)(t % Wo); t /= Wo;
        const int yo = (int)(t % Ho);
        const int b = (int)(t / Ho);
        const __half ninf = __ushort_as_half((unsigned short)0xFC00);
        const __half2 n2 = __halves2half2(ninf, ninf);
        uint4 m;
        __half2* mm = reinterpret_cast<__half2*>(&m);
        mm[0] = n2; mm[1] = n2; mm[2] = n2; mm[3] = n2;
        for (int dy = 0; dy < k; ++dy) {
            const int yi = yo * s - p + dy;
            if (yi < 0 || yi >= H) continue;
            for (int dx = 0; dx < k; ++dx) {
                const int xi = xo * s - p + dx;
                if (xi < 0 || xi >= W) continue;
                const size_t r = ((size_t)b * Hp + (yi + 1)) * Wp + (xi + 1);
                m = hmax8(m, *reinterpret_cast<const uint4*>(in + r * in_ld + cg * 8));
            }
        }
        const size_t orow = ((size_t)b * Hop + (yo + 1)) * Wop + (xo + 1);
        *reinterpret_cast<uint4*>(out + orow * out_ld + cg * 8) = m;
    }
}

int launch_maxpool(const __half* in, int in_ld, int B, int H, int W, int C, int k, int s, int p, __half* out, int out_ld,
                   int Ho, int Wo, cudaStream_t st) {
    ADAS_CHECK(C % 8 == 0 && in_ld % 8 == 0 && out_ld % 8 == 0, "maxpool: channel alignment");
    const long long total = (long long)B * Ho * Wo * (C / 8);
    int blocks = grid_for(total, 256);
    if (blocks > 148 * 32) blocks = 148 * 32;
    maxpool_kernel<<<blocks, 256, 0, st>>>(in, in_ld, B, H, W, C, k, s, p, out, out_ld, Ho, Wo);
    count_launch();
    ADAS_CUDA(cudaGetLastError());
    return 0;
}

// ---- nearest upsample x2 into a channel slice of the consumer's concat buffer ---------------------
__global__ void upsample2x_kernel(const __half* __restrict__ in, int in_ld, int B, int H, int W, int C,
                                  __half* __restrict__ out, int out_ld) {
    const int c8 = C >> 3;
    const int Ho = 2 * H, Wo = 2 * W;
    const long long total = (long long)B * Ho * Wo * c8;
    const int Hp = H + 2, Wp = W + 2, Hop = Ho + 2, Wop = Wo + 2;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int cg = (int)(i % c8);
        long long t = i / c8;
        const int xo = (int)(t % Wo); t /= Wo;
        const int yo = (int)(t % Ho);
        const int b = (int)(t / Ho);
        const size_t r = ((size_t)b * Hp + (yo / 2 + 1)) * Wp + (xo / 2 + 1);
        const size_t orow = ((size_t)b * Hop + (yo + 1)) * Wop + (xo + 1);
        *reinterpret_cast<uint4*>(out + orow * out_ld + cg * 8) = *reinterpret_cast<const uint4*>(in + r * in_ld + cg * 8);
    }
}

int launch_upsample2x(const __half* in, int in_ld, int B, int H, int W, int C, __half* out, int out_ld, cudaStream_t st) {
    ADAS_CHECK(C % 8 == 0 && in_ld % 8 == 0 && out_ld % 8 == 0, "upsample: channel alignment");
    const long long total = (long long)B * 4 * H * W * (C / 8);
    int blocks = grid_for(total, 256);
    if (blocks > 148 * 32) blocks = 148 * 32;
    upsample2x_kernel<<<blocks, 256, 0, st>>>(in, in_ld, B, H, W, C, out, out_ld);
    count_launch();
    ADAS_CUDA(cudaGetLastError());
    return 0;
}

// ---- LayerNorm over a feature row (one CTA per row), fp32 statistics ------------------------------
// Block-wide sums of a and b (fixed order: lanes, then warps), returned to every thread.  The leading barrier lets the kernel call
// it twice on the same shared buffer: nobody overwrites it before every thread has read the previous result.
__device__ __forceinline__ void block_sum2(float& a, float& b, float (*red)[32]) {
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
    }
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) { red[0][w] = a; red[1][w] = b; }
    __syncthreads();
    if (w == 0) {
        a = (l < (int)(blockDim.x >> 5)) ? red[0][l] : 0.f;
        b = (l < (int)(blockDim.x >> 5)) ? red[1][l] : 0.f;
        for (int o = 16; o > 0; o >>= 1) {
            a += __shfl_xor_sync(0xffffffffu, a, o);
            b += __shfl_xor_sync(0xffffffffu, b, o);
        }
        if (l == 0) { red[0][0] = a; red[1][0] = b; }
    }
    __syncthreads();
    a = red[0][0];
    b = red[1][0];
}

// Two passes over the row (the UFLD slab is 10 KB, re-read from L1): the mean, then the squared deviations from it.  The one-pass
// E[x^2] - mean^2 loses the variance to cancellation once |mean| / std nears 100 (pool-conv features with a large bias).  The
// d_len - d_norm structural entries of the slab are zeros (plan.h), so the second pass skips zero entries and adds the real ones
// among them back as (Dn - nonzeros) * mean^2.
__global__ void layernorm_kernel(const __half* __restrict__ in, int in_ld, int D, int Dn, const float* __restrict__ gamma,
                                 const float* __restrict__ beta, float eps, __half* __restrict__ out, int out_ld) {
    const int row = blockIdx.x;
    const __half* x = in + (size_t)row * in_ld;
    __shared__ float red[2][32];
    float s = 0.f, unused = 0.f;
    for (int i = threadIdx.x; i < D; i += blockDim.x) s += __half2float(x[i]);
    block_sum2(s, unused, red);
    const float mean = s / Dn;
    float q = 0.f, nz = 0.f;
    for (int i = threadIdx.x; i < D; i += blockDim.x) {
        const float v = __half2float(x[i]);
        if (v != 0.f) {
            const float d = v - mean;
            q += d * d;
            nz += 1.f;
        }
    }
    block_sum2(q, nz, red);
    const float var = fmaxf((q + ((float)Dn - nz) * mean * mean) / Dn, 0.f);
    const float rstd = rsqrtf(var + eps);
    for (int i = threadIdx.x; i < D; i += blockDim.x) {
        const float v = (__half2float(x[i]) - mean) * rstd * gamma[i] + beta[i];
        out[(size_t)row * out_ld + i] = __float2half_rn(v);
    }
}

int launch_layernorm(const __half* in, int in_ld, int rows, int d_len, int d_norm, const float* gamma, const float* beta,
                     float eps, __half* out, int out_ld, cudaStream_t st) {
    layernorm_kernel<<<rows, 256, 0, st>>>(in, in_ld, d_len, d_norm, gamma, beta, eps, out, out_ld);
    count_launch();
    ADAS_CUDA(cudaGetLastError());
    return 0;
}

// ---- fp32 NCHW input binding -> fp16 padded NHWC (C padded to out_ld, extra channels zero) ------------
__global__ void nchw_to_padded_kernel(const float* __restrict__ in, int B, int C, int H, int W, __half* __restrict__ out,
                                      int out_ld) {
    const long long total = (long long)B * H * W;
    const int Hp = H + 2, Wp = W + 2;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int x = (int)(i % W);
        long long t = i / W;
        const int y = (int)(t % H);
        const int b = (int)(t / H);
        const size_t orow = ((size_t)b * Hp + (y + 1)) * Wp + (x + 1);
        for (int c = 0; c < out_ld; ++c) {
            float v = 0.f;
            if (c < C) v = in[(((size_t)b * C + c) * H + y) * W + x];
            out[orow * out_ld + c] = __float2half_rn(v);
        }
    }
}

int launch_nchw_to_padded(const float* in, int B, int C, int H, int W, __half* out, int out_ld, cudaStream_t st) {
    const long long total = (long long)B * H * W;
    int blocks = grid_for(total, 256);
    if (blocks > 148 * 16) blocks = 148 * 16;
    nchw_to_padded_kernel<<<blocks, 256, 0, st>>>(in, B, C, H, W, out, out_ld);
    count_launch();
    ADAS_CUDA(cudaGetLastError());
    return 0;
}

// ---- 7x7 stride-2 stem re-layout ---------------------------------------------------------------------
// Q[b][yy = j][xo+1][p*32 + kx*4 + c] = img[b][2j-1+p][2xo+kx-3][c]   (j = 0 .. Ho, p = 0,1, kx = 0..6, c = 0..3; kx = 7 is zero)
// written on the padded grid of the stem OUTPUT (Ho x Wo): row yy = j holds the input-row pair (2j-1, 2j).  One thread writes the
// 16 bytes of two horizontal taps (kx, kx+1) of one pair half; the image (4 MB per frame) stays in L2 while it is re-read.
__global__ void stempack_kernel(const __half* __restrict__ img, int B, int H, int W, __half* __restrict__ q) {
    const int Ho = H >> 1, Wo = W >> 1;
    const long long total = (long long)B * (Ho + 1) * Wo * 8;     // 8 chunks of 16 B per Q pixel
    const int Hp = H + 2, Wp = W + 2, Hop = Ho + 2, Wop = Wo + 2;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int ch = (int)(i & 7);                 // chunk: p = ch >> 2, kx pair = (ch & 3) * 2
        long long t = i >> 3;
        const int xo = (int)(t % Wo); t /= Wo;
        const int j = (int)(t % (Ho + 1));
        const int b = (int)(t / (Ho + 1));
        const int pp = ch >> 2, kx0 = (ch & 3) * 2;
        const int y = 2 * j - 1 + pp;
        uint2 v0 = make_uint2(0u, 0u), v1 = make_uint2(0u, 0u);
        if (y >= 0 && y < H) {
            const int x0 = 2 * xo + kx0 - 3, x1 = x0 + 1;
            const __half* row = img + ((size_t)b * Hp + (y + 1)) * Wp * 4;
            if (x0 >= 0 && x0 < W) v0 = *reinterpret_cast<const uint2*>(row + (size_t)(x0 + 1) * 4);
            if (kx0 + 1 < 7 && x1 >= 0 && x1 < W) v1 = *reinterpret_cast<const uint2*>(row + (size_t)(x1 + 1) * 4);
        }
        const size_t orow = ((size_t)b * Hop + j) * Wop + (xo + 1);
        *reinterpret_cast<uint4*>(q + orow * 64 + ch * 8) = make_uint4(v0.x, v0.y, v1.x, v1.y);
    }
}

int launch_stempack(const __half* img, int B, int H, int W, __half* q, cudaStream_t st) {
    const long long total = (long long)B * (H / 2 + 1) * (W / 2) * 8;
    int blocks = grid_for(total, 256);
    if (blocks > 148 * 16) blocks = 148 * 16;
    stempack_kernel<<<blocks, 256, 0, st>>>(img, B, H, W, q);
    count_launch();
    ADAS_CUDA(cudaGetLastError());
    return 0;
}

int launch_zero_rows(__half* buf, int ld, int C, int row0, int nrows, cudaStream_t st) {
    ADAS_CUDA(cudaMemset2DAsync(buf + (size_t)row0 * ld, (size_t)ld * 2, 0, (size_t)C * 2, nrows, st));
    return 0;
}

}  // namespace adas

namespace adas {
// ---- fully connected layer at small batch: weight-streaming kernel ------------------------------------------------------------
// Replaces the first Linear of the UFLDv2 head (exportLib/ultrafastLaneV2/model_culane.py:35-37, `cls` Sequential) at the batch
// sizes the pipeline uses: out[b][n] = act(bias[n] + sum_k x[b][k] * W[n][k]).  At batch <= 32 the layer is a stream of the
// weight matrix (FC1: 2048 x 4992 fp16 = 20 MB, L2-resident): the swap-AB tensor-core GEMM had 8 CTAs for it (47.8 us, 0.43 TB/s).
// One CTA owns FC_F output features and 8 batch rows; its 8 warps split K, lanes stride over 16-byte chunks (8 independent weight
// loads per lane per step), fp32 accumulation, fixed-order reduction (xor-shuffle over lanes, then warps in ascending order).  Every (b, n) value is computed by the same instruction sequence whatever the batch size (batch rows are independent
// accumulators), so per-frame results do not depend on the batch.
static constexpr int FC_F = 8;          // output features per CTA
static constexpr int FC_WARPS = 8;      // each warp owns one K slice of all FC_F features (many independent 16-byte loads in flight)

__global__ void __launch_bounds__(32 * FC_WARPS)
fc_stream_kernel(const __half* __restrict__ x, int x_ld, int batch, const __half* __restrict__ W, int K, int N, const float* __restrict__ bias,
                 int act, void* __restrict__ out, int out_ld, int out_f32) {
    __shared__ float part[FC_WARPS][FC_F][8];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n0 = blockIdx.x * FC_F;
    const int b0 = blockIdx.y * 8;
    const int nb = min(8, batch - b0);
    // K slice of this warp, in 8-element (16-byte) chunks
    const int chunks = K >> 3;
    const int per = (chunks + FC_WARPS - 1) / FC_WARPS;
    const int c0 = warp * per, c1 = min(chunks, c0 + per);
    float acc[FC_F][8];
#pragma unroll
    for (int f = 0; f < FC_F; ++f)
#pragma unroll
        for (int b = 0; b < 8; ++b) acc[f][b] = 0.f;
    for (int c = c0 + lane; c < c1; c += 32) {
        const int k = c << 3;
        uint4 w4[FC_F];
#pragma unroll
        for (int f = 0; f < FC_F; ++f) {
            const int n = min(n0 + f, N - 1);
            w4[f] = __ldg(reinterpret_cast<const uint4*>(W + (size_t)n * K + k));
        }
#pragma unroll
        for (int b = 0; b < 8; ++b) {
            if (b < nb) {
                const uint4 x4 = __ldg(reinterpret_cast<const uint4*>(x + (size_t)(b0 + b) * x_ld + k));
                const __half2* xh = reinterpret_cast<const __half2*>(&x4);
                float2 xf[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) xf[j] = __half22float2(xh[j]);
#pragma unroll
                for (int f = 0; f < FC_F; ++f) {
                    const __half2* wh = reinterpret_cast<const __half2*>(&w4[f]);
                    float a = acc[f][b];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float2 wf = __half22float2(wh[j]);
                        a = fmaf(wf.x, xf[j].x, a);
                        a = fmaf(wf.y, xf[j].y, a);
                    }
                    acc[f][b] = a;
                }
            }
        }
    }
    // fixed-order reduction: lanes (xor tree), then warps (ascending) -- the same sequence whatever the batch size
#pragma unroll
    for (int f = 0; f < FC_F; ++f)
#pragma unroll
        for (int b = 0; b < 8; ++b) {
            float v = acc[f][b];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == 0) part[warp][f][b] = v;
        }
    __syncthreads();
    if (threadIdx.x < FC_F * 8) {
        const int f = threadIdx.x >> 3, b = threadIdx.x & 7;
        const int n = n0 + f;
        if (n < N && b < nb) {
            float v = 0.f;
#pragma unroll
            for (int w = 0; w < FC_WARPS; ++w) v += part[w][f][b];
            v += bias ? bias[n] : 0.f;
            if (act == 1) v = v / (1.f + __expf(-v));
            else if (act == 2) v = fmaxf(v, 0.f);
            const size_t o = (size_t)(b0 + b) * out_ld + n;
            if (out_f32) reinterpret_cast<float*>(out)[o] = v;
            else reinterpret_cast<__half*>(out)[o] = __float2half_rn(v);
        }
    }
}

int launch_fc_stream(const __half* x, int x_ld, int batch, const __half* W, int K, int N, const float* bias, int act, void* out, int out_ld,
                     int out_f32, cudaStream_t st) {
    ADAS_CHECK(K % 8 == 0 && x_ld % 8 == 0, "fc_stream: K (%d) and the activation row stride (%d) must be multiples of 8", K, x_ld);
    dim3 grid((N + FC_F - 1) / FC_F, (batch + 7) / 8, 1);
    fc_stream_kernel<<<grid, 32 * FC_WARPS, 0, st>>>(x, x_ld, batch, W, K, N, bias, act, out, out_ld, out_f32);
    count_launch();
    ADAS_CUDA(cudaGetLastError());
    return 0;
}
}  // namespace adas
