// mortal_b200 — fused elementwise kernels for the policy-net inference path (mortal/model.py ResBlock / ChannelAttention,
// restated in mortal_b200/model.py). The convolutions stay with cuDNN (tcgen05 implicit-GEMM kernels); what PyTorch runs
// between them as 5-6 separate bandwidth-bound passes per block (BatchNorm affine, Mish, two pooling reductions, gate
// multiply, residual add) is done here in three: one 16-byte vector of 8 bf16 channels per thread, NHWC
// (channels-last) activations [B, L, C], fp32 math, one rounding to bf16 at the end.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>

namespace mjx_nn {

struct alignas(16) Vec8 { __nv_bfloat162 v[4]; };

__device__ __forceinline__ float mish_f(float x) {
    // x * tanh(softplus(x)) = x * n / (n + 2) with n = e^x (e^x + 2): tanh(log(1 + e)) = ((1 + e)^2 - 1) / ((1 + e)^2 + 1).
    // One exponential and one reciprocal on the SFU instead of log1pf + tanhf (which made the pass ALU-bound at 4x its HBM time);
    // the ~1e-6 relative error is far below the bf16 rounding of the result. For x > 20 the quotient is 1 in fp32.
    const float e = __expf(fminf(x, 20.f));
    const float n = e * (e + 2.f);
    return x > 20.f ? x : x * __fdividef(n, n + 2.f);
}
__device__ __forceinline__ float bf16_round(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }

// per-thread channel group: the launch's thread count is a multiple of c8 (nn_grid_for), so a thread meets the same 8 channels in
// every iteration of its grid-stride loop and keeps their scale / bias in registers (16 scalar loads per vector otherwise made the
// pass L1-bound at a third of the HBM rate)
__device__ __forceinline__ void ld8(const float* __restrict__ p, float* o) {  // 32-byte aligned
    const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p) + 1);
    o[0] = a.x; o[1] = a.y; o[2] = a.z; o[3] = a.w; o[4] = b.x; o[5] = b.y; o[6] = b.z; o[7] = b.w;
}
struct Affine8 { float s[8], b[8]; };
__device__ __forceinline__ Affine8 load_affine8(const float* __restrict__ scale, const float* __restrict__ bias, int cv) {
    Affine8 a;
    const float4 s0 = __ldg(reinterpret_cast<const float4*>(scale) + 2 * cv), s1 = __ldg(reinterpret_cast<const float4*>(scale) + 2 * cv + 1);
    const float4 b0 = __ldg(reinterpret_cast<const float4*>(bias) + 2 * cv), b1 = __ldg(reinterpret_cast<const float4*>(bias) + 2 * cv + 1);
    a.s[0] = s0.x; a.s[1] = s0.y; a.s[2] = s0.z; a.s[3] = s0.w; a.s[4] = s1.x; a.s[5] = s1.y; a.s[6] = s1.z; a.s[7] = s1.w;
    a.b[0] = b0.x; a.b[1] = b0.y; a.b[2] = b0.z; a.b[3] = b0.w; a.b[4] = b1.x; a.b[5] = b1.y; a.b[6] = b1.z; a.b[7] = b1.w;
    return a;
}
__device__ __forceinline__ Vec8 affine_mish8(const Vec8& in, const Affine8& A) {
    Vec8 o;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const float2 f = __bfloat1622float2(in.v[k]);
        o.v[k] = __floats2bfloat162_rn(mish_f(fmaf(f.x, A.s[2 * k], A.b[2 * k])), mish_f(fmaf(f.y, A.s[2 * k + 1], A.b[2 * k + 1])));
    }
    return o;
}

// out = mish(x * scale[c] + bias[c]); gridDim.x * blockDim.x is a multiple of c8
__global__ void __launch_bounds__(256) k_affine_mish(const Vec8* __restrict__ x, const float* __restrict__ scale,
                                                     const float* __restrict__ bias, Vec8* __restrict__ out, size_t n_vec, int c8) {
    const size_t t0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
    const Affine8 A = load_affine8(scale, bias, (int)(t0 % (size_t)c8));
    size_t v = t0;
    for (; v + stride < n_vec; v += 2 * stride) {  // two independent vectors in flight per thread
        const Vec8 i0 = x[v], i1 = x[v + stride];
        out[v] = affine_mish8(i0, A);
        out[v + stride] = affine_mish8(i1, A);
    }
    if (v < n_vec) out[v] = affine_mish8(x[v], A);
}

// avg[b, c] = mean_l x[b, l, c], mx[b, c] = max_l x[b, l, c]   (ChannelAttention pooling)
__global__ void __launch_bounds__(256) k_pool(const Vec8* __restrict__ x, Vec8* __restrict__ avg, Vec8* __restrict__ mx,
                                              int batch, int length, int c8) {
    const size_t n = (size_t)batch * c8;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const size_t b = i / c8;
        const int cv = (int)(i - b * c8);
        float s[8], m[8];
#pragma unroll
        for (int k = 0; k < 8; k++) { s[k] = 0.f; m[k] = -3.402823466e+38f; }
        const Vec8* p = x + b * (size_t)length * c8 + cv;
        for (int l = 0; l < length; l++) {
            const Vec8 in = p[(size_t)l * c8];
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const float2 f = __bfloat1622float2(in.v[k]);
                s[2 * k] += f.x; s[2 * k + 1] += f.y;
                m[2 * k] = fmaxf(m[2 * k], f.x); m[2 * k + 1] = fmaxf(m[2 * k + 1], f.y);
            }
        }
        Vec8 oa, om;
        const float inv = 1.f / (float)length;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            oa.v[k] = __floats2bfloat162_rn(s[2 * k] * inv, s[2 * k + 1] * inv);
            om.v[k] = __floats2bfloat162_rn(m[2 * k], m[2 * k + 1]);
        }
        avg[i] = oa;
        mx[i] = om;
    }
}

// out = y * gate[b, c] + x   (channel gate + residual)
__global__ void __launch_bounds__(256) k_gate_residual(const Vec8* __restrict__ y, const Vec8* __restrict__ gate,
                                                       const Vec8* __restrict__ x, Vec8* __restrict__ out, size_t n_vec,
                                                       int length, int c8) {
    const size_t per_b = (size_t)length * c8;
    for (size_t v = (size_t)blockIdx.x * blockDim.x + threadIdx.x; v < n_vec; v += (size_t)gridDim.x * blockDim.x) {
        const size_t b = v / per_b;
        const int cv = (int)(v % (size_t)c8);
        const Vec8 yy = y[v], xx = x[v], g = gate[b * c8 + cv];
        Vec8 o;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const float2 fy = __bfloat1622float2(yy.v[k]), fx = __bfloat1622float2(xx.v[k]), fg = __bfloat1622float2(g.v[k]);
            o.v[k] = __floats2bfloat162_rn(fmaf(fy.x, fg.x, fx.x), fmaf(fy.y, fg.y, fx.y));
        }
        out[v] = o;
    }
}

// Channel attention of one batch row by ONE warp (mortal/model.py ChannelAttention): mean / max over the L positions, the gate MLP
// (C -> H -> C, shared by both pooled vectors), sigmoid -> gate[b, c] bf16. Lane cv < c8 owns channels 8 cv .. 8 cv + 7 (c8 <= 32;
// lanes past c8 idle), a position is c8 consecutive 16-byte loads of the warp and eight positions are in flight per lane; the MLP
// weights (w1 [H][C] and w2 TRANSPOSED to [H][C], 2 x 9 KB at C = 192) are read through L1 as two float4 per lane and use.
// fp32 throughout (the bf16 pipeline this replaces rounded the pooled vectors, the hidden layer and the logits); the gate is stored as bf16.
__global__ void __launch_bounds__(256) k_pool_gate(const Vec8* __restrict__ y, const float* __restrict__ w1, const float* __restrict__ b1,
                                                   const float* __restrict__ w2t, const float* __restrict__ b2, Vec8* __restrict__ gate,
                                                   int batch, int length, int c8, int hidden) {
    const int C = c8 * 8;
    const int lane = threadIdx.x & 31, warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
    const bool act = lane < c8;
    const int cv = act ? lane : 0;
    const float inv_len = 1.f / (float)length;
    for (int b = warp; b < batch; b += nwarps) {
        const Vec8* row = y + (size_t)b * length * c8 + cv;
        float s[8], m[8];
#pragma unroll
        for (int k = 0; k < 8; k++) { s[k] = 0.f; m[k] = -3.402823466e+38f; }
        if (act) {
#pragma unroll 8
            for (int l = 0; l < length; l++) {
                const Vec8 in = row[(size_t)l * c8];
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const float2 f = __bfloat1622float2(in.v[k]);
                    s[2 * k] += f.x; s[2 * k + 1] += f.y;
                    m[2 * k] = fmaxf(m[2 * k], f.x); m[2 * k + 1] = fmaxf(m[2 * k + 1], f.y);
                }
            }
        }
#pragma unroll
        for (int k = 0; k < 8; k++) { s[k] = act ? s[k] * inv_len : 0.f; m[k] = act ? m[k] : 0.f; }
        float oa[8], om[8];
#pragma unroll
        for (int k = 0; k < 8; k++) { oa[k] = __ldg(b2 + cv * 8 + k); om[k] = oa[k]; }
        for (int j = 0; j < hidden; j++) {
            float wj[8], vj[8];
            ld8(w1 + j * C + cv * 8, wj);
            ld8(w2t + j * C + cv * 8, vj);
            float pa = 0.f, pm = 0.f;
#pragma unroll
            for (int k = 0; k < 8; k++) { pa = fmaf(wj[k], s[k], pa); pm = fmaf(wj[k], m[k], pm); }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) { pa += __shfl_xor_sync(0xffffffffu, pa, o); pm += __shfl_xor_sync(0xffffffffu, pm, o); }
            const float bj = __ldg(b1 + j);
            const float ha = mish_f(pa + bj), hm = mish_f(pm + bj);
#pragma unroll
            for (int k = 0; k < 8; k++) { oa[k] = fmaf(vj[k], ha, oa[k]); om[k] = fmaf(vj[k], hm, om[k]); }
        }
        if (act) {
            Vec8 g;
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const float z0 = oa[2 * k] + om[2 * k], z1 = oa[2 * k + 1] + om[2 * k + 1];
                g.v[k] = __floats2bfloat162_rn(1.f / (1.f + __expf(-z0)), 1.f / (1.f + __expf(-z1)));
            }
            gate[(size_t)b * c8 + cv] = g;
        }
    }
}

// x_out = y * gate[b, c] + x and a_out = mish(x_out * scale[c] + bias[c]) (the next block's pre-activation) in one streaming pass;
// gridDim.x * blockDim.x is a multiple of c8 (see k_affine_mish)
__global__ void __launch_bounds__(256) k_gate_residual_mish(const Vec8* __restrict__ y, const Vec8* __restrict__ gate, const Vec8* __restrict__ x,
                                                            const float* __restrict__ scale, const float* __restrict__ bias,
                                                            Vec8* __restrict__ x_out, Vec8* __restrict__ a_out, size_t n_vec, int length, int c8) {
    const size_t t0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
    const int cv = (int)(t0 % (size_t)c8);
    const Affine8 A = load_affine8(scale, bias, cv);
    const size_t per_b = (size_t)length * c8;
    for (size_t v = t0; v < n_vec; v += stride) {
        const Vec8 yy = y[v], xx = x[v], g = gate[(v / per_b) * c8 + cv];
        Vec8 xo;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const float2 fy = __bfloat1622float2(yy.v[k]), fx = __bfloat1622float2(xx.v[k]), fg = __bfloat1622float2(g.v[k]);
            xo.v[k] = __floats2bfloat162_rn(fmaf(fy.x, fg.x, fx.x), fmaf(fy.y, fg.y, fx.y));
        }
        x_out[v] = xo;
        a_out[v] = affine_mish8(xo, A);
    }
}

// The network's first step as one pass: observations f32 [batch, channels, length] (libriichi's layout: one row of `length` floats
// per channel) -> bf16 channels-last [batch, length, cpad] with the channel count padded with zeros to a multiple of 64, which is
// what the stem convolution's implicit GEMM wants (PyTorch + cuDNN otherwise run a cast, a layout copy and two padding kernels).
// One CTA = 64 channels of one observation through a shared-memory tile.
// GATHER: output row b is observation rows[b] for b < *count and all zeros past it (a per-engine batch converted straight from the
// environment's observation buffer; the zero rows pad the batch to the bucket a CUDA graph was captured for).
constexpr int NHWC_TC = 64;
template <bool GATHER>
__global__ void __launch_bounds__(256) k_obs_to_nhwc(const float* __restrict__ obs, __nv_bfloat16* __restrict__ out, int channels, int length,
                                                     int cpad, const int* __restrict__ rows, const int* __restrict__ count) {
    extern __shared__ float tile[];  // [NHWC_TC][length + 1]
    const int chunks = cpad / NHWC_TC;
    const int b = blockIdx.x / chunks, c0 = (blockIdx.x - b * chunks) * NHWC_TC;
    int nc = max(0, min(NHWC_TC, channels - c0));  // real channels in this chunk
    size_t src_row = b;
    if constexpr (GATHER) {
        if (b < *count) src_row = (size_t)rows[b];
        else nc = 0;
    }
    const float* src = obs + (src_row * channels + c0) * length;
    const int pitch = length + 1;
    for (int i = threadIdx.x; i < nc * length; i += blockDim.x) {
        const int c = i / length, l = i - c * length;
        tile[c * pitch + l] = src[i];
    }
    __syncthreads();
    __nv_bfloat162* dst = reinterpret_cast<__nv_bfloat162*>(out + ((size_t)b * length) * cpad + c0);
    for (int i = threadIdx.x; i < length * (NHWC_TC / 2); i += blockDim.x) {
        const int l = i / (NHWC_TC / 2), c = (i - l * (NHWC_TC / 2)) * 2;
        const float a = c < nc ? tile[c * pitch + l] : 0.f, bb = c + 1 < nc ? tile[(c + 1) * pitch + l] : 0.f;
        dst[(size_t)l * (cpad / 2) + c / 2] = __floats2bfloat162_rn(a, bb);
    }
}

}  // namespace mjx_nn
