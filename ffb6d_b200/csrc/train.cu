// train.cu -- training-mode pieces of the fusion / RandLA 1x1 layers (sm_100a): batch-statistics
// BatchNorm around the tensor-core GEMMs of fusion_mlp.cu, and the backward of attentive pooling.
//
// Reference layer: pt_utils.Conv2d = conv1x1(bias=False) -> BatchNorm2d -> ReLU / LeakyReLU / none
// (models/pytorch_utils.py:75-129 for the fusion layers, models/RandLA/pytorch_utils.py:35-111 for
// RandLA: eps 1e-6, momentum 0.99).  In training mode BatchNorm normalises with the statistics of the
// batch, which sit between the GEMM and the activation, so the layer runs as
//     z = W * cat(x1, x2)                      ffb6d_fusion_mlp_fwd_ex (tcgen05), z kept for the backward
//     (mean, var) per channel over B x P       bn_stats_kernel + bn_finalize_kernel (also the running stats)
//     y = act((z - mean) * gamma / sqrt(var + eps) + beta)      bn_apply_kernel
// and backwards
//     g' = g * act'(y);  dbeta = sum g';  dgamma = sum g' * xhat           bn_bwd_reduce_kernel
//     dz = gamma * invstd * (g' - dbeta / n - xhat * dgamma / n)            bn_bwd_apply_kernel
//     dW = dz * X^T (ffb6d_fusion_mlp_wgrad),  dX = W^T * dz (the forward GEMM with the transposed weight).
// These kernels are HBM bound: every element of z / g is read once per pass with 128-bit loads; the
// per-channel sums are accumulated in fp32 per thread (<= a few hundred terms) and in fp64 across
// threads, CTAs and frames.
#include "common.cuh"

#include <algorithm>

namespace ffb6d {

constexpr int BN_THREADS = 256;

__device__ __forceinline__ double block_sum(double v, double *red)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) red[wid] = v;
    __syncthreads();
    double t = 0.0;
    for (int w = 0; w < BN_THREADS / 32; ++w) t += red[w];
    return t;
}

// partial[c][s] = (sum, sum of squares) of z[:, c, chunk s] over all frames
__global__ void __launch_bounds__(BN_THREADS)
bn_stats_kernel(const float *__restrict__ z, int B, int C, int P, int chunk, int nsplit, double *__restrict__ partial)
{
    __shared__ double red[BN_THREADS / 32];
    const int c = blockIdx.y, s = blockIdx.x;
    const int p0 = s * chunk, p1 = min(P, p0 + chunk);
    float a = 0.f, q = 0.f;
    const bool vec = ((P & 3) == 0) && ((chunk & 3) == 0) && ((reinterpret_cast<uintptr_t>(z) & 15) == 0);
    for (int b = 0; b < B; ++b) {
        const float *row = z + ((size_t)b * C + c) * P;
        if (vec) {
            for (int p = p0 + 4 * threadIdx.x; p < p1; p += 4 * BN_THREADS) {
                const float4 v = __ldg(reinterpret_cast<const float4 *>(row + p));
                a += (v.x + v.y) + (v.z + v.w);
                q += (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
            }
        } else {
            for (int p = p0 + threadIdx.x; p < p1; p += BN_THREADS) {
                const float v = __ldg(row + p);
                a += v;
                q += v * v;
            }
        }
    }
    const double A = block_sum((double)a, red), Q = block_sum((double)q, red);
    if (threadIdx.x == 0) {
        partial[((size_t)c * nsplit + s) * 2] = A;
        partial[((size_t)c * nsplit + s) * 2 + 1] = Q;
    }
}

// stats[c] = (mean, invstd, gamma * invstd, beta); running statistics updated like torch.nn.BatchNorm2d
__global__ void __launch_bounds__(BN_THREADS)
bn_finalize_kernel(const double *__restrict__ partial, int C, int nsplit, double n, float eps, float momentum,
                   const float *__restrict__ gamma, const float *__restrict__ beta, float *__restrict__ running_mean,
                   float *__restrict__ running_var, float4 *__restrict__ stats)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    double A = 0.0, Q = 0.0;
    for (int s = 0; s < nsplit; ++s) {
        A += partial[((size_t)c * nsplit + s) * 2];
        Q += partial[((size_t)c * nsplit + s) * 2 + 1];
    }
    const double mean = A / n;
    double var = Q / n - mean * mean;   // biased, as BatchNorm normalises with
    if (var < 0.0) var = 0.0;
    const float invstd = (float)(1.0 / sqrt(var + (double)eps));
    const float g = gamma ? gamma[c] : 1.f;
    stats[c] = make_float4((float)mean, invstd, g * invstd, beta ? beta[c] : 0.f);
    if (running_mean) running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * (float)mean;
    if (running_var) {
        const double unbiased = n > 1.0 ? var * n / (n - 1.0) : var;
        running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unbiased;
    }
}

__device__ __forceinline__ float act_fwd(float y, int act, float slope)
{
    if (act == 1) return fmaxf(y, 0.f);
    if (act == 2) return y > 0.f ? y : y * slope;
    return y;
}

// y = act((z - mean) * scale + beta), one (frame, channel) row per blockIdx.y
__global__ void __launch_bounds__(BN_THREADS)
bn_apply_kernel(const float *__restrict__ z, const float4 *__restrict__ stats, int C, int P, int act, float slope,
                float *__restrict__ y)
{
    const size_t row = blockIdx.x;
    const float4 st = stats[row % C];
    const float *src = z + row * P;
    float *dst = y + row * P;
    const bool vec = ((P & 3) == 0) && ((reinterpret_cast<uintptr_t>(z) & 15) == 0) && ((reinterpret_cast<uintptr_t>(y) & 15) == 0);
    if (vec) {
        for (int p = 4 * (blockIdx.y * BN_THREADS + threadIdx.x); p < P; p += 4 * BN_THREADS * gridDim.y) {
            float4 v = __ldg(reinterpret_cast<const float4 *>(src + p));
            v.x = act_fwd(__fmaf_rn(v.x - st.x, st.z, st.w), act, slope);
            v.y = act_fwd(__fmaf_rn(v.y - st.x, st.z, st.w), act, slope);
            v.z = act_fwd(__fmaf_rn(v.z - st.x, st.z, st.w), act, slope);
            v.w = act_fwd(__fmaf_rn(v.w - st.x, st.z, st.w), act, slope);
            *reinterpret_cast<float4 *>(dst + p) = v;
        }
    } else {
        for (int p = blockIdx.y * BN_THREADS + threadIdx.x; p < P; p += BN_THREADS * gridDim.y)
            dst[p] = act_fwd(__fmaf_rn(__ldg(src + p) - st.x, st.z, st.w), act, slope);
    }
}

__device__ __forceinline__ float act_grad(float g, float ypre, int act, float slope)
{
    if (act == 1) return ypre > 0.f ? g : 0.f;
    if (act == 2) return ypre > 0.f ? g : g * slope;
    return g;
}

// partial[c][s] = (sum g', sum g' * xhat) over all frames of chunk s
__global__ void __launch_bounds__(BN_THREADS)
bn_bwd_reduce_kernel(const float *__restrict__ z, const float *__restrict__ g, const float4 *__restrict__ stats, int B, int C,
                     int P, int chunk, int nsplit, int act, float slope, double *__restrict__ partial)
{
    __shared__ double red[BN_THREADS / 32];
    const int c = blockIdx.y, s = blockIdx.x;
    const int p0 = s * chunk, p1 = min(P, p0 + chunk);
    const float4 st = stats[c];
    float a = 0.f, q = 0.f;
    for (int b = 0; b < B; ++b) {
        const float *zr = z + ((size_t)b * C + c) * P, *gr = g + ((size_t)b * C + c) * P;
        for (int p = p0 + threadIdx.x; p < p1; p += BN_THREADS) {
            const float d = __ldg(zr + p) - st.x;
            const float gp = act_grad(__ldg(gr + p), __fmaf_rn(d, st.z, st.w), act, slope);
            a += gp;
            q += gp * (d * st.y);
        }
    }
    const double A = block_sum((double)a, red), Q = block_sum((double)q, red);
    if (threadIdx.x == 0) {
        partial[((size_t)c * nsplit + s) * 2] = A;
        partial[((size_t)c * nsplit + s) * 2 + 1] = Q;
    }
}

// sums[c] = (dbeta, dgamma); also written to grad_beta / grad_gamma
__global__ void __launch_bounds__(BN_THREADS)
bn_bwd_finalize_kernel(const double *__restrict__ partial, int C, int nsplit, float2 *__restrict__ sums,
                       float *__restrict__ grad_gamma, float *__restrict__ grad_beta)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    double A = 0.0, Q = 0.0;
    for (int s = 0; s < nsplit; ++s) {
        A += partial[((size_t)c * nsplit + s) * 2];
        Q += partial[((size_t)c * nsplit + s) * 2 + 1];
    }
    sums[c] = make_float2((float)A, (float)Q);
    if (grad_beta) grad_beta[c] = (float)A;
    if (grad_gamma) grad_gamma[c] = (float)Q;
}

// dz = scale * (g' - dbeta / n - xhat * dgamma / n)
__global__ void __launch_bounds__(BN_THREADS)
bn_bwd_apply_kernel(const float *__restrict__ z, const float *__restrict__ g, const float4 *__restrict__ stats,
                    const float2 *__restrict__ sums, int C, int P, float inv_n, int act, float slope, float *__restrict__ dz)
{
    const size_t row = blockIdx.x;
    const int c = (int)(row % C);
    const float4 st = stats[c];
    const float2 sm = sums[c];
    const float mb = sm.x * inv_n, mg = sm.y * inv_n;
    const float *zr = z + row * P, *gr = g + row * P;
    float *dr = dz + row * P;
    for (int p = blockIdx.y * BN_THREADS + threadIdx.x; p < P; p += BN_THREADS * gridDim.y) {
        const float d = __ldg(zr + p) - st.x;
        const float gp = act_grad(__ldg(gr + p), __fmaf_rn(d, st.z, st.w), act, slope);
        dr[p] = st.z * (gp - mb - (d * st.y) * mg);
    }
}

// ------------------------------------------------------------------ BatchNorm split at the reduction (SyncBatchNorm)
// The entry points ffb6d_bn_train_{stats,apply,bwd_stats,bwd_apply} run the kernels above with the per-channel fp64
// sums handed to the caller in between, so that they can be all-reduced across ranks.  Each kernel below repeats the
// arithmetic of its single-GPU counterpart expression for expression: at one rank the split path is bit-identical.

// sums[c] = (sum over s of partial[c][s]) in ascending s, as bn_finalize_kernel / bn_bwd_finalize_kernel add them;
// with grad_beta / grad_gamma, also their float roundings (the local dbeta, dgamma)
__global__ void __launch_bounds__(BN_THREADS)
bn_partial_sums_kernel(const double *__restrict__ partial, int C, int nsplit, double *__restrict__ sums,
                       float *__restrict__ grad_gamma, float *__restrict__ grad_beta)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    double A = 0.0, Q = 0.0;
    for (int s = 0; s < nsplit; ++s) {
        A += partial[((size_t)c * nsplit + s) * 2];
        Q += partial[((size_t)c * nsplit + s) * 2 + 1];
    }
    sums[2 * (size_t)c] = A;
    sums[2 * (size_t)c + 1] = Q;
    if (grad_beta) grad_beta[c] = (float)A;
    if (grad_gamma) grad_gamma[c] = (float)Q;
}

// bn_finalize_kernel with the partials already added up (sums[c] = (sum z, sum z^2) over n elements of all ranks)
__global__ void __launch_bounds__(BN_THREADS)
bn_finalize_sums_kernel(const double *__restrict__ sums, int C, double n, float eps, float momentum,
                        const float *__restrict__ gamma, const float *__restrict__ beta, float *__restrict__ running_mean,
                        float *__restrict__ running_var, float4 *__restrict__ stats)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const double A = sums[2 * (size_t)c], Q = sums[2 * (size_t)c + 1];
    const double mean = A / n;
    double var = Q / n - mean * mean;
    if (var < 0.0) var = 0.0;
    const float invstd = (float)(1.0 / sqrt(var + (double)eps));
    const float g = gamma ? gamma[c] : 1.f;
    stats[c] = make_float4((float)mean, invstd, g * invstd, beta ? beta[c] : 0.f);
    if (running_mean) running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * (float)mean;
    if (running_var) {
        const double unbiased = n > 1.0 ? var * n / (n - 1.0) : var;
        running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unbiased;
    }
}

// bn_bwd_apply_kernel reading the fp64 sums (sum g', sum g' * xhat) of all ranks, rounded to float as
// bn_bwd_finalize_kernel rounds them
__global__ void __launch_bounds__(BN_THREADS)
bn_bwd_apply_sums_kernel(const float *__restrict__ z, const float *__restrict__ g, const float4 *__restrict__ stats,
                         const double *__restrict__ sums, int C, int P, float inv_n, int act, float slope,
                         float *__restrict__ dz)
{
    const size_t row = blockIdx.x;
    const int c = (int)(row % C);
    const float4 st = stats[c];
    const float2 sm = make_float2((float)sums[2 * (size_t)c], (float)sums[2 * (size_t)c + 1]);
    const float mb = sm.x * inv_n, mg = sm.y * inv_n;
    const float *zr = z + row * P, *gr = g + row * P;
    float *dr = dz + row * P;
    for (int p = blockIdx.y * BN_THREADS + threadIdx.x; p < P; p += BN_THREADS * gridDim.y) {
        const float d = __ldg(zr + p) - st.x;
        const float gp = act_grad(__ldg(gr + p), __fmaf_rn(d, st.z, st.w), act, slope);
        dr[p] = st.z * (gp - mb - (d * st.y) * mg);
    }
}

// activation backward alone (a layer without BatchNorm but with an activation): dz = g * act'(z)
__global__ void __launch_bounds__(BN_THREADS)
act_bwd_kernel(const float *__restrict__ z, const float *__restrict__ g, long long n, int act, float slope, float *__restrict__ dz)
{
    for (long long i = (long long)blockIdx.x * BN_THREADS + threadIdx.x; i < n; i += (long long)gridDim.x * BN_THREADS)
        dz[i] = act_grad(__ldg(g + i), __ldg(z + i), act, slope);
}

// ------------------------------------------------------------------ attentive pooling backward
// forward: out[b,c,n] = sum_k f[k] * s[k], s = softmax_k(att)   (models/RandLA/RandLANet.py:245-248)
// backward: df[k] = g * s[k];  datt[k] = s[k] * g * (f[k] - out).  One thread per (b, c, n); with KT = 16 the
// thread's 64-byte rows of f / att / df / datt move as four 128-bit accesses each and exp is evaluated once.
template <int KT>
__global__ void __launch_bounds__(256)
att_pool_bwd_kernel(const float *__restrict__ f1, int C1, const float *__restrict__ f2, int C2, const float *__restrict__ att,
                    const float *__restrict__ gout, int N, int K, float *__restrict__ gf1, float *__restrict__ gf2,
                    float *__restrict__ gatt, long long total)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // (b*C + c)*N + n
    if (t >= total) return;
    const int C = C1 + C2;
    const int n = (int)(t % N);
    const int c = (int)((t / N) % C);
    const int b = (int)(t / ((long long)N * C));
    const size_t foff = (c < C1) ? (((size_t)b * C1 + c) * N + n) * K : (((size_t)b * C2 + (c - C1)) * N + n) * K;
    const float *fp = (c < C1) ? f1 + foff : f2 + foff;
    float *gfp = (c < C1) ? gf1 + foff : gf2 + foff;
    const float *ap = att + (size_t)t * K;
    float *gap = gatt + (size_t)t * K;
    const float g = __ldg(gout + t);
    if constexpr (KT > 0) {
        float fv[KT], av[KT];
#pragma unroll
        for (int q = 0; q < KT / 4; ++q) {
            const float4 u = __ldg(reinterpret_cast<const float4 *>(fp) + q), v = __ldg(reinterpret_cast<const float4 *>(ap) + q);
            fv[4 * q] = u.x; fv[4 * q + 1] = u.y; fv[4 * q + 2] = u.z; fv[4 * q + 3] = u.w;
            av[4 * q] = v.x; av[4 * q + 1] = v.y; av[4 * q + 2] = v.z; av[4 * q + 3] = v.w;
        }
        float m = av[0];
#pragma unroll
        for (int k = 1; k < KT; ++k) m = fmaxf(m, av[k]);
        float den = 0.f;
#pragma unroll
        for (int k = 0; k < KT; ++k) {
            av[k] = expf(av[k] - m);
            den += av[k];
        }
        float out = 0.f;
#pragma unroll
        for (int k = 0; k < KT; ++k) {
            av[k] = av[k] / den;
            out += fv[k] * av[k];
        }
#pragma unroll
        for (int q = 0; q < KT / 4; ++q) {
            float4 a, d;
            a.x = g * av[4 * q]; a.y = g * av[4 * q + 1]; a.z = g * av[4 * q + 2]; a.w = g * av[4 * q + 3];
            d.x = a.x * (fv[4 * q] - out); d.y = a.y * (fv[4 * q + 1] - out);
            d.z = a.z * (fv[4 * q + 2] - out); d.w = a.w * (fv[4 * q + 3] - out);
            reinterpret_cast<float4 *>(gfp)[q] = a;
            reinterpret_cast<float4 *>(gap)[q] = d;
        }
    } else {
        float m = __ldg(ap);
        for (int k = 1; k < K; ++k) m = fmaxf(m, __ldg(ap + k));
        float den = 0.f;
        for (int k = 0; k < K; ++k) den += expf(__ldg(ap + k) - m);
        float out = 0.f;
        for (int k = 0; k < K; ++k) out += __ldg(fp + k) * (expf(__ldg(ap + k) - m) / den);
        for (int k = 0; k < K; ++k) {
            const float s = expf(__ldg(ap + k) - m) / den;
            gfp[k] = g * s;
            gap[k] = s * g * (__ldg(fp + k) - out);
        }
    }
}

// ------------------------------------------------------------------ weight gradient of NARROW layers
// dW[co, ci] = sum_{b,p} dz[b, co, p] * x[b, ci, p] for Co, Ci <= 64 (the RandLA layers on [B, C, N, K] tensors:
// 10 -> 16 ... 64 -> 64 channels over millions of positions).  A 128 x 128 tensor-core tile would be > 90 % padding
// there and the k-loop latency bound; this is a streaming reduction instead: a CTA takes a run of positions, stages
// 64-position slabs of dz and x in shared memory (coalesced along p) and every thread accumulates a 4 x 4 block of
// dW in registers (fp32 FMA); CTA partials are added to dW with atomics.
constexpr int WS_TP = 64;    // positions per slab
// T = tile edge (16, 32, 64: the smallest that holds Co and Ci); a thread owns a (T/16) x (T/16) block of dW and
// walks the slab four positions at a time with 128-bit shared-memory loads.
template <int T>
__global__ void __launch_bounds__(256)
wgrad_small_kernel(const float *__restrict__ dz, const float *__restrict__ x1, int C1, const float *__restrict__ x2, int C2,
                   float *__restrict__ dw, int Co, int P, int B, int slabs_per_cta)
{
    constexpr int R = T / 16;                    // rows of dz / x per thread
    constexpr int LD = WS_TP + 4;                // row stride: 16-byte aligned rows, conflict-free 128-bit loads
    __shared__ __align__(16) float sz[T * LD], sx[T * LD];
    const int Ci = C1 + C2;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;     // dW rows R*ty .., columns R*tx ..
    float acc[R][R];
#pragma unroll
    for (int i = 0; i < R; ++i)
#pragma unroll
        for (int j = 0; j < R; ++j) acc[i][j] = 0.f;
    const long long slabs_per_frame = (P + WS_TP - 1) / WS_TP, total = slabs_per_frame * B;
    const long long s0 = (long long)blockIdx.x * slabs_per_cta, s1 = min(total, s0 + slabs_per_cta);
    for (long long sl = s0; sl < s1; ++sl) {
        const int b = (int)(sl / slabs_per_frame), p0 = (int)(sl % slabs_per_frame) * WS_TP;
        __syncthreads();
        for (int t = threadIdx.x; t < T * WS_TP; t += 256) {
            const int r = t / WS_TP, p = t % WS_TP;
            const bool in = p0 + p < P;
            sz[r * LD + p] = (in && r < Co) ? __ldg(dz + ((size_t)b * Co + r) * P + p0 + p) : 0.f;
            float v = 0.f;
            if (in && r < Ci) v = (r < C1) ? __ldg(x1 + ((size_t)b * C1 + r) * P + p0 + p) : __ldg(x2 + ((size_t)b * C2 + (r - C1)) * P + p0 + p);
            sx[r * LD + p] = v;
        }
        __syncthreads();
#pragma unroll 4
        for (int p = 0; p < WS_TP; p += 4) {
            float4 a[R], c[R];
#pragma unroll
            for (int i = 0; i < R; ++i) {
                a[i] = *reinterpret_cast<const float4 *>(sz + (R * ty + i) * LD + p);
                c[i] = *reinterpret_cast<const float4 *>(sx + (R * tx + i) * LD + p);
            }
#pragma unroll
            for (int i = 0; i < R; ++i)
#pragma unroll
                for (int j = 0; j < R; ++j)
                    acc[i][j] = fmaf(a[i].x, c[j].x, fmaf(a[i].y, c[j].y, fmaf(a[i].z, c[j].z, fmaf(a[i].w, c[j].w, acc[i][j]))));
        }
    }
#pragma unroll
    for (int i = 0; i < R; ++i)
#pragma unroll
        for (int j = 0; j < R; ++j) {
            const int co = R * ty + i, ci = R * tx + j;
            if (co < Co && ci < Ci && acc[i][j] != 0.f) atomicAdd(dw + (size_t)co * Ci + ci, acc[i][j]);
        }
}

static void split_plan(int64_t C, int64_t P, int &chunk, int &nsplit)
{
    // enough CTAs to fill the machine twice, chunks of whole 1024-element strides
    int64_t want = std::max<int64_t>(1, ceil_div(2 * (int64_t)num_sms(), C));
    int64_t ch = ceil_div(ceil_div(P, want), 1024) * 1024;
    if (ch < 1024) ch = 1024;
    chunk = (int)ch;
    nsplit = (int)ceil_div(P, ch);
}

// narrow layers (Co, Ci <= 64) of ffb6d_fusion_mlp_wgrad: CUDA-core streaming reduction
int wgrad_small_launch(const float *grad_z, const float *x1, int64_t C1, const float *x2, int64_t C2, int64_t B, int64_t Co,
                      int64_t P, float *grad_w, cudaStream_t st_in)
{
    cudaStream_t st = st_in;
    const long long slabs = ceil_div(P, WS_TP) * B;
    const int per = (int)std::max<long long>(1, ceil_div(slabs, 4ll * num_sms()));
    const unsigned grid = (unsigned)ceil_div(slabs, per);
    const int64_t m = std::max<int64_t>(Co, C1 + C2);
    if (m <= 16)
        wgrad_small_kernel<16><<<grid, 256, 0, st>>>(grad_z, x1, (int)C1, C2 ? x2 : nullptr, (int)C2, grad_w, (int)Co, (int)P, (int)B, per);
    else if (m <= 32)
        wgrad_small_kernel<32><<<grid, 256, 0, st>>>(grad_z, x1, (int)C1, C2 ? x2 : nullptr, (int)C2, grad_w, (int)Co, (int)P, (int)B, per);
    else
        wgrad_small_kernel<64><<<grid, 256, 0, st>>>(grad_z, x1, (int)C1, C2 ? x2 : nullptr, (int)C2, grad_w, (int)Co, (int)P, (int)B, per);
    FFB6D_LAUNCH_OK("wgrad_small_kernel");
    return FFB6D_OK;
}

}  // namespace ffb6d

using namespace ffb6d;

extern "C" {

size_t ffb6d_bn_workspace_bytes(int64_t C, int64_t P)
{
    if (C < 1 || P < 1) return 0;
    int chunk, nsplit;
    split_plan(C, P, chunk, nsplit);
    return align_up((size_t)C * nsplit * 2 * sizeof(double), 256) + align_up((size_t)C * sizeof(float2), 256);
}

int ffb6d_bn_train_fwd(const float *z, int64_t B, int64_t C, int64_t P, const float *gamma, const float *beta, float eps,
                       float momentum, float *running_mean, float *running_var, int act, float negative_slope,
                       float *stats, float *y, void *workspace, size_t workspace_bytes, ffb6d_stream_t stream)
{
    FFB6D_CHECK_ARG(B >= 1 && C >= 1 && P >= 1 && B < 65536 && C <= 65535 && P < (1ll << 31) && B * C < (1ll << 31),
                    "bn_train_fwd: bad size");
    FFB6D_CHECK_ARG(z && stats && y && workspace, "bn_train_fwd: null pointer");
    FFB6D_CHECK_ARG(act >= 0 && act <= 2, "bn_train_fwd: act=%d", act);
    FFB6D_CHECK_ARG(workspace_bytes >= ffb6d_bn_workspace_bytes(C, P), "bn_train_fwd: workspace too small");
    FFB6D_CHECK_ARG((reinterpret_cast<uintptr_t>(stats) & 15) == 0, "bn_train_fwd: stats must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    int chunk, nsplit;
    split_plan(C, P, chunk, nsplit);
    double *partial = (double *)workspace;
    bn_stats_kernel<<<dim3((unsigned)nsplit, (unsigned)C), BN_THREADS, 0, st>>>(z, (int)B, (int)C, (int)P, chunk, nsplit, partial);
    FFB6D_LAUNCH_OK("bn_stats_kernel");
    bn_finalize_kernel<<<(unsigned)ceil_div(C, BN_THREADS), BN_THREADS, 0, st>>>(
        partial, (int)C, nsplit, (double)B * (double)P, eps, momentum, gamma, beta, running_mean, running_var, (float4 *)stats);
    FFB6D_LAUNCH_OK("bn_finalize_kernel");
    const unsigned gx = (unsigned)std::min<int64_t>(ceil_div(P, 4 * BN_THREADS), 64);
    bn_apply_kernel<<<dim3((unsigned)(B * C), gx), BN_THREADS, 0, st>>>(z, (const float4 *)stats, (int)C, (int)P, act,
                                                                        negative_slope, y);
    FFB6D_LAUNCH_OK("bn_apply_kernel");
    return FFB6D_OK;
}

int ffb6d_bn_train_bwd(const float *z, const float *grad_y, const float *stats, int64_t B, int64_t C, int64_t P, int act,
                       float negative_slope, float *grad_gamma, float *grad_beta, float *grad_z, void *workspace,
                       size_t workspace_bytes, ffb6d_stream_t stream)
{
    FFB6D_CHECK_ARG(B >= 1 && C >= 1 && P >= 1 && B < 65536 && C <= 65535 && P < (1ll << 31) && B * C < (1ll << 31),
                    "bn_train_bwd: bad size");
    FFB6D_CHECK_ARG(z && grad_y && stats && grad_z && workspace, "bn_train_bwd: null pointer");
    FFB6D_CHECK_ARG(workspace_bytes >= ffb6d_bn_workspace_bytes(C, P), "bn_train_bwd: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    int chunk, nsplit;
    split_plan(C, P, chunk, nsplit);
    double *partial = (double *)workspace;
    float2 *sums = (float2 *)((char *)workspace + align_up((size_t)C * nsplit * 2 * sizeof(double), 256));
    bn_bwd_reduce_kernel<<<dim3((unsigned)nsplit, (unsigned)C), BN_THREADS, 0, st>>>(
        z, grad_y, (const float4 *)stats, (int)B, (int)C, (int)P, chunk, nsplit, act, negative_slope, partial);
    FFB6D_LAUNCH_OK("bn_bwd_reduce_kernel");
    bn_bwd_finalize_kernel<<<(unsigned)ceil_div(C, BN_THREADS), BN_THREADS, 0, st>>>(partial, (int)C, nsplit, sums, grad_gamma,
                                                                                    grad_beta);
    FFB6D_LAUNCH_OK("bn_bwd_finalize_kernel");
    const unsigned gx = (unsigned)std::min<int64_t>(ceil_div(P, BN_THREADS), 64);
    bn_bwd_apply_kernel<<<dim3((unsigned)(B * C), gx), BN_THREADS, 0, st>>>(
        z, grad_y, (const float4 *)stats, sums, (int)C, (int)P, (float)(1.0 / ((double)B * (double)P)), act, negative_slope, grad_z);
    FFB6D_LAUNCH_OK("bn_bwd_apply_kernel");
    return FFB6D_OK;
}

#define FFB6D_BN_SIZES_OK(who)                                                                                           \
    FFB6D_CHECK_ARG(B >= 1 && C >= 1 && P >= 1 && B < 65536 && C <= 65535 && P < (1ll << 31) && B * C < (1ll << 31), \
                    who ": bad size")
#define FFB6D_BN_COUNT_OK(who)                                                                                   \
    FFB6D_CHECK_ARG(count >= (double)B * (double)P && count < 9.007199254740992e15, who ": count %g outside [B*P = %lld, 2^53)", \
                    count, (long long)(B * P))

int ffb6d_bn_train_stats(const float *z, int64_t B, int64_t C, int64_t P, double *sums, void *workspace,
                         size_t workspace_bytes, ffb6d_stream_t stream)
{
    FFB6D_BN_SIZES_OK("bn_train_stats");
    FFB6D_CHECK_ARG(z && sums && workspace, "bn_train_stats: null pointer");
    FFB6D_CHECK_ARG((reinterpret_cast<uintptr_t>(sums) & 7) == 0, "bn_train_stats: sums must be 8-byte aligned");
    FFB6D_CHECK_ARG(workspace_bytes >= ffb6d_bn_workspace_bytes(C, P), "bn_train_stats: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    int chunk, nsplit;
    split_plan(C, P, chunk, nsplit);
    double *partial = (double *)workspace;
    bn_stats_kernel<<<dim3((unsigned)nsplit, (unsigned)C), BN_THREADS, 0, st>>>(z, (int)B, (int)C, (int)P, chunk, nsplit, partial);
    FFB6D_LAUNCH_OK("bn_stats_kernel");
    bn_partial_sums_kernel<<<(unsigned)ceil_div(C, BN_THREADS), BN_THREADS, 0, st>>>(partial, (int)C, nsplit, sums, nullptr,
                                                                                    nullptr);
    FFB6D_LAUNCH_OK("bn_partial_sums_kernel");
    return FFB6D_OK;
}

int ffb6d_bn_train_apply(const float *z, int64_t B, int64_t C, int64_t P, const double *sums, double count,
                         const float *gamma, const float *beta, float eps, float momentum, float *running_mean,
                         float *running_var, int act, float negative_slope, float *stats, float *y, ffb6d_stream_t stream)
{
    FFB6D_BN_SIZES_OK("bn_train_apply");
    FFB6D_CHECK_ARG(z && sums && stats && y, "bn_train_apply: null pointer");
    FFB6D_CHECK_ARG(act >= 0 && act <= 2, "bn_train_apply: act=%d", act);
    FFB6D_BN_COUNT_OK("bn_train_apply");
    FFB6D_CHECK_ARG((reinterpret_cast<uintptr_t>(sums) & 7) == 0, "bn_train_apply: sums must be 8-byte aligned");
    FFB6D_CHECK_ARG((reinterpret_cast<uintptr_t>(stats) & 15) == 0, "bn_train_apply: stats must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    bn_finalize_sums_kernel<<<(unsigned)ceil_div(C, BN_THREADS), BN_THREADS, 0, st>>>(
        sums, (int)C, count, eps, momentum, gamma, beta, running_mean, running_var, (float4 *)stats);
    FFB6D_LAUNCH_OK("bn_finalize_sums_kernel");
    const unsigned gx = (unsigned)std::min<int64_t>(ceil_div(P, 4 * BN_THREADS), 64);
    bn_apply_kernel<<<dim3((unsigned)(B * C), gx), BN_THREADS, 0, st>>>(z, (const float4 *)stats, (int)C, (int)P, act,
                                                                        negative_slope, y);
    FFB6D_LAUNCH_OK("bn_apply_kernel");
    return FFB6D_OK;
}

int ffb6d_bn_train_bwd_stats(const float *z, const float *grad_y, const float *stats, int64_t B, int64_t C, int64_t P,
                             int act, float negative_slope, double *sums, float *grad_gamma, float *grad_beta,
                             void *workspace, size_t workspace_bytes, ffb6d_stream_t stream)
{
    FFB6D_BN_SIZES_OK("bn_train_bwd_stats");
    FFB6D_CHECK_ARG(z && grad_y && stats && sums && workspace, "bn_train_bwd_stats: null pointer");
    FFB6D_CHECK_ARG(act >= 0 && act <= 2, "bn_train_bwd_stats: act=%d", act);
    FFB6D_CHECK_ARG((reinterpret_cast<uintptr_t>(sums) & 7) == 0, "bn_train_bwd_stats: sums must be 8-byte aligned");
    FFB6D_CHECK_ARG((reinterpret_cast<uintptr_t>(stats) & 15) == 0, "bn_train_bwd_stats: stats must be 16-byte aligned");
    FFB6D_CHECK_ARG(workspace_bytes >= ffb6d_bn_workspace_bytes(C, P), "bn_train_bwd_stats: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    int chunk, nsplit;
    split_plan(C, P, chunk, nsplit);
    double *partial = (double *)workspace;
    bn_bwd_reduce_kernel<<<dim3((unsigned)nsplit, (unsigned)C), BN_THREADS, 0, st>>>(
        z, grad_y, (const float4 *)stats, (int)B, (int)C, (int)P, chunk, nsplit, act, negative_slope, partial);
    FFB6D_LAUNCH_OK("bn_bwd_reduce_kernel");
    bn_partial_sums_kernel<<<(unsigned)ceil_div(C, BN_THREADS), BN_THREADS, 0, st>>>(partial, (int)C, nsplit, sums, grad_gamma,
                                                                                    grad_beta);
    FFB6D_LAUNCH_OK("bn_partial_sums_kernel");
    return FFB6D_OK;
}

int ffb6d_bn_train_bwd_apply(const float *z, const float *grad_y, const float *stats, const double *sums, double count,
                             int64_t B, int64_t C, int64_t P, int act, float negative_slope, float *grad_z,
                             ffb6d_stream_t stream)
{
    FFB6D_BN_SIZES_OK("bn_train_bwd_apply");
    FFB6D_CHECK_ARG(z && grad_y && stats && sums && grad_z, "bn_train_bwd_apply: null pointer");
    FFB6D_CHECK_ARG(act >= 0 && act <= 2, "bn_train_bwd_apply: act=%d", act);
    FFB6D_BN_COUNT_OK("bn_train_bwd_apply");
    FFB6D_CHECK_ARG((reinterpret_cast<uintptr_t>(sums) & 7) == 0, "bn_train_bwd_apply: sums must be 8-byte aligned");
    FFB6D_CHECK_ARG((reinterpret_cast<uintptr_t>(stats) & 15) == 0, "bn_train_bwd_apply: stats must be 16-byte aligned");
    const unsigned gx = (unsigned)std::min<int64_t>(ceil_div(P, BN_THREADS), 64);
    bn_bwd_apply_sums_kernel<<<dim3((unsigned)(B * C), gx), BN_THREADS, 0, (cudaStream_t)stream>>>(
        z, grad_y, (const float4 *)stats, sums, (int)C, (int)P, (float)(1.0 / count), act, negative_slope, grad_z);
    FFB6D_LAUNCH_OK("bn_bwd_apply_sums_kernel");
    return FFB6D_OK;
}

#undef FFB6D_BN_SIZES_OK
#undef FFB6D_BN_COUNT_OK

int ffb6d_act_bwd(const float *z, const float *grad_y, int64_t n, int act, float negative_slope, float *grad_z,
                  ffb6d_stream_t stream)
{
    FFB6D_CHECK_ARG(n >= 0 && act >= 0 && act <= 2, "act_bwd: bad argument");
    if (n == 0) return FFB6D_OK;
    FFB6D_CHECK_ARG(z && grad_y && grad_z, "act_bwd: null pointer");
    const unsigned blocks = (unsigned)std::min<int64_t>(ceil_div(n, BN_THREADS), 8 * (int64_t)num_sms());
    act_bwd_kernel<<<blocks, BN_THREADS, 0, (cudaStream_t)stream>>>(z, grad_y, (long long)n, act, negative_slope, grad_z);
    FFB6D_LAUNCH_OK("act_bwd_kernel");
    return FFB6D_OK;
}

int ffb6d_att_pool_bwd(const float *f1, int64_t C1, const float *f2, int64_t C2, const float *att, const float *grad_out,
                       int64_t B, int64_t N, int K, float *grad_f1, float *grad_f2, float *grad_att, ffb6d_stream_t stream)
{
    FFB6D_CHECK_ARG(B >= 0 && C1 >= 1 && C2 >= 0 && N >= 0, "att_pool_bwd: bad size");
    FFB6D_CHECK_ARG(K >= 1 && K <= FFB6D_MAX_K, "att_pool_bwd: K=%d outside [1,%d]", K, FFB6D_MAX_K);
    if (B == 0 || N == 0) return FFB6D_OK;
    FFB6D_CHECK_ARG(f1 && att && grad_out && grad_f1 && grad_att && (C2 == 0 || (f2 && grad_f2)), "att_pool_bwd: null pointer");
    const long long total = (long long)B * (C1 + C2) * N;
    const bool v16 = K == 16 && ((reinterpret_cast<uintptr_t>(f1) | reinterpret_cast<uintptr_t>(f2) | reinterpret_cast<uintptr_t>(att) |
                                  reinterpret_cast<uintptr_t>(grad_f1) | reinterpret_cast<uintptr_t>(grad_f2) |
                                  reinterpret_cast<uintptr_t>(grad_att)) & 15) == 0;
    if (v16)
        att_pool_bwd_kernel<16><<<(unsigned)ceil_div(total, 256), 256, 0, (cudaStream_t)stream>>>(
            f1, (int)C1, f2, (int)C2, att, grad_out, (int)N, K, grad_f1, grad_f2, grad_att, total);
    else
        att_pool_bwd_kernel<0><<<(unsigned)ceil_div(total, 256), 256, 0, (cudaStream_t)stream>>>(
            f1, (int)C1, f2, (int)C2, att, grad_out, (int)N, K, grad_f1, grad_f2, grad_att, total);
    FFB6D_LAUNCH_OK("att_pool_bwd_kernel");
    return FFB6D_OK;
}

}  // extern "C"
