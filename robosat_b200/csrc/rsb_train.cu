// Training-path helper kernels around the tensor-core convolutions (HBM-bound elementwise / reduction work):
// train-mode BatchNorm (batch statistics, running-stat update, apply, backward), ReLU / max-pool / final-1x1
// backward, and the fp32-master <-> fp16-packed weight conversions run every optimiser step.
//
// Reference semantics: nn.BatchNorm2d in training mode (torchvision resnet50 inside robosat/unet.py:122-130):
// biased batch variance for normalisation, running_var updated with the unbiased estimate, momentum 0.1, eps 1e-5;
// autograd of conv / relu / max_pool2d / interpolate / cat triggered by loss.backward() (robosat/tools/train.py:186).
// All activations and activation gradients are NHWC fp16 (gradients carry the loss scale), reductions run in
// fp32 per thread and fp64 across blocks, parameter gradients are fp32.

#include <cuda_fp16.h>

#include "../../include/rsb200.h"
#include "rsb_host.h"

namespace rsb {

static inline unsigned tr_blocks(int64_t total, int block, int cap = 148 * 16) {
    int64_t b = (total + block - 1) / block;
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    return static_cast<unsigned>(b);
}

// grid of the channel reductions: every block folds >= 8 row groups (4 per iteration in flight), at most 4 blocks per SM
static inline unsigned reduce_blocks(int64_t M, int C) {
    const int rows_per_iter = 256 / (C / 8);
    return tr_blocks((M + rows_per_iter * 8 - 1) / (rows_per_iter * 8), 1, 148 * 4);
}

// Programmatic dependent launch: the training step is a chain of ~650 mostly small kernels, so the launch gap (scheduling the
// next grid only after the previous one has drained) is a visible part of it. Chained kernels are launched with the
// programmatic-stream-serialization attribute; each lets its successor be scheduled as soon as its own blocks are resident
// (launch_dependents) and touches global memory only after the predecessor has completed and flushed (wait). For a normal
// launch both instructions are no-ops.
__device__ __forceinline__ void pdl_sync() {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
}

template <typename... KArgs, typename... Args>
static cudaError_t launch_chained(bool chained, void (*kern)(KArgs...), unsigned grid, unsigned block, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = chained ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

__device__ __forceinline__ void load8(const __half* p, float (&v)[8]) {
    const uint4 q = __ldg(reinterpret_cast<const uint4*>(p));
    const __half2* h = reinterpret_cast<const __half2*>(&q);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float2 f = __half22float2(h[i]);
        v[2 * i] = f.x;
        v[2 * i + 1] = f.y;
    }
}
__device__ __forceinline__ void store8(__half* p, const float (&v)[8]) {
    uint4 q;
    __half2* h = reinterpret_cast<__half2*>(&q);
#pragma unroll
    for (int i = 0; i < 4; ++i) h[i] = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
    *reinterpret_cast<uint4*>(p) = q;
}

// ------------------------------------------------------------------------------------------------
// per-channel sums over M rows of an NHWC fp16 tensor [M][C]; two fused reductions:
//   KIND 0 (forward stats)   : s0 += z            s1 += z*z
//   KIND 1 (BN backward)     : g = dy * (y > 0 or no mask); s0 += g ; s1 += g * z   (raw: consumers turn it into
//                              sum g*zhat = (s1 - mean*s0) * invstd, which keeps mean / invstd out of the streaming loop)
// 256 threads: C/8 threads cover one row (8 channels = 16 bytes each), 256/(C/8) rows per iteration, two iterations in
// flight per thread. Block totals go to one of kRedSlots replicated fp64 accumulators (slot = block % kRedSlots) so that
// at most blocks/kRedSlots atomics queue up on an address; consumers add the slots.
static constexpr int kRedSlots = 8;

// Scratch layout (doubles): [kRedSlots][2][C] accumulators | 1 arrival counter | 1 pad | (as floats) 3*C coefficients.
// The LAST block to finish (arrival counter) folds the slots and does the per-channel epilogue, so no extra launch is needed:
//   KIND 0: BatchNorm finalize (mean / invstd / folded scale+shift, running statistics)      -- when tail.gamma != NULL
//   KIND 1: dgamma / dbeta and the coefficients A, B, D of dz = A*g + B*z + D for bn_bwd_apply_kernel
struct RedTail {
    const float* gamma;
    const float* beta;
    float* running_mean;
    float* running_var;
    int64_t* num_batches;
    float* mean;    // KIND 0: out; KIND 1: in
    float* invstd;  // KIND 0: out; KIND 1: in
    float* scale;
    float* shift;
    float* dgamma;
    float* dbeta;
    float eps, momentum, inv_scale;
    int self_clean;  // the last block leaves the accumulator slots and the arrival counter zeroed for the next call (no memset launch)
    const int* frozen;  // strict plans: *frozen != 0 (weights past the plan's exponents) -> running statistics left untouched
};

__device__ __forceinline__ double red_slots(const double* sums, int which, int c, int C) {
    double t = 0.0;
#pragma unroll
    for (int sl = 0; sl < kRedSlots; ++sl) t += __ldcg(&sums[(static_cast<int64_t>(sl) * 2 + which) * C + c]);
    return t;
}

// ZMASK: the ReLU mask of a plain relu(bn(z)) output is re-derived from z instead of reading y: bn_apply_kernel rounds
// o = fma(z, scale, shift) to fp16, and half(o) > 0 exactly when o > 2^-25 (round-to-nearest-even), so the mask is bit-identical.
static constexpr float kHalfPositive = 0x1p-25f;

template <int KIND, bool ZMASK = false>
__global__ void __launch_bounds__(256, 2) channel_reduce_kernel(const __half* __restrict__ a, const __half* __restrict__ y, const __half* __restrict__ z,
                                                             double* __restrict__ sums, int64_t M, int C, const RedTail tail,
                                                             const float* __restrict__ msc = nullptr, const float* __restrict__ msh = nullptr) {
    __shared__ float sh0[256 * 8];
    __shared__ float sh1[256 * 8];
    pdl_sync();
    const int tpr = C / 8;
    const int rows_per_iter = 256 / tpr;
    const int col = (threadIdx.x % tpr) * 8;
    const int rsub = threadIdx.x / tpr;
    float acc0[8], acc1[8], zsc[8], zsh[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        acc0[i] = acc1[i] = 0.f;
        zsc[i] = ZMASK ? msc[col + i] : 0.f;
        zsh[i] = ZMASK ? msh[col + i] : 0.f;
    }
    const int64_t step = static_cast<int64_t>(gridDim.x) * rows_per_iter;
    auto zmask = [&](const float (&zz)[8], float (&yy)[8]) {
#pragma unroll
        for (int i = 0; i < 8; ++i) yy[i] = fmaf(zz[i], zsc[i], zsh[i]) > kHalfPositive ? 1.f : 0.f;
    };
    auto fold = [&](const float (&v)[8], const float (&zz)[8], const float (&yy)[8], bool masked) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            if (KIND == 0) {
                acc0[i] += v[i];
                acc1[i] = fmaf(v[i], v[i], acc1[i]);
            } else {
                const float g = (masked && !(yy[i] > 0.f)) ? 0.f : v[i];
                acc0[i] += g;
                acc1[i] = fmaf(g, zz[i], acc1[i]);
            }
        }
    };
    int64_t r = static_cast<int64_t>(blockIdx.x) * rows_per_iter + rsub;
    // Main loop: FOUR row groups per iteration, all 16-byte loads issued (raw, 4 registers each) before the first conversion:
    // 8-12 loads x 16 B in flight per thread. With two in flight a block kept ~8 KB outstanding and the passes ran at 37-53 % of
    // the HBM peak (Little's law wants ~45 KB per SM); see profiles/r2_train.md.
    auto raw = [](const __half* p) { return __ldg(reinterpret_cast<const uint4*>(p)); };
    auto cvt = [](const uint4& q, float (&v)[8]) {
        const __half2* h = reinterpret_cast<const __half2*>(&q);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float2 f = __half22float2(h[i]);
            v[2 * i] = f.x;
            v[2 * i + 1] = f.y;
        }
    };
    const bool use_y = !ZMASK && y != nullptr;
    for (; r + 3 * step < M; r += 4 * step) {
        uint4 qa[4], qz[4], qy[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) qa[u] = raw(a + (r + u * step) * C + col);
        if (KIND == 1) {
#pragma unroll
            for (int u = 0; u < 4; ++u) qz[u] = raw(z + (r + u * step) * C + col);
            if (use_y) {
#pragma unroll
                for (int u = 0; u < 4; ++u) qy[u] = raw(y + (r + u * step) * C + col);
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            float v0[8], z0[8], y0[8];
            cvt(qa[u], v0);
            if (KIND == 1) {
                cvt(qz[u], z0);
                if (ZMASK) zmask(z0, y0);
                else if (use_y) cvt(qy[u], y0);
            }
            fold(v0, z0, y0, ZMASK || y != nullptr);
        }
    }
    for (; r + step < M; r += 2 * step) {
        float v0[8], v1[8], z0[8], z1[8], y0[8], y1[8];
        load8(a + r * C + col, v0);
        load8(a + (r + step) * C + col, v1);
        if (KIND == 1) {
            load8(z + r * C + col, z0);
            load8(z + (r + step) * C + col, z1);
            if (ZMASK) {
                zmask(z0, y0);
                zmask(z1, y1);
            } else if (y) {
                load8(y + r * C + col, y0);
                load8(y + (r + step) * C + col, y1);
            }
        }
        fold(v0, z0, y0, ZMASK || y != nullptr);
        fold(v1, z1, y1, ZMASK || y != nullptr);
    }
    if (r < M) {
        float v0[8], z0[8], y0[8];
        load8(a + r * C + col, v0);
        if (KIND == 1) {
            load8(z + r * C + col, z0);
            if (ZMASK) zmask(z0, y0);
            else if (y) load8(y + r * C + col, y0);
        }
        fold(v0, z0, y0, ZMASK || y != nullptr);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        sh0[threadIdx.x * 8 + i] = acc0[i];
        sh1[threadIdx.x * 8 + i] = acc1[i];
    }
    __syncthreads();
    // threads 0..C-1 (at most 2048 channels -> loop) fold the row-groups
    double* s0 = sums + static_cast<int64_t>(blockIdx.x % kRedSlots) * 2 * C;
    double* s1 = s0 + C;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        const int t0 = c / 8, e = c % 8;
        float a0 = 0.f, a1 = 0.f;
        for (int g = 0; g < rows_per_iter; ++g) {
            a0 += sh0[(g * tpr + t0) * 8 + e];
            a1 += sh1[(g * tpr + t0) * 8 + e];
        }
        atomicAdd(&s0[c], static_cast<double>(a0));
        atomicAdd(&s1[c], static_cast<double>(a1));
    }
    if (tail.gamma == nullptr) return;
    // ---- last block: per-channel epilogue
    __shared__ bool is_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned* counter = reinterpret_cast<unsigned*>(sums + static_cast<int64_t>(kRedSlots) * 2 * C);
        is_last = atomicAdd(counter, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    const double dM = static_cast<double>(M);
    if (KIND == 0 && threadIdx.x == 0 && tail.num_batches) *tail.num_batches += 1;
    float* coef = reinterpret_cast<float*>(sums + static_cast<int64_t>(kRedSlots) * 2 * C + 2);
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        const double t0 = red_slots(sums, 0, c, C), t1 = red_slots(sums, 1, c, C);
        if (KIND == 0) {
            const double mean = t0 / dM;
            double var = t1 / dM - mean * mean;
            if (var < 0) var = 0;
            const float invstd = static_cast<float>(1.0 / sqrt(var + static_cast<double>(tail.eps)));
            const float sc = tail.gamma[c] * invstd;
            tail.mean[c] = static_cast<float>(mean);
            tail.invstd[c] = invstd;
            tail.scale[c] = sc;
            tail.shift[c] = tail.beta[c] - static_cast<float>(mean) * sc;
            if (tail.running_mean) {
                const double unbiased = dM > 1 ? var * dM / (dM - 1.0) : var;
                tail.running_mean[c] = (1.f - tail.momentum) * tail.running_mean[c] + tail.momentum * static_cast<float>(mean);
                tail.running_var[c] = (1.f - tail.momentum) * tail.running_var[c] + tail.momentum * static_cast<float>(unbiased);
            }
        } else {
            const float is = tail.invstd[c], ga = tail.gamma[c], mu = tail.mean[c];
            const double sgzh = (t1 - static_cast<double>(mu) * t0) * static_cast<double>(is);  // sum of g * zhat
            tail.dgamma[c] = static_cast<float>(sgzh) * tail.inv_scale;
            tail.dbeta[c] = static_cast<float>(t0) * tail.inv_scale;
            const float mg = static_cast<float>(t0 / dM), mgz = static_cast<float>(sgzh / dM);
            coef[c] = ga * is;                                        // A
            coef[C + c] = -ga * is * is * mgz;                        // B
            coef[2 * C + c] = -ga * is * mg + ga * is * is * mu * mgz;  // D
        }
        if (tail.self_clean) {
#pragma unroll
            for (int sl = 0; sl < kRedSlots; ++sl) {
                sums[(static_cast<int64_t>(sl) * 2 + 0) * C + c] = 0.0;
                sums[(static_cast<int64_t>(sl) * 2 + 1) * C + c] = 0.0;
            }
        }
    }
    if (tail.self_clean && threadIdx.x == 0) *reinterpret_cast<unsigned*>(sums + static_cast<int64_t>(kRedSlots) * 2 * C) = 0u;
}

// ------------------------------------------------------------------------------------------------
// Batch statistics from the per-quarter-tile partial sums a STATS convolution wrote (rsb_conv_desc.stats): P is an fp32
// matrix [R][L], L = 2*C (row = one 32-pixel quarter of a tile: C sums, then C sums of squares). Column sums go to the same
// replicated fp64 accumulators as channel_reduce_kernel<0> ([slot][2][C] == [slot][L]) and the last block runs the same
// BatchNorm finalize, so the op reads 1/8 of the bytes of z instead of all of z.
__global__ void __launch_bounds__(256) partial_reduce_kernel(const float* __restrict__ P, double* __restrict__ sums, int64_t R, int L, int C, int64_t M,
                                                            const RedTail tail) {
    __shared__ float4 sh[256];
    pdl_sync();
    const int tpr = L / 4 < 256 ? L / 4 : 256;  // threads per row, one float4 each
    const int rows_per_iter = 256 / tpr;
    const int col = blockIdx.y * tpr * 4 + (threadIdx.x % tpr) * 4;
    const int rsub = threadIdx.x / tpr;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    const int64_t step = static_cast<int64_t>(gridDim.x) * rows_per_iter;
    int64_t r = static_cast<int64_t>(blockIdx.x) * rows_per_iter + rsub;
    auto ld = [&](int64_t row) { return __ldg(reinterpret_cast<const float4*>(P + row * L + col)); };
    auto add = [&](const float4& v) {
        acc.x += v.x;
        acc.y += v.y;
        acc.z += v.z;
        acc.w += v.w;
    };
    for (; r + 3 * step < R; r += 4 * step) {
        const float4 a = ld(r), b = ld(r + step), c = ld(r + 2 * step), d = ld(r + 3 * step);
        add(a);
        add(b);
        add(c);
        add(d);
    }
    for (; r < R; r += step) add(ld(r));
    sh[threadIdx.x] = acc;
    __syncthreads();
    if (threadIdx.x < tpr) {
        float4 t = sh[threadIdx.x];
        for (int g = 1; g < rows_per_iter; ++g) {
            const float4 v = sh[g * tpr + threadIdx.x];
            t.x += v.x;
            t.y += v.y;
            t.z += v.z;
            t.w += v.w;
        }
        double* s = sums + static_cast<int64_t>(blockIdx.x % kRedSlots) * L + col;
        atomicAdd(&s[0], static_cast<double>(t.x));
        atomicAdd(&s[1], static_cast<double>(t.y));
        atomicAdd(&s[2], static_cast<double>(t.z));
        atomicAdd(&s[3], static_cast<double>(t.w));
    }
    // ---- last block (of the whole 2-D grid): BatchNorm finalize, as in channel_reduce_kernel<0>
    __shared__ bool is_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned* counter = reinterpret_cast<unsigned*>(sums + static_cast<int64_t>(kRedSlots) * 2 * C);
        is_last = atomicAdd(counter, 1u) == gridDim.x * gridDim.y - 1;
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    const double dM = static_cast<double>(M);
    if (threadIdx.x == 0 && tail.num_batches) *tail.num_batches += 1;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        const double t0 = red_slots(sums, 0, c, C), t1 = red_slots(sums, 1, c, C);
        const double mean = t0 / dM;
        double var = t1 / dM - mean * mean;
        if (var < 0) var = 0;
        const float invstd = static_cast<float>(1.0 / sqrt(var + static_cast<double>(tail.eps)));
        const float sc = tail.gamma[c] * invstd;
        tail.mean[c] = static_cast<float>(mean);
        tail.invstd[c] = invstd;
        tail.scale[c] = sc;
        tail.shift[c] = tail.beta[c] - static_cast<float>(mean) * sc;
        if (tail.running_mean) {
            const double unbiased = dM > 1 ? var * dM / (dM - 1.0) : var;
            tail.running_mean[c] = (1.f - tail.momentum) * tail.running_mean[c] + tail.momentum * static_cast<float>(mean);
            tail.running_var[c] = (1.f - tail.momentum) * tail.running_var[c] + tail.momentum * static_cast<float>(unbiased);
        }
        if (tail.self_clean) {
#pragma unroll
            for (int sl = 0; sl < kRedSlots; ++sl) {
                sums[(static_cast<int64_t>(sl) * 2 + 0) * C + c] = 0.0;
                sums[(static_cast<int64_t>(sl) * 2 + 1) * C + c] = 0.0;
            }
        }
    }
    if (tail.self_clean && threadIdx.x == 0) *reinterpret_cast<unsigned*>(sums + static_cast<int64_t>(kRedSlots) * 2 * C) = 0u;
}

// mean / invstd / folded scale+shift from the batch sums, running-stat update (momentum, unbiased variance)
__global__ void bn_finalize_kernel(const double* __restrict__ sums, const float* __restrict__ gamma,
                                   const float* __restrict__ beta, float* __restrict__ running_mean, float* __restrict__ running_var,
                                   int64_t* __restrict__ num_batches, float* __restrict__ mean_out, float* __restrict__ invstd_out,
                                   float* __restrict__ scale_out, float* __restrict__ shift_out, int C, double M, float eps, float momentum) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c == 0 && num_batches) *num_batches += 1;
    if (c >= C) return;
    const double mean = red_slots(sums, 0, c, C) / M;
    double var = red_slots(sums, 1, c, C) / M - mean * mean;
    if (var < 0) var = 0;
    const float invstd = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
    const float sc = gamma[c] * invstd;
    mean_out[c] = static_cast<float>(mean);
    invstd_out[c] = invstd;
    scale_out[c] = sc;
    shift_out[c] = beta[c] - static_cast<float>(mean) * sc;
    if (running_mean) {
        const double unbiased = M > 1 ? var * M / (M - 1.0) : var;
        running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * static_cast<float>(mean);
        running_var[c] = (1.f - momentum) * running_var[c] + momentum * static_cast<float>(unbiased);
    }
}

// y = relu?(z * scale + shift (+ res)). The grid stride (blocks * 256) is a multiple of C/8 (C/8 divides 256), so every
// thread keeps the same 8 channels for its whole loop and holds their coefficients in registers.
__global__ void bn_apply_kernel(const __half* __restrict__ z, const float* __restrict__ scale, const float* __restrict__ shift,
                                const __half* __restrict__ res, __half* __restrict__ y, int64_t M, int C, int relu) {
    pdl_sync();
    const int C8 = C / 8;
    const int64_t total = M * C8;
    const int64_t i0 = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    const int col = static_cast<int>(i0 % C8) * 8;
    float sc[8], sh[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        sc[e] = scale[col + e];
        sh[e] = shift[col + e];
    }
    const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
    auto finish = [&](int64_t i, const uint4& qz, const uint4& qr) {
        float v[8], r[8];
        const __half2* hz = reinterpret_cast<const __half2*>(&qz);
        const __half2* hr = reinterpret_cast<const __half2*>(&qr);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float2 f = __half22float2(hz[e]), g = __half22float2(hr[e]);
            v[2 * e] = f.x;
            v[2 * e + 1] = f.y;
            r[2 * e] = g.x;
            r[2 * e + 1] = g.y;
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            float o = fmaf(v[e], sc[e], sh[e]);
            if (res) o += r[e];
            v[e] = relu ? fmaxf(o, 0.f) : o;
        }
        store8(y + i * 8, v);
    };
    int64_t i = i0;
    // four 16-byte units (eight with a residual) in flight per thread before the first conversion
    for (; i + 3 * stride < total; i += 4 * stride) {
        uint4 qz[4], qr[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) qz[u] = __ldg(reinterpret_cast<const uint4*>(z + (i + u * stride) * 8));
#pragma unroll
        for (int u = 0; u < 4; ++u) qr[u] = res ? __ldg(reinterpret_cast<const uint4*>(res + (i + u * stride) * 8)) : make_uint4(0, 0, 0, 0);
#pragma unroll
        for (int u = 0; u < 4; ++u) finish(i + u * stride, qz[u], qr[u]);
    }
    for (; i < total; i += stride) {
        const uint4 qz = __ldg(reinterpret_cast<const uint4*>(z + i * 8));
        const uint4 qr = res ? __ldg(reinterpret_cast<const uint4*>(res + i * 8)) : make_uint4(0, 0, 0, 0);
        finish(i, qz, qr);
    }
}

// dz = gamma*invstd * (g - sum_g/M - zhat * sum_gzhat/M) = A*g + B*z + D per channel, g = dy * (y > 0);
// optionally also writes g (identity-branch gradient). Per-channel coefficients live in registers (see bn_apply_kernel);
// two 16-byte units per thread are in flight per iteration.
template <bool ZMASK>
__global__ void __launch_bounds__(256, 2) bn_bwd_apply_kernel(const __half* __restrict__ dy, const __half* __restrict__ y, const __half* __restrict__ z,
                                                              const float* __restrict__ coef, __half* __restrict__ dz, __half* __restrict__ g_out,
                                                              int64_t M, int C, const float* __restrict__ msc, const float* __restrict__ msh) {
    pdl_sync();
    const int C8 = C / 8;
    const int64_t total = M * C8;
    const int64_t i0 = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    const int col = static_cast<int>(i0 % C8) * 8;
    float A[8], B[8], D[8], zsc[8], zsh[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        A[e] = coef[col + e];
        B[e] = coef[C + col + e];
        D[e] = coef[2 * C + col + e];
        zsc[e] = ZMASK ? msc[col + e] : 0.f;
        zsh[e] = ZMASK ? msh[col + e] : 0.f;
    }
    const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
    auto finish = [&](int64_t i, float (&g)[8], const float (&zz)[8], const float (&yy)[8]) {
        if (ZMASK) {
#pragma unroll
            for (int e = 0; e < 8; ++e) g[e] = fmaf(zz[e], zsc[e], zsh[e]) > kHalfPositive ? g[e] : 0.f;
        } else if (y) {
#pragma unroll
            for (int e = 0; e < 8; ++e) g[e] = yy[e] > 0.f ? g[e] : 0.f;
        }
        if (g_out) store8(g_out + i * 8, g);
        float o[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) o[e] = fmaf(A[e], g[e], fmaf(B[e], zz[e], D[e]));
        store8(dz + i * 8, o);
    };
    int64_t i = i0;
    // four units per iteration, all raw 16-byte loads (8-12 per thread) issued before the first conversion
    auto cvt = [](const uint4& q, float (&v)[8]) {
        const __half2* h = reinterpret_cast<const __half2*>(&q);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float2 f = __half22float2(h[e]);
            v[2 * e] = f.x;
            v[2 * e + 1] = f.y;
        }
    };
    const bool use_y = !ZMASK && y != nullptr;
    for (; i + 3 * stride < total; i += 4 * stride) {
        uint4 qg[4], qz[4], qy[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) qg[u] = __ldg(reinterpret_cast<const uint4*>(dy + (i + u * stride) * 8));
#pragma unroll
        for (int u = 0; u < 4; ++u) qz[u] = __ldg(reinterpret_cast<const uint4*>(z + (i + u * stride) * 8));
        if (use_y) {
#pragma unroll
            for (int u = 0; u < 4; ++u) qy[u] = __ldg(reinterpret_cast<const uint4*>(y + (i + u * stride) * 8));
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            float g0[8], z0[8], y0[8];
            cvt(qg[u], g0);
            cvt(qz[u], z0);
            if (use_y) cvt(qy[u], y0);
            finish(i + u * stride, g0, z0, y0);
        }
    }
    for (; i + stride < total; i += 2 * stride) {
        float g0[8], g1[8], z0[8], z1[8], y0[8], y1[8];
        load8(dy + i * 8, g0);
        load8(dy + (i + stride) * 8, g1);
        load8(z + i * 8, z0);
        load8(z + (i + stride) * 8, z1);
        if (!ZMASK && y) {
            load8(y + i * 8, y0);
            load8(y + (i + stride) * 8, y1);
        }
        finish(i, g0, z0, y0);
        finish(i + stride, g1, z1, y1);
    }
    if (i < total) {
        float g0[8], z0[8], y0[8];
        load8(dy + i * 8, g0);
        load8(z + i * 8, z0);
        if (!ZMASK && y) load8(y + i * 8, y0);
        finish(i, g0, z0, y0);
    }
}

// out = a * (y > 0) (+ b): ReLU backward with an optional second gradient stream (skip connection fan-in)
__global__ void relu_bwd_kernel(const __half* __restrict__ a, const __half* __restrict__ b, const __half* __restrict__ y,
                                __half* __restrict__ out, int64_t total8) {
    pdl_sync();
    const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
    auto finish = [&](int64_t i, const uint4& qa, const uint4& qb, const uint4& qy) {
        float g[8];
        const __half2* ha = reinterpret_cast<const __half2*>(&qa);
        const __half2* hb = reinterpret_cast<const __half2*>(&qb);
        const __half2* hy = reinterpret_cast<const __half2*>(&qy);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            float2 f = __half22float2(ha[e]);
            if (b) {
                const float2 h = __half22float2(hb[e]);
                f.x += h.x;
                f.y += h.y;
            }
            if (y) {
                const float2 m = __half22float2(hy[e]);
                f.x = m.x > 0.f ? f.x : 0.f;
                f.y = m.y > 0.f ? f.y : 0.f;
            }
            g[2 * e] = f.x;
            g[2 * e + 1] = f.y;
        }
        store8(out + i * 8, g);
    };
    const uint4 zero = make_uint4(0, 0, 0, 0);
    int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    for (; i + 3 * stride < total8; i += 4 * stride) {  // four units (up to twelve 16-byte loads) in flight per thread
        uint4 qa[4], qb[4], qy[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) qa[u] = __ldg(reinterpret_cast<const uint4*>(a + (i + u * stride) * 8));
#pragma unroll
        for (int u = 0; u < 4; ++u) qb[u] = b ? __ldg(reinterpret_cast<const uint4*>(b + (i + u * stride) * 8)) : zero;
#pragma unroll
        for (int u = 0; u < 4; ++u) qy[u] = y ? __ldg(reinterpret_cast<const uint4*>(y + (i + u * stride) * 8)) : zero;
#pragma unroll
        for (int u = 0; u < 4; ++u) finish(i + u * stride, qa[u], qb[u], qy[u]);
    }
    for (; i < total8; i += stride)
        finish(i, __ldg(reinterpret_cast<const uint4*>(a + i * 8)), b ? __ldg(reinterpret_cast<const uint4*>(b + i * 8)) : zero,
               y ? __ldg(reinterpret_cast<const uint4*>(y + i * 8)) : zero);
}

// max-pool backward: dx[h][w] = sum over the windows that contain (h, w) and whose argmax is (h, w) (first max wins, like ATen)
__global__ void maxpool_bwd_kernel(const __half* __restrict__ x, const __half* __restrict__ dy, __half* __restrict__ dx, int N, int H, int W,
                                   int C, int k, int s, int p, int OH, int OW) {
    const int C8 = C / 8;
    const int64_t total = static_cast<int64_t>(N) * H * W * C8;
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int c8 = static_cast<int>(i % C8);
        int64_t r = i / C8;
        const int w = static_cast<int>(r % W);
        r /= W;
        const int h = static_cast<int>(r % H);
        const int n = static_cast<int>(r / H);
        float xv[8], acc[8];
        load8(x + i * 8, xv);
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[e] = 0.f;
        // windows (oh, ow) covering this input pixel
        const int oh_lo = max(0, (h + p - k + s) / s), oh_hi = min(OH - 1, (h + p) / s);
        const int ow_lo = max(0, (w + p - k + s) / s), ow_hi = min(OW - 1, (w + p) / s);
        for (int oh = oh_lo; oh <= oh_hi; ++oh) {
            for (int ow = ow_lo; ow <= ow_hi; ++ow) {
                // is (h, w) the first maximum of window (oh, ow)?
                bool first[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) first[e] = true;
                for (int dyy = 0; dyy < k; ++dyy) {
                    const int hh = oh * s - p + dyy;
                    if (hh < 0 || hh >= H) continue;
                    for (int dxx = 0; dxx < k; ++dxx) {
                        const int ww = ow * s - p + dxx;
                        if (ww < 0 || ww >= W || (hh == h && ww == w)) continue;
                        float o[8];
                        load8(x + ((static_cast<int64_t>(n) * H + hh) * W + ww) * C + c8 * 8, o);
                        const bool before = (hh < h) || (hh == h && ww < w);
#pragma unroll
                        for (int e = 0; e < 8; ++e) {
                            if (o[e] > xv[e] || (before && o[e] == xv[e])) first[e] = false;
                        }
                    }
                }
                float g[8];
                load8(dy + ((static_cast<int64_t>(n) * OH + oh) * OW + ow) * C + c8 * 8, g);
#pragma unroll
                for (int e = 0; e < 8; ++e) acc[e] += first[e] ? g[e] : 0.f;
            }
        }
        store8(dx + i * 8, acc);
    }
}

// Two-pass variant (what the engine uses): pass 1 recomputes, once per pooling window, the position (dy*k + dx) of its
// first maximum; pass 2 gathers, per input pixel, the gradients of the <= ceil(k/s)^2 windows whose argmax it is.
__global__ void maxpool_argmax_kernel(const __half* __restrict__ x, uint8_t* __restrict__ idx, int N, int H, int W, int C, int k, int s, int p,
                                      int OH, int OW) {
    const int C8 = C / 8;
    const int64_t total = static_cast<int64_t>(N) * OH * OW * C8;
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int c8 = static_cast<int>(i % C8);
        int64_t r = i / C8;
        const int ow = static_cast<int>(r % OW);
        r /= OW;
        const int oh = static_cast<int>(r % OH);
        const int n = static_cast<int>(r / OH);
        float best[8];
        uint32_t pos[8];
        bool any = false;
        for (int dyy = 0; dyy < k; ++dyy) {
            const int hh = oh * s - p + dyy;
            if (hh < 0 || hh >= H) continue;
            for (int dxx = 0; dxx < k; ++dxx) {
                const int ww = ow * s - p + dxx;
                if (ww < 0 || ww >= W) continue;
                float v[8];
                load8(x + ((static_cast<int64_t>(n) * H + hh) * W + ww) * C + c8 * 8, v);
                const uint32_t q = static_cast<uint32_t>(dyy * k + dxx);
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    if (!any || v[e] > best[e]) {
                        best[e] = v[e];
                        pos[e] = q;
                    }
                }
                any = true;
            }
        }
        uint2 o;
        o.x = pos[0] | (pos[1] << 8) | (pos[2] << 16) | (pos[3] << 24);
        o.y = pos[4] | (pos[5] << 8) | (pos[6] << 16) | (pos[7] << 24);
        *reinterpret_cast<uint2*>(idx + i * 8) = o;
    }
}

__global__ void maxpool_bwd_gather_kernel(const uint8_t* __restrict__ idx, const __half* __restrict__ dy, __half* __restrict__ dx, int N, int H,
                                          int W, int C, int k, int s, int p, int OH, int OW) {
    const int C8 = C / 8;
    const int64_t total = static_cast<int64_t>(N) * H * W * C8;
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int c8 = static_cast<int>(i % C8);
        int64_t r = i / C8;
        const int w = static_cast<int>(r % W);
        r /= W;
        const int h = static_cast<int>(r % H);
        const int n = static_cast<int>(r / H);
        float acc[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[e] = 0.f;
        const int oh_lo = max(0, (h + p - k + s) / s), oh_hi = min(OH - 1, (h + p) / s);
        const int ow_lo = max(0, (w + p - k + s) / s), ow_hi = min(OW - 1, (w + p) / s);
        for (int oh = oh_lo; oh <= oh_hi; ++oh) {
            for (int ow = ow_lo; ow <= ow_hi; ++ow) {
                const int64_t o = ((static_cast<int64_t>(n) * OH + oh) * OW + ow) * C + c8 * 8;
                const uint32_t me = static_cast<uint32_t>((h - (oh * s - p)) * k + (w - (ow * s - p)));
                const uint2 q = __ldg(reinterpret_cast<const uint2*>(idx + o));
                float g[8];
                load8(dy + o, g);
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    const uint32_t a = ((e < 4 ? q.x : q.y) >> (8 * (e & 3))) & 0xffu;
                    acc[e] += a == me ? g[e] : 0.f;
                }
            }
        }
        store8(dx + i * 8, acc);
    }
}

// final 1x1 conv (32 -> C classes, with bias) forward: logits fp32 NCHW from NHWC fp16 activations (unet.py:141)
__global__ void final_fwd_kernel(const __half* __restrict__ y5, const float* __restrict__ w, const float* __restrict__ b,
                                 float* __restrict__ logits, int64_t P, int64_t HW, int classes) {
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < P; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        float v[32];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float t[8];
            load8(y5 + i * 32 + j * 8, t);
#pragma unroll
            for (int e = 0; e < 8; ++e) v[j * 8 + e] = t[e];
        }
        const int64_t n = i / HW, pix = i % HW;
        for (int k = 0; k < classes; ++k) {
            float s = b[k];
#pragma unroll
            for (int c = 0; c < 32; ++c) s = fmaf(w[k * 32 + c], v[c], s);
            logits[(n * classes + k) * HW + pix] = s;
        }
    }
}

// final 1x1 backward, input gradient: dy5[p][c] = loss_scale * sum_k dlogits[p][k] * w[k][c]  (fp16; dec5's ReLU mask is applied later)
__global__ void final_bwd_dx_kernel(const float* __restrict__ dlogits, const float* __restrict__ w, __half* __restrict__ dy5,
                                    float loss_scale, int64_t P, int64_t HW, int classes) {
    __shared__ float sw[8 * 32];
    for (int i = threadIdx.x; i < classes * 32; i += blockDim.x) sw[i] = w[i];
    __syncthreads();
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < P; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int64_t n = i / HW, pix = i % HW;
        float d[32];
#pragma unroll
        for (int c = 0; c < 32; ++c) d[c] = 0.f;
        for (int k = 0; k < classes; ++k) {
            const float g = dlogits[(n * classes + k) * HW + pix] * loss_scale;
#pragma unroll
            for (int c = 0; c < 32; ++c) d[c] = fmaf(g, sw[k * 32 + c], d[c]);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float t[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) t[e] = d[j * 8 + e];
            store8(dy5 + i * 32 + j * 8, t);
        }
    }
}

// final 1x1 backward, parameter gradients for ONE class k: dW[k][c] = sum_p dlogits[p][k] * y5[p][c], db[k] = sum_p dlogits[p][k]
__global__ void final_bwd_dw_kernel(const float* __restrict__ dlogits, const __half* __restrict__ y5, double* __restrict__ dw_acc,
                                    double* __restrict__ db_acc, int k, int64_t P, int64_t HW, int classes) {
    float ldw[32];
    float ldb = 0.f;
#pragma unroll
    for (int c = 0; c < 32; ++c) ldw[c] = 0.f;
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < P; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int64_t n = i / HW, pix = i % HW;
        const float g = dlogits[(n * classes + k) * HW + pix];
        ldb += g;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float t[8];
            load8(y5 + i * 32 + j * 8, t);
#pragma unroll
            for (int e = 0; e < 8; ++e) ldw[j * 8 + e] = fmaf(g, t[e], ldw[j * 8 + e]);
        }
    }
    // warp reduce, then one fp64 atomic per warp and channel
#pragma unroll
    for (int c = 0; c < 32; ++c) {
        float v = ldw[c];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) == 0) atomicAdd(&dw_acc[k * 32 + c], static_cast<double>(v));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ldb += __shfl_xor_sync(0xffffffffu, ldb, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(&db_acc[k], static_cast<double>(ldb));
}

__global__ void f64_to_f32_kernel(const double* __restrict__ src, float* __restrict__ dst, int n, float mul) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = static_cast<float>(src[i]) * mul;
}

// ------------------------------------------------------------------------------------------------
// fp32 master weights -> fp16 packed operand matrices, and packed fp32 gradients -> fp32 OIHW gradients.
// A packed matrix is [rows][K]; `map` gives, for every packed element, up to 4 source indices into the OIHW tensor
// (-1 = none): forward packs gather one element, the upsample phases sum up to four taps. The same map drives the
// gradient scatter (packed gradient element added to each of its sources).
__global__ void pack_gather_kernel(const float* __restrict__ src, const int32_t* __restrict__ map, __half* __restrict__ dst, int64_t n) {
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int4 m = __ldg(reinterpret_cast<const int4*>(map) + i);
        float v = 0.f;
        if (m.x >= 0) v += src[m.x];
        if (m.y >= 0) v += src[m.y];
        if (m.z >= 0) v += src[m.z];
        if (m.w >= 0) v += src[m.w];
        dst[i] = __float2half_rn(v);
    }
}

// the common case of the same re-pack: every packed element has ONE source (all layouts but the pre-summed nearest-x2 taps).
// 8 elements per thread: 32 bytes of map, 8 gathers, one 16-byte store (the 4-index map costs 16 bytes per element).
__global__ void pack_gather1_kernel(const float* __restrict__ src, const int32_t* __restrict__ map, __half* __restrict__ dst, int64_t n8) {
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n8; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int4 m0 = __ldg(reinterpret_cast<const int4*>(map) + 2 * i);
        const int4 m1 = __ldg(reinterpret_cast<const int4*>(map) + 2 * i + 1);
        const int idx[8] = {m0.x, m0.y, m0.z, m0.w, m1.x, m1.y, m1.z, m1.w};
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = idx[j] >= 0 ? __ldg(src + idx[j]) : 0.f;
        store8(dst + 8 * i, v);
    }
}

__global__ void unpack_scatter_kernel(const float* __restrict__ packed_grad, const int32_t* __restrict__ map, float* __restrict__ grad,
                                      int64_t n, float mul) {
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int4 m = __ldg(reinterpret_cast<const int4*>(map) + i);
        const float g = packed_grad[i] * mul;
        if (m.x >= 0) atomicAdd(&grad[m.x], g);
        if (m.y >= 0) atomicAdd(&grad[m.y], g);
        if (m.z >= 0) atomicAdd(&grad[m.z], g);
        if (m.w >= 0) atomicAdd(&grad[m.w], g);
    }
}

// Deterministic form of the same scatter: one thread per OIHW gradient element, which GATHERS its (at most four) packed
// contributions in index order -- the nearest-x2 phases route every 3x3 weight into four packed elements, and adding those with
// atomics made the last bits of the decoder gradients depend on the thread schedule.
__global__ void unpack_gather_kernel(const float* __restrict__ packed_grad, const int32_t* __restrict__ dst_idx, const int32_t* __restrict__ inv,
                                     float* __restrict__ grad, int64_t n, float mul) {
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int4 m = __ldg(reinterpret_cast<const int4*>(inv) + i);
        float g = 0.f;
        if (m.x >= 0) g += packed_grad[m.x];
        if (m.y >= 0) g += packed_grad[m.y];
        if (m.z >= 0) g += packed_grad[m.z];
        if (m.w >= 0) g += packed_grad[m.w];
        grad[dst_idx[i]] = g * mul;
    }
}

// dst_i[j] += alpha * src_i[j] over a table of (src, dst, n) fp32 segments, one block per segment: the whole network's
// parameter gradients are added into the caller's .grad tensors in one launch (instead of one autograd add per tensor).
__global__ void multi_axpy_kernel(const int64_t* __restrict__ table, float alpha) {
    const int64_t* t = table + static_cast<int64_t>(blockIdx.x) * 3;
    const float* __restrict__ src = reinterpret_cast<const float*>(t[0]);
    float* __restrict__ dst = reinterpret_cast<float*>(t[1]);
    const int n = static_cast<int>(t[2]);
    for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] += alpha * src[i];
}

// ------------------------------------------------------------------------------------------------
// Strict-precision training forward. Every forward activation is an fp16 (hi, lo) pair in two planes `plane` elements apart,
// value = hi + lo (exact in fp32), with hi = half(v) and lo = half(v - hi) as the split convolutions write them.

// v -> (hi, lo) of v * scale; `bad` when hi would not be a finite fp16 (|v * scale| rounds past 65504, or v is inf / NaN)
__device__ __forceinline__ bool split_scaled(float v, float scale, __half& hi, __half& lo) {
    const float vs = v * scale;
    hi = __float2half_rn(vs);
    lo = __float2half_rn(vs - __half2float(hi));
    return !(fabsf(vs) < 65520.f);
}

__device__ __forceinline__ void split8(const float (&v)[8], __half* hi, __half* lo) {
    __align__(16) __half h[8];
    __align__(16) __half l[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        h[e] = __float2half_rn(v[e]);
        l[e] = __float2half_rn(v[e] - __half2float(h[e]));
    }
    *reinterpret_cast<uint4*>(hi) = *reinterpret_cast<const uint4*>(h);
    *reinterpret_cast<uint4*>(lo) = *reinterpret_cast<const uint4*>(l);
}

// 8 channels of a pair as fp32 values hi + lo
__device__ __forceinline__ void load8_pair(const __half* p, int64_t plane, float (&v)[8]) {
    float l[8];
    load8(p, v);
    load8(p + plane, l);
#pragma unroll
    for (int e = 0; e < 8; ++e) v[e] += l[e];
}

// fp32 master weights -> split packed operand [2][n] (hi plane, lo plane at + plane) of w * scale, scale = 2^e fixed per layer.
// Elements whose scaled hi is not a finite fp16 are counted in *overflow (the plan's exponent no longer fits the weights).
__global__ void pack_gather_split_kernel(const float* __restrict__ src, const int32_t* __restrict__ map, __half* __restrict__ dst, int64_t plane,
                                         int64_t n, float scale, int* __restrict__ overflow) {
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int4 m = __ldg(reinterpret_cast<const int4*>(map) + i);
        float v = 0.f;
        if (m.x >= 0) v += src[m.x];
        if (m.y >= 0) v += src[m.y];
        if (m.z >= 0) v += src[m.z];
        if (m.w >= 0) v += src[m.w];
        __half h, l;
        if (split_scaled(v, scale, h, l)) atomicAdd(overflow, 1);
        dst[i] = h;
        dst[plane + i] = l;
    }
}

__global__ void pack_gather1_split_kernel(const float* __restrict__ src, const int32_t* __restrict__ map, __half* __restrict__ dst, int64_t plane,
                                          int64_t n8, float scale, int* __restrict__ overflow) {
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n8; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int4 m0 = __ldg(reinterpret_cast<const int4*>(map) + 2 * i);
        const int4 m1 = __ldg(reinterpret_cast<const int4*>(map) + 2 * i + 1);
        const int idx[8] = {m0.x, m0.y, m0.z, m0.w, m1.x, m1.y, m1.z, m1.w};
        __align__(16) __half h[8];
        __align__(16) __half l[8];
        int bad = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) bad += split_scaled(idx[j] >= 0 ? __ldg(src + idx[j]) : 0.f, scale, h[j], l[j]) ? 1 : 0;
        if (bad) atomicAdd(overflow, bad);
        *reinterpret_cast<uint4*>(dst + 8 * i) = *reinterpret_cast<const uint4*>(h);
        *reinterpret_cast<uint4*>(dst + plane + 8 * i) = *reinterpret_cast<const uint4*>(l);
    }
}

// BatchNorm finalize of one channel from the folded slot sums (what channel_reduce_kernel<0>'s last block does)
__device__ __forceinline__ void bn_finalize_channel(double* sums, int c, int C, double dM, const RedTail& tail) {
    const double t0 = red_slots(sums, 0, c, C), t1 = red_slots(sums, 1, c, C);
    const double mean = t0 / dM;
    double var = t1 / dM - mean * mean;
    if (var < 0) var = 0;
    const float invstd = static_cast<float>(1.0 / sqrt(var + static_cast<double>(tail.eps)));
    const float sc = tail.gamma[c] * invstd;
    tail.mean[c] = static_cast<float>(mean);
    tail.invstd[c] = invstd;
    tail.scale[c] = sc;
    tail.shift[c] = tail.beta[c] - static_cast<float>(mean) * sc;
    if (tail.running_mean && !(tail.frozen && *tail.frozen)) {
        const double unbiased = dM > 1 ? var * dM / (dM - 1.0) : var;
        tail.running_mean[c] = (1.f - tail.momentum) * tail.running_mean[c] + tail.momentum * static_cast<float>(mean);
        tail.running_var[c] = (1.f - tail.momentum) * tail.running_var[c] + tail.momentum * static_cast<float>(unbiased);
    }
    if (tail.self_clean) {
#pragma unroll
        for (int sl = 0; sl < kRedSlots; ++sl) {
            sums[(static_cast<int64_t>(sl) * 2 + 0) * C + c] = 0.0;
            sums[(static_cast<int64_t>(sl) * 2 + 1) * C + c] = 0.0;
        }
    }
}

// Batch statistics of a two-plane z: per-channel sums of v = hi + lo and of v*v, accumulated in fp64 from the first add on
// (fp32 partial sums would cost the statistics the precision the split forward buys), same slots / last-block finalize as
// channel_reduce_kernel<0>. Thread mapping as there: C/8 threads per row, 256/(C/8) rows per iteration.
__global__ void __launch_bounds__(256) bn_stats_split_kernel(const __half* __restrict__ z, int64_t plane, double* __restrict__ sums, int64_t M, int C,
                                                             const RedTail tail) {
    __shared__ double sh0[256 * 8];
    __shared__ double sh1[256 * 8];
    pdl_sync();
    const int tpr = C / 8;
    const int rows_per_iter = 256 / tpr;
    const int col = (threadIdx.x % tpr) * 8;
    const int rsub = threadIdx.x / tpr;
    double acc0[8], acc1[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc0[i] = acc1[i] = 0.0;
    const int64_t step = static_cast<int64_t>(gridDim.x) * rows_per_iter;
    auto fold = [&](const float (&v)[8]) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const double d = static_cast<double>(v[i]);
            acc0[i] += d;
            acc1[i] = fma(d, d, acc1[i]);
        }
    };
    int64_t r = static_cast<int64_t>(blockIdx.x) * rows_per_iter + rsub;
    for (; r + step < M; r += 2 * step) {
        float v0[8], v1[8];
        load8_pair(z + r * C + col, plane, v0);
        load8_pair(z + (r + step) * C + col, plane, v1);
        fold(v0);
        fold(v1);
    }
    if (r < M) {
        float v0[8];
        load8_pair(z + r * C + col, plane, v0);
        fold(v0);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        sh0[threadIdx.x * 8 + i] = acc0[i];
        sh1[threadIdx.x * 8 + i] = acc1[i];
    }
    __syncthreads();
    double* s0 = sums + static_cast<int64_t>(blockIdx.x % kRedSlots) * 2 * C;
    double* s1 = s0 + C;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        const int t0 = c / 8, e = c % 8;
        double a0 = 0.0, a1 = 0.0;
        for (int g = 0; g < rows_per_iter; ++g) {
            a0 += sh0[(g * tpr + t0) * 8 + e];
            a1 += sh1[(g * tpr + t0) * 8 + e];
        }
        atomicAdd(&s0[c], a0);
        atomicAdd(&s1[c], a1);
    }
    __shared__ bool is_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned* counter = reinterpret_cast<unsigned*>(sums + static_cast<int64_t>(kRedSlots) * 2 * C);
        is_last = atomicAdd(counter, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    if (threadIdx.x == 0 && tail.num_batches && !(tail.frozen && *tail.frozen)) *tail.num_batches += 1;
    for (int c = threadIdx.x; c < C; c += blockDim.x) bn_finalize_channel(sums, c, C, static_cast<double>(M), tail);
    if (tail.self_clean && threadIdx.x == 0) *reinterpret_cast<unsigned*>(sums + static_cast<int64_t>(kRedSlots) * 2 * C) = 0u;
}

// y = relu?(z*scale + shift (+ res)) in fp32 from two-plane z and residual, written as a (hi, lo) pair. Channel mapping as
// bn_apply_kernel (every thread keeps the same 8 channels for its whole loop).
__global__ void bn_apply_split_kernel(const __half* __restrict__ z, int64_t zplane, const float* __restrict__ scale, const float* __restrict__ shift,
                                      const __half* __restrict__ res, int64_t rplane, __half* __restrict__ y, int64_t yplane, int64_t M, int C,
                                      int relu) {
    pdl_sync();
    const int C8 = C / 8;
    const int64_t total = M * C8;
    const int64_t i0 = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    const int col = static_cast<int>(i0 % C8) * 8;
    float sc[8], sh[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        sc[e] = scale[col + e];
        sh[e] = shift[col + e];
    }
    const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
    for (int64_t i = i0; i < total; i += stride) {
        float v[8], r[8];
        load8_pair(z + i * 8, zplane, v);
        if (res) load8_pair(res + i * 8, rplane, r);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            float o = fmaf(v[e], sc[e], sh[e]);
            if (res) o += r[e];
            v[e] = relu ? fmaxf(o, 0.f) : o;
        }
        split8(v, y + i * 8, y + yplane + i * 8);
    }
}

// max-pool arg-max of two-plane x: the window position (dy*k + dx, row-major scan) of the FIRST element whose hi + lo equals the
// window's maximum -- ties, including pairs whose hi planes tie and whose lo planes decide, resolve like ATen's max_pool2d
// (first maximum in scan order) on the fp32 values. rsb_maxpool_nhwc_split takes its maximum over the same values.
__global__ void maxpool_argmax_split_kernel(const __half* __restrict__ x, int64_t plane, uint8_t* __restrict__ idx, int N, int H, int W, int C, int k,
                                            int s, int p, int OH, int OW) {
    const int C8 = C / 8;
    const int64_t total = static_cast<int64_t>(N) * OH * OW * C8;
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int c8 = static_cast<int>(i % C8);
        int64_t r = i / C8;
        const int ow = static_cast<int>(r % OW);
        r /= OW;
        const int oh = static_cast<int>(r % OH);
        const int n = static_cast<int>(r / OH);
        float best[8];
        uint32_t pos[8];
        bool any = false;
        for (int dyy = 0; dyy < k; ++dyy) {
            const int hh = oh * s - p + dyy;
            if (hh < 0 || hh >= H) continue;
            for (int dxx = 0; dxx < k; ++dxx) {
                const int ww = ow * s - p + dxx;
                if (ww < 0 || ww >= W) continue;
                float v[8];
                load8_pair(x + ((static_cast<int64_t>(n) * H + hh) * W + ww) * C + c8 * 8, plane, v);
                const uint32_t q = static_cast<uint32_t>(dyy * k + dxx);
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    if (!any || v[e] > best[e]) {
                        best[e] = v[e];
                        pos[e] = q;
                    }
                }
                any = true;
            }
        }
        uint2 o;
        o.x = pos[0] | (pos[1] << 8) | (pos[2] << 16) | (pos[3] << 24);
        o.y = pos[4] | (pos[5] << 8) | (pos[6] << 16) | (pos[7] << 24);
        *reinterpret_cast<uint2*>(idx + i * 8) = o;
    }
}

// final 1x1 conv forward on two-plane dec5 activations: the fp32 values hi + lo contracted with the fp32 weights in fp32.
// *overflow != 0: the plan's packed weights are not finite, and neither are the logits (NaN): the loss and the gradients of the
// step follow, so the guarded optimiser skips it (a ReLU may have turned the non-finite activations into finite garbage on the way)
__global__ void final_fwd_split_kernel(const __half* __restrict__ y5, int64_t plane, const float* __restrict__ w, const float* __restrict__ b,
                                       const int* __restrict__ overflow, float* __restrict__ logits, int64_t P, int64_t HW, int classes) {
    const bool poisoned = overflow && *overflow;
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < P; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        float v[32];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float t[8];
            load8_pair(y5 + i * 32 + j * 8, plane, t);
#pragma unroll
            for (int e = 0; e < 8; ++e) v[j * 8 + e] = t[e];
        }
        const int64_t n = i / HW, pix = i % HW;
        for (int k = 0; k < classes; ++k) {
            float s = b[k];
#pragma unroll
            for (int c = 0; c < 32; ++c) s = fmaf(w[k * 32 + c], v[c], s);
            logits[(n * classes + k) * HW + pix] = poisoned ? __int_as_float(0x7fc00000) : s;
        }
    }
}

}  // namespace rsb

using namespace rsb;

#define RSB_LAUNCH_CHECK(what)                                            \
    do {                                                                  \
        cudaError_t e__ = cudaGetLastError();                             \
        if (e__ != cudaSuccess) return set_cuda_error(e__, what);         \
    } while (0)

static bool bad_c(int C) { return C <= 0 || (C % 8) || (C > 2048) || (256 % (C / 8 > 256 ? 256 : C / 8)); }

extern "C" int rsb_bn_stats(const void* z, double* sums, int64_t M, int32_t C, void* stream) {
    if (!z || !sums || M <= 0 || bad_c(C) || C < 64) return set_error(RSB_E_INVALID, "bn_stats: bad arguments (C in 64..2048, power of two)");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cudaError_t e = cudaMemsetAsync(sums, 0, sizeof(double) * (2 * C * kRedSlots + 2), st);
    if (e != cudaSuccess) return set_cuda_error(e, "bn_stats memset");
    RedTail tail = {};
    channel_reduce_kernel<0><<<reduce_blocks(M, C), 256, 0, st>>>(static_cast<const __half*>(z), nullptr, nullptr, sums, M, C, tail);
    RSB_LAUNCH_CHECK("bn_stats launch");
    return RSB_OK;
}

static int bn_stats_finalize_impl(const void* z, double* sums, const float* gamma, const float* beta, float* running_mean, float* running_var,
                                  int64_t* num_batches, float* mean, float* invstd, float* scale, float* shift, int64_t M, int32_t C, float eps,
                                  float momentum, void* stream, bool chained) {
    if (!z || !sums || !gamma || !beta || !mean || !invstd || !scale || !shift || M <= 0 || bad_c(C) || C < 64)
        return set_error(RSB_E_INVALID, "bn_stats_finalize: bad arguments (C in 64..2048, power of two)");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (!chained) {
        cudaError_t e = cudaMemsetAsync(sums, 0, sizeof(double) * (2 * C * kRedSlots + 2), st);
        if (e != cudaSuccess) return set_cuda_error(e, "bn_stats_finalize memset");
    }
    RedTail tail = {};
    tail.gamma = gamma;
    tail.beta = beta;
    tail.running_mean = running_mean;
    tail.running_var = running_var;
    tail.num_batches = num_batches;
    tail.mean = mean;
    tail.invstd = invstd;
    tail.scale = scale;
    tail.shift = shift;
    tail.eps = eps;
    tail.momentum = momentum;
    tail.self_clean = chained ? 1 : 0;
    cudaError_t e = launch_chained(chained, channel_reduce_kernel<0, false>, reduce_blocks(M, C), 256, st, static_cast<const __half*>(z),
                                   static_cast<const __half*>(nullptr), static_cast<const __half*>(nullptr), sums, M, static_cast<int>(C), tail,
                                   static_cast<const float*>(nullptr), static_cast<const float*>(nullptr));
    if (e != cudaSuccess) return set_cuda_error(e, "bn_stats_finalize launch");
    return RSB_OK;
}

extern "C" int rsb_bn_stats_finalize(const void* z, double* sums, const float* gamma, const float* beta, float* running_mean, float* running_var,
                                     int64_t* num_batches, float* mean, float* invstd, float* scale, float* shift, int64_t M, int32_t C, float eps,
                                     float momentum, void* stream) {
    return bn_stats_finalize_impl(z, sums, gamma, beta, running_mean, running_var, num_batches, mean, invstd, scale, shift, M, C, eps, momentum, stream,
                                  false);
}

extern "C" int rsb_bn_stats_finalize_chained(const void* z, double* sums, const float* gamma, const float* beta, float* running_mean,
                                             float* running_var, int64_t* num_batches, float* mean, float* invstd, float* scale, float* shift,
                                             int64_t M, int32_t C, float eps, float momentum, void* stream) {
    return bn_stats_finalize_impl(z, sums, gamma, beta, running_mean, running_var, num_batches, mean, invstd, scale, shift, M, C, eps, momentum, stream,
                                  true);
}

extern "C" int rsb_bn_partials_finalize(const float* partials, int64_t rows, double* sums, const float* gamma, const float* beta, float* running_mean,
                                        float* running_var, int64_t* num_batches, float* mean, float* invstd, float* scale, float* shift, int64_t M,
                                        int32_t C, float eps, float momentum, int32_t chained, void* stream) {
    if (!partials || rows <= 0 || !sums || !gamma || !beta || !mean || !invstd || !scale || !shift || M <= 0 || bad_c(C) || C < 32 ||
        (reinterpret_cast<uintptr_t>(partials) & 15))
        return set_error(RSB_E_INVALID, "bn_partials_finalize: bad arguments (C in 32..2048, power of two; partials 16B aligned)");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (!chained) {
        cudaError_t e = cudaMemsetAsync(sums, 0, sizeof(double) * (2 * C * kRedSlots + 2), st);
        if (e != cudaSuccess) return set_cuda_error(e, "bn_partials_finalize memset");
    }
    RedTail tail = {};
    tail.gamma = gamma;
    tail.beta = beta;
    tail.running_mean = running_mean;
    tail.running_var = running_var;
    tail.num_batches = num_batches;
    tail.mean = mean;
    tail.invstd = invstd;
    tail.scale = scale;
    tail.shift = shift;
    tail.eps = eps;
    tail.momentum = momentum;
    tail.self_clean = chained ? 1 : 0;
    const int L = 2 * C;
    const int tpr = L / 4 < 256 ? L / 4 : 256;
    const int colblocks = L / (tpr * 4);
    const int rows_per_iter = 256 / tpr;
    int64_t bx = (rows + rows_per_iter * 4 - 1) / (rows_per_iter * 4);
    const int64_t cap = (2 * num_sms() + colblocks - 1) / colblocks;
    if (bx > cap) bx = cap;
    if (bx < 1) bx = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(static_cast<unsigned>(bx), static_cast<unsigned>(colblocks));
    cfg.blockDim = dim3(256);
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = chained ? 1 : 0;
    cudaError_t e = cudaLaunchKernelEx(&cfg, partial_reduce_kernel, partials, sums, rows, L, static_cast<int>(C), M, tail);
    if (e != cudaSuccess) return set_cuda_error(e, "bn_partials_finalize launch");
    return RSB_OK;
}

extern "C" int rsb_bn_finalize(const double* sums, const float* gamma, const float* beta, float* running_mean, float* running_var,
                               int64_t* num_batches, float* mean, float* invstd, float* scale, float* shift, int32_t C, int64_t M,
                               float eps, float momentum, void* stream) {
    if (!sums || !gamma || !beta || !mean || !invstd || !scale || !shift || C <= 0 || M <= 0) return set_error(RSB_E_INVALID, "bn_finalize: bad arguments");
    bn_finalize_kernel<<<(C + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(sums, gamma, beta, running_mean, running_var,
                                                                                   num_batches, mean, invstd, scale, shift, C,
                                                                                   static_cast<double>(M), eps, momentum);
    RSB_LAUNCH_CHECK("bn_finalize launch");
    return RSB_OK;
}

static int bn_apply_impl(const void* z, const float* scale, const float* shift, const void* residual, void* y, int64_t M, int32_t C, int32_t relu,
                         void* stream, bool chained) {
    if (!z || !scale || !shift || !y || M <= 0 || C <= 0 || (C % 8)) return set_error(RSB_E_INVALID, "bn_apply: bad arguments");
    cudaError_t e = launch_chained(chained, bn_apply_kernel, tr_blocks(M * (C / 8), 256), 256, static_cast<cudaStream_t>(stream),
                                   static_cast<const __half*>(z), scale, shift, static_cast<const __half*>(residual), static_cast<__half*>(y), M,
                                   static_cast<int>(C), static_cast<int>(relu));
    if (e != cudaSuccess) return set_cuda_error(e, "bn_apply launch");
    return RSB_OK;
}

extern "C" int rsb_bn_apply(const void* z, const float* scale, const float* shift, const void* residual, void* y, int64_t M, int32_t C,
                            int32_t relu, void* stream) {
    return bn_apply_impl(z, scale, shift, residual, y, M, C, relu, stream, false);
}

extern "C" int rsb_bn_apply_chained(const void* z, const float* scale, const float* shift, const void* residual, void* y, int64_t M, int32_t C,
                                    int32_t relu, void* stream) {
    return bn_apply_impl(z, scale, shift, residual, y, M, C, relu, stream, true);
}

static int bn_backward_impl(const void* dy, const void* y, const void* z, const float* mean, const float* invstd, const float* gamma,
                            const float* mask_scale, const float* mask_shift, double* sums, void* dz, void* g_out, float* dgamma, float* dbeta,
                            float inv_loss_scale, int64_t M, int32_t C, void* stream, bool chained) {
    if (!dy || !z || !mean || !invstd || !gamma || !sums || !dz || !dgamma || !dbeta || M <= 0 || bad_c(C) || C < 64)
        return set_error(RSB_E_INVALID, "bn_backward: bad arguments");
    if ((mask_scale != nullptr) != (mask_shift != nullptr) || (mask_scale && y))
        return set_error(RSB_E_INVALID, "bn_backward: pass either y, or mask_scale + mask_shift, or neither");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (!chained) {
        cudaError_t e = cudaMemsetAsync(sums, 0, sizeof(double) * (2 * C * kRedSlots + 2), st);
        if (e != cudaSuccess) return set_cuda_error(e, "bn_backward memset");
    }
    RedTail tail = {};
    tail.gamma = gamma;
    tail.mean = const_cast<float*>(mean);
    tail.invstd = const_cast<float*>(invstd);
    tail.dgamma = dgamma;
    tail.dbeta = dbeta;
    tail.inv_scale = inv_loss_scale;
    tail.self_clean = chained ? 1 : 0;
    const __half* dyh = static_cast<const __half*>(dy);
    const __half* yh = static_cast<const __half*>(y);
    const __half* zh = static_cast<const __half*>(z);
    const float* coef = reinterpret_cast<const float*>(sums + static_cast<int64_t>(kRedSlots) * 2 * C + 2);
    const unsigned ablocks = tr_blocks((M * (C / 8) + 3) / 4, 256);
    const __half* nullh = nullptr;
    const float* nullf = nullptr;
    cudaError_t e;
    if (mask_scale) {
        e = launch_chained(chained, channel_reduce_kernel<1, true>, reduce_blocks(M, C), 256, st, dyh, nullh, zh, sums, M, static_cast<int>(C), tail, mask_scale,
                           mask_shift);
        if (e == cudaSuccess)
            e = launch_chained(chained, bn_bwd_apply_kernel<true>, ablocks, 256, st, dyh, nullh, zh, coef, static_cast<__half*>(dz), static_cast<__half*>(g_out),
                               M, static_cast<int>(C), mask_scale, mask_shift);
    } else {
        e = launch_chained(chained, channel_reduce_kernel<1, false>, reduce_blocks(M, C), 256, st, dyh, yh, zh, sums, M, static_cast<int>(C), tail, nullf, nullf);
        if (e == cudaSuccess)
            e = launch_chained(chained, bn_bwd_apply_kernel<false>, ablocks, 256, st, dyh, yh, zh, coef, static_cast<__half*>(dz), static_cast<__half*>(g_out),
                               M, static_cast<int>(C), nullf, nullf);
    }
    if (e != cudaSuccess) return set_cuda_error(e, "bn_backward launch");
    return RSB_OK;
}

extern "C" int rsb_bn_backward(const void* dy, const void* y, const void* z, const float* mean, const float* invstd, const float* gamma,
                               const float* mask_scale, const float* mask_shift, double* sums, void* dz, void* g_out, float* dgamma, float* dbeta,
                               float inv_loss_scale, int64_t M, int32_t C, void* stream) {
    return bn_backward_impl(dy, y, z, mean, invstd, gamma, mask_scale, mask_shift, sums, dz, g_out, dgamma, dbeta, inv_loss_scale, M, C, stream, false);
}

extern "C" int rsb_bn_backward_chained(const void* dy, const void* y, const void* z, const float* mean, const float* invstd, const float* gamma,
                                       const float* mask_scale, const float* mask_shift, double* sums, void* dz, void* g_out, float* dgamma,
                                       float* dbeta, float inv_loss_scale, int64_t M, int32_t C, void* stream) {
    return bn_backward_impl(dy, y, z, mean, invstd, gamma, mask_scale, mask_shift, sums, dz, g_out, dgamma, dbeta, inv_loss_scale, M, C, stream, true);
}

extern "C" int rsb_relu_backward(const void* a, const void* b, const void* y, void* out, int64_t n, void* stream) {
    if (!a || !out || n <= 0 || (n % 8)) return set_error(RSB_E_INVALID, "relu_backward: bad arguments");
    relu_bwd_kernel<<<tr_blocks(n / 8, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __half*>(a), static_cast<const __half*>(b), static_cast<const __half*>(y), static_cast<__half*>(out), n / 8);
    RSB_LAUNCH_CHECK("relu_backward launch");
    return RSB_OK;
}

extern "C" int rsb_maxpool_backward(const void* x, const void* dy, void* dx, void* argmax_scratch, int32_t N, int32_t H, int32_t W, int32_t C,
                                    int32_t k, int32_t s, int32_t p, void* stream) {
    if (!x || !dy || !dx || N <= 0 || H <= 0 || W <= 0 || C <= 0 || (C % 8) || k < 1 || k > 15 || s < 1 || p < 0)
        return set_error(RSB_E_INVALID, "maxpool_backward: bad arguments");
    const int OH = (H + 2 * p - k) / s + 1, OW = (W + 2 * p - k) / s + 1;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (argmax_scratch) {
        uint8_t* idx = static_cast<uint8_t*>(argmax_scratch);
        maxpool_argmax_kernel<<<tr_blocks(static_cast<int64_t>(N) * OH * OW * (C / 8), 256), 256, 0, st>>>(static_cast<const __half*>(x), idx, N, H, W,
                                                                                                          C, k, s, p, OH, OW);
        RSB_LAUNCH_CHECK("maxpool_argmax launch");
        maxpool_bwd_gather_kernel<<<tr_blocks(static_cast<int64_t>(N) * H * W * (C / 8), 256), 256, 0, st>>>(
            idx, static_cast<const __half*>(dy), static_cast<__half*>(dx), N, H, W, C, k, s, p, OH, OW);
        RSB_LAUNCH_CHECK("maxpool_bwd_gather launch");
        return RSB_OK;
    }
    maxpool_bwd_kernel<<<tr_blocks(static_cast<int64_t>(N) * H * W * (C / 8), 256), 256, 0, st>>>(
        static_cast<const __half*>(x), static_cast<const __half*>(dy), static_cast<__half*>(dx), N, H, W, C, k, s, p, OH, OW);
    RSB_LAUNCH_CHECK("maxpool_backward launch");
    return RSB_OK;
}

extern "C" int rsb_final_forward(const void* y5, const float* w, const float* b, float* logits, int32_t N, int32_t HW, int32_t classes,
                                 void* stream) {
    if (!y5 || !w || !b || !logits || N <= 0 || HW <= 0 || classes < 1 || classes > 8) return set_error(RSB_E_INVALID, "final_forward: bad arguments");
    const int64_t P = static_cast<int64_t>(N) * HW;
    final_fwd_kernel<<<tr_blocks(P, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const __half*>(y5), w, b, logits, P, HW, classes);
    RSB_LAUNCH_CHECK("final_forward launch");
    return RSB_OK;
}

extern "C" int rsb_final_backward(const float* dlogits, const void* y5, const float* w, void* dy5, double* acc, float* dw, float* db,
                                  float loss_scale, int32_t N, int32_t HW, int32_t classes, void* stream) {
    if (!dlogits || !y5 || !w || !dy5 || !acc || !dw || !db || N <= 0 || HW <= 0 || classes < 1 || classes > 8)
        return set_error(RSB_E_INVALID, "final_backward: bad arguments");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cudaError_t e = cudaMemsetAsync(acc, 0, sizeof(double) * (classes * 32 + 8), st);
    if (e != cudaSuccess) return set_cuda_error(e, "final_backward memset");
    const int64_t P = static_cast<int64_t>(N) * HW;
    final_bwd_dx_kernel<<<tr_blocks(P, 256), 256, 0, st>>>(dlogits, w, static_cast<__half*>(dy5), loss_scale, P, HW, classes);
    for (int k = 0; k < classes; ++k)
        final_bwd_dw_kernel<<<tr_blocks(P, 256, 148 * 2), 256, 0, st>>>(dlogits, static_cast<const __half*>(y5), acc, acc + classes * 32, k, P, HW, classes);
    f64_to_f32_kernel<<<(classes * 32 + 127) / 128, 128, 0, st>>>(acc, dw, classes * 32, 1.0f);
    f64_to_f32_kernel<<<1, 128, 0, st>>>(acc + classes * 32, db, classes, 1.0f);
    RSB_LAUNCH_CHECK("final_backward launch");
    return RSB_OK;
}

extern "C" int rsb_pack_weights(const float* src, const int32_t* map4, void* dst, int64_t n, void* stream) {
    if (!src || !map4 || !dst || n <= 0) return set_error(RSB_E_INVALID, "pack_weights: bad arguments");
    pack_gather_kernel<<<tr_blocks(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(src, map4, static_cast<__half*>(dst), n);
    RSB_LAUNCH_CHECK("pack_weights launch");
    return RSB_OK;
}

extern "C" int rsb_pack_weights1(const float* src, const int32_t* map1, void* dst, int64_t n, void* stream) {
    if (!src || !map1 || !dst || n <= 0 || (n % 8) || (reinterpret_cast<uintptr_t>(dst) & 15) || (reinterpret_cast<uintptr_t>(map1) & 15))
        return set_error(RSB_E_INVALID, "pack_weights1: bad arguments (n a multiple of 8, map and dst 16B aligned)");
    pack_gather1_kernel<<<tr_blocks(n / 8, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(src, map1, static_cast<__half*>(dst), n / 8);
    RSB_LAUNCH_CHECK("pack_weights1 launch");
    return RSB_OK;
}

extern "C" int rsb_unpack_grads(const float* packed_grad, const int32_t* map4, float* grad, int64_t n, float mul, void* stream) {
    if (!packed_grad || !map4 || !grad || n <= 0) return set_error(RSB_E_INVALID, "unpack_grads: bad arguments");
    unpack_scatter_kernel<<<tr_blocks(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(packed_grad, map4, grad, n, mul);
    RSB_LAUNCH_CHECK("unpack_grads launch");
    return RSB_OK;
}

extern "C" int rsb_unpack_grads_gather(const float* packed_grad, const int32_t* dst_idx, const int32_t* inv4, float* grad, int64_t n, float mul,
                                       void* stream) {
    if (!packed_grad || !dst_idx || !inv4 || !grad || n <= 0) return set_error(RSB_E_INVALID, "unpack_grads_gather: bad arguments");
    int64_t blocks = (n + 255) / 256;
    if (blocks > 65535) blocks = 65535;
    unpack_gather_kernel<<<static_cast<unsigned>(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(packed_grad, dst_idx, inv4, grad, n, mul);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? RSB_OK : set_cuda_error(e, "unpack_gather launch");
}

extern "C" int rsb_multi_axpy(const int64_t* table, int32_t segments, float alpha, void* stream) {
    if (!table || segments < 0) return set_error(RSB_E_INVALID, "multi_axpy: bad arguments");
    if (segments == 0) return RSB_OK;
    multi_axpy_kernel<<<static_cast<unsigned>(segments), 256, 0, static_cast<cudaStream_t>(stream)>>>(table, alpha);
    RSB_LAUNCH_CHECK("multi_axpy launch");
    return RSB_OK;
}

// ------------------------------------------------------------------------------------------------ strict-precision training forward
// every entry point validates its arguments first (RSB_E_INVALID on any host), then needs an sm_100 device (RSB_E_NODEVICE)
static bool bad_plane(const void* p, int64_t plane) { return !p || plane <= 0 || (plane % 8) || (reinterpret_cast<uintptr_t>(p) & 15); }

static int pack_split_impl(const float* src, const int32_t* map, void* dst, int64_t plane, int64_t n, float scale, int32_t* overflow, void* stream,
                           bool single) {
    if (!src || !map || !dst || !overflow || n <= 0 || plane < n || !(scale > 0.f) || !isfinite(scale))
        return set_error(RSB_E_INVALID, "pack_weights_split: bad arguments (plane >= n, scale a positive finite number)");
    if (single && ((n % 8) || (plane % 8) || (reinterpret_cast<uintptr_t>(dst) & 15) || (reinterpret_cast<uintptr_t>(map) & 15)))
        return set_error(RSB_E_INVALID, "pack_weights1_split: n and plane multiples of 8, map and dst 16B aligned");
    int rc = rsb_device_ok();
    if (rc != RSB_OK) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (single)
        pack_gather1_split_kernel<<<tr_blocks(n / 8, 256), 256, 0, st>>>(src, map, static_cast<__half*>(dst), plane, n / 8, scale, overflow);
    else
        pack_gather_split_kernel<<<tr_blocks(n, 256), 256, 0, st>>>(src, map, static_cast<__half*>(dst), plane, n, scale, overflow);
    RSB_LAUNCH_CHECK("pack_weights_split launch");
    return RSB_OK;
}

extern "C" int rsb_pack_weights_split(const float* src, const int32_t* map4, void* dst, int64_t plane, int64_t n, float scale, int32_t* overflow,
                                      void* stream) {
    return pack_split_impl(src, map4, dst, plane, n, scale, overflow, stream, false);
}

extern "C" int rsb_pack_weights1_split(const float* src, const int32_t* map1, void* dst, int64_t plane, int64_t n, float scale, int32_t* overflow,
                                       void* stream) {
    return pack_split_impl(src, map1, dst, plane, n, scale, overflow, stream, true);
}

static int bn_stats_split_impl(const void* z, int64_t plane, double* sums, const float* gamma, const float* beta, float* running_mean, float* running_var,
                               int64_t* num_batches, float* mean, float* invstd, float* scale, float* shift, int64_t M, int32_t C, float eps,
                               float momentum, const int32_t* overflow, void* stream, bool chained) {
    if (bad_plane(z, plane) || !sums || !gamma || !beta || !mean || !invstd || !scale || !shift || M <= 0 || bad_c(C) || C < 64)
        return set_error(RSB_E_INVALID, "bn_stats_finalize_split: bad arguments (C in 64..2048, power of two; plane a multiple of 8)");
    int rc = rsb_device_ok();
    if (rc != RSB_OK) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (!chained) {
        cudaError_t e = cudaMemsetAsync(sums, 0, sizeof(double) * (2 * C * kRedSlots + 2), st);
        if (e != cudaSuccess) return set_cuda_error(e, "bn_stats_finalize_split memset");
    }
    RedTail tail = {};
    tail.gamma = gamma;
    tail.beta = beta;
    tail.running_mean = running_mean;
    tail.running_var = running_var;
    tail.num_batches = num_batches;
    tail.mean = mean;
    tail.invstd = invstd;
    tail.scale = scale;
    tail.shift = shift;
    tail.eps = eps;
    tail.momentum = momentum;
    tail.self_clean = chained ? 1 : 0;
    tail.frozen = overflow;
    cudaError_t e = launch_chained(chained, bn_stats_split_kernel, reduce_blocks(M, C), 256, st, static_cast<const __half*>(z), plane, sums, M,
                                   static_cast<int>(C), tail);
    if (e != cudaSuccess) return set_cuda_error(e, "bn_stats_finalize_split launch");
    return RSB_OK;
}

extern "C" int rsb_bn_stats_finalize_split(const void* z, int64_t plane, double* sums, const float* gamma, const float* beta, float* running_mean,
                                           float* running_var, int64_t* num_batches, float* mean, float* invstd, float* scale, float* shift, int64_t M,
                                           int32_t C, float eps, float momentum, const int32_t* overflow, void* stream) {
    return bn_stats_split_impl(z, plane, sums, gamma, beta, running_mean, running_var, num_batches, mean, invstd, scale, shift, M, C, eps, momentum,
                               overflow, stream, false);
}

extern "C" int rsb_bn_stats_finalize_split_chained(const void* z, int64_t plane, double* sums, const float* gamma, const float* beta,
                                                   float* running_mean, float* running_var, int64_t* num_batches, float* mean, float* invstd,
                                                   float* scale, float* shift, int64_t M, int32_t C, float eps, float momentum,
                                                   const int32_t* overflow, void* stream) {
    return bn_stats_split_impl(z, plane, sums, gamma, beta, running_mean, running_var, num_batches, mean, invstd, scale, shift, M, C, eps, momentum,
                               overflow, stream, true);
}

static int bn_apply_split_impl(const void* z, int64_t z_plane, const float* scale, const float* shift, const void* residual, int64_t res_plane, void* y,
                               int64_t y_plane, int64_t M, int32_t C, int32_t relu, void* stream, bool chained) {
    if (bad_plane(z, z_plane) || bad_plane(y, y_plane) || (residual && bad_plane(residual, res_plane)) || !scale || !shift || M <= 0 || C <= 0 ||
        (C % 8) || (256 % (C / 8 > 256 ? 256 : C / 8)))
        return set_error(RSB_E_INVALID, "bn_apply_split: bad arguments (C a multiple of 8 with C/8 dividing 256; planes multiples of 8)");
    int rc = rsb_device_ok();
    if (rc != RSB_OK) return rc;
    cudaError_t e = launch_chained(chained, bn_apply_split_kernel, tr_blocks(M * (C / 8), 256), 256, static_cast<cudaStream_t>(stream),
                                   static_cast<const __half*>(z), z_plane, scale, shift, static_cast<const __half*>(residual), res_plane,
                                   static_cast<__half*>(y), y_plane, M, static_cast<int>(C), static_cast<int>(relu));
    if (e != cudaSuccess) return set_cuda_error(e, "bn_apply_split launch");
    return RSB_OK;
}

extern "C" int rsb_bn_apply_split(const void* z, int64_t z_plane, const float* scale, const float* shift, const void* residual, int64_t res_plane,
                                  void* y, int64_t y_plane, int64_t M, int32_t C, int32_t relu, void* stream) {
    return bn_apply_split_impl(z, z_plane, scale, shift, residual, res_plane, y, y_plane, M, C, relu, stream, false);
}

extern "C" int rsb_bn_apply_split_chained(const void* z, int64_t z_plane, const float* scale, const float* shift, const void* residual,
                                          int64_t res_plane, void* y, int64_t y_plane, int64_t M, int32_t C, int32_t relu, void* stream) {
    return bn_apply_split_impl(z, z_plane, scale, shift, residual, res_plane, y, y_plane, M, C, relu, stream, true);
}

extern "C" int rsb_maxpool_backward_split(const void* x, int64_t x_plane, const void* dy, void* dx, void* argmax_scratch, int32_t N, int32_t H,
                                          int32_t W, int32_t C, int32_t k, int32_t s, int32_t p, void* stream) {
    if (bad_plane(x, x_plane) || !dy || !dx || !argmax_scratch || N <= 0 || H <= 0 || W <= 0 || C <= 0 || (C % 8) || k < 1 || k > 15 || s < 1 ||
        p < 0 || 2 * p > k)
        return set_error(RSB_E_INVALID, "maxpool_backward_split: bad arguments (argmax scratch required; C and x_plane multiples of 8)");
    int rc = rsb_device_ok();
    if (rc != RSB_OK) return rc;
    const int OH = (H + 2 * p - k) / s + 1, OW = (W + 2 * p - k) / s + 1;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    uint8_t* idx = static_cast<uint8_t*>(argmax_scratch);
    maxpool_argmax_split_kernel<<<tr_blocks(static_cast<int64_t>(N) * OH * OW * (C / 8), 256), 256, 0, st>>>(static_cast<const __half*>(x), x_plane,
                                                                                                            idx, N, H, W, C, k, s, p, OH, OW);
    RSB_LAUNCH_CHECK("maxpool_argmax_split launch");
    maxpool_bwd_gather_kernel<<<tr_blocks(static_cast<int64_t>(N) * H * W * (C / 8), 256), 256, 0, st>>>(
        idx, static_cast<const __half*>(dy), static_cast<__half*>(dx), N, H, W, C, k, s, p, OH, OW);
    RSB_LAUNCH_CHECK("maxpool_bwd_gather launch");
    return RSB_OK;
}

extern "C" int rsb_final_forward_split(const void* y5, int64_t plane, const float* w, const float* b, const int32_t* overflow, float* logits,
                                       int32_t N, int32_t HW, int32_t classes, void* stream) {
    if (bad_plane(y5, plane) || !w || !b || !logits || N <= 0 || HW <= 0 || classes < 1 || classes > 8)
        return set_error(RSB_E_INVALID, "final_forward_split: bad arguments");
    int rc = rsb_device_ok();
    if (rc != RSB_OK) return rc;
    const int64_t P = static_cast<int64_t>(N) * HW;
    final_fwd_split_kernel<<<tr_blocks(P, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const __half*>(y5), plane, w, b, overflow, logits,
                                                                                             P, HW, classes);
    RSB_LAUNCH_CHECK("final_forward_split launch");
    return RSB_OK;
}
