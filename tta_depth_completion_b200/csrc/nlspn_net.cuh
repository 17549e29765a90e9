// Channel-generic kernels of the NLSPN network around the tcgen05 convolutions (SURVEY.md section 8 row a18):
//   stem            conv1_rgb (3->48) + conv1_dep (1->16), bias, LeakyReLU(0.2)          nlspnmodel_adapt.py:385-388, 866-867
//   chan_stats      per-channel sum / sum of squares of an NHWC bf16 map (train-mode BatchNorm statistics; every BatchNorm2d of
//                   the network uses batch statistics after adapt_parameters('meta_bn'), src/nlspn_model_adapt.py:322-337)
//   bn_finalize     -> mean, rstd, scale = gamma*rstd, shift = beta - mean*scale (+ running statistics for the BatchNorm1d heads)
//   bn_act          y = act(x*scale + shift [+ residual | + residual*rscale + rshift])    common.py:45-80, torchvision BasicBlock
//   bn_bwd_*        g = (dyA + dyB) * act'(y);  d gamma = sum g*xhat, d beta = sum g;  dx = gamma*rstd*(g - mean(g) - xhat*mean(g*xhat))
//   conv8to24       prop_layer.conv_offset_aff (fp32, 3x3) and its data gradient              nlspnmodel_adapt.py:219-224, 259
//   thin_grad_pack  gradients of (pred_init, guide, confidence) through LeakyReLU / identity / sigmoid -> NHWC bf16 [.,64]
//   wgrad48         weight gradient of the adapted 48->48 meta conv (persistent CTAs, mma.sync, pixels = K)   :1370-1374
// All NHWC bf16 maps have channel counts that are multiples of 64; every elementwise thread moves 16 B (8 channels).
// Memory-bound kernels: algorithmic bytes = 2 B per element read / written, stated per kernel in DESIGN.md.
#pragma once
#include "common.cuh"
#include "peer_comm.cuh"

namespace ptta {

__device__ __forceinline__ void load8(const bf16* p, float (&f)[8]) {
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(p));
    const uint32_t* u = reinterpret_cast<const uint32_t*>(&v);
#pragma unroll
    for (int j = 0; j < 4; ++j) { const float2 t = unpack_bf162(u[j]); f[2 * j] = t.x; f[2 * j + 1] = t.y; }
}
__device__ __forceinline__ void unpack8(const uint4& v, float (&f)[8]) {
    const uint32_t* u = reinterpret_cast<const uint32_t*>(&v);
#pragma unroll
    for (int j = 0; j < 4; ++j) { const float2 t = unpack_bf162(u[j]); f[2 * j] = t.x; f[2 * j + 1] = t.y; }
}
__device__ __forceinline__ void store8(bf16* p, const float (&f)[8]) {
    uint4 v;
    v.x = pack_bf162(f[0], f[1]); v.y = pack_bf162(f[2], f[3]); v.z = pack_bf162(f[4], f[5]); v.w = pack_bf162(f[6], f[7]);
    *reinterpret_cast<uint4*>(p) = v;
}
__device__ __forceinline__ void load8f(const float* p, float (&f)[8]) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p) + 1);
    f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
}
// activation codes: 0 none, 1 ReLU, 2 LeakyReLU(0.2)
__device__ __forceinline__ float act_fwd(float v, int act) { return act == 1 ? fmaxf(v, 0.f) : (act == 2 ? (v > 0.f ? v : 0.2f * v) : v); }
__device__ __forceinline__ float act_der(float y, int act) { return act == 1 ? (y > 0.f ? 1.f : 0.f) : (act == 2 ? (y > 0.f ? 1.f : 0.2f) : 1.f); }

// ---- stem --------------------------------------------------------------------------------------------------------------------
// image fp32 NCHW [N,3,H,W] (null = the zero image of the second encoder pass, nlspnmodel_adapt.py:907), depth fp32 [N,1,H,W]
// -> out NHWC bf16 [N,H,W,64]: channels 0..47 = LeakyReLU(conv1_rgb), 48..63 = LeakyReLU(conv1_dep)
__global__ void __launch_bounds__(128) nl_stem_kernel(const float* __restrict__ image, const float* __restrict__ depth,
                                                      const float* __restrict__ w_rgb, const float* __restrict__ b_rgb,
                                                      const float* __restrict__ w_dep, const float* __restrict__ b_dep,
                                                      const float* __restrict__ scale, const float* __restrict__ shift,
                                                      bf16* __restrict__ out, int N, int H, int W, int n_src) {
    PDL_SYNC();
    __shared__ float s_w[27 * 48 + 9 * 16];      // [ci*9+tap][48] then [tap][16]
    __shared__ float s_b[64];
    for (int i = threadIdx.x; i < 27 * 48; i += blockDim.x) { const int co = i % 48, r = i / 48; s_w[i] = w_rgb[co * 27 + r]; }
    for (int i = threadIdx.x; i < 9 * 16; i += blockDim.x) { const int co = i % 16, r = i / 16; s_w[27 * 48 + i] = w_dep[co * 9 + r]; }
    if (threadIdx.x < 64) s_b[threadIdx.x] = threadIdx.x < 48 ? b_rgb[threadIdx.x] : b_dep[threadIdx.x - 48];
    __syncthreads();
    // image normalisation (x * scale + shift per channel) folded in; zero padding applies to the normalised image
    float nsc[3], nsh[3];
#pragma unroll
    for (int ci = 0; ci < 3; ++ci) { nsc[ci] = scale ? scale[ci] : 1.f; nsh[ci] = shift ? shift[ci] : 0.f; }
    const long long HW = (long long)H * W, total = (long long)N * HW;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int x = idx % W, y = (idx / W) % H, n_out = idx / HW;
    // pair mode (n_src < N): output images n_src .. N-1 are the zero-image copies of images 0 .. n_src-1 (same sparse depth)
    const int n = n_out % n_src;
    const bool has_image = image != nullptr && n_out < n_src;
    float acc[64];
#pragma unroll
    for (int c = 0; c < 64; ++c) acc[c] = s_b[c];
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
        const int gy = y + ky - 1;
        if (gy < 0 || gy >= H) continue;
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
            const int gx = x + kx - 1;
            if (gx < 0 || gx >= W) continue;
            const long long o = (long long)gy * W + gx;
            const int tap = ky * 3 + kx;
            if (has_image) {
#pragma unroll
                for (int ci = 0; ci < 3; ++ci) {
                    const float v = fmaf(__ldg(image + ((long long)n * 3 + ci) * HW + o), nsc[ci], nsh[ci]);
                    const float* wr = s_w + (ci * 9 + tap) * 48;
#pragma unroll
                    for (int c = 0; c < 48; ++c) acc[c] = fmaf(v, wr[c], acc[c]);
                }
            }
            const float d = __ldg(depth + (long long)n * HW + o);
            const float* wd = s_w + 27 * 48 + tap * 16;
#pragma unroll
            for (int c = 0; c < 16; ++c) acc[48 + c] = fmaf(d, wd[c], acc[48 + c]);
        }
    }
    bf16* dst = out + idx * 64;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        float f[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) { const float v = acc[q * 8 + j]; f[j] = v > 0.f ? v : 0.2f * v; }
        store8(dst + q * 8, f);
    }
}

// ---- per-channel reductions ----------------------------------------------------------------------------------------------------
// grid (blocks_p, C/64), 256 threads = 32 pixel lanes x 8 channel groups of 8.  partial[(blk*2 + s)*C + c]
// MODE 0: (sum x, sum x^2).  MODE 1: g = (dyA [+ dyB]) * act'(y): (sum g, sum g*xhat), xhat = (x - mean)*rstd
template <int MODE>
__global__ void __launch_bounds__(256) chan_reduce_kernel(const bf16* __restrict__ x, long long ldx, const bf16* __restrict__ dyA, long long ldA,
                                                          const bf16* __restrict__ dyB, long long ldB, const bf16* __restrict__ y, int act,
                                                          const float* __restrict__ mean, const float* __restrict__ rstd, long long P, int C,
                                                          float* __restrict__ partial) {
    PDL_SYNC();
    // blockIdx.z = statistics group (independent row ranges of P rows each, e.g. the real / zero-image halves of a merged batch)
    x += (long long)blockIdx.z * P * ldx;
    partial += (size_t)blockIdx.z * gridDim.x * 2 * C;
    __shared__ float sh[2][8][64];
    const int cg = threadIdx.x & 7, pl = threadIdx.x >> 3, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c0 = blockIdx.y * 64 + cg * 8;
    float s[8], q[8], mu[8], rs[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { s[j] = 0.f; q[j] = 0.f; }
    if (MODE == 1) { load8f(mean + c0, mu); load8f(rstd + c0, rs); }
    // U pixels per iteration: all their loads are issued before the first use (the kernel is a latency-bound stream otherwise)
    constexpr int U = MODE == 0 ? 4 : 2;
    const long long stride = (long long)gridDim.x * 32;
    for (long long p0 = (long long)blockIdx.x * 32 + pl; p0 < P; p0 += stride * U) {
        uint4 rx[U], ra[U], rb[U], ry[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const long long p = p0 + u * stride;
            const bool ok = p < P;
            const uint4 z = make_uint4(0u, 0u, 0u, 0u);
            rx[u] = ok ? __ldg(reinterpret_cast<const uint4*>(x + p * ldx + c0)) : z;
            if (MODE == 1) {
                ra[u] = ok ? __ldg(reinterpret_cast<const uint4*>(dyA + p * ldA + c0)) : z;
                rb[u] = (ok && dyB) ? __ldg(reinterpret_cast<const uint4*>(dyB + p * ldB + c0)) : z;
                ry[u] = (ok && act) ? __ldg(reinterpret_cast<const uint4*>(y + p * (long long)C + c0)) : z;
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (p0 + u * stride >= P) break;
            float xv[8];
            unpack8(rx[u], xv);
            if (MODE == 0) {
#pragma unroll
                for (int j = 0; j < 8; ++j) { s[j] += xv[j]; q[j] = fmaf(xv[j], xv[j], q[j]); }
            } else {
                float g[8];
                unpack8(ra[u], g);
                if (dyB) {
                    float b[8];
                    unpack8(rb[u], b);
#pragma unroll
                    for (int j = 0; j < 8; ++j) g[j] += b[j];
                }
                if (act) {
                    float yv[8];
                    unpack8(ry[u], yv);
#pragma unroll
                    for (int j = 0; j < 8; ++j) g[j] *= act_der(yv[j], act);
                }
#pragma unroll
                for (int j = 0; j < 8; ++j) { s[j] += g[j]; q[j] = fmaf(g[j], (xv[j] - mu[j]) * rs[j], q[j]); }
            }
        }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        s[j] += __shfl_xor_sync(0xffffffffu, s[j], 8); s[j] += __shfl_xor_sync(0xffffffffu, s[j], 16);
        q[j] += __shfl_xor_sync(0xffffffffu, q[j], 8); q[j] += __shfl_xor_sync(0xffffffffu, q[j], 16);
    }
    if (lane < 8) {
#pragma unroll
        for (int j = 0; j < 8; ++j) { sh[0][warp][cg * 8 + j] = s[j]; sh[1][warp][cg * 8 + j] = q[j]; }
    }
    __syncthreads();
    if (threadIdx.x < 128) {
        const int which = threadIdx.x >> 6, c = threadIdx.x & 63;
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) t += sh[which][w][c];
        partial[((size_t)blockIdx.x * 2 + which) * C + blockIdx.y * 64 + c] = t;
    }
}

// 1024 threads = 32 block-slices x 32 channels: every warp load is one coalesced 128 B row of the partial table, four rows in
// flight per thread (the loop is a chain of L2 round trips otherwise); the slices are combined through shared memory in a fixed
// order (deterministic).  Returns the totals to the threads of slice 0.
__device__ __forceinline__ bool partial_sums(const float* __restrict__ partial, int nblk, int C, int& c, double& s, double& q) {
    __shared__ double sh[2][32][32];
    const int lane = threadIdx.x & 31, slice = threadIdx.x >> 5;
    c = blockIdx.x * 32 + lane;
    s = 0.0; q = 0.0;
    if (c < C) {
        int b = slice;
        for (; b + 96 < nblk; b += 128) {
            float v[8];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                v[2 * u] = partial[((size_t)(b + 32 * u) * 2) * C + c];
                v[2 * u + 1] = partial[((size_t)(b + 32 * u) * 2 + 1) * C + c];
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) { s += (double)v[2 * u]; q += (double)v[2 * u + 1]; }
        }
        for (; b < nblk; b += 32) { s += (double)partial[((size_t)b * 2) * C + c]; q += (double)partial[((size_t)b * 2 + 1) * C + c]; }
    }
    sh[0][slice][lane] = s; sh[1][slice][lane] = q;
    __syncthreads();
    if (slice != 0 || c >= C) return false;
#pragma unroll
    for (int k = 1; k < 32; ++k) { s += sh[0][k][lane]; q += sh[1][k][lane]; }
    return true;
}

// per channel, from the totals (s, q) = (sum x, sum x^2) over `count` rows
__device__ __forceinline__ void bn_finalize2_channel(int c, double s, double q, long long count, const float* __restrict__ gamma,
                                                     const float* __restrict__ beta, float eps, float* __restrict__ mean, float* __restrict__ rstd,
                                                     float* __restrict__ scale, float* __restrict__ shift, float* __restrict__ run_mean,
                                                     float* __restrict__ run_var, long long* __restrict__ nbt, float momentum) {
    const double m = s / (double)count;
    double var = q / (double)count - m * m;
    if (var < 0.0) var = 0.0;
    const float r = (float)(1.0 / sqrt(var + (double)eps));
    mean[c] = (float)m; rstd[c] = r;
    const float sc = gamma[c] * r;
    scale[c] = sc; shift[c] = beta[c] - (float)m * sc;
    if (run_mean) {
        run_mean[c] = (1.f - momentum) * run_mean[c] + momentum * (float)m;
        const double unb = count > 1 ? var * (double)count / (double)(count - 1) : var;
        run_var[c] = (1.f - momentum) * run_var[c] + momentum * (float)unb;
        if (nbt && c == 0) *nbt += 1;
    }
}

__global__ void __launch_bounds__(1024) bn_finalize2_kernel(const float* __restrict__ partial, int nblk, long long count, int C,
                                                           const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                                                           float* __restrict__ mean, float* __restrict__ rstd, float* __restrict__ scale,
                                                           float* __restrict__ shift, float* __restrict__ run_mean, float* __restrict__ run_var,
                                                           long long* __restrict__ nbt, float momentum, float* __restrict__ sums_out) {
    PDL_SYNC();
    int c;
    double s, q;
    partial += (size_t)blockIdx.y * nblk * 2 * C;                     // statistics group
    const int go = blockIdx.y * C;
    mean += go; rstd += go; scale += go; shift += go;
    if (!partial_sums(partial, nblk, C, c, s, q)) return;
    if (sums_out) { sums_out[c] = (float)s; return; }          // plain column sums (bias gradients)
    bn_finalize2_channel(c, s, q, count, gamma, beta, eps, mean, rstd, scale, shift, run_mean, run_var, nbt, momentum);
}

// shared-model mode (SyncBatchNorm): the same statistics over the batches of ALL ranks -- the rank's (sum x, sum x^2) per channel are
// exchanged through peer memory (peer_comm.cuh) and added in rank order, count = local rows x world.  Every thread of every block reaches
// the exchange, so the early exit of the non-owner threads comes after it.  One statistics group (gridDim.y == 1).
__global__ void __launch_bounds__(1024) bn_finalize2_sync_kernel(const float* __restrict__ partial, int nblk, long long count, int C,
                                                                const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                                                                float* __restrict__ mean, float* __restrict__ rstd, float* __restrict__ scale,
                                                                float* __restrict__ shift, float* __restrict__ run_mean, float* __restrict__ run_var,
                                                                long long* __restrict__ nbt, float momentum, const PeerComm comm, int xid) {
    PDL_SYNC();
    int c;
    double s, q;
    const bool owner = partial_sums(partial, nblk, C, c, s, q);
    bn_sums_all_ranks(comm, xid, C, owner, c, s, q);
    if (!owner) return;
    bn_finalize2_channel(c, s, q, count * comm.world, gamma, beta, eps, mean, rstd, scale, shift, run_mean, run_var, nbt, momentum);
}

__device__ __forceinline__ void bn_bwd_finalize2_channel(int c, double sg, double sgx, long long count, const float* __restrict__ gamma,
                                                         const float* __restrict__ rstd, float* __restrict__ k0, float* __restrict__ k1,
                                                         float* __restrict__ k2) {
    const float a = gamma[c] * rstd[c];
    k0[c] = a; k1[c] = (float)((double)a * sg / (double)count); k2[c] = (float)((double)a * sgx / (double)count);
}

__global__ void __launch_bounds__(1024) bn_bwd_finalize2_kernel(const float* __restrict__ partial, int nblk, long long count, int C,
                                                               const float* __restrict__ gamma, const float* __restrict__ rstd,
                                                               float* __restrict__ dgamma, float* __restrict__ dbeta, float* __restrict__ k0,
                                                               float* __restrict__ k1, float* __restrict__ k2) {
    PDL_SYNC();
    int c;
    double sg, sgx;
    if (!partial_sums(partial, nblk, C, c, sg, sgx)) return;
    if (dgamma) dgamma[c] = (float)sgx;
    if (dbeta) dbeta[c] = (float)sg;
    bn_bwd_finalize2_channel(c, sg, sgx, count, gamma, rstd, k0, k1, k2);
}

// shared-model mode: d gamma / d beta stay the LOCAL sums (the gradient all-reduce averages them, as DDP does -- the global sums would
// scale them by the world size); the data gradient uses the means over the global batch (torch SyncBatchNorm backward all-reduces
// sum_dy / sum_dy_xmu only).  Every thread of every block reaches the exchange.
__global__ void __launch_bounds__(1024) bn_bwd_finalize2_sync_kernel(const float* __restrict__ partial, int nblk, long long count, int C,
                                                                    const float* __restrict__ gamma, const float* __restrict__ rstd,
                                                                    float* __restrict__ dgamma, float* __restrict__ dbeta, float* __restrict__ k0,
                                                                    float* __restrict__ k1, float* __restrict__ k2, const PeerComm comm, int xid) {
    PDL_SYNC();
    int c;
    double sg, sgx;
    const bool owner = partial_sums(partial, nblk, C, c, sg, sgx);
    if (owner) {
        if (dgamma) dgamma[c] = (float)sgx;
        if (dbeta) dbeta[c] = (float)sg;
    }
    bn_sums_all_ranks(comm, xid, C, owner, c, sg, sgx);
    if (!owner) return;
    bn_bwd_finalize2_channel(c, sg, sgx, count * comm.world, gamma, rstd, k0, k1, k2);
}

// ---- elementwise -----------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) bn_act_kernel(const bf16* __restrict__ x, const float* __restrict__ scale, const float* __restrict__ shift,
                                                     const bf16* __restrict__ res, long long ldr, const float* __restrict__ rscale,
                                                     const float* __restrict__ rshift, bf16* __restrict__ y, long long P, int C, int act,
                                                     long long rows_per_group) {
    PDL_SYNC();
    // rows_per_group > 0: row p uses the scale / shift vectors of group p / rows_per_group (merged real | zero-image batch)
    // two 16-byte elements per thread, `half` apart, loads first (more bytes in flight per thread)
    const int c8n = C >> 3;
    const long long total = P * c8n, half = (total + 1) >> 1;
    const long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i0 >= half) return;
    long long idx[2] = {i0, i0 + half};
    uint4 rx[2], rr[2];
    long long pp[2]; int cc[2]; bool ok[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
        ok[u] = idx[u] < total;
        pp[u] = ok[u] ? idx[u] / c8n : 0;
        cc[u] = ok[u] ? (int)(idx[u] - pp[u] * c8n) * 8 : 0;
        rx[u] = __ldg(reinterpret_cast<const uint4*>(x + pp[u] * C + cc[u]));
        if (res) rr[u] = __ldg(reinterpret_cast<const uint4*>(res + pp[u] * ldr + cc[u]));
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
        if (!ok[u]) continue;
        const int c0 = cc[u];
        const int gofs = rows_per_group > 0 ? (int)(pp[u] / rows_per_group) * C : 0;
        float v[8], sc[8], sh[8];
        unpack8(rx[u], v);
        load8f(scale + gofs + c0, sc); load8f(shift + gofs + c0, sh);
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = fmaf(v[j], sc[j], sh[j]);
        if (res) {
            float r[8];
            unpack8(rr[u], r);
            if (rscale) {
                load8f(rscale + gofs + c0, sc); load8f(rshift + gofs + c0, sh);
#pragma unroll
                for (int j = 0; j < 8; ++j) r[j] = fmaf(r[j], sc[j], sh[j]);
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] += r[j];
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = act_fwd(v[j], act);
        store8(y + pp[u] * C + c0, v);
    }
}

// dx = k0*g - k1 - xhat*k2 (bf16); optionally gskip = g (the gradient that flows on through the residual connection)
__global__ void __launch_bounds__(256) bn_bwd_apply2_kernel(const bf16* __restrict__ dyA, long long ldA, const bf16* __restrict__ dyB, long long ldB,
                                                            const bf16* __restrict__ y, int act, const bf16* __restrict__ x,
                                                            const float* __restrict__ mean, const float* __restrict__ rstd,
                                                            const float* __restrict__ k0, const float* __restrict__ k1, const float* __restrict__ k2,
                                                            bf16* __restrict__ dx, bf16* __restrict__ gskip, long long P, int C) {
    PDL_SYNC();
    const int c8n = C >> 3;
    const long long total = P * c8n, half = (total + 1) >> 1;
    const long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i0 >= half) return;
    long long idx[2] = {i0, i0 + half};
    uint4 ra[2], rb[2], ry[2], rx[2];
    long long pp[2]; int cc[2]; bool ok[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
        ok[u] = idx[u] < total;
        pp[u] = ok[u] ? idx[u] / c8n : 0;
        cc[u] = ok[u] ? (int)(idx[u] - pp[u] * c8n) * 8 : 0;
        ra[u] = __ldg(reinterpret_cast<const uint4*>(dyA + pp[u] * ldA + cc[u]));
        if (dyB) rb[u] = __ldg(reinterpret_cast<const uint4*>(dyB + pp[u] * ldB + cc[u]));
        if (act) ry[u] = __ldg(reinterpret_cast<const uint4*>(y + pp[u] * C + cc[u]));
        if (dx) rx[u] = __ldg(reinterpret_cast<const uint4*>(x + pp[u] * C + cc[u]));
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
        if (!ok[u]) continue;
        const long long p = pp[u];
        const int c0 = cc[u];
        float g[8];
        unpack8(ra[u], g);
        if (dyB) {
            float b[8];
            unpack8(rb[u], b);
#pragma unroll
            for (int j = 0; j < 8; ++j) g[j] += b[j];
        }
        if (act) {
            float yv[8];
            unpack8(ry[u], yv);
#pragma unroll
            for (int j = 0; j < 8; ++j) g[j] *= act_der(yv[j], act);
        }
        if (gskip) store8(gskip + p * C + c0, g);
        if (dx) {
            float xv[8], mu[8], rs[8], a0[8], a1[8], a2[8], o[8];
            unpack8(rx[u], xv);
            load8f(mean + c0, mu); load8f(rstd + c0, rs); load8f(k0 + c0, a0); load8f(k1 + c0, a1); load8f(k2 + c0, a2);
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = a0[j] * g[j] - a1[j] - (xv[j] - mu[j]) * rs[j] * a2[j];
            store8(dx + p * C + c0, o);
        }
    }
}

// out = a + b (+ c), each with its own pixel stride
__global__ void __launch_bounds__(256) add3_kernel(const bf16* __restrict__ a, long long lda, const bf16* __restrict__ b, long long ldb,
                                                   const bf16* __restrict__ c, long long ldc, bf16* __restrict__ out, long long P, int C) {
    PDL_SYNC();
    const int c8n = C >> 3;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= P * c8n) return;
    const long long p = idx / c8n;
    const int c0 = (int)(idx - p * c8n) * 8;
    float v[8], t[8];
    load8(a + p * lda + c0, v);
    load8(b + p * ldb + c0, t);
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] += t[j];
    if (c) {
        load8(c + p * ldc + c0, t);
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] += t[j];
    }
    store8(out + p * C + c0, v);
}

// out = max(y, 0) (nlspnmodel_adapt.py:901);  backward: g_y = g_out * [y > 0]
__global__ void clamp0_kernel(const float* __restrict__ y, float* __restrict__ out, long long n) {
    PDL_SYNC();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = fmaxf(y[i], 0.f);
}
__global__ void clamp_range_kernel(const float* __restrict__ x, float* __restrict__ out, float lo, float hi, long long n) {
    PDL_SYNC();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = fminf(fmaxf(x[i], lo), hi);
}
__global__ void mask_pos_kernel(const float* __restrict__ g, const float* __restrict__ y, float* __restrict__ out, long long n) {
    PDL_SYNC();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = y[i] > 0.f ? g[i] : 0.f;
}

// gradients wrt the three thin heads' pre-activation outputs, as one NHWC bf16 [N,H,W,64] operand (channels >= 10 zero):
//   ch 0 = g_pred * LeakyReLU'(pred_init), ch 1..8 = g_guide, ch 9 = g_conf * conf*(1-conf)
__global__ void __launch_bounds__(256) thin_grad_pack_kernel(const float* __restrict__ g_pred, const float* __restrict__ pred_init,
                                                             const float* __restrict__ g_guide, const float* __restrict__ g_conf,
                                                             const float* __restrict__ conf, bf16* __restrict__ out, int N, long long HW) {
    PDL_SYNC();
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= N * HW) return;
    const long long n = idx / HW, o = idx - n * HW;
    float f[16];
    f[0] = g_pred[idx] * (pred_init[idx] > 0.f ? 1.f : 0.2f);
#pragma unroll
    for (int k = 0; k < 8; ++k) f[1 + k] = g_guide[(n * 8 + k) * HW + o];
    const float cf = conf[idx];
    f[9] = g_conf[idx] * cf * (1.f - cf);
#pragma unroll
    for (int k = 10; k < 16; ++k) f[k] = 0.f;
    bf16* dst = out + idx * 64;
    float lo[8], hi[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { lo[j] = f[j]; hi[j] = f[8 + j]; }
    store8(dst, lo); store8(dst + 8, hi);
    const uint4 z = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
    for (int q = 2; q < 8; ++q) *reinterpret_cast<uint4*>(dst + q * 8) = z;
}

// ---- prop_layer.conv_offset_aff: Conv2d(8, 24, 3, 1, 1) in fp32 on planar maps -------------------------------------------------------
// forward: in [N,8,H,W] -> out [N,24,H,W];  TRANSPOSED: in = g_out [N,24,H,W] -> out = g_in [N,8,H,W] (data gradient)
template <bool TRANSPOSED>
__global__ void __launch_bounds__(128) conv8to24_kernel(const float* __restrict__ in, const float* __restrict__ w, const float* __restrict__ bias,
                                                        float* __restrict__ out, int N, int H, int W) {
    PDL_SYNC();
    constexpr int CI = TRANSPOSED ? 24 : 8, CO = TRANSPOSED ? 8 : 24;
    __shared__ float s_w[9 * CI * CO];          // [tap][ci][co]
    for (int i = threadIdx.x; i < 9 * CI * CO; i += blockDim.x) {
        const int co = i % CO, ci = (i / CO) % CI, tap = i / (CO * CI);
        // weight tensor is [24][8][3][3]; the data gradient reads it transposed with flipped taps
        s_w[i] = TRANSPOSED ? w[(ci * 8 + co) * 9 + (8 - tap)] : w[(co * 8 + ci) * 9 + tap];
    }
    __syncthreads();
    const long long HW = (long long)H * W;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= N * HW) return;
    const int x = idx % W, y = (idx / W) % H, n = idx / HW;
    float acc[CO];
#pragma unroll
    for (int c = 0; c < CO; ++c) acc[c] = (!TRANSPOSED && bias) ? bias[c] : 0.f;
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
        const int gy = y + ky - 1;
        if (gy < 0 || gy >= H) continue;
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
            const int gx = x + kx - 1;
            if (gx < 0 || gx >= W) continue;
            const float* src = in + (long long)n * CI * HW + (long long)gy * W + gx;
            const float* wr = s_w + (ky * 3 + kx) * CI * CO;
#pragma unroll
            for (int ci = 0; ci < CI; ++ci) {
                const float v = __ldg(src + ci * HW);
#pragma unroll
                for (int c = 0; c < CO; ++c) acc[c] = fmaf(v, wr[ci * CO + c], acc[c]);
            }
        }
    }
#pragma unroll
    for (int c = 0; c < CO; ++c) out[((long long)n * CO + c) * HW + (long long)y * W + x] = acc[c];
}

// ---- weight gradient of the 48->48 meta conv -----------------------------------------------------------------------------------------
// dW[co][ci][ky][kx] = sum_p g[p][co] * X[p + (ky-1, kx-1)][ci] over NHWC bf16 maps with 64 stored channels (48 used).
// Persistent CTAs of 9 warps: warp t owns tap t and keeps its 48x48 fp32 block in registers (3 m16 x 6 n8 mma tiles) while
// the CTA walks over 16x16 pixel tiles (halo 18x18x64 + gradient tile 256x64 staged in swizzled shared memory; both operands
// read with ldmatrix.trans: pixels are the K dimension).  Partials [cta][9][48][48] are summed in a fixed order.
struct Wgrad48Cfg {
    static const int HALO_BYTES = 18 * 18 * 128;     // 41472
    static const int G_BYTES = 256 * 128;            // 32768
    static const int STAGE = HALO_BYTES + G_BYTES;   // one tile's operands
    static const int SMEM = 2 * STAGE;               // double buffered: tile t+1 is fetched with cp.async while tile t is multiplied
    static const int THREADS = 288;
};
__device__ __forceinline__ int swz128(int row, int chunk) { return row * 128 + ((chunk ^ (row & 7)) << 4); }

// cp.async (zero-fill outside the image) of one tile's halo (18x18 pixels of the conv input) and gradient tile (16x16 pixels)
__device__ __forceinline__ void wgrad48_fetch(unsigned char* stage, const bf16* __restrict__ xin, const bf16* __restrict__ gout, int tile, int tiles_x,
                                              int tiles_y, int H, int W, int tid) {
    const int n = tile / (tiles_y * tiles_x), r = tile - n * tiles_y * tiles_x;
    const int y0 = (r / tiles_x) * 16, x0 = (r % tiles_x) * 16;
    const uint32_t hs = smem_u32(stage), gs = hs + Wgrad48Cfg::HALO_BYTES;
    const bf16* in_n = xin + (size_t)n * H * W * 64;
    for (int i = tid; i < 18 * 18 * 8; i += Wgrad48Cfg::THREADS) {
        const int pix = i >> 3, c = i & 7;
        const int hy = pix / 18, hx = pix - hy * 18;
        const int gy = y0 - 1 + hy, gx = x0 - 1 + hx;
        const bool ok = gy >= 0 && gy < H && gx >= 0 && gx < W;
        cp_async16(hs + swz128(pix, c), ok ? in_n + ((size_t)gy * W + gx) * 64 + c * 8 : in_n, ok);
    }
    const bf16* g_n = gout + (size_t)n * H * W * 64;
    for (int i = tid; i < 256 * 8; i += Wgrad48Cfg::THREADS) {
        const int pix = i >> 3, c = i & 7;
        const int gy = y0 + (pix >> 4), gx = x0 + (pix & 15);
        const bool ok = gy < H && gx < W;
        cp_async16(gs + swz128(pix, c), ok ? g_n + ((size_t)gy * W + gx) * 64 + c * 8 : g_n, ok);
    }
    cp_async_commit();
}

__global__ void __launch_bounds__(Wgrad48Cfg::THREADS, 1) wgrad48_kernel(const bf16* __restrict__ xin, const bf16* __restrict__ gout,
                                                                        float* __restrict__ partial, int N, int H, int W) {
    PDL_SYNC();
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tiles_x = (W + 15) / 16, tiles_y = (H + 15) / 16;
    const int total = N * tiles_y * tiles_x;
    const int ky = warp / 3, kx = warp - ky * 3;
    const int a_k = (lane & 7) + (lane >> 4) * 8, a_mc = (lane >> 3) & 1;
    const int b_k = (lane & 7) + ((lane >> 3) & 1) * 8, b_nc = lane >> 4;
    float acc[3][6][4];
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = 0; b < 6; ++b)
#pragma unroll
            for (int c = 0; c < 4; ++c) acc[a][b][c] = 0.f;
    int buf = 0;
    if ((int)blockIdx.x < total) wgrad48_fetch(smem, xin, gout, blockIdx.x, tiles_x, tiles_y, H, W, tid);
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x, buf ^= 1) {
        const int next = tile + gridDim.x;
        if (next < total) {
            wgrad48_fetch(smem + (buf ^ 1) * Wgrad48Cfg::STAGE, xin, gout, next, tiles_x, tiles_y, H, W, tid);
            cp_async_wait<1>();                       // this tile's group has landed, the next one may still be in flight
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();
        const uint32_t hb = smem_u32(smem + buf * Wgrad48Cfg::STAGE), gb = hb + Wgrad48Cfg::HALO_BYTES;
#pragma unroll 2
        for (int ks = 0; ks < 16; ++ks) {             // one tile row of 16 pixels per k16 step
            uint32_t a[3][4], b[12];
#pragma unroll
            for (int mt = 0; mt < 3; ++mt) ldmatrix_x4_trans(a[mt][0], a[mt][1], a[mt][2], a[mt][3], gb + swz128(ks * 16 + a_k, mt * 2 + a_mc));
            const int prow = (ks + ky) * 18 + (b_k + kx);
#pragma unroll
            for (int h = 0; h < 3; ++h) ldmatrix_x4_trans(b[h * 4], b[h * 4 + 1], b[h * 4 + 2], b[h * 4 + 3], hb + swz128(prow, h * 2 + b_nc));
#pragma unroll
            for (int mt = 0; mt < 3; ++mt)
#pragma unroll
                for (int nt = 0; nt < 6; ++nt) mma_bf16_16816(acc[mt][nt], a[mt], b[nt * 2], b[nt * 2 + 1]);
        }
        __syncthreads();                              // everyone is done with this buffer before the fetch after next overwrites it
    }
    const int c_row = lane >> 2, c_col = (lane & 3) * 2;
    float* part = partial + ((size_t)blockIdx.x * 9 + warp) * 48 * 48;
#pragma unroll
    for (int mt = 0; mt < 3; ++mt)
#pragma unroll
        for (int half = 0; half < 2; ++half)
#pragma unroll
            for (int nt = 0; nt < 6; ++nt) {
                const int co = mt * 16 + c_row + half * 8, ci = nt * 8 + c_col;
                *reinterpret_cast<float2*>(part + co * 48 + ci) = make_float2(acc[mt][nt][half * 2], acc[mt][nt][half * 2 + 1]);
            }
}

// dw[co][ci][tap] (Conv2d layout [48][48][3][3]) = sum over CTAs of partial[cta][tap][co][ci]
__global__ void __launch_bounds__(256) wgrad48_reduce_kernel(const float* __restrict__ partial, float* __restrict__ dw, int nblocks) {
    PDL_SYNC();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 9 * 48 * 48) return;
    float s = 0.f;
    for (int b = 0; b < nblocks; ++b) s += partial[(size_t)b * 9 * 48 * 48 + i];
    const int tap = i / (48 * 48), rem = i - tap * 48 * 48, co = rem / 48, ci = rem - co * 48;
    dw[(co * 48 + ci) * 9 + tap] = s;
}

// ---- evaluation metrics on the device (src/eval_utils.py:117-175 as used by src/tta_main.py:760-798) ------------------------------
// mask = gt > 0 and min <= gt <= max; MAE / RMSE on 1000*depth (mm), iMAE / iRMSE on 1 / (0.001*depth + 1e-9) (1/km)
// partial[blk][5] (double): sum |d|, sum d^2, sum |id|, sum id^2, count
__global__ void __launch_bounds__(256) eval_metrics_kernel(const float* __restrict__ out, const float* __restrict__ gt, long long n, float min_d,
                                                           float max_d, double* __restrict__ partial) {
    PDL_SYNC();
    __shared__ double sh[32];
    double a = 0.0, b = 0.0, c = 0.0, d = 0.0, cnt = 0.0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float g = gt[i], o = out[i];
        if (g > 0.f && !(g < min_d) && !(g > max_d)) {
            const float e = 1000.f * g - 1000.f * o;
            const float ie = 1.f / (0.001f * g + 1e-9f) - 1.f / (0.001f * o + 1e-9f);
            a += (double)fabsf(e); b += (double)(e * e); c += (double)fabsf(ie); d += (double)(ie * ie); cnt += 1.0;
        }
    }
    const double r0 = block_sum_d(a, sh), r1 = block_sum_d(b, sh), r2 = block_sum_d(c, sh), r3 = block_sum_d(d, sh), r4 = block_sum_d(cnt, sh);
    if (threadIdx.x == 0) {
        double* o5 = partial + (size_t)blockIdx.x * 5;
        o5[0] = r0; o5[1] = r1; o5[2] = r2; o5[3] = r3; o5[4] = r4;
    }
}
// result[5] (float): mae, rmse, imae, irmse, number of evaluated pixels
__global__ void __launch_bounds__(256) eval_metrics_finalize_kernel(const double* __restrict__ partial, int nblk, float* __restrict__ result) {
    PDL_SYNC();
    __shared__ double sh[32];
    double v[5] = {0, 0, 0, 0, 0};
    for (int b = threadIdx.x; b < nblk; b += blockDim.x)
        for (int k = 0; k < 5; ++k) v[k] += partial[(size_t)b * 5 + k];
    double t[5];
    for (int k = 0; k < 5; ++k) t[k] = block_sum_d(v[k], sh);
    if (threadIdx.x == 0) {
        const double c = t[4];
        result[0] = (float)(t[0] / c); result[1] = (float)sqrt(t[1] / c); result[2] = (float)(t[2] / c); result[3] = (float)sqrt(t[3] / c);
        result[4] = (float)c;
    }
}

// ---- input stage (src/data_utils.py:134-200 load_image / load_depth_with_validity_map + the crop of src/datasets.py:83-170) -------
// decoded 8-bit RGB (HWC) and 16-bit depth PNG payloads -> fp32 NCHW image in [0, 255], depth = png / multiplier (<= 0 -> 0) and the
// binary validity map, cropped to (h, w) at (y0, x0): the frames cross PCIe in their native compact types (3.2x fewer bytes)
__global__ void __launch_bounds__(256) input_stage_kernel(const unsigned char* __restrict__ img, const unsigned short* __restrict__ dep,
                                                          float* __restrict__ image, float* __restrict__ depth, float* __restrict__ validity,
                                                          int N, int H0, int W0, int y0, int x0, int h, int w, float multiplier) {
    PDL_SYNC();
    const long long hw = (long long)h * w;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= N * hw) return;
    const int n = (int)(idx / hw);
    const long long o = idx - n * hw;
    const int y = (int)(o / w), x = (int)(o - (long long)y * w);
    const long long src = ((long long)n * H0 + (y0 + y)) * W0 + (x0 + x);
#pragma unroll
    for (int c = 0; c < 3; ++c) image[((long long)n * 3 + c) * hw + o] = (float)img[src * 3 + c];
    float z = (float)dep[src] / multiplier;
    if (z <= 0.f) z = 0.f;
    depth[idx] = z;
    validity[idx] = z > 0.f ? 1.f : z;
}

}  // namespace ptta
