// Memory-bound kernels of the ProxyTTA step: pre-processing, pyramid, 1<->32 channel stems, bilinear
// x2 (and its adjoint), BatchNorm pieces, losses, Adam.  All fp32 arithmetic; 32-channel maps are
// NHWC bf16, single-channel maps fp32 [N,H,W].
#pragma once
#include "common.cuh"
#include "peer_comm.cuh"
#include <math_constants.h>

namespace ptta {

// -------------------------------------------------------------------------------------------------
// a1 + a2: validity map (src/tta_main.py:583-586) and OutlierRemoval(7, 1.5)
// (src/net_utils.py:766-811).  Invalid / out-of-image samples are +inf in the 7x7 min window, which
// gives bit-identical results to the reference's 10*max(d) fill without its global reduction.
// -------------------------------------------------------------------------------------------------
#define OR_TX 32
#define OR_TY 8
__global__ void __launch_bounds__(OR_TX * OR_TY) outlier_removal_kernel(const float* __restrict__ d, float* __restrict__ d_out,
                                                                        float* __restrict__ v_out, int H, int W, int ksize, float thr) {
    PDL_SYNC();
    extern __shared__ float s_or[];
    const int pad = ksize / 2;
    const int SW = OR_TX + 2 * pad, SH = OR_TY + 2 * pad;
    const int n = blockIdx.z;
    const int x0 = blockIdx.x * OR_TX, y0 = blockIdx.y * OR_TY;
    const float* dn = d + (size_t)n * H * W;
    const int tid = threadIdx.y * OR_TX + threadIdx.x;
    for (int i = tid; i < SW * SH; i += OR_TX * OR_TY) {
        int sy = i / SW, sx = i - sy * SW;
        int gy = y0 - pad + sy, gx = x0 - pad + sx;
        float f = CUDART_INF_F;
        if (gy >= 0 && gy < H && gx >= 0 && gx < W) {
            float val = dn[(size_t)gy * W + gx];
            float vm = val > 0.f ? 1.f : val;          // validity map
            f = vm <= 0.f ? CUDART_INF_F : val;
        }
        s_or[i] = f;
    }
    __syncthreads();
    int x = x0 + threadIdx.x, y = y0 + threadIdx.y;
    if (x >= W || y >= H) return;
    float val = dn[(size_t)y * W + x];
    float vm = val > 0.f ? 1.f : val;
    float keep = 1.f;
    if (vm != 0.f) {
        float m = CUDART_INF_F;
        for (int j = 0; j < ksize; ++j)
            for (int i = 0; i < ksize; ++i) m = fminf(m, s_or[(threadIdx.y + j) * SW + threadIdx.x + i]);
        keep = (m < val - thr) ? 0.f : 1.f;
    }
    float vo = vm * keep;
    size_t o = (size_t)n * H * W + (size_t)y * W + x;
    v_out[o] = vo;
    d_out[o] = val * vo;
}

// -------------------------------------------------------------------------------------------------
// a3 + a6: clamp(d, 0, cap) (src/external_model_adapt.py:103-108) and the validity-normalised
// average-pool pyramid (network_exp_msg_chn_adapt.py:479,487,492).  One thread per /4 cell.
// -------------------------------------------------------------------------------------------------
__global__ void pyramid_kernel(const float* __restrict__ d, float* __restrict__ dc, float* __restrict__ d2, float* __restrict__ d4,
                               int N, int H, int W, float cap, int do_clamp) {
    PDL_SYNC();
    int H4 = H / 4, W4 = W / 4;
    long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)N * H4 * W4) return;
    int x4 = idx % W4;
    int y4 = (idx / W4) % H4;
    int n = idx / ((long long)W4 * H4);
    const float* dn = d + (size_t)n * H * W;
    float* dcn = dc + (size_t)n * H * W;
    float v[4][4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        float4 r = *reinterpret_cast<const float4*>(dn + (size_t)(y4 * 4 + j) * W + x4 * 4);
        if (do_clamp) {
            r.x = fminf(fmaxf(r.x, 0.f), cap); r.y = fminf(fmaxf(r.y, 0.f), cap);
            r.z = fminf(fmaxf(r.z, 0.f), cap); r.w = fminf(fmaxf(r.w, 0.f), cap);
        }
        *reinterpret_cast<float4*>(dcn + (size_t)(y4 * 4 + j) * W + x4 * 4) = r;
        v[j][0] = r.x; v[j][1] = r.y; v[j][2] = r.z; v[j][3] = r.w;
    }
    float s4 = 0.f, c4 = 0.f;
    int H2 = H / 2, W2 = W / 2;
#pragma unroll
    for (int by = 0; by < 2; ++by)
#pragma unroll
        for (int bx = 0; bx < 2; ++bx) {
            float s = 0.f, c = 0.f;
#pragma unroll
            for (int j = 0; j < 2; ++j)
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    float t = v[by * 2 + j][bx * 2 + i];
                    s += t;
                    c += t > 0.f ? 1.f : 0.f;
                }
            s4 += s; c4 += c;
            d2[(size_t)n * H2 * W2 + (size_t)(y4 * 2 + by) * W2 + x4 * 2 + bx] = (s * 0.25f) / (c * 0.25f + 0.0001f);
        }
    d4[(size_t)n * H4 * W4 + (size_t)y4 * W4 + x4] = (s4 * 0.0625f) / (c4 * 0.0625f + 0.0001f);
}

// -------------------------------------------------------------------------------------------------
// a4: pad-to-/16 + flip-pad ensembling of MsgChnModel_Adapt.forward (src/msg_chn_model_adapt.py:54-197).  An N x C x Hu x Wu
// input becomes a 2N x C x H x W batch: copy 0 padded at the top / right, copy 1 padded at the bottom / left; the two
// predictions are cropped back and averaged.  pad_pair(scale = 0.5, fill = 0) is also the exact adjoint of unpad_mean.
// -------------------------------------------------------------------------------------------------
__global__ void pad_pair_kernel(const float* __restrict__ src, float* __restrict__ dst, int Nu, int C, int Hu, int Wu, int H, int W, float scale,
                                float f0, float f1, float f2) {
    PDL_SYNC();
    const long long total = 2LL * Nu * C * H * W;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int x = idx % W, y = (idx / W) % H, c = (idx / ((long long)W * H)) % C, n2 = idx / ((long long)W * H * C);
    const int copy = n2 / Nu, n = n2 - copy * Nu;
    const int pt = H - Hu, pr = W - Wu;
    const int sy = copy == 0 ? y - pt : y, sx = copy == 0 ? x : x - pr;
    float v = c == 0 ? f0 : (c == 1 ? f1 : f2);
    if (sy >= 0 && sy < Hu && sx >= 0 && sx < Wu) v = scale * __ldg(src + (((long long)n * C + c) * Hu + sy) * Wu + sx);
    dst[idx] = v;
}
__global__ void unpad_mean_kernel(const float* __restrict__ src, float* __restrict__ dst, int Nu, int Hu, int Wu, int H, int W) {
    PDL_SYNC();
    const long long total = (long long)Nu * Hu * Wu;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int x = idx % Wu, y = (idx / Wu) % Hu, n = idx / ((long long)Wu * Hu);
    const int pt = H - Hu, pr = W - Wu;
    const float a = __ldg(src + ((long long)n * H + (y + pt)) * W + x);
    const float b = __ldg(src + ((long long)(Nu + n) * H + y) * W + (x + pr));
    dst[idx] = 0.5f * (a + b);      // torch.mean over the stacked pair (msg_chn_model_adapt.py:116-121)
}

// -------------------------------------------------------------------------------------------------
// Stem: {1,2,3} fp32 planes -> 32 channels bf16 NHWC, 3x3 s1 p1 (init.0 of every encoder,
// network_exp_msg_chn_adapt.py:172,220).  Each plane has its own pointer / batch stride and an
// affine (x*scale + shift) so that image normalisation (src/transforms.py:669-712) and the
// cat((d, up2(pred))) of the cascade (network_exp_msg_chn_adapt.py:494,501) need no extra pass.
// With CIN=1, pre-flipped weights and a ReLU mask it is also the data-gradient of the 32->1
// prediction conv.
// -------------------------------------------------------------------------------------------------
struct StemParams {
    const float* plane[3];
    long long batch_stride[3];
    float scale[3], shift[3];
    const float* w;      // [32][CIN][3][3]
    const float* bias;   // [32] or null
    const bf16* mask;    // relu mask (NHWC 32) or null
    bf16* out;
    int N, H, W;
    int relu_out;        // store ReLU(result): every consumer of an init.0 output applies ReLU first
};

template <int CIN>
__global__ void __launch_bounds__(128) stem_conv_kernel(const StemParams p) {
    PDL_SYNC();
    __shared__ float s_w[CIN * 9 * 32];   // [ci][tap][co]
    __shared__ float s_b[32];
    __shared__ __align__(16) unsigned char s_stage[4][2048];   // per warp: 32 pixels x 64 B (mask in, result out)
    for (int i = threadIdx.x; i < CIN * 9 * 32; i += blockDim.x) {
        int co = i & 31, r = i >> 5;       // r = ci*9 + tap
        s_w[i] = p.w[(size_t)co * CIN * 9 + r];
    }
    if (threadIdx.x < 32) s_b[threadIdx.x] = p.bias ? p.bias[threadIdx.x] : 0.f;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long total = (long long)p.N * p.H * p.W;
    const long long idx0 = (long long)blockIdx.x * blockDim.x + warp * 32;   // first pixel of this warp (pixels are contiguous in NHWC)
    if (idx0 >= total) return;
    const int nvalid = (int)min((long long)32, total - idx0);
    const long long idx = idx0 + lane;
    const bool valid = lane < nvalid;
    unsigned char* stage = s_stage[warp];
    const int swz = (lane >> 1) & 3;
    // each warp instruction moves 512 contiguous bytes; lane l then owns pixel l's 64 B (16 B chunks XOR-swizzled: conflict-free)
    if (p.mask) {
        const uint4* src = reinterpret_cast<const uint4*>(p.mask + (size_t)idx0 * 32);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int i = k * 32 + lane, px = i >> 2, c = i & 3;
            if (px < nvalid) *reinterpret_cast<uint4*>(stage + px * 64 + ((c ^ ((px >> 1) & 3)) << 4)) = __ldg(src + i);
        }
        __syncwarp();
    }
    float acc[32];
#pragma unroll
    for (int c = 0; c < 32; ++c) acc[c] = s_b[c];
    if (valid) {
        const int x = idx % p.W;
        const int y = (idx / p.W) % p.H;
        const int n = idx / ((long long)p.W * p.H);
#pragma unroll
        for (int ci = 0; ci < CIN; ++ci) {
            const float* pl = p.plane[ci] + (size_t)n * p.batch_stride[ci];
#pragma unroll
            for (int ky = 0; ky < 3; ++ky) {
                int gy = y + ky - 1;
                if (gy < 0 || gy >= p.H) continue;
#pragma unroll
                for (int kx = 0; kx < 3; ++kx) {
                    int gx = x + kx - 1;
                    if (gx < 0 || gx >= p.W) continue;
                    float v = __ldg(pl + (size_t)gy * p.W + gx) * p.scale[ci] + p.shift[ci];
                    const float* wr = s_w + (ci * 9 + ky * 3 + kx) * 32;
#pragma unroll
                    for (int c = 0; c < 32; ++c) acc[c] = fmaf(v, wr[c], acc[c]);
                }
            }
        }
        if (p.mask) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                uint4 mv = *reinterpret_cast<const uint4*>(stage + lane * 64 + ((q ^ swz) << 4));
                const uint32_t* mu = reinterpret_cast<const uint32_t*>(&mv);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float2 m = unpack_bf162(mu[j]);
                    if (!(m.x > 0.f)) acc[q * 8 + j * 2] = 0.f;
                    if (!(m.y > 0.f)) acc[q * 8 + j * 2 + 1] = 0.f;
                }
            }
        }
        if (p.relu_out) {
#pragma unroll
            for (int c = 0; c < 32; ++c) acc[c] = fmaxf(acc[c], 0.f);
        }
    }
    __syncwarp();                       // every lane is done with the staged mask
    if (valid) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            uint4 ov;
            ov.x = pack_bf162(acc[q * 8 + 0], acc[q * 8 + 1]);
            ov.y = pack_bf162(acc[q * 8 + 2], acc[q * 8 + 3]);
            ov.z = pack_bf162(acc[q * 8 + 4], acc[q * 8 + 5]);
            ov.w = pack_bf162(acc[q * 8 + 6], acc[q * 8 + 7]);
            *reinterpret_cast<uint4*>(stage + lane * 64 + ((q ^ swz) << 4)) = ov;
        }
    }
    __syncwarp();
    uint4* dst = reinterpret_cast<uint4*>(p.out + (size_t)idx0 * 32);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int i = k * 32 + lane, px = i >> 2, c = i & 3;
        if (px < nvalid) dst[i] = *reinterpret_cast<const uint4*>(stage + px * 64 + ((c ^ ((px >> 1) & 3)) << 4));
    }
}

// Same operator, PX (2 or 4) consecutive pixels of a row per thread (W % PX == 0): every weight read from shared memory (one 16 B
// broadcast load = 4 output channels) feeds 4*PX FMAs instead of 4, the 3 x (PX+2) input window is loaded once per plane, and the
// thread's PX x 64 B of bf16 output leave through a warp-private swizzled staging tile as 512 B coalesced stores.  The kernel is bound by
// the fp32 FMA pipe (864 FMA per pixel for the 3-plane image stem: 10 us at 352x1216 at 100 % issue rate); tensor cores are not an
// option here because the depth planes need fp32 inputs (metres with millimetre resolution: bf16 / tf32 would quantise a 40 m sample
// by 12 cm / 2 cm).  PX = 2 with 4 blocks per SM: 16 warps hide the shared-memory latency of the weight loads (ncu on the PX = 4, 2
// blocks per SM form: 36 % issue-slot utilisation, 2 warps per scheduler, 5.4 cycles per issued instruction).
template <int CIN, int PX>
__global__ void __launch_bounds__(128, PX == 2 ? 4 : 2) stem_convp_kernel(const StemParams p) {
    PDL_SYNC();
    constexpr int TB = PX * 64;                         // bytes of output per thread
    constexpr int NCH = PX * 4;                         // 16 B chunks per thread
    __shared__ __align__(16) float s_w[CIN * 9 * 32];   // [ci][tap][co]
    __shared__ float s_b[32];
    __shared__ __align__(16) unsigned char s_stage[4][32 * TB];   // per warp: 32 threads x TB
    for (int i = threadIdx.x; i < CIN * 9 * 32; i += blockDim.x) {
        int co = i & 31, r = i >> 5;       // r = ci*9 + tap
        s_w[i] = p.w[(size_t)co * CIN * 9 + r];
    }
    if (threadIdx.x < 32) s_b[threadIdx.x] = p.bias ? p.bias[threadIdx.x] : 0.f;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int wq = p.W / PX;
    const long long total = (long long)p.N * p.H * wq;                          // groups; group q covers NHWC pixels PX*q .. PX*q+PX-1
    const long long q0 = (long long)blockIdx.x * blockDim.x + warp * 32;
    if (q0 >= total) return;
    const int nvalid = (int)min((long long)32, total - q0);
    const long long q = q0 + lane;
    const bool valid = lane < nvalid;
    unsigned char* stage = s_stage[warp];
    float acc[PX][32];
#pragma unroll
    for (int px = 0; px < PX; ++px)
#pragma unroll
        for (int c = 0; c < 32; ++c) acc[px][c] = s_b[c];
    if (valid) {
        const int x = (int)(q % wq) * PX;
        const int y = (int)((q / wq) % p.H);
        const long long n = q / ((long long)wq * p.H);
#pragma unroll
        for (int ci = 0; ci < CIN; ++ci) {
            const float* pl = p.plane[ci] + n * p.batch_stride[ci];
            const float sc = p.scale[ci], sh = p.shift[ci];
#pragma unroll
            for (int ky = 0; ky < 3; ++ky) {
                const int gy = y + ky - 1;
                if (gy < 0 || gy >= p.H) continue;                               // zero padding of the (normalised) input
                const float* row = pl + (size_t)gy * p.W + x;
                float v[PX + 2];
                v[0] = x > 0 ? fmaf(__ldg(row - 1), sc, sh) : 0.f;
                if (PX == 4) {
                    const float4 c4 = __ldg(reinterpret_cast<const float4*>(row));
                    v[1] = fmaf(c4.x, sc, sh); v[2] = fmaf(c4.y, sc, sh); v[PX - 1] = fmaf(c4.z, sc, sh); v[PX] = fmaf(c4.w, sc, sh);
                } else {
                    const float2 c2 = __ldg(reinterpret_cast<const float2*>(row));
                    v[1] = fmaf(c2.x, sc, sh); v[2] = fmaf(c2.y, sc, sh);
                }
                v[PX + 1] = x + PX < p.W ? fmaf(__ldg(row + PX), sc, sh) : 0.f;
#pragma unroll
                for (int kx = 0; kx < 3; ++kx) {
                    const float4* wr = reinterpret_cast<const float4*>(s_w + (ci * 9 + ky * 3 + kx) * 32);
#pragma unroll
                    for (int c4i = 0; c4i < 8; ++c4i) {
                        const float4 w4 = wr[c4i];
#pragma unroll
                        for (int px = 0; px < PX; ++px) {
                            const float a = v[px + kx];
                            acc[px][c4i * 4 + 0] = fmaf(a, w4.x, acc[px][c4i * 4 + 0]);
                            acc[px][c4i * 4 + 1] = fmaf(a, w4.y, acc[px][c4i * 4 + 1]);
                            acc[px][c4i * 4 + 2] = fmaf(a, w4.z, acc[px][c4i * 4 + 2]);
                            acc[px][c4i * 4 + 3] = fmaf(a, w4.w, acc[px][c4i * 4 + 3]);
                        }
                    }
                }
            }
        }
        const uint4* mrow = p.mask ? reinterpret_cast<const uint4*>(p.mask + (size_t)q * (PX * 32)) : nullptr;    // PX pixels x 32 channels
#pragma unroll
        for (int px = 0; px < PX; ++px) {
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                float* a = &acc[px][g * 8];
                if (mrow) {
                    const uint4 mv = __ldg(mrow + px * 4 + g);
                    const uint32_t* mu = reinterpret_cast<const uint32_t*>(&mv);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float2 m = unpack_bf162(mu[j]);
                        if (!(m.x > 0.f)) a[j * 2] = 0.f;
                        if (!(m.y > 0.f)) a[j * 2 + 1] = 0.f;
                    }
                }
                if (p.relu_out) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) a[j] = fmaxf(a[j], 0.f);
                }
                uint4 ov;
                ov.x = pack_bf162(a[0], a[1]); ov.y = pack_bf162(a[2], a[3]);
                ov.z = pack_bf162(a[4], a[5]); ov.w = pack_bf162(a[6], a[7]);
                const int k = px * 4 + g;
                *reinterpret_cast<uint4*>(stage + lane * TB + ((k ^ (lane & (NCH - 1))) << 4)) = ov;
            }
        }
    }
    __syncwarp();
    uint4* dst = reinterpret_cast<uint4*>(p.out + (size_t)q0 * (PX * 32));
#pragma unroll
    for (int j = 0; j < NCH; ++j) {
        const int i = j * 32 + lane, r = i / NCH, c = i % NCH;
        if (r < nvalid) dst[i] = *reinterpret_cast<const uint4*>(stage + r * TB + ((c ^ (r & (NCH - 1))) << 4));
    }
}

// The engine's form: weights and bias travel BY VALUE in the kernel parameters (constant bank), so every FMA takes its weight as a
// constant operand and the inner loop is FMAs only -- no shared-memory weight loads (a 16 B broadcast load costs the shared pipe
// four wavefronts: with one per 8 / 16 FMAs that pipe, not the FMA pipe, set the speed of the kernels above), no staging barrier.
// The layers it serves are frozen ('meta' adapt mode), so the host copy taken at pack time stays valid; a re-pack re-captures the graph.
struct StemCParams {
    const float* plane[3];
    long long batch_stride[3];
    float scale[3], shift[3];
    const bf16* mask;    // relu mask (NHWC 32) or null
    bf16* out;
    int N, H, W;
    int relu_out;
    float bias[32];
    float w[3 * 9 * 32]; // [ci][tap][co]
};

template <int CIN, int PX>
__global__ void __launch_bounds__(128, 4) stem_convc_kernel(const __grid_constant__ StemCParams p) {
    PDL_SYNC();
    constexpr int TB = PX * 64, NCH = PX * 4;
    __shared__ __align__(16) unsigned char s_stage[4][32 * TB];   // per warp: 32 threads x TB
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int wq = p.W / PX;
    const long long total = (long long)p.N * p.H * wq;
    const long long q0 = (long long)blockIdx.x * blockDim.x + warp * 32;
    if (q0 >= total) return;
    const int nvalid = (int)min((long long)32, total - q0);
    const long long q = q0 + lane;
    const bool valid = lane < nvalid;
    unsigned char* stage = s_stage[warp];
    float acc[PX][32];
#pragma unroll
    for (int px = 0; px < PX; ++px)
#pragma unroll
        for (int c = 0; c < 32; ++c) acc[px][c] = p.bias[c];
    if (valid) {
        const int x = (int)(q % wq) * PX;
        const int y = (int)((q / wq) % p.H);
        const long long n = q / ((long long)wq * p.H);
        // the whole 3 x (PX+2) x CIN input window first (all loads in flight together: one exposed memory latency per thread, hidden by
        // the FMA phases of the other warps), then FMAs only
        float vin[CIN][3][PX + 2];
#pragma unroll
        for (int ci = 0; ci < CIN; ++ci) {
            const float* pl = p.plane[ci] + n * p.batch_stride[ci];
            const float sc = p.scale[ci], sh = p.shift[ci];
#pragma unroll
            for (int ky = 0; ky < 3; ++ky) {
                const int gy = y + ky - 1;
                const bool rin = gy >= 0 && gy < p.H;                             // outside: zero padding of the (normalised) input
                const float* row = pl + (size_t)(rin ? gy : y) * p.W + x;
                float* v = vin[ci][ky];
                v[0] = (rin && x > 0) ? fmaf(__ldg(row - 1), sc, sh) : 0.f;
                if (PX == 4) {
                    const float4 c4 = __ldg(reinterpret_cast<const float4*>(row));
                    v[1] = fmaf(c4.x, sc, sh); v[2] = fmaf(c4.y, sc, sh); v[PX - 1] = fmaf(c4.z, sc, sh); v[PX] = fmaf(c4.w, sc, sh);
                } else {
                    const float2 c2 = __ldg(reinterpret_cast<const float2*>(row));
                    v[1] = fmaf(c2.x, sc, sh); v[2] = fmaf(c2.y, sc, sh);
                }
                v[PX + 1] = (rin && x + PX < p.W) ? fmaf(__ldg(row + PX), sc, sh) : 0.f;
                if (!rin) {
#pragma unroll
                    for (int k = 1; k <= PX; ++k) v[k] = 0.f;
                }
            }
        }
#pragma unroll
        for (int ci = 0; ci < CIN; ++ci) {
#pragma unroll
            for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
                for (int kx = 0; kx < 3; ++kx) {
#pragma unroll
                    for (int c = 0; c < 32; ++c) {
                        const float wv = p.w[(ci * 9 + ky * 3 + kx) * 32 + c];      // constant-bank operand
#pragma unroll
                        for (int px = 0; px < PX; ++px) acc[px][c] = fmaf(vin[ci][ky][px + kx], wv, acc[px][c]);
                    }
                }
            }
        }
        const uint4* mrow = p.mask ? reinterpret_cast<const uint4*>(p.mask + (size_t)q * (PX * 32)) : nullptr;
#pragma unroll
        for (int px = 0; px < PX; ++px) {
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                float* a = &acc[px][g * 8];
                if (mrow) {
                    const uint4 mv = __ldg(mrow + px * 4 + g);
                    const uint32_t* mu = reinterpret_cast<const uint32_t*>(&mv);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float2 m = unpack_bf162(mu[j]);
                        if (!(m.x > 0.f)) a[j * 2] = 0.f;
                        if (!(m.y > 0.f)) a[j * 2 + 1] = 0.f;
                    }
                }
                if (p.relu_out) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) a[j] = fmaxf(a[j], 0.f);
                }
                uint4 ov;
                ov.x = pack_bf162(a[0], a[1]); ov.y = pack_bf162(a[2], a[3]);
                ov.z = pack_bf162(a[4], a[5]); ov.w = pack_bf162(a[6], a[7]);
                const int k = px * 4 + g;
                *reinterpret_cast<uint4*>(stage + lane * TB + ((k ^ (lane & (NCH - 1))) << 4)) = ov;
            }
        }
    }
    __syncwarp();
    uint4* dst = reinterpret_cast<uint4*>(p.out + (size_t)q0 * (PX * 32));
#pragma unroll
    for (int j = 0; j < NCH; ++j) {
        const int i = j * 32 + lane, r = i / NCH, c = i % NCH;
        if (r < nvalid) dst[i] = *reinterpret_cast<const uint4*>(stage + r * TB + ((c ^ (r & (NCH - 1))) << 4));
    }
}

// W must be even; `cin` selects the instantiation
inline void launch_stem_const(const StemCParams& p, int cin, cudaStream_t st) {
    const long long tot = (long long)p.N * p.H * p.W;
    const int blocks = cdiv(tot / 2, 128);
    if (cin == 1) launch_k(stem_convc_kernel<1, 2>, blocks, 128, 0, st, p);
    else if (cin == 2) launch_k(stem_convc_kernel<2, 2>, blocks, 128, 0, st, p);
    else launch_k(stem_convc_kernel<3, 2>, blocks, 128, 0, st, p);
}

// launches the 2-pixel kernel when the row length allows it, the 1-pixel kernel otherwise
inline void launch_stem(const StemParams& p, int cin, cudaStream_t st) {
    const long long tot = (long long)p.N * p.H * p.W;
    if ((p.W & 1) == 0) {
        const int blocks = cdiv(tot / 2, 128);
        if (cin == 1) launch_k(stem_convp_kernel<1, 2>, blocks, 128, 0, st, p);
        else if (cin == 2) launch_k(stem_convp_kernel<2, 2>, blocks, 128, 0, st, p);
        else launch_k(stem_convp_kernel<3, 2>, blocks, 128, 0, st, p);
    } else {
        const int blocks = cdiv(tot, 128);
        if (cin == 1) launch_k(stem_conv_kernel<1>, blocks, 128, 0, st, p);
        else if (cin == 2) launch_k(stem_conv_kernel<2>, blocks, 128, 0, st, p);
        else launch_k(stem_conv_kernel<3>, blocks, 128, 0, st, p);
    }
}

// -------------------------------------------------------------------------------------------------
// 32 -> 1 channel 3x3 s1 p1 conv: the prediction layer prdct.3 (network_exp_msg_chn_adapt.py:289)
// with ReLU-on-load, and -- with pre-flipped weights, no ReLU, accumulate -- the data-gradient of a
// stem with respect to one of its input planes.  out = [acc_prev +] conv(in) + bias [+ add].
// -------------------------------------------------------------------------------------------------
// Block = a 32 x 8 tile of output pixels: the (34 x 10) input halo (zero padded) is staged in shared memory with coalesced
// 16 B loads (ReLU applied on the way in), then every thread reads its 9 x 64 B taps conflict-free.
// Launch: grid (cdiv(W, 32), cdiv(H, 8), N), block (32, 8).
#define HEADC_TW 32
#define HEADC_TH 8
__global__ void __launch_bounds__(HEADC_TW * HEADC_TH) head_conv_kernel(const bf16* __restrict__ in, const float* __restrict__ w /*[9][32]*/,
                                                        float bias, const float* __restrict__ add, float* __restrict__ out,
                                                        int N, int H, int W, int relu_in, int accumulate) {
    PDL_SYNC();
    __shared__ float s_w[9 * 32];
    __shared__ __align__(16) unsigned char s_in[(HEADC_TH + 2) * (HEADC_TW + 2) * 64];
    const int tid = threadIdx.y * HEADC_TW + threadIdx.x;
    for (int i = tid; i < 288; i += HEADC_TW * HEADC_TH) s_w[i] = w[i];
    const int x0 = blockIdx.x * HEADC_TW, y0 = blockIdx.y * HEADC_TH, n = blockIdx.z;
    const bf16* inn = in + (size_t)n * H * W * 32;
    const bf162 z = __floats2bfloat162_rn(0.f, 0.f);
    for (int i = tid; i < (HEADC_TH + 2) * (HEADC_TW + 2) * 4; i += HEADC_TW * HEADC_TH) {
        const int c = i & 3, px = (i >> 2) % (HEADC_TW + 2), ry = (i >> 2) / (HEADC_TW + 2);
        const int gy = y0 + ry - 1, gx = x0 + px - 1;
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (gy >= 0 && gy < H && gx >= 0 && gx < W) {
            v = __ldg(reinterpret_cast<const uint4*>(inn + ((size_t)gy * W + gx) * 32) + c);
            if (relu_in) {
                bf162* h = reinterpret_cast<bf162*>(&v);
#pragma unroll
                for (int j = 0; j < 4; ++j) h[j] = __hmax2(h[j], z);
            }
        }
        const int row = ry * (HEADC_TW + 2) + px;
        *reinterpret_cast<uint4*>(s_in + row * 64 + ((c ^ ((row >> 1) & 3)) << 4)) = v;
    }
    __syncthreads();
    const int x = x0 + threadIdx.x, y = y0 + threadIdx.y;
    if (x >= W || y >= H) return;
    float acc = bias;
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
            const int row = (threadIdx.y + ky) * (HEADC_TW + 2) + threadIdx.x + kx;
            const float* wr = s_w + (ky * 3 + kx) * 32;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                uint4 v = *reinterpret_cast<const uint4*>(s_in + row * 64 + ((q ^ ((row >> 1) & 3)) << 4));
                const uint32_t* u = reinterpret_cast<const uint32_t*>(&v);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float2 f = unpack_bf162(u[j]);
                    acc = fmaf(f.x, wr[q * 8 + j * 2], acc);
                    acc = fmaf(f.y, wr[q * 8 + j * 2 + 1], acc);
                }
            }
        }
    }
    const size_t idx = ((size_t)n * H + y) * W + x;
    if (add) acc += add[idx];
    if (accumulate) acc += out[idx];
    out[idx] = acc;
}

// The engine's form of the 32 -> 1 conv: the same tile scheme with the weights BY VALUE in the kernel parameters (constant-bank FMA
// operands instead of 72 shared-memory weight loads per output pixel).  A vertical-strip variant (4 outputs per thread, each staged pixel
// unpacked once for the three rows it feeds) was measured at 36 us against 24 us for this form at 352x1216: register pressure made the
// compiler redo the unpacking per tap.  Launch: grid (cdiv(W, 32), cdiv(H, 8), N), block (32, 8).
struct HeadCParams {
    const bf16* in; const float* add; float* out;
    int N, H, W, relu_in, accumulate;
    float bias;
    float w[9 * 32];     // [tap][ci]
};
__global__ void __launch_bounds__(HEADC_TW * HEADC_TH) head_convc_kernel(const __grid_constant__ HeadCParams p) {
    PDL_SYNC();
    __shared__ __align__(16) unsigned char s_in[(HEADC_TH + 2) * (HEADC_TW + 2) * 64];
    const int x0 = blockIdx.x * HEADC_TW, y0 = blockIdx.y * HEADC_TH, n = blockIdx.z;
    const bf16* inn = p.in + (size_t)n * p.H * p.W * 32;
    const bf162 z = __floats2bfloat162_rn(0.f, 0.f);
    // halo: warp w stages rows w, w+8; lane j walks the row's 34 x 4 sixteen-byte chunks (no integer division on the way)
    for (int ry = threadIdx.y; ry < HEADC_TH + 2; ry += HEADC_TH) {
        const int gy = y0 + ry - 1;
        const bool rin = gy >= 0 && gy < p.H;
        const bf16* grow = inn + (size_t)(rin ? gy : 0) * p.W * 32;
        for (int j = threadIdx.x; j < (HEADC_TW + 2) * 4; j += 32) {
            const int c = j & 3, px = j >> 2;
            const int gx = x0 + px - 1;
            uint4 v = make_uint4(0u, 0u, 0u, 0u);
            if (rin && gx >= 0 && gx < p.W) {
                v = __ldg(reinterpret_cast<const uint4*>(grow + (size_t)gx * 32) + c);
                if (p.relu_in) {
                    bf162* h = reinterpret_cast<bf162*>(&v);
#pragma unroll
                    for (int k = 0; k < 4; ++k) h[k] = __hmax2(h[k], z);
                }
            }
            const int row = ry * (HEADC_TW + 2) + px;
            *reinterpret_cast<uint4*>(s_in + row * 64 + ((c ^ ((row >> 1) & 3)) << 4)) = v;
        }
    }
    __syncthreads();
    const int x = x0 + threadIdx.x, y = y0 + threadIdx.y;
    if (x >= p.W || y >= p.H) return;
    float acc = p.bias;
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
            const int row = (threadIdx.y + ky) * (HEADC_TW + 2) + threadIdx.x + kx;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const uint4 v = *reinterpret_cast<const uint4*>(s_in + row * 64 + ((q ^ ((row >> 1) & 3)) << 4));
                const uint32_t* u = reinterpret_cast<const uint32_t*>(&v);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float2 f = unpack_bf162(u[j]);
                    acc = fmaf(f.x, p.w[(ky * 3 + kx) * 32 + q * 8 + j * 2], acc);
                    acc = fmaf(f.y, p.w[(ky * 3 + kx) * 32 + q * 8 + j * 2 + 1], acc);
                }
            }
        }
    }
    const size_t idx = ((size_t)n * p.H + y) * p.W + x;
    if (p.add) acc += p.add[idx];
    if (p.accumulate) acc += p.out[idx];
    p.out[idx] = acc;
}

// -------------------------------------------------------------------------------------------------
// bilinear x2, align_corners=True (F.interpolate; SURVEY Appendix B), fp32 coordinates as ATen's
// upsample_bilinear2d: scale = (in-1)/(out-1), src = scale*dst, i0 = int(src), lambda = src - i0.
// -------------------------------------------------------------------------------------------------
__device__ __forceinline__ void up2_coord(int dst, int in_size, float scale, int& i0, int& i1, float& l0, float& l1) {
    float src = scale * (float)dst;
    i0 = (int)src;
    if (i0 > in_size - 1) i0 = in_size - 1;
    i1 = i0 + ((i0 < in_size - 1) ? 1 : 0);
    l1 = src - (float)i0;
    l0 = 1.f - l1;
}
__host__ __device__ __forceinline__ float up2_scale(int in_size) {
    int out_size = 2 * in_size;
    return out_size > 1 ? (float)(in_size - 1) / (float)(out_size - 1) : 0.f;
}

// out[y][x] = up2(a [+ b])[y][x] [+ c[y][x]]     (a, b: [N,h,w]; out, c: [N,2h,2w])
__global__ void up2_1ch_kernel(const float* __restrict__ a, const float* __restrict__ b, const float* __restrict__ c,
                               float* __restrict__ out, int N, int h, int w) {
    PDL_SYNC();
    int H = 2 * h, W = 2 * w;
    long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)N * H * W) return;
    int x = idx % W;
    int y = (idx / W) % H;
    int n = idx / ((long long)W * H);
    int y0, y1, x0, x1; float ly0, ly1, lx0, lx1;
    up2_coord(y, h, up2_scale(h), y0, y1, ly0, ly1);
    up2_coord(x, w, up2_scale(w), x0, x1, lx0, lx1);
    size_t base = (size_t)n * h * w;
    float v00 = a[base + (size_t)y0 * w + x0], v01 = a[base + (size_t)y0 * w + x1];
    float v10 = a[base + (size_t)y1 * w + x0], v11 = a[base + (size_t)y1 * w + x1];
    if (b) {
        v00 += b[base + (size_t)y0 * w + x0]; v01 += b[base + (size_t)y0 * w + x1];
        v10 += b[base + (size_t)y1 * w + x0]; v11 += b[base + (size_t)y1 * w + x1];
    }
    float r = ly0 * (lx0 * v00 + lx1 * v01) + ly1 * (lx0 * v10 + lx1 * v11);
    if (c) r += c[idx];
    out[idx] = r;
}

// weight with which destination index t reads source index s along one axis
__device__ __forceinline__ float up2_adj_weight(int t, int s, int in_size, float scale) {
    int i0, i1; float l0, l1;
    up2_coord(t, in_size, scale, i0, i1, l0, l1);
    float wgt = 0.f;
    if (i0 == s) wgt += l0;
    if (i1 == s) wgt += l1;
    return wgt;
}

// adjoint: gl[s] [+]= sum_t w(t,s) * gh[t]        (gh: [N,2h,2w] -> gl: [N,h,w])
__global__ void up2_1ch_adj_kernel(const float* __restrict__ gh, float* __restrict__ gl, int N, int h, int w, int accumulate) {
    PDL_SYNC();
    long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)N * h * w) return;
    int x = idx % w;
    int y = (idx / w) % h;
    int n = idx / ((long long)w * h);
    int H = 2 * h, W = 2 * w;
    float sy = up2_scale(h), sx = up2_scale(w);
    float wy[6], wx[6];
    int ty0 = 2 * y - 2, tx0 = 2 * x - 2;
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        int t = ty0 + j;
        wy[j] = (t >= 0 && t < H) ? up2_adj_weight(t, y, h, sy) : 0.f;
        t = tx0 + j;
        wx[j] = (t >= 0 && t < W) ? up2_adj_weight(t, x, w, sx) : 0.f;
    }
    const float* g = gh + (size_t)n * H * W;
    float acc = 0.f;
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        if (wy[j] == 0.f) continue;
        float row = 0.f;
#pragma unroll
        for (int i = 0; i < 6; ++i)
            if (wx[i] != 0.f) row += wx[i] * g[(size_t)(ty0 + j) * W + tx0 + i];
        acc += wy[j] * row;
    }
    if (accumulate) acc += gl[idx];
    gl[idx] = acc;
}

// 32-channel NHWC bf16: out[p] = x[p] + up2(half)[p]   (thread = pixel x 8 channels)
// out2 (optional) additionally receives ReLU(out): the stride-2 tensor-core conv that consumes it has no ReLU-on-load
__global__ void add_up2_c32_kernel(const bf16* __restrict__ x, const bf16* __restrict__ half, bf16* __restrict__ out, int N, int h, int w,
                                   bf16* __restrict__ out2) {
    PDL_SYNC();
    int H = 2 * h, W = 2 * w;
    long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)N * H * W * 4) return;
    int q = idx & 3;
    long long pix = idx >> 2;
    int xx = pix % W;
    int yy = (pix / W) % H;
    int n = pix / ((long long)W * H);
    int y0, y1, x0, x1; float ly0, ly1, lx0, lx1;
    up2_coord(yy, h, up2_scale(h), y0, y1, ly0, ly1);
    up2_coord(xx, w, up2_scale(w), x0, x1, lx0, lx1);
    const bf16* hb = half + (size_t)n * h * w * 32 + q * 8;
    uint4 a00 = __ldg(reinterpret_cast<const uint4*>(hb + ((size_t)y0 * w + x0) * 32));
    uint4 a01 = __ldg(reinterpret_cast<const uint4*>(hb + ((size_t)y0 * w + x1) * 32));
    uint4 a10 = __ldg(reinterpret_cast<const uint4*>(hb + ((size_t)y1 * w + x0) * 32));
    uint4 a11 = __ldg(reinterpret_cast<const uint4*>(hb + ((size_t)y1 * w + x1) * 32));
    uint4 xv = *reinterpret_cast<const uint4*>(x + (size_t)pix * 32 + q * 8);
    const uint32_t *u00 = reinterpret_cast<const uint32_t*>(&a00), *u01 = reinterpret_cast<const uint32_t*>(&a01);
    const uint32_t *u10 = reinterpret_cast<const uint32_t*>(&a10), *u11 = reinterpret_cast<const uint32_t*>(&a11);
    const uint32_t* ux = reinterpret_cast<const uint32_t*>(&xv);
    uint4 ov; uint32_t* uo = reinterpret_cast<uint32_t*>(&ov);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        float2 f00 = unpack_bf162(u00[j]), f01 = unpack_bf162(u01[j]), f10 = unpack_bf162(u10[j]), f11 = unpack_bf162(u11[j]);
        float2 fx = unpack_bf162(ux[j]);
        float r0 = ly0 * (lx0 * f00.x + lx1 * f01.x) + ly1 * (lx0 * f10.x + lx1 * f11.x);
        float r1 = ly0 * (lx0 * f00.y + lx1 * f01.y) + ly1 * (lx0 * f10.y + lx1 * f11.y);
        uo[j] = pack_bf162(fx.x + r0, fx.y + r1);
    }
    *reinterpret_cast<uint4*>(out + (size_t)pix * 32 + q * 8) = ov;
    if (out2) {
        const bf162 z = __floats2bfloat162_rn(0.f, 0.f);
        bf162* h2 = reinterpret_cast<bf162*>(&ov);
#pragma unroll
        for (int j = 0; j < 4; ++j) h2[j] = __hmax2(h2[j], z);
        *reinterpret_cast<uint4*>(out2 + (size_t)pix * 32 + q * 8) = ov;
    }
}

// adjoint for 32-channel maps: gl[s] [+]= sum_t w(t,s) gh[t]
__global__ void up2_c32_adj_kernel(const bf16* __restrict__ gh, bf16* __restrict__ gl, int N, int h, int w, int accumulate) {
    PDL_SYNC();
    long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)N * h * w * 4) return;
    int q = idx & 3;
    long long pix = idx >> 2;
    int x = pix % w;
    int y = (pix / w) % h;
    int n = pix / ((long long)w * h);
    int H = 2 * h, W = 2 * w;
    float sy = up2_scale(h), sx = up2_scale(w);
    float wy[6], wx[6];
    int ty0 = 2 * y - 2, tx0 = 2 * x - 2;
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        int t = ty0 + j;
        wy[j] = (t >= 0 && t < H) ? up2_adj_weight(t, y, h, sy) : 0.f;
        t = tx0 + j;
        wx[j] = (t >= 0 && t < W) ? up2_adj_weight(t, x, w, sx) : 0.f;
    }
    const bf16* g = gh + (size_t)n * H * W * 32 + q * 8;
    float acc[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[c] = 0.f;
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        if (wy[j] == 0.f) continue;
#pragma unroll
        for (int i = 0; i < 6; ++i) {
            float wgt = wy[j] * wx[i];
            if (wgt == 0.f) continue;
            uint4 v = __ldg(reinterpret_cast<const uint4*>(g + ((size_t)(ty0 + j) * W + tx0 + i) * 32));
            const uint32_t* u = reinterpret_cast<const uint32_t*>(&v);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                float2 f = unpack_bf162(u[k]);
                acc[k * 2] = fmaf(wgt, f.x, acc[k * 2]);
                acc[k * 2 + 1] = fmaf(wgt, f.y, acc[k * 2 + 1]);
            }
        }
    }
    bf16* o = gl + (size_t)pix * 32 + q * 8;
    if (accumulate) {
        uint4 v = *reinterpret_cast<const uint4*>(o);
        const uint32_t* u = reinterpret_cast<const uint32_t*>(&v);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float2 f = unpack_bf162(u[k]);
            acc[k * 2] += f.x; acc[k * 2 + 1] += f.y;
        }
    }
    uint4 ov;
    ov.x = pack_bf162(acc[0], acc[1]); ov.y = pack_bf162(acc[2], acc[3]);
    ov.z = pack_bf162(acc[4], acc[5]); ov.w = pack_bf162(acc[6], acc[7]);
    *reinterpret_cast<uint4*>(o) = ov;
}

// out = a + b, optionally ReLU'd (bf16, n multiple of 8)
__global__ void ew_add_kernel(const bf16* __restrict__ a, const bf16* __restrict__ b, bf16* __restrict__ out, long long n8, int relu) {
    PDL_SYNC();
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n8) return;
    uint4 av = reinterpret_cast<const uint4*>(a)[i], bv = reinterpret_cast<const uint4*>(b)[i];
    const uint32_t *ua = reinterpret_cast<const uint32_t*>(&av), *ub = reinterpret_cast<const uint32_t*>(&bv);
    uint4 ov; uint32_t* uo = reinterpret_cast<uint32_t*>(&ov);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        float2 fa = unpack_bf162(ua[j]), fb = unpack_bf162(ub[j]);
        float s0 = fa.x + fb.x, s1 = fa.y + fb.y;
        if (relu) { s0 = fmaxf(s0, 0.f); s1 = fmaxf(s1, 0.f); }
        uo[j] = pack_bf162(s0, s1);
    }
    reinterpret_cast<uint4*>(out)[i] = ov;
}

// The three skip sums of a decoder (network_exp_msg_chn_adapt.py:301-303: x2 = dx2 + cx2, x1 = dx1 + cx1, x0 = dx0 + cx0) in one
// launch; the /4-resolution sum x2 is also written through a ReLU (the transposed conv that reads it has no ReLU-on-load).
struct DecSumsParams { const bf16* a[3]; const bf16* b[3]; bf16* out[3]; bf16* out0_relu; long long n8[3]; };
__global__ void dec_sums_kernel(const DecSumsParams p) {
    PDL_SYNC();
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    int k = 0;
    if (i >= p.n8[0]) { i -= p.n8[0]; k = 1; if (i >= p.n8[1]) { i -= p.n8[1]; k = 2; if (i >= p.n8[2]) return; } }
    const uint4 av = reinterpret_cast<const uint4*>(p.a[k])[i], bv = reinterpret_cast<const uint4*>(p.b[k])[i];
    const uint32_t *ua = reinterpret_cast<const uint32_t*>(&av), *ub = reinterpret_cast<const uint32_t*>(&bv);
    uint4 ov, rv; uint32_t *uo = reinterpret_cast<uint32_t*>(&ov), *ur = reinterpret_cast<uint32_t*>(&rv);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float2 fa = unpack_bf162(ua[j]), fb = unpack_bf162(ub[j]);
        const float s0 = fa.x + fb.x, s1 = fa.y + fb.y;
        uo[j] = pack_bf162(s0, s1);
        ur[j] = pack_bf162(fmaxf(s0, 0.f), fmaxf(s1, 0.f));
    }
    reinterpret_cast<uint4*>(p.out[k])[i] = ov;
    if (k == 0 && p.out0_relu) reinterpret_cast<uint4*>(p.out0_relu)[i] = rv;
}

// -------------------------------------------------------------------------------------------------
// BatchNorm (train mode: batch statistics, biased variance for normalisation, unbiased for the
// running estimate, momentum 0.1 -- nn.BatchNorm2d/1d as used at network_exp_msg_chn_adapt.py:28-36
// and :1089-1098).  Tensors are [rows][C] bf16 (NHWC maps or the R x 512 head matrices).
//   col_stats        : per-block partial sums, double:  mode 0: (sum x, sum x^2)
//                                                       mode 1: (sum dy, sum dy*xhat)  [BN backward]
//   bn_finalize      : partials -> mean/invstd/scale/shift (+ running-stat update)
//   bn_apply         : y = act(x*scale + shift) [+ residual]
//   bn_bwd_finalize  : partials -> dgamma, dbeta, and the three coefficient vectors of dx
//   bn_bwd_apply     : dx = k0[c]*dy - k1[c] - xhat*k2[c]
// `relu_mask`: the incoming dy is first multiplied by [x*scale+shift > 0] (the ReLU that follows BN
// in the MLP heads), so no masked copy of dy is ever written.
// -------------------------------------------------------------------------------------------------
struct BnParams {
    const float* gamma; const float* beta;
    float* running_mean; float* running_var; long long* num_batches_tracked;
    float* mean; float* invstd; float* scale; float* shift;
    float* uvar;          // optional: unbiased batch variance (what a deferred running-statistics update needs)
    float momentum, eps;
};

// The per-channel arithmetic of the two finalize steps, written with explicit roundings (no fused multiply-add left to the compiler) so that
// the stand-alone finalize kernels and the finalize fused into col_stats give bit-identical vectors.
__device__ __forceinline__ void bn_forward_channel(const BnParams& p, int ch, double a, double b, long long count) {
    const double cnt = (double)count;
    const double m = __ddiv_rn(a, cnt);
    double var = __dsub_rn(__ddiv_rn(b, cnt), __dmul_rn(m, m));
    if (var < 0.0) var = 0.0;
    const float invstd = (float)__ddiv_rn(1.0, sqrt(__dadd_rn(var, (double)p.eps)));
    const float mf = (float)m;
    p.mean[ch] = mf;
    p.invstd[ch] = invstd;
    const float sc = __fmul_rn(p.gamma[ch], invstd);
    p.scale[ch] = sc;
    p.shift[ch] = __fsub_rn(p.beta[ch], __fmul_rn(mf, sc));
    const double unbiased = count > 1 ? __ddiv_rn(__dmul_rn(var, cnt), (double)(count - 1)) : var;
    if (p.uvar) p.uvar[ch] = (float)unbiased;
    if (p.running_mean) {
        const float keep = __fsub_rn(1.f, p.momentum);
        p.running_mean[ch] = __fadd_rn(__fmul_rn(keep, p.running_mean[ch]), __fmul_rn(p.momentum, mf));
        p.running_var[ch] = __fadd_rn(__fmul_rn(keep, p.running_var[ch]), __fmul_rn(p.momentum, (float)unbiased));
    }
    if (ch == 0 && p.num_batches_tracked) *p.num_batches_tracked += 1;
}
// a, b: the sums over the batch the data gradient uses (all ranks in shared-model mode); count likewise
__device__ __forceinline__ void bn_backward_channel(int ch, double a, double b, long long count, const float* __restrict__ gamma,
                                                    const float* __restrict__ invstd, float* __restrict__ k0, float* __restrict__ k1,
                                                    float* __restrict__ k2) {
    const float g = __fmul_rn(gamma[ch], invstd[ch]);
    const double cnt = (double)count;
    k0[ch] = g;
    k1[ch] = (float)__ddiv_rn(__dmul_rn((double)g, a), cnt);
    k2[ch] = (float)__ddiv_rn(__dmul_rn((double)g, b), cnt);
}

// sum of partial[k][slot][ch] over k for 32 channels per block: thread (cx = tid & 31, ks = tid >> 5) adds slice ks of the
// partial list (256 B coalesced reads, four independent loads in flight), the FIN_SLICES slices are combined through shared
// memory in a fixed order (deterministic).  Returns the totals (a: slot 0, b: slot 1) in the threads with ks == 0; launch
// with FIN_THREADS threads, cdiv(C, 32) blocks.
#define FIN_SLICES 32
#define FIN_THREADS (32 * FIN_SLICES)
__device__ __forceinline__ bool block_reduce_partials(const double* __restrict__ partial, int nblk, int C, int nslots, int& ch, double& a, double& b) {
    __shared__ double sh[2][FIN_SLICES][32];
    const int cx = threadIdx.x & 31, ks = threadIdx.x >> 5;
    ch = blockIdx.x * 32 + cx;
    a = 0.0; b = 0.0;
    if (ch < C) {
        double a4[4] = {0.0, 0.0, 0.0, 0.0}, b4[4] = {0.0, 0.0, 0.0, 0.0};
        int k = ks;
        for (; k + 3 * FIN_SLICES < nblk; k += 4 * FIN_SLICES) {
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                a4[u] += partial[((size_t)(k + u * FIN_SLICES) * 2 + 0) * C + ch];
                if (nslots > 1) b4[u] += partial[((size_t)(k + u * FIN_SLICES) * 2 + 1) * C + ch];
            }
        }
        for (; k < nblk; k += FIN_SLICES) {
            a4[0] += partial[((size_t)k * 2 + 0) * C + ch];
            if (nslots > 1) b4[0] += partial[((size_t)k * 2 + 1) * C + ch];
        }
        a = (a4[0] + a4[1]) + (a4[2] + a4[3]);
        b = (b4[0] + b4[1]) + (b4[2] + b4[3]);
    }
    sh[0][ks][cx] = a; sh[1][ks][cx] = b;
    __syncthreads();
    if (ks != 0 || ch >= C) return false;
#pragma unroll
    for (int k = 1; k < FIN_SLICES; ++k) { a += sh[0][k][cx]; b += sh[1][k][cx]; }
    return true;
}

#define STATS_ROWS_PER_BLOCK 64
// Fused finalize (single-GPU path): instead of a separate bn_finalize / bn_bwd_finalize launch, the LAST blocks of col_stats to finish
// turn the partial sums into the per-channel vectors.  Every block takes a ticket when its partials are written; the blocks holding the
// last G tickets (G = number of 32-channel groups, at most the grid size) wait until all tickets are out -- every other block has then
// published its partials -- and each finalises one group: the same slices, the same summation order and the same arithmetic as the
// stand-alone finalize kernels, so the vectors are bit-identical to theirs.  At most G blocks ever wait and every block they wait for is
// already running or does not need their slot, so the wait cannot deadlock.  The last finaliser resets the two counters.
struct StatsFin {
    int kind;                     // 0: none, 1: forward (BnParams), 2: backward (dgamma / dbeta / k0 / k1 / k2)
    unsigned int* counters;       // [2]: tickets, finished finalisers (zero between launches)
    long long count;
    BnParams p;
    const float* gamma; const float* invstd; float* dgamma; float* dbeta; float* k0; float* k1; float* k2;
};
__device__ __forceinline__ void stats_fused_finalize(const StatsFin& fin, const double* __restrict__ partial, int nblk, int C, double* scratch);

__global__ void __launch_bounds__(256) col_stats_kernel(const bf16* __restrict__ x, const bf16* __restrict__ dy, double* __restrict__ partial,
                                                        long long rows, int C, int mode, const float* __restrict__ mean,
                                                        const float* __restrict__ invstd, const float* __restrict__ scale,
                                                        const float* __restrict__ shift, int relu_mask, const StatsFin fin) {
    PDL_SYNC();
    extern __shared__ double s_red[];   // [256][2]... reduced per chunk below
    const int CH = C / 8;
    const int step = 256 / CH;
    const int c = threadIdx.x % CH, r0 = threadIdx.x / CH;
    long long row_begin = (long long)blockIdx.x * STATS_ROWS_PER_BLOCK;
    long long row_end = row_begin + STATS_ROWS_PER_BLOCK;
    if (row_end > rows) row_end = rows;
    float s0[8], s1[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { s0[j] = 0.f; s1[j] = 0.f; }
    float mu[8], is[8], sc[8], sh[8];
    if (mode == 1) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            mu[j] = mean[c * 8 + j]; is[j] = invstd[c * 8 + j];
            sc[j] = relu_mask ? scale[c * 8 + j] : 0.f; sh[j] = relu_mask ? shift[c * 8 + j] : 0.f;
        }
    }
#pragma unroll 4
    for (long long r = row_begin + r0; r < row_end; r += step) {
        uint4 xv = __ldg(reinterpret_cast<const uint4*>(x + (size_t)r * C + c * 8));
        const uint32_t* ux = reinterpret_cast<const uint32_t*>(&xv);
        if (mode == 0) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float2 f = unpack_bf162(ux[j]);
                s0[j * 2] += f.x; s0[j * 2 + 1] += f.y;
                s1[j * 2] = fmaf(f.x, f.x, s1[j * 2]); s1[j * 2 + 1] = fmaf(f.y, f.y, s1[j * 2 + 1]);
            }
        } else {
            uint4 gv = __ldg(reinterpret_cast<const uint4*>(dy + (size_t)r * C + c * 8));
            const uint32_t* ug = reinterpret_cast<const uint32_t*>(&gv);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float2 f = unpack_bf162(ux[j]), g = unpack_bf162(ug[j]);
                if (relu_mask) {
                    if (!(f.x * sc[j * 2] + sh[j * 2] > 0.f)) g.x = 0.f;
                    if (!(f.y * sc[j * 2 + 1] + sh[j * 2 + 1] > 0.f)) g.y = 0.f;
                }
                float xh0 = (f.x - mu[j * 2]) * is[j * 2], xh1 = (f.y - mu[j * 2 + 1]) * is[j * 2 + 1];
                s0[j * 2] += g.x; s0[j * 2 + 1] += g.y;
                s1[j * 2] = fmaf(g.x, xh0, s1[j * 2]); s1[j * 2 + 1] = fmaf(g.y, xh1, s1[j * 2 + 1]);
            }
        }
    }
    // reduce over the `step` threads that share a channel chunk
    double* sh0 = s_red;                 // [step][C]
    double* sh1 = s_red + (size_t)step * C;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        sh0[(size_t)r0 * C + c * 8 + j] = (double)s0[j];
        sh1[(size_t)r0 * C + c * 8 + j] = (double)s1[j];
    }
    __syncthreads();
    for (int ch = threadIdx.x; ch < C; ch += 256) {
        double a = 0.0, b = 0.0;
        for (int k = 0; k < step; ++k) { a += sh0[(size_t)k * C + ch]; b += sh1[(size_t)k * C + ch]; }
        partial[((size_t)blockIdx.x * 2 + 0) * C + ch] = a;
        partial[((size_t)blockIdx.x * 2 + 1) * C + ch] = b;
    }
    if (fin.kind) stats_fused_finalize(fin, partial, (int)gridDim.x, C, s_red);      // s_red (32 KB) is free again: reused for the slice sums
}


// one 32-channel group finalised by a 256-thread block: thread (cx = tid & 31, w = tid >> 5) computes slices ks = w, w + 8, w + 16, w + 24 of
// the FIN_SLICES = 32 slice sums exactly as block_reduce_partials does with 1024 threads (same loop, same 4-way split, same pairing), then
// the owner thread adds the 32 slices in the same order
__device__ __forceinline__ bool group_reduce_partials_256(const double* __restrict__ partial, int nblk, int C, int group, int& ch, double& a, double& b,
                                                          double (*sh)[FIN_SLICES][32]) {
    const int cx = threadIdx.x & 31, w = threadIdx.x >> 5;
    ch = group * 32 + cx;
    for (int ks = w; ks < FIN_SLICES; ks += 8) {
        double sa = 0.0, sb = 0.0;
        if (ch < C) {
            double a4[4] = {0.0, 0.0, 0.0, 0.0}, b4[4] = {0.0, 0.0, 0.0, 0.0};
            int k = ks;
            for (; k + 3 * FIN_SLICES < nblk; k += 4 * FIN_SLICES) {
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    a4[u] += partial[((size_t)(k + u * FIN_SLICES) * 2 + 0) * C + ch];
                    b4[u] += partial[((size_t)(k + u * FIN_SLICES) * 2 + 1) * C + ch];
                }
            }
            for (; k < nblk; k += FIN_SLICES) {
                a4[0] += partial[((size_t)k * 2 + 0) * C + ch];
                b4[0] += partial[((size_t)k * 2 + 1) * C + ch];
            }
            sa = (a4[0] + a4[1]) + (a4[2] + a4[3]);
            sb = (b4[0] + b4[1]) + (b4[2] + b4[3]);
        }
        sh[0][ks][cx] = sa; sh[1][ks][cx] = sb;
    }
    __syncthreads();
    a = sh[0][0][cx]; b = sh[1][0][cx];
    const bool owner = w == 0 && ch < C;
    if (owner) {
#pragma unroll
        for (int k = 1; k < FIN_SLICES; ++k) { a += sh[0][k][cx]; b += sh[1][k][cx]; }
    }
    __syncthreads();            // the shared slices are reused by the block's next group
    return owner;
}

__device__ __forceinline__ void stats_fused_finalize(const StatsFin& fin, const double* __restrict__ partial, int nblk, int C, double* scratch) {
    double (*fsh)[FIN_SLICES][32] = reinterpret_cast<double (*)[FIN_SLICES][32]>(scratch);      // 2 x 32 x 32 doubles = 16 KB
    __shared__ unsigned int s_ticket;
    __threadfence();                                   // this block's partials are visible device-wide before its ticket is
    __syncthreads();
    if (threadIdx.x == 0) s_ticket = atomicAdd(fin.counters, 1u);
    __syncthreads();
    const int G = (C + 31) / 32, F = G < nblk ? G : nblk;          // F finaliser blocks: the holders of the last F tickets
    const int first = nblk - F;
    if ((int)s_ticket < first) return;
    if (threadIdx.x == 0) {
        while (*reinterpret_cast<volatile unsigned int*>(fin.counters) < (unsigned int)nblk) { }
        __threadfence();
    }
    __syncthreads();
    for (int g = (int)s_ticket - first; g < G; g += F) {
        int ch; double a, b;
        const bool owner = group_reduce_partials_256(partial, nblk, C, g, ch, a, b, fsh);
        if (!owner) continue;
        if (fin.kind == 1) {
            bn_forward_channel(fin.p, ch, a, b, fin.count);
        } else {
            if (fin.dbeta) fin.dbeta[ch] = (float)a;
            if (fin.dgamma) fin.dgamma[ch] = (float)b;
            bn_backward_channel(ch, a, b, fin.count, fin.gamma, fin.invstd, fin.k0, fin.k1, fin.k2);
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(fin.counters + 1, 1u) == (unsigned int)(F - 1)) { fin.counters[0] = 0u; fin.counters[1] = 0u; __threadfence(); }
    }
}

__global__ void __launch_bounds__(FIN_THREADS) bn_finalize_kernel(const double* __restrict__ partial, int nblk, long long count, int C, BnParams p, int training,
                                                                  const PeerComm comm, int xid) {
    PDL_SYNC();
    int ch; double a, b;
    if (training) {
        const bool owner = block_reduce_partials(partial, nblk, C, 2, ch, a, b);
        if (comm.world > 1) {                                   // batch statistics over the global batch (SyncBatchNorm)
            bn_sums_all_ranks(comm, xid, C, owner, ch, a, b);
            count *= comm.world;
        }
        if (!owner) return;
        bn_forward_channel(p, ch, a, b, count);
    } else {
        ch = blockIdx.x * 32 + (threadIdx.x & 31);
        if ((threadIdx.x >> 5) != 0 || ch >= C) return;
        float invstd = 1.f / sqrtf(p.running_var[ch] + p.eps);
        p.mean[ch] = p.running_mean[ch];
        p.invstd[ch] = invstd;
        float sc = p.gamma[ch] * invstd;
        p.scale[ch] = sc;
        p.shift[ch] = p.beta[ch] - p.running_mean[ch] * sc;
    }
}

// deferred running-statistics update (momentum form of nn.BatchNorm) from statistics computed earlier on another stream:
// keeps the reference's update ORDER (real image first, zero image second) while the zero-image branch runs ahead
__global__ void bn_running_update_kernel(const float* __restrict__ mean, const float* __restrict__ uvar, float* __restrict__ running_mean,
                                         float* __restrict__ running_var, long long* __restrict__ num_batches_tracked, int C, float momentum) {
    PDL_SYNC();
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch < C) {
        running_mean[ch] = (1.f - momentum) * running_mean[ch] + momentum * mean[ch];
        running_var[ch] = (1.f - momentum) * running_var[ch] + momentum * uvar[ch];
    }
    if (ch == 0 && num_batches_tracked) *num_batches_tracked += 1;
}

// y = act(x*scale+shift) [+ res];  act: 0 none, 1 relu
// thread = one 8-channel chunk x EW_ROWS rows (rows interleaved across the block's row groups: coalesced 16 B accesses);
// the per-channel vectors are read once per thread.  Launch: blockDim 256, grid cdiv(rows, (256 / (C/8)) * EW_ROWS).
#define EW_ROWS 8
__global__ void __launch_bounds__(256) bn_apply_kernel(const bf16* __restrict__ x, const bf16* __restrict__ res, bf16* __restrict__ y, long long rows, int C,
                                const float* __restrict__ scale, const float* __restrict__ shift, int act) {
    PDL_SYNC();
    const int CH = C / 8, step = 256 / CH;
    const int c = threadIdx.x % CH, r0 = threadIdx.x / CH;
    float sc[8], sh[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { sc[j] = scale[c * 8 + j]; sh[j] = shift[c * 8 + j]; }
    const long long rb = (long long)blockIdx.x * step * EW_ROWS + r0;
#pragma unroll
    for (int k = 0; k < EW_ROWS; ++k) {
        const long long r = rb + (long long)k * step;
        if (r >= rows) break;
        const size_t i = (size_t)r * CH + c;
        uint4 xv = reinterpret_cast<const uint4*>(x)[i];
        const uint32_t* ux = reinterpret_cast<const uint32_t*>(&xv);
        uint4 rv = make_uint4(0u, 0u, 0u, 0u);
        if (res) rv = reinterpret_cast<const uint4*>(res)[i];
        const uint32_t* ur = reinterpret_cast<const uint32_t*>(&rv);
        uint4 ov; uint32_t* uo = reinterpret_cast<uint32_t*>(&ov);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float2 f = unpack_bf162(ux[j]);
            f.x = f.x * sc[j * 2] + sh[j * 2];
            f.y = f.y * sc[j * 2 + 1] + sh[j * 2 + 1];
            if (act == 1) { f.x = fmaxf(f.x, 0.f); f.y = fmaxf(f.y, 0.f); }
            if (res) { float2 rr = unpack_bf162(ur[j]); f.x += rr.x; f.y += rr.y; }
            uo[j] = pack_bf162(f.x, f.y);
        }
        reinterpret_cast<uint4*>(y)[i] = ov;
    }
}

// dgamma = sum dy*xhat, dbeta = sum dy;  dx = k0*dy - k1 - xhat*k2 with
//   k0 = gamma*invstd, k1 = k0*mean(dy), k2 = k0*mean(dy*xhat)
__global__ void __launch_bounds__(FIN_THREADS) bn_bwd_finalize_kernel(const double* __restrict__ partial, int nblk, long long count, int C,
                                       const float* __restrict__ gamma, const float* __restrict__ invstd,
                                       float* __restrict__ dgamma, float* __restrict__ dbeta,
                                       float* __restrict__ k0, float* __restrict__ k1, float* __restrict__ k2, const PeerComm comm, int xid) {
    PDL_SYNC();
    int ch; double a, b;
    const bool owner = block_reduce_partials(partial, nblk, C, 2, ch, a, b);
    // parameter gradients stay LOCAL sums (the gradient all-reduce averages them, as DDP does); the data gradient uses the means over
    // the global batch (torch SyncBatchNorm backward: all_reduce of sum_dy / sum_dy_xmu only)
    if (owner) {
        if (dbeta) dbeta[ch] = (float)a;
        if (dgamma) dgamma[ch] = (float)b;
    }
    if (comm.world > 1) {
        bn_sums_all_ranks(comm, xid, C, owner, ch, a, b);
        count *= comm.world;
    }
    if (!owner) return;
    bn_backward_channel(ch, a, b, count, gamma, invstd, k0, k1, k2);
}

__global__ void __launch_bounds__(256) bn_bwd_apply_kernel(const bf16* __restrict__ dy, const bf16* __restrict__ x, bf16* __restrict__ dx, long long rows, int C,
                                    const float* __restrict__ mean, const float* __restrict__ invstd, const float* __restrict__ k0,
                                    const float* __restrict__ k1, const float* __restrict__ k2, const float* __restrict__ scale,
                                    const float* __restrict__ shift, int relu_mask) {
    PDL_SYNC();
    const int CH = C / 8, step = 256 / CH;
    const int c = threadIdx.x % CH, r0 = threadIdx.x / CH;
    float mu[8], is[8], a0[8], a1[8], a2[8], sc[8], sh[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int ch = c * 8 + j;
        mu[j] = mean[ch]; is[j] = invstd[ch]; a0[j] = k0[ch]; a1[j] = k1[ch]; a2[j] = k2[ch];
        sc[j] = relu_mask ? scale[ch] : 0.f; sh[j] = relu_mask ? shift[ch] : 0.f;
    }
    const long long rb = (long long)blockIdx.x * step * EW_ROWS + r0;
#pragma unroll
    for (int k = 0; k < EW_ROWS; ++k) {
        const long long r = rb + (long long)k * step;
        if (r >= rows) break;
        const size_t i = (size_t)r * CH + c;
        uint4 xv = reinterpret_cast<const uint4*>(x)[i], gv = reinterpret_cast<const uint4*>(dy)[i];
        const uint32_t *ux = reinterpret_cast<const uint32_t*>(&xv), *ug = reinterpret_cast<const uint32_t*>(&gv);
        uint4 ov; uint32_t* uo = reinterpret_cast<uint32_t*>(&ov);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float2 f = unpack_bf162(ux[j]), g = unpack_bf162(ug[j]);
            if (relu_mask) {
                if (!(f.x * sc[j * 2] + sh[j * 2] > 0.f)) g.x = 0.f;
                if (!(f.y * sc[j * 2 + 1] + sh[j * 2 + 1] > 0.f)) g.y = 0.f;
            }
            float xh0 = (f.x - mu[j * 2]) * is[j * 2], xh1 = (f.y - mu[j * 2 + 1]) * is[j * 2 + 1];
            float o0 = a0[j * 2] * g.x - a1[j * 2] - xh0 * a2[j * 2];
            float o1 = a0[j * 2 + 1] * g.y - a1[j * 2 + 1] - xh1 * a2[j * 2 + 1];
            uo[j] = pack_bf162(o0, o1);
        }
        reinterpret_cast<uint4*>(dx)[i] = ov;
    }
}

// column sums of a [rows][C] bf16 matrix into fp32 (bias gradients): out[c] = sum_r x[r][c]; uses col_stats partials (mode 0, slot 0)
__global__ void __launch_bounds__(FIN_THREADS) colsum_finalize_kernel(const double* __restrict__ partial, int nblk, int C, float* __restrict__ out) {
    PDL_SYNC();
    int ch; double a, b;
    if (!block_reduce_partials(partial, nblk, C, 1, ch, a, b)) return;
    out[ch] = (float)a;
}

// -------------------------------------------------------------------------------------------------
// a13-a15: the three TTA losses (src/loss_utils.py:116-169,624-638; src/external_model_adapt.py:371-441)
//   map part : masked sparse-depth L1 (per-image normalisation, no epsilon) + edge-aware smoothness on
//              the RAW [0,255] image; one reduction pass + one gradient pass over the full-res maps
//   cos part : mean_r(2 - 2 <e/|e|, r/|r|>) over the two R x 512 head outputs, warp per row
//   finalize : device-side `if loss_cos < 0.3: w_cos = 0` gate (a host sync in the reference)
// Partial layout (doubles): map: [N][nblk][4] = {sum v|d-p|, sum v, sum wx|dx|, sum wy|dy|}; cos: [nblk]
// -------------------------------------------------------------------------------------------------
#define LOSS_BLOCK 256
__global__ void __launch_bounds__(LOSS_BLOCK) loss_map_reduce_kernel(const float* __restrict__ pred, const float* __restrict__ d,
                                                                     const float* __restrict__ v, const float* __restrict__ img,
                                                                     double* __restrict__ partial, int H, int W, float cap, int do_clamp) {
    PDL_SYNC();
    __shared__ double sh[32];
    const int n = blockIdx.y;
    const long long HW = (long long)H * W;
    const float* pn = pred + n * HW; const float* dn = d + n * HW; const float* vn = v + n * HW;
    const float* in = img + n * HW * 3;
    double s_sd = 0.0, s_v = 0.0, s_x = 0.0, s_y = 0.0;
    const int hw = (int)HW;                 // one image: < 2^31 pixels (32-bit index math: the 64-bit div / mod cost more than the loads)
    for (int i = blockIdx.x * LOSS_BLOCK + threadIdx.x; i < hw; i += gridDim.x * LOSS_BLOCK) {
        const int y = i / W, x = i - y * W;
        float p0 = pn[i];
        float dd = dn[i];
        if (do_clamp) dd = fminf(fmaxf(dd, 0.f), cap);
        float vv = vn[i];
        s_sd += (double)(vv * fabsf(dd - p0));
        s_v += (double)vv;
        if (x < W - 1) {
            float g = fabsf(in[i] - in[i + 1]) + fabsf(in[HW + i] - in[HW + i + 1]) + fabsf(in[2 * HW + i] - in[2 * HW + i + 1]);
            s_x += (double)(expf(-g / 3.f) * fabsf(p0 - pn[i + 1]));
        }
        if (y < H - 1) {
            float g = fabsf(in[i] - in[i + W]) + fabsf(in[HW + i] - in[HW + i + W]) + fabsf(in[2 * HW + i] - in[2 * HW + i + W]);
            s_y += (double)(expf(-g / 3.f) * fabsf(p0 - pn[i + W]));
        }
    }
    double r0 = block_sum_d(s_sd, sh), r1 = block_sum_d(s_v, sh), r2 = block_sum_d(s_x, sh), r3 = block_sum_d(s_y, sh);
    if (threadIdx.x == 0) {
        double* o = partial + ((size_t)n * gridDim.x + blockIdx.x) * 4;
        o[0] = r0; o[1] = r1; o[2] = r2; o[3] = r3;
    }
}

// rowstat[r] = {dot, |e|^2, |r|^2}; partial[blk] = sum over its rows of (2 - 2 cos)
__global__ void __launch_bounds__(256) loss_cos_rows_kernel(const bf16* __restrict__ emb, const bf16* __restrict__ ref, float* __restrict__ rowstat,
                                                            double* __restrict__ partial, long long R, int D) {
    PDL_SYNC();
    __shared__ double sh[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double local = 0.0;
    for (long long r = (long long)blockIdx.x * 8 + warp; r < R; r += (long long)gridDim.x * 8) {
        const bf16* e = emb + (size_t)r * D; const bf16* f = ref + (size_t)r * D;
        float dot = 0.f, ne = 0.f, nr = 0.f;
        for (int c = lane * 8; c < D; c += 256) {
            uint4 ev = __ldg(reinterpret_cast<const uint4*>(e + c)), fv = __ldg(reinterpret_cast<const uint4*>(f + c));
            const uint32_t *ue = reinterpret_cast<const uint32_t*>(&ev), *uf = reinterpret_cast<const uint32_t*>(&fv);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float2 a = unpack_bf162(ue[j]), b = unpack_bf162(uf[j]);
                dot = fmaf(a.x, b.x, dot); dot = fmaf(a.y, b.y, dot);
                ne = fmaf(a.x, a.x, ne); ne = fmaf(a.y, a.y, ne);
                nr = fmaf(b.x, b.x, nr); nr = fmaf(b.y, b.y, nr);
            }
        }
        dot = warp_sum(dot); ne = warp_sum(ne); nr = warp_sum(nr);
        if (lane == 0) {
            rowstat[r * 3 + 0] = dot; rowstat[r * 3 + 1] = ne; rowstat[r * 3 + 2] = nr;
            float den = fmaxf(sqrtf(ne), 1e-12f) * fmaxf(sqrtf(nr), 1e-12f);
            local += (double)(2.f - 2.f * dot / den);
        }
    }
    double tot = block_sum_d(local, sh);
    if (threadIdx.x == 0) partial[blockIdx.x] = tot;
}

struct LossScalars {   // device-resident result block
    float loss, loss_sparse_depth, loss_smooth, loss_cos, w_cos_eff;
    float inv_count[64];   // 1 / sum(v) per image (N <= 64)
};

__global__ void __launch_bounds__(256) loss_finalize_kernel(const double* __restrict__ map_partial, int map_blocks, const double* __restrict__ cos_partial,
                                     int cos_blocks, int N, int H, int W, long long R, float w_sd, float w_sm, float w_cos,
                                     float cos_gate, LossScalars* out) {
    PDL_SYNC();
    __shared__ double sh[32];
    __shared__ double s_sd;
    double sx = 0.0, sy = 0.0;
    if (threadIdx.x == 0) s_sd = 0.0;
    for (int n = 0; n < N; ++n) {
        double a = 0.0, b = 0.0, cx = 0.0, cy = 0.0;
        for (int k = threadIdx.x; k < map_blocks; k += 256) {
            const double* p = map_partial + ((size_t)n * map_blocks + k) * 4;
            a += p[0]; b += p[1]; cx += p[2]; cy += p[3];
        }
        a = block_sum_d(a, sh); b = block_sum_d(b, sh); cx = block_sum_d(cx, sh); cy = block_sum_d(cy, sh);
        if (threadIdx.x == 0) {
            float fa = (float)a, fb = (float)b;
            s_sd += (double)(fa / fb);               // no epsilon: an empty frame yields NaN, as in the reference
            if (n < 64) out->inv_count[n] = 1.f / fb;
            sx += cx; sy += cy;
        }
    }
    double c = 0.0;
    for (int k = threadIdx.x; k < cos_blocks; k += 256) c += cos_partial[k];
    c = block_sum_d(c, sh);
    if (threadIdx.x != 0) return;
    float l_sd = (float)(s_sd / N);
    float l_sm = (float)(sx / ((double)N * H * (W - 1))) + (float)(sy / ((double)N * (H - 1) * W));
    float l_cos = R > 0 ? (float)(c / (double)R) : 0.f;
    float w_eff = (l_cos < cos_gate) ? 0.f : w_cos;
    out->loss_sparse_depth = l_sd;
    out->loss_smooth = l_sm;
    out->loss_cos = l_cos;
    out->w_cos_eff = w_eff;
    out->loss = w_sd * l_sd + w_sm * l_sm + w_eff * l_cos;
}

// d loss / d pred  (upstream gradient `gscale` of the scalar loss, 1 for plain backward())
__global__ void loss_map_grad_kernel(const float* __restrict__ pred, const float* __restrict__ d, const float* __restrict__ v,
                                     const float* __restrict__ img, float* __restrict__ gpred, const LossScalars* __restrict__ ls,
                                     int N, int H, int W, float cap, int do_clamp, float w_sd, float w_sm, float gscale) {
    PDL_SYNC();
    const long long HW = (long long)H * W;
    long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= N * HW) return;
    int n = idx / HW;
    long long i = idx - n * HW;
    int x = i % W, y = i / W;
    const float* pn = pred + n * HW; const float* in = img + n * HW * 3;
    float p0 = pn[i];
    float dd = d[idx];
    if (do_clamp) dd = fminf(fmaxf(dd, 0.f), cap);
    float diff = p0 - dd;
    float sgn = diff > 0.f ? 1.f : (diff < 0.f ? -1.f : 0.f);
    float g = w_sd * v[idx] * sgn * ls->inv_count[n] / (float)N;
    float cx = w_sm / ((float)N * H * (W - 1)), cy = w_sm / ((float)N * (H - 1) * W);
    if (x < W - 1) {
        float e = fabsf(in[i] - in[i + 1]) + fabsf(in[HW + i] - in[HW + i + 1]) + fabsf(in[2 * HW + i] - in[2 * HW + i + 1]);
        float dx = p0 - pn[i + 1];
        g += cx * expf(-e / 3.f) * (dx > 0.f ? 1.f : (dx < 0.f ? -1.f : 0.f));
    }
    if (x > 0) {
        float e = fabsf(in[i - 1] - in[i]) + fabsf(in[HW + i - 1] - in[HW + i]) + fabsf(in[2 * HW + i - 1] - in[2 * HW + i]);
        float dx = pn[i - 1] - p0;
        g -= cx * expf(-e / 3.f) * (dx > 0.f ? 1.f : (dx < 0.f ? -1.f : 0.f));
    }
    if (y < H - 1) {
        float e = fabsf(in[i] - in[i + W]) + fabsf(in[HW + i] - in[HW + i + W]) + fabsf(in[2 * HW + i] - in[2 * HW + i + W]);
        float dy = p0 - pn[i + W];
        g += cy * expf(-e / 3.f) * (dy > 0.f ? 1.f : (dy < 0.f ? -1.f : 0.f));
    }
    if (y > 0) {
        float e = fabsf(in[i - W] - in[i]) + fabsf(in[HW + i - W] - in[HW + i]) + fabsf(in[2 * HW + i - W] - in[2 * HW + i]);
        float dy = pn[i - W] - p0;
        g -= cy * expf(-e / 3.f) * (dy > 0.f ? 1.f : (dy < 0.f ? -1.f : 0.f));
    }
    gpred[idx] = g * gscale;
}

// d loss / d ref = w_eff * (-2/R) * (ehat - cos*rhat) / max(|r|, eps)
// wrt_emb = 0: gradient with respect to `ref` (the loss is symmetric in its two arguments: wrt_emb = 1 swaps their roles and writes the
// gradient with respect to `emb` -- needed when the heads' BatchNorm affine pairs are adapted, NLSPN 'meta_bn' after convert_syncbn)
__global__ void __launch_bounds__(256) loss_cos_grad_kernel(const bf16* __restrict__ emb, const bf16* __restrict__ ref, const float* __restrict__ rowstat,
                                                            const LossScalars* __restrict__ ls, bf16* __restrict__ gref, long long R, int D, float gscale,
                                                            int wrt_emb = 0) {
    PDL_SYNC();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const float coef = ls->w_cos_eff * (-2.f / (float)R) * gscale;
    for (long long r = (long long)blockIdx.x * 8 + warp; r < R; r += (long long)gridDim.x * 8) {
        float dot = rowstat[r * 3], ne = fmaxf(sqrtf(rowstat[r * 3 + 1]), 1e-12f), nr = fmaxf(sqrtf(rowstat[r * 3 + 2]), 1e-12f);
        const bf16* e = emb + (size_t)r * D; const bf16* f = ref + (size_t)r * D;
        if (wrt_emb) { const float t = ne; ne = nr; nr = t; const bf16* tp = e; e = f; f = tp; }
        float cs = dot / (ne * nr);
        float a = coef / (ne * nr), b = coef * cs / (nr * nr);
        bf16* o = gref + (size_t)r * D;
        for (int c = lane * 8; c < D; c += 256) {
            uint4 ev = __ldg(reinterpret_cast<const uint4*>(e + c)), fv = __ldg(reinterpret_cast<const uint4*>(f + c));
            const uint32_t *ue = reinterpret_cast<const uint32_t*>(&ev), *uf = reinterpret_cast<const uint32_t*>(&fv);
            uint4 ov; uint32_t* uo = reinterpret_cast<uint32_t*>(&ov);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float2 x = unpack_bf162(ue[j]), y = unpack_bf162(uf[j]);
                uo[j] = pack_bf162(a * x.x - b * y.x, a * x.y - b * y.y);
            }
            *reinterpret_cast<uint4*>(o + c) = ov;
        }
    }
}

// -------------------------------------------------------------------------------------------------
// f3: losses of the source-domain preparation stages
//   stage 1 (src/msg_chn_model_adapt.py:224-264, src/loss_utils.py:266-287): gt' = clamp(gt, 0, max_predict), v = [gt' > 0],
//            loss = mean_n( sum v (pred - gt')^2 / sum v );   partial layout (doubles): [N][nblk][4] = {sum v (pred-gt')^2, sum v, -, -}
//   stage 2 (src/external_model_adapt.py:524-540): mean_r(2 - 2 cos(emb_r, ref_r)) -- loss_cos_rows_kernel + this finalize, no gate
// -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(LOSS_BLOCK) l2_loss_reduce_kernel(const float* __restrict__ pred, const float* __restrict__ gt,
                                                                    double* __restrict__ partial, int HW, float max_predict) {
    PDL_SYNC();
    __shared__ double sh[32];
    const int n = blockIdx.y;
    const float* pn = pred + (size_t)n * HW; const float* gn = gt + (size_t)n * HW;
    double s_l = 0.0, s_v = 0.0;
    for (int i = blockIdx.x * LOSS_BLOCK + threadIdx.x; i < HW; i += gridDim.x * LOSS_BLOCK) {
        const float g = fminf(fmaxf(gn[i], 0.f), max_predict);
        if (g > 0.f) {
            const float d = pn[i] - g;
            s_l += (double)(d * d);
            s_v += 1.0;
        }
    }
    double r0 = block_sum_d(s_l, sh), r1 = block_sum_d(s_v, sh);
    if (threadIdx.x == 0) {
        double* o = partial + ((size_t)n * gridDim.x + blockIdx.x) * 4;
        o[0] = r0; o[1] = r1; o[2] = 0.0; o[3] = 0.0;
    }
}

__global__ void __launch_bounds__(256) l2_loss_finalize_kernel(const double* __restrict__ partial, int nblk, int N, LossScalars* out) {
    PDL_SYNC();
    __shared__ double sh[32];
    double tot = 0.0;
    for (int n = 0; n < N; ++n) {
        double a = 0.0, b = 0.0;
        for (int k = threadIdx.x; k < nblk; k += 256) {
            const double* p = partial + ((size_t)n * nblk + k) * 4;
            a += p[0]; b += p[1];
        }
        a = block_sum_d(a, sh); b = block_sum_d(b, sh);
        if (threadIdx.x == 0) {
            const float fa = (float)a, fb = (float)b;
            tot += (double)(fa / fb);                   // no epsilon, as in the reference
            if (n < 64) out->inv_count[n] = 1.f / fb;
        }
    }
    if (threadIdx.x != 0) return;
    out->loss = (float)(tot / N);
    out->loss_sparse_depth = 0.f; out->loss_smooth = 0.f; out->loss_cos = 0.f; out->w_cos_eff = 0.f;
}

// d loss / d pred = gscale * 2 v (pred - gt') / (N sum_n v)
__global__ void l2_loss_grad_kernel(const float* __restrict__ pred, const float* __restrict__ gt, float* __restrict__ gpred,
                                    const LossScalars* __restrict__ ls, int N, int HW, float max_predict, float gscale) {
    PDL_SYNC();
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)N * HW) return;
    const int n = (int)(idx / HW);
    const float g = fminf(fmaxf(gt[idx], 0.f), max_predict);
    float r = 0.f;
    if (g > 0.f) r = gscale * 2.f * (pred[idx] - g) * ls->inv_count[n] / (float)N;
    gpred[idx] = r;
}

__global__ void __launch_bounds__(256) cos_loss_finalize_kernel(const double* __restrict__ cos_partial, int cos_blocks, long long R, LossScalars* out) {
    PDL_SYNC();
    __shared__ double sh[32];
    double c = 0.0;
    for (int k = threadIdx.x; k < cos_blocks; k += 256) c += cos_partial[k];
    c = block_sum_d(c, sh);
    if (threadIdx.x != 0) return;
    const float l_cos = R > 0 ? (float)(c / (double)R) : 0.f;
    out->loss = l_cos; out->loss_cos = l_cos; out->loss_sparse_depth = 0.f; out->loss_smooth = 0.f;
    out->w_cos_eff = 1.f;                               // loss_cos_grad_kernel scales with it
}

// EMA copy of the projector (network_exp_msg_chn_adapt.py:701-703): t = t * tau + s * (1 - tau), two products and one sum like the
// reference's tensor expression (no fused multiply-add, so the result is bit-identical)
struct EmaParams { float* t[8]; const float* s[8]; long long n[8]; int count; float tau, one_minus_tau; };
__global__ void __launch_bounds__(256) ema_update_kernel(const EmaParams p) {
    PDL_SYNC();
    const int k = blockIdx.y;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n[k]) return;
    p.t[k][i] = __fadd_rn(__fmul_rn(p.t[k][i], p.tau), __fmul_rn(p.s[k][i], p.one_minus_tau));
}

// -------------------------------------------------------------------------------------------------
// a17: fused multi-tensor Adam (torch.optim.Adam, amsgrad=False; src/tta_main.py:341-346,633).
// One launch over a chunk table covering every adapted tensor; hyper-parameters and the step count
// live on the device so the launch is CUDA-graph friendly.
// -------------------------------------------------------------------------------------------------
struct AdamHyper { float lr, beta1, beta2, eps, weight_decay, one_minus_beta1, one_minus_beta2; int step; double beta1_d, beta2_d, lr_d; };
struct AdamChunk { float* p; const float* g; float* m; float* v; int n; };
#define ADAM_CHUNK 2048
#define ADAM_MAX_CHUNKS 1024

// torch's single-tensor formulation: exp_avg.lerp_(g, 1-b1); exp_avg_sq.mul_(b2).addcmul_(g, g, value=1-b2);
// denom = sqrt(v)/sqrt(bc2) + eps; p.addcdiv_(m, denom, value=-lr/bc1)   (1-b computed in double, as torch does)
__device__ __forceinline__ void adam_update(float& p, float g, float& m, float& v, float b2, float omb1, float omb2, float eps, float wd,
                                            float step_size, float bc2_sqrt) {
    if (wd != 0.f) g = fmaf(wd, p, g);
    m = fmaf(omb1, g - m, m);
    v = b2 * v + omb2 * g * g;
    float denom = sqrtf(v) / bc2_sqrt + eps;
    p = p - step_size * (m / denom);
}

__global__ void __launch_bounds__(256) adam_kernel(const AdamChunk* __restrict__ chunks, const AdamHyper* __restrict__ hy) {
    PDL_SYNC();
    const AdamChunk ck = chunks[blockIdx.x];
    const int t = hy->step + 1;
    const double bc1 = 1.0 - pow(hy->beta1_d, (double)t);
    const double bc2 = 1.0 - pow(hy->beta2_d, (double)t);
    const float step_size = (float)(hy->lr_d / bc1);
    const float bc2_sqrt = (float)sqrt(bc2);
    const float b2 = hy->beta2, omb1 = hy->one_minus_beta1, omb2 = hy->one_minus_beta2, eps = hy->eps, wd = hy->weight_decay;
    for (int i = threadIdx.x; i < ck.n; i += 256) {
        float p = ck.p[i], m = ck.m[i], v = ck.v[i];
        adam_update(p, ck.g[i], m, v, b2, omb1, omb2, eps, wd, step_size, bc2_sqrt);
        ck.p[i] = p; ck.m[i] = m; ck.v[i] = v;
    }
}
__global__ void adam_advance_kernel(AdamHyper* hy) {
    PDL_SYNC(); hy->step += 1; }

// end of a step: the next step's exchanges use the next tag
__global__ void comm_advance_kernel(PeerComm c) {
    PDL_SYNC();
    if (threadIdx.x == 0 && blockIdx.x == 0) *reinterpret_cast<volatile uint32_t*>(c.base[c.rank] + comm_epoch_off()) += 1u;
}

// Shared-model mode: mean all-reduce of the adapted-parameter gradients FUSED with the Adam update, one launch, one-shot over NVLink
// peer memory.  Block = one chunk of the chunk table (as adam_kernel): it copies its part of the local gradient into the rank's slot, the
// ranks rendezvous (peer_comm.cuh), and every block then sums the W copies of its chunk in rank order (bit-identical on all ranks),
// scales by 1/W, writes the averaged gradient back (what DDP leaves in .grad) and applies Adam.  g_base: start of the flat gradient
// buffer the chunk pointers point into.
__global__ void __launch_bounds__(256) adam_allreduce_kernel(const AdamChunk* __restrict__ chunks, const AdamHyper* __restrict__ hy, const PeerComm comm,
                                                             int xid, const float* __restrict__ g_base) {
    PDL_SYNC();
    const AdamChunk ck = chunks[blockIdx.x];
    const uint32_t tag = comm_tag(comm);
    const size_t off = comm_grad_off((int)(tag & 1u), comm.grad_floats), idx0 = (size_t)(ck.g - g_base);
    float* mine = reinterpret_cast<float*>(comm.base[comm.rank] + off) + idx0;
    for (int i = threadIdx.x; i < ck.n; i += 256) mine[i] = ck.g[i];
    comm_publish_and_wait(comm, xid, tag);
    const int t = hy->step + 1;
    const double bc1 = 1.0 - pow(hy->beta1_d, (double)t);
    const double bc2 = 1.0 - pow(hy->beta2_d, (double)t);
    const float step_size = (float)(hy->lr_d / bc1);
    const float bc2_sqrt = (float)sqrt(bc2);
    const float b2 = hy->beta2, omb1 = hy->one_minus_beta1, omb2 = hy->one_minus_beta2, eps = hy->eps, wd = hy->weight_decay;
    const float inv_w = 1.f / (float)comm.world;
    for (int i = threadIdx.x; i < ck.n; i += 256) {
        float g = 0.f;
        for (int r = 0; r < comm.world; ++r) g += ld_volatile_f32(reinterpret_cast<const float*>(comm.base[r] + off) + idx0 + i);
        g *= inv_w;
        const_cast<float*>(ck.g)[i] = g;
        float p = ck.p[i], m = ck.m[i], v = ck.v[i];
        adam_update(p, g, m, v, b2, omb1, omb2, eps, wd, step_size, bc2_sqrt);
        ck.p[i] = p; ck.m[i] = m; ck.v[i] = v;
    }
}

// -------------------------------------------------------------------------------------------------
// weight packing: fp32 parameter -> bf16 [tap][O][I] operand of conv3x3_mma
//   dst[(tap*O + o)*I + i] = src[o*s_o + i*s_i + tap']   tap' = flip ? 8 - tap : tap
// -------------------------------------------------------------------------------------------------
__global__ void pack_conv_weight_kernel(const float* __restrict__ src, bf16* __restrict__ dst, int O, int I, int s_o, int s_i, int flip) {
    PDL_SYNC();
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= 9 * O * I) return;
    int i = idx % I;
    int o = (idx / I) % O;
    int tap = idx / (I * O);
    int ts = flip ? 8 - tap : tap;
    dst[idx] = __float2bfloat16_rn(src[(size_t)o * s_o + (size_t)i * s_i + ts]);
}
// generic 2-D cast with optional transpose: dst[r][c] = src[r*s_r + c*s_c]
__global__ void pack_matrix_kernel(const float* __restrict__ src, bf16* __restrict__ dst, int rows, int cols, int s_r, int s_c) {
    PDL_SYNC();
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= rows * cols) return;
    int c = idx % cols, r = idx / cols;
    dst[idx] = __float2bfloat16_rn(src[(size_t)r * s_r + (size_t)c * s_c]);
}
// head conv weights: dst[tap][c] = src[c*s_c + tap'] (fp32)
// Two Linear layers with nothing between them (proj.3 then pred.0: network_exp_msg_chn_adapt.py:1089-1098, emb = pred(proj(z))) are ONE
// Linear layer: W = W2 W1, b = W2 b1 + b2.  Computed in fp32 at pack time (both layers are frozen), rounded to bf16 once.
// out[o][i] = sum_k w2[o][k] w1[k][i];  launch: grid (cdiv(n_in, 256), n_out), block 256
__global__ void fuse_linear_kernel(const float* __restrict__ w2, const float* __restrict__ b2, const float* __restrict__ w1,
                                   const float* __restrict__ b1, bf16* __restrict__ w_out, float* __restrict__ b_out, int n_out, int n_mid, int n_in) {
    PDL_SYNC();
    const int i = blockIdx.x * blockDim.x + threadIdx.x, o = blockIdx.y;
    if (i >= n_in) return;
    const float* r2 = w2 + (size_t)o * n_mid;
    float acc = 0.f;
    for (int k = 0; k < n_mid; ++k) acc = fmaf(__ldg(r2 + k), __ldg(w1 + (size_t)k * n_in + i), acc);
    w_out[(size_t)o * n_in + i] = __float2bfloat16_rn(acc);
    if (i == 0) {
        float bb = b2[o];
        for (int k = 0; k < n_mid; ++k) bb = fmaf(r2[k], b1[k], bb);
        b_out[o] = bb;
    }
}

__global__ void pack_head_weight_kernel(const float* __restrict__ src, float* __restrict__ dst, int s_c, int flip) {
    PDL_SYNC();
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= 288) return;
    int c = idx & 31, tap = idx >> 5;
    dst[idx] = src[(size_t)c * s_c + (flip ? 8 - tap : tap)];
}
// stem-shaped fp32 weights for the 1->32 data gradient of prdct.3: dst[c][tap] = src[c*9 + (8 - tap)]
__global__ void pack_flip9_kernel(const float* __restrict__ src, float* __restrict__ dst, int n) {
    PDL_SYNC();
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n * 9) return;
    int tap = idx % 9, c = idx / 9;
    dst[idx] = src[(size_t)c * 9 + (8 - tap)];
}

// misc
__global__ void fill_kernel(float* p, float v, long long n) {
    PDL_SYNC();
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}
__global__ void bf16_to_f32_kernel(const bf16* __restrict__ s, float* __restrict__ d, long long n) {
    PDL_SYNC();
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) d[i] = __bfloat162float(s[i]);
}
__global__ void f32_to_bf16_kernel(const float* __restrict__ s, bf16* __restrict__ d, long long n) {
    PDL_SYNC();
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) d[i] = __float2bfloat16_rn(s[i]);
}

}  // namespace ptta
