// Eval-time hole filling of the NLSPN prediction: skimage.restoration.inpaint_biharmonic (0.18 / 0.19) of every pixel that is
// exactly 0, per sample, solved exactly in fp64 on the device (src/nlspn_model_adapt.py:124-127 -> src/data_utils.py:327-354).
//
// One equation per hole p: sum_q c_p(q) u(q) = 0 with c_p = laplace(laplace(delta_p)) (scipy.ndimage, mode 'reflect') on the 5x5
// window around p clipped to the image; known pixels go to the right-hand side.  The operator is (Dy + Dx)^2 with 1-D second
// differences whose reflect rule only depends on how far p is from each border (0, 1, >= 2), so c_p is built from three 1-D
// profiles per axis (InpaintStencil, made once on the host).  The matrix is symmetric positive definite, borders included.
//
// Holes couple only within stencil reach (offsets (0,+-1), (+-1,0), (+-1,+-1), (0,+-2), (+-2,0)), so the system splits into the
// connected components of that adjacency; solving them one by one equals skimage's per-region and global solves.
// Per component: cut it into slabs of two grid lines across the axis that minimises sum b_k^3 (b_k unknowns in slab k).  The
// stencil reaches two lines, so the matrix is block tridiagonal; each slab is eliminated as one dense row block
// [A_kk | A_k,k+1 | r_k] (upper block Cholesky: the row block becomes [U_kk | U_k,k+1 | y_k]), then a backward substitution.
//
// Launches (fixed, independent of the number of holes or components): plan = memset + scan; solve = memset + init + union +
// flatten + stats + solve.  The solve kernel is persistent: its CTAs take components from a device work list.
#pragma once
#include "common.cuh"

namespace ptta {

constexpr int INPAINT_SOLVE_CTAS = 296;
constexpr int INPAINT_THREADS = 256;

// p[class][order][offset + 2]: 1-D profile of delta (order 0), D delta (1) and D D delta (2) on a window clipped to the image;
// class = 3 * min(dist to low border, 2) + min(dist to high border, 2); zero outside the window
struct InpaintStencil { signed char p[9][3][5]; };

// order-preserving float -> uint32 key (atomicMin / atomicMax on the bit pattern)
__device__ __forceinline__ unsigned int inpaint_key(float f) {
    const unsigned int u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float inpaint_unkey(unsigned int k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// summary[4 s + {0, 1, 2}] = {holes, ~key(min known), key(max known)} of sample s (zeroed by the caller)
__global__ void __launch_bounds__(256) inpaint_scan_kernel(const float* __restrict__ depth, long long hw, unsigned int* __restrict__ summary) {
    PDL_SYNC();
    const int s = blockIdx.y;
    const float* d = depth + (long long)s * hw;
    unsigned int holes = 0, nlo = 0, hi = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < hw; i += (long long)gridDim.x * blockDim.x) {
        const float v = d[i];
        if (v == 0.f) {
            ++holes;
        } else {
            const unsigned int k = inpaint_key(v);
            nlo = max(nlo, ~k);
            hi = max(hi, k);
        }
    }
    holes = __reduce_add_sync(0xffffffffu, holes);
    nlo = __reduce_max_sync(0xffffffffu, nlo);
    hi = __reduce_max_sync(0xffffffffu, hi);
    if ((threadIdx.x & 31) == 0) {
        if (holes) atomicAdd(&summary[4 * s], holes);
        if (nlo) atomicMax(&summary[4 * s + 1], nlo);
        if (hi) atomicMax(&summary[4 * s + 2], hi);
    }
}

__device__ __forceinline__ int uf_find(const int* parent, int a) {
    int p = __ldcg(parent + a);
    while (p != a) { a = p; p = __ldcg(parent + a); }
    return a;
}

// union by smaller index: every root is the smallest pixel index of its set
__device__ __forceinline__ void uf_union(int* parent, int a, int b) {
    while (true) {
        a = uf_find(parent, a);
        b = uf_find(parent, b);
        if (a == b) return;
        if (a < b) { const int t = a; a = b; b = t; }
        const int old = atomicMin(parent + a, b);
        if (old == a) return;
        a = old;
    }
}

// label[p] = p for a hole, -1 otherwise
__global__ void __launch_bounds__(256) inpaint_init_kernel(const float* __restrict__ depth, long long total, int* __restrict__ label) {
    PDL_SYNC();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x)
        label[i] = depth[i] == 0.f ? (int)i : -1;
}

__global__ void __launch_bounds__(256) inpaint_union_kernel(int* label, long long total, int h, int w) {
    PDL_SYNC();
    const int dy[6] = {0, 0, 1, 1, 1, 2}, dx[6] = {1, 2, -1, 0, 1, 0};     // the forward half of the stencil-reach adjacency
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        if (__ldcg(label + i) < 0) continue;
        const int x = (int)(i % w), y = (int)((i / w) % h);
#pragma unroll
        for (int t = 0; t < 6; ++t) {
            const int yy = y + dy[t], xx = x + dx[t];
            if (yy >= h || xx < 0 || xx >= w) continue;
            const long long q = i + (long long)dy[t] * w + dx[t];
            if (__ldcg(label + q) >= 0) uf_union(label, (int)i, (int)q);
        }
    }
}

// comp[c] = {root, count, y0, y1, x0, x1}; counters[0] = number of components
__global__ void __launch_bounds__(256) inpaint_flatten_kernel(int* label, long long total, int* __restrict__ index, int* __restrict__ comp,
                                                              int* __restrict__ counters) {
    PDL_SYNC();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        if (__ldcg(label + i) < 0) continue;
        const int r = uf_find(label, (int)i);
        if (r == (int)i) {
            const int c = atomicAdd(&counters[0], 1);
            int* cr = comp + 6 * (long long)c;
            cr[0] = r; cr[1] = 0; cr[2] = 0x7fffffff; cr[3] = -1; cr[4] = 0x7fffffff; cr[5] = -1;
            index[i] = c;
        } else {
            label[i] = r;
        }
    }
}

__global__ void __launch_bounds__(256) inpaint_stats_kernel(const int* __restrict__ label, long long total, int h, int w,
                                                            const int* __restrict__ index, int* __restrict__ comp) {
    PDL_SYNC();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int r = label[i];
        if (r < 0) continue;
        int* cr = comp + 6 * (long long)index[r];
        const int x = (int)(i % w), y = (int)((i / w) % h);
        atomicAdd(&cr[1], 1);
        atomicMin(&cr[2], y); atomicMax(&cr[3], y);
        atomicMin(&cr[4], x); atomicMax(&cr[5], x);
    }
}

struct InpaintSolveArgs {
    float* depth;
    const unsigned int* summary;
    const int* label;
    int* index;                 // pixel -> unknown index within its component (overwrites the flatten kernel's root -> component id)
    const int* comp;
    int* counters;              // [0] components, [1] work ticket
    unsigned long long* bump;   // arena doubles handed out
    unsigned long long arena_doubles;
    double* arena;
    int* status;                // 1: non-positive pivot, 2: workspace too small
    int* scratch;               // per CTA: histY[sy_max], histX[sx_max] (padded to even), off[s_max + 2 & ~1], foff[s_max + 1] (long long)
    long long scratch_ints;
    int h, w, sy_max, sx_max, s_max;
    InpaintStencil st;
};

__device__ __forceinline__ int inpaint_class(int pos, int len) { return 3 * min(pos, 2) + min(len - 1 - pos, 2); }

// block-wide exclusive prefix of a 0/1 flag in thread order; returns the prefix, *total gets the block's count
__device__ __forceinline__ int block_prefix(bool flag, int* sh_warp, int* total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const unsigned int b = __ballot_sync(0xffffffffu, flag);
    __syncthreads();
    if (lane == 0) sh_warp[wid] = __popc(b);
    __syncthreads();
    int before = 0, all = 0;
    for (int k = 0; k < INPAINT_THREADS / 32; ++k) {
        before += k < wid ? sh_warp[k] : 0;
        all += sh_warp[k];
    }
    *total = all;
    return before + __popc(b & ((1u << lane) - 1u));
}

__global__ void __launch_bounds__(INPAINT_THREADS, 1) inpaint_solve_kernel(const InpaintSolveArgs a) {
    PDL_SYNC();
    __shared__ int sh_ticket, sh_axis, sh_bad;
    __shared__ unsigned long long sh_base;
    __shared__ int sh_warp[INPAINT_THREADS / 32];
    __shared__ double sh_red[32];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int h = a.h, w = a.w;
    const long long hw = (long long)h * w;
    int* histY = a.scratch + (long long)blockIdx.x * a.scratch_ints;
    int* histX = histY + a.sy_max;
    int* off = histY + ((a.sy_max + a.sx_max + 1) & ~1);
    long long* foff = reinterpret_cast<long long*>(off + ((a.s_max + 2) & ~1));

    while (true) {
        if (tid == 0) sh_ticket = atomicAdd(&a.counters[1], 1);
        __syncthreads();
        const int c = sh_ticket;
        if (c >= __ldcg(&a.counters[0])) break;
        const int* cr = a.comp + 6 * (long long)c;
        const int root = cr[0], n = cr[1], y0 = cr[2], y1 = cr[3], x0 = cr[4], x1 = cr[5];
        const int s = (int)(root / hw);
        const long long base_px = (long long)s * hw;
        const float lo = inpaint_unkey(~a.summary[4 * s + 1]), hi = inpaint_unkey(a.summary[4 * s + 2]);
        const int bh = y1 - y0 + 1, bw = x1 - x0 + 1, sy = (bh + 1) / 2, sx = (bw + 1) / 2;

        // slab populations along both axes
        for (int k = tid; k < sy; k += INPAINT_THREADS) histY[k] = 0;
        for (int k = tid; k < sx; k += INPAINT_THREADS) histX[k] = 0;
        __syncthreads();
        for (long long t = tid; t < (long long)bh * bw; t += INPAINT_THREADS) {
            const int y = y0 + (int)(t / bw), x = x0 + (int)(t % bw);
            if (__ldcg(a.label + base_px + (long long)y * w + x) == root) {
                atomicAdd(&histY[(y - y0) >> 1], 1);
                atomicAdd(&histX[(x - x0) >> 1], 1);
            }
        }
        __syncthreads();
        double cy = 0.0, cx = 0.0;
        for (int k = tid; k < sy; k += INPAINT_THREADS) { const double b = __ldcg(&histY[k]); cy += b * b * b; }
        for (int k = tid; k < sx; k += INPAINT_THREADS) { const double b = __ldcg(&histX[k]); cx += b * b * b; }
        cy = block_sum_d(cy, sh_red);
        cx = block_sum_d(cx, sh_red);
        if (tid == 0) sh_axis = cy <= cx ? 0 : 1;     // 0: slabs are pairs of rows
        __syncthreads();
        const int axis = sh_axis;
        const int S = axis == 0 ? sy : sx;
        const int* hist = axis == 0 ? histY : histX;
        if (tid == 0) {
            long long f = 0;
            int o = 0;
            for (int k = 0; k < S; ++k) {
                const int b = __ldcg(&hist[k]), bn = k + 1 < S ? __ldcg(&hist[k + 1]) : 0;
                off[k] = o; foff[k] = f;
                o += b;
                f += (long long)b * (b + bn + 1);
            }
            off[S] = o; foff[S] = f;
            const unsigned long long need = 2ull * n + (unsigned long long)f;
            const unsigned long long base = atomicAdd(a.bump, need);
            sh_bad = base + need > a.arena_doubles ? 2 : 0;
            sh_base = base;
        }
        __syncthreads();
        if (sh_bad) {                                   // cannot happen when the workspace has ptta_inpaint_workspace_bytes
            if (tid == 0) atomicMax(a.status, 2);
            continue;
        }
        int* pix = reinterpret_cast<int*>(a.arena + sh_base);          // n ints in the first n doubles
        double* xv = a.arena + sh_base + n;
        double* M = a.arena + sh_base + 2 * (long long)n;
        const int line0 = axis == 0 ? y0 : x0, len = axis == 0 ? bw : bh, pos0 = axis == 0 ? x0 : y0;

        // number the unknowns slab by slab (within a slab: line-major, then along the line)
        for (int k = 0; k < S; ++k) {
            int run = off[k];
            const int cells = 2 * len;
            for (int t0 = 0; t0 < cells; t0 += INPAINT_THREADS) {
                const int t = t0 + tid;
                const int line = line0 + 2 * k + t / len, pos = pos0 + t % len;
                long long p = -1;
                if (t < cells && line <= (axis == 0 ? y1 : x1)) {
                    const long long q = base_px + (axis == 0 ? (long long)line * w + pos : (long long)pos * w + line);
                    if (__ldcg(a.label + q) == root) p = q;
                }
                int total;
                const int pre = block_prefix(p >= 0, sh_warp, &total);
                if (p >= 0) { pix[run + pre] = (int)p; a.index[p] = run + pre; }
                run += total;
            }
        }
        if (tid == 0) sh_bad = 0;
        __syncthreads();

        // block Cholesky, slab by slab: row block k = [A_kk | A_k,k+1 | r_k], row stride W = b + bn + 1
        for (int k = 0; k < S; ++k) {
            const int ok = off[k], b = off[k + 1] - ok, bn = k + 1 < S ? off[k + 2] - off[k + 1] : 0;
            const int W = b + bn + 1;
            double* Mk = M + foff[k];
            for (long long t = tid; t < (long long)b * W; t += INPAINT_THREADS) Mk[t] = 0.0;
            __syncthreads();
            for (int i = tid; i < b; i += INPAINT_THREADS) {
                const long long p = pix[ok + i];
                const int y = (int)((p - base_px) / w), x = (int)((p - base_px) % w);
                const int ccy = inpaint_class(y, h), ccx = inpaint_class(x, w);
                double rhs = 0.0;
                for (int ddy = -2; ddy <= 2; ++ddy) {
                    const int py0 = a.st.p[ccy][0][ddy + 2], py1 = a.st.p[ccy][1][ddy + 2], py2 = a.st.p[ccy][2][ddy + 2];
                    if (!(py0 | py1 | py2)) continue;
                    for (int ddx = -2; ddx <= 2; ++ddx) {
                        const int coef = py2 * a.st.p[ccx][0][ddx + 2] + 2 * py1 * a.st.p[ccx][1][ddx + 2] + py0 * a.st.p[ccx][2][ddx + 2];
                        if (coef == 0) continue;
                        const long long q = p + (long long)ddy * w + ddx;
                        if (__ldcg(a.label + q) >= 0) {               // a hole within reach: an unknown of this component
                            const int j = __ldcg(a.index + q);
                            const int ks = ((axis == 0 ? y + ddy : x + ddx) - line0) >> 1;
                            if (ks == k) Mk[(long long)i * W + (j - ok)] = coef;
                            else if (ks == k + 1) Mk[(long long)i * W + b + (j - off[k + 1])] = coef;
                        } else {
                            rhs -= coef * (double)a.depth[q];
                        }
                    }
                }
                Mk[(long long)i * W + W - 1] = rhs;
            }
            __syncthreads();
            if (k > 0) {                                   // Schur complement of the previous slab: [A_kk | r_k] -= U_k-1,k^T [U_k-1,k | y_k-1]
                const int bp = off[k] - off[k - 1], Wp = bp + W - bn;
                const double* Mp = M + foff[k - 1];
                for (int i = wid; i < b; i += INPAINT_THREADS / 32) {
                    for (int l = i + lane; l <= b; l += 32) {
                        const int cl = l < b ? l : W - 1;
                        double acc = 0.0;
                        for (int m = 0; m < bp; ++m) acc += Mp[(long long)m * Wp + bp + i] * Mp[(long long)m * Wp + bp + l];
                        Mk[(long long)i * W + cl] -= acc;
                    }
                }
                __syncthreads();
            }
            for (int j = 0; j < b; ++j) {                  // right-looking elimination of the row block (unscaled rows)
                const double* rj = Mk + (long long)j * W;
                const double piv = rj[j];
                if (!(piv > 0.0)) { if (tid == 0) sh_bad = 1; }
                const double inv = 1.0 / piv;
                for (int i = j + 1 + wid; i < b; i += INPAINT_THREADS / 32) {
                    double* ri = Mk + (long long)i * W;
                    const double f = rj[i] * inv;
                    for (int l = i + lane; l < W; l += 32) ri[l] -= f * rj[l];
                }
                __syncthreads();
            }
            for (int j = wid; j < b; j += INPAINT_THREADS / 32) {   // scale row j by 1 / sqrt(pivot): U rows
                double* rj = Mk + (long long)j * W;
                const double sc = 1.0 / sqrt(rj[j]);
                __syncwarp();
                for (int l = j + lane; l < W; l += 32) rj[l] *= sc;
            }
            __syncthreads();
        }

        // backward substitution: U_kk x_k = y_k - U_k,k+1 x_k+1
        for (int k = S - 1; k >= 0; --k) {
            const int ok = off[k], b = off[k + 1] - ok, bn = k + 1 < S ? off[k + 2] - off[k + 1] : 0;
            const int W = b + bn + 1;
            const double* Mk = M + foff[k];
            for (int i = wid; i < b; i += INPAINT_THREADS / 32) {
                double acc = 0.0;
                for (int l = lane; l < bn; l += 32) acc += Mk[(long long)i * W + b + l] * xv[off[k + 1] + l];
                acc = warp_sum_d(acc);
                if (lane == 0) xv[ok + i] = Mk[(long long)i * W + W - 1] - acc;
            }
            __syncthreads();
            if (wid == 0) {
                for (int j = b - 1; j >= 0; --j) {
                    const double xj = xv[ok + j] / Mk[(long long)j * W + j];
                    __syncwarp();
                    if (lane == 0) xv[ok + j] = xj;
                    for (int i = lane; i < j; i += 32) xv[ok + i] -= Mk[(long long)i * W + j] * xj;
                    __syncwarp();
                }
            }
            __syncthreads();
        }

        // clip to the sample's known range (np.clip keeps NaN), store fp32 in place; a failed factorisation leaves NaN
        const bool bad = sh_bad != 0;
        for (int i = tid; i < n; i += INPAINT_THREADS) {
            double v = xv[i];
            v = v < (double)lo ? (double)lo : (v > (double)hi ? (double)hi : v);
            a.depth[pix[i]] = bad ? __int_as_float(0x7fc00000) : (float)v;
        }
        if (bad && tid == 0) atomicMax(a.status, 1);
        __syncthreads();
    }
}

// ---- host side ----------------------------------------------------------------------------------------------------------------
static InpaintStencil inpaint_make_stencil() {
    InpaintStencil st = {};
    for (int lo = 0; lo < 3; ++lo)
        for (int hi = 0; hi < 3; ++hi) {
            const int L = lo + hi + 1;
            int v[3][5] = {};
            v[0][lo] = 1;
            for (int o = 1; o < 3; ++o)                    // scipy.ndimage.correlate1d([1, -2, 1], mode='reflect') on the clipped window
                for (int i = 0; i < L; ++i)
                    v[o][i] = v[o - 1][i > 0 ? i - 1 : 0] - 2 * v[o - 1][i] + v[o - 1][i + 1 < L ? i + 1 : L - 1];
            for (int o = 0; o < 3; ++o)
                for (int i = 0; i < L; ++i) st.p[3 * lo + hi][o][i - lo + 2] = (signed char)v[o][i];
        }
    return st;
}

struct InpaintLayout {
    size_t label, index, comp, counters, scratch, arena, total;
    long long scratch_ints;
    int sy_max, sx_max, s_max;
};

static InpaintLayout inpaint_layout(int n, int h, int w, unsigned long long arena_doubles) {
    InpaintLayout L;
    const size_t px = (size_t)n * h * w;
    L.sy_max = (h + 1) / 2; L.sx_max = (w + 1) / 2;
    L.s_max = L.sy_max > L.sx_max ? L.sy_max : L.sx_max;
    L.scratch_ints = (((long long)L.sy_max + L.sx_max + 1) / 2 * 2 + ((L.s_max + 2) & ~1) + 2LL * (L.s_max + 1) + 63) & ~63LL;
    auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
    L.label = 0;
    L.index = up(L.label + px * 4);
    L.comp = up(L.index + px * 4);
    L.counters = up(L.comp + px * 24);
    L.scratch = up(L.counters + 64);
    L.arena = up(L.scratch + (size_t)INPAINT_SOLVE_CTAS * L.scratch_ints * 4);
    L.total = L.arena + arena_doubles * 8;
    return L;
}

// arena doubles a component of n unknowns takes: pix + x (2n) + sum_k b_k (b_k + b_k+1 + 1) <= 3n + 2 sum_k b_k^2.  On the chosen axis
// sum b^3 <= n (2m)^2 with m = min(h, w) (either axis has b_k <= 2 x its line length), so by Cauchy-Schwarz sum b^2 <= sqrt(n sum b^3)
// <= 2 m n, and sum b^2 <= n^2 trivially: a sample with `holes` holes needs at most holes (3 + 2 min(holes, 2m)) doubles.
static unsigned long long inpaint_arena_doubles(const unsigned int* summary_host, int n, int h, int w) {
    const unsigned long long m2 = 2ull * (unsigned long long)(h < w ? h : w);
    unsigned long long d = 0;
    for (int s = 0; s < n; ++s) {
        const unsigned long long c = summary_host[4 * s];
        d += c * (3 + 2 * (c < m2 ? c : m2));
    }
    return d;
}

}  // namespace ptta
