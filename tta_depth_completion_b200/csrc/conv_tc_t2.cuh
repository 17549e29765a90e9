// 3x3 TRANSPOSED stride-2 32->32 NHWC bf16 convolution on tcgen05 -- the up-sampling layers of every MSG-CHN decoder
// (network_exp_msg_chn_adapt.py:276-283: ConvTranspose2d(32, 32, 3, 2, 1, 1) in dec{1,2}.1) and, with the matching packed weights,
// the data gradient of the stride-2 Conv2d layers of the encoders (:175-185).  Same machinery as conv_tc.cuh (TMA-fed
// SWIZZLE_128B pixel-pair rows, scatter-form accumulation in TMEM with first-touch MMAs, elect.sync issue, TMA-store epilogue
// with two warps per TMEM lane quarter); what changes is the geometry:
//
//   out[2y-1+ky][2x-1+kx] += in[y][x] . W[ky][kx]     (pad 1, output_padding 1: the output is exactly 2H x 2W)
//
//   horizontally, input pixel pair j = (pixels 2j, 2j+1) owns the output quad 4j .. 4j+3 -- four accumulator banks:
//       out[4j]   = even(j) . W[kx=1]
//       out[4j+1] = even(j) . W[kx=2] + odd(j)    . W[kx=0]
//       out[4j+2] = odd(j)  . W[kx=1]
//       out[4j+3] = odd(j)  . W[kx=2] + even(j+1) . W[kx=0]
//   (even / odd / next-even are descriptor start offsets 0 / 64 / 128 B into the staged row: one halo pair on the right);
//   vertically, input row i feeds output rows 2i-1 (ky = 0), 2i (ky = 1) and 2i+1 (ky = 2): the three taps are stacked along N
//   (weights arranged [kx][ky*32 + cout][cin]).  Row 2i gets its only contribution from input row i, row 2i+1 its first one,
//   so for those two (N = 64, neighbouring TMEM slots) the first MMA of every bank runs with accumulate = 0; row 2i-1 (N = 32)
//   always accumulates and is complete afterwards.  Every input row is read once; 12 + 12 MMAs per input row of 256 pixels
//   produce two output rows of 512 pixels.
//
// TMEM: 4 banks x 4 output-row slots x 32 columns = all 512 columns.  A CTA walks a contiguous range of the (image, strip,
// input row) sequence and reads one extra input row at the end of each segment (its ky = 0 tap completes the last odd output row).
#pragma once
#include "conv_tc.cuh"

namespace ptta {

// OPS: the instantiation that reads mask / add.  It gives up four input-row slots (still eight output rows of look-ahead: an input
// row feeds two output rows) for one staging tile per epilogue warp and operand.
template <bool OPS = false>
struct ConvTcT2Cfg {
    static const int RB = OPS ? 4 : 8;            // input-row slots in the shared-memory ring
    static const int NSLOT = 4;                   // output-row accumulator slots per bank
    static const int BOXP = 130;                  // pixel pairs per staged row (the stride-1 kernel's tensor map; 129 are used)
    static const int ROW_BYTES = BOXP * 128;
    static const int SLOT_BYTES = 17408;
    static const int W_BYTES = 9 * 32 * 64;
    static const int OUT_TILE = 8192;             // one TMEM lane quarter's output row: 64 output pixel pairs x 128 B (one TMA store box)
    static const int STAGE_BYTES = 4 * 2 * OUT_TILE;   // 4 quarters x double buffer
    static const int OP_TILE = 32 * 128;          // one epilogue warp's share of an output row of one operand: 32 lanes x 2 pixels x 64 B
    static const int OP_BYTES = OPS ? 8 * 2 * OP_TILE : 0;     // [warp][mask | add]
    static const int BAR_BYTES = 1024;
    static const int SMEM = 1024 + RB * SLOT_BYTES + W_BYTES + STAGE_BYTES + OP_BYTES + BAR_BYTES;
    static const int THREADS = 320;               // warp 0 TMA producer | warp 1 MMA issuer | warps 2-9 epilogue
    static_assert(SMEM <= 232448, "conv3x3_tc_t2: shared memory over the 227 KB a block can opt into");
};

// [tap][cout][cin] bf16 (tap = ky*3 + kx of the ConvTranspose2d weight as the mma.sync MODE_T2 kernel reads it) -> the kernel's
// shared-memory weight image: row = kx*96 + ky*32 + cout, 64 B rows, SWIZZLE_64B chunk order
__global__ void pack_conv_weight_tc_t2_kernel(const bf16* __restrict__ pack, bf16* __restrict__ image) {
    PDL_SYNC();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 9 * 32 * 4) return;
    const int row = i >> 2, c = i & 3;
    const int kx = row / 96, rem = row - kx * 96;
    const int ky = rem / 32, co = rem & 31;
    uint4 v = *reinterpret_cast<const uint4*>(pack + (size_t)((ky * 3 + kx) * 32 + co) * 32 + c * 8);
    *reinterpret_cast<uint4*>(reinterpret_cast<unsigned char*>(image) + row * 64 + ((c ^ ((row >> 1) & 3)) << 4)) = v;
}

// p.H, p.W: INPUT size (W even); output 2H x 2W.  p.rows_per_cta / p.total_rows count INPUT rows.
// The thread's two output pixels are 128 contiguous bytes of every output-shaped map, at a 256 B stride between lanes.  Loaded by
// the thread itself, every request of a mask / add row touches 32 lines; instead the warp copies its 32 x 128 B of each operand row
// with cp.async, eight lanes per 128 B (4 lines per request), into a tile swizzled by lane (chunk c of lane l at
// l * 128 + ((c ^ (l & 7)) << 4)), issued before the accumulator wait, and each thread reads its own 128 B back.
template <bool OPS>
__global__ void __launch_bounds__(ConvTcT2Cfg<>::THREADS, 1) conv3x3_tc_t2_kernel(const __grid_constant__ CUtensorMap tmap_in,
                                                                                  const __grid_constant__ CUtensorMap tmap_out, const ConvTcParams p) {
    typedef ConvTcT2Cfg<OPS> C;
    extern __shared__ unsigned char smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    unsigned char* smem = smem_raw + (smem_base - smem_u32(smem_raw));
    const uint32_t rows_s = smem_base;
    const uint32_t w_s = smem_base + C::RB * C::SLOT_BYTES;
    const uint32_t stage_s = w_s + C::W_BYTES;
    const uint32_t op_s = stage_s + C::STAGE_BYTES;          // OPS: [epilogue warp][mask | add][OP_TILE]
    const uint32_t bar_s = op_s + C::OP_BYTES;
    const uint32_t row_full = bar_s;                         // [RB]    TMA      -> MMA
    const uint32_t row_free = bar_s + 8 * C::RB;             // [RB]    MMA      -> producer
    const uint32_t slot_full = bar_s + 16 * C::RB;           // [NSLOT] MMA      -> epilogue
    const uint32_t slot_empty = slot_full + 8 * C::NSLOT;    // [NSLOT] epilogue -> MMA (8 arrivals)
    const uint32_t w_full = slot_empty + 8 * C::NSLOT;
    const uint32_t tmem_slot = w_full + 8;
    const uint32_t bias_s = tmem_slot + 8;                   // 32 floats
    volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem + (tmem_slot - smem_base));
    float* bias_sm = reinterpret_cast<float*>(smem + (bias_s - smem_base));

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (warp == 0 && lane == 0) {
        tc::prefetch_tmap(&tmap_in);
        tc::prefetch_tmap(&tmap_out);
        for (int i = 0; i < C::RB; ++i) {
            tc::mbar_init(row_full + 8 * i, 1);
            tc::mbar_init(row_free + 8 * i, 1);
        }
        for (int i = 0; i < C::NSLOT; ++i) {
            tc::mbar_init(slot_full + 8 * i, 1);
            tc::mbar_init(slot_empty + 8 * i, 8);
        }
        tc::mbar_init(w_full, 1);
        tc::fence_barrier_init();
    }
    if (warp == 1) tc::tmem_alloc(tmem_slot, 512);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;
    PDL_SYNC();      // nothing above touches global data
    if (warp == 2) bias_sm[lane] = p.bias ? __ldg(p.bias + lane) : 0.f;

    const int lin0 = min(blockIdx.x * p.rows_per_cta, p.total_rows), lin1 = min(lin0 + p.rows_per_cta, p.total_rows);
    const int Ho = 2 * p.H, Wo = 2 * p.W;

    if (warp == 0) {
        // =========================== TMA producer ===========================
        if (elect_one()) {
            tc::mbar_arrive_expect_tx(w_full, C::W_BYTES);
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(w_s), "l"(p.w), "r"((uint32_t)C::W_BYTES), "r"(w_full) : "memory");
        }
        __syncwarp();
        uint32_t r = 0;
        for (int lin = lin0; lin < lin1;) {
            const int col = lin / p.H, y0 = lin - col * p.H, y1 = min(p.H, y0 + (lin1 - lin));
            const int n = col / p.strips, sx = col - n * p.strips;
            for (int yy = y0; yy <= y1; ++yy, ++r) {                // y1 itself: halo row (zero-filled below the image)
                const uint32_t slot = r % C::RB;
                tc::mbar_wait(row_free + 8 * slot, ((r / C::RB) & 1) ^ 1);
                if (elect_one()) {
                    tc::mbar_arrive_expect_tx(row_full + 8 * slot, C::ROW_BYTES);
                    tc::tma_load_4d(rows_s + slot * C::SLOT_BYTES, &tmap_in, row_full + 8 * slot, 0, sx * 128, yy, n);
                }
                __syncwarp();
            }
            lin += y1 - y0;
        }
    } else if (warp == 1) {
        // =========================== MMA issuer ===========================
        const uint32_t idesc32 = tc::make_idesc_bf16(128, 32), idesc64 = tc::make_idesc_bf16(128, 64);
        const uint64_t da0 = make_desc_sw128(0), db0 = tc::make_desc_sw64(0, 512, 0);
        const uint32_t a_hi = (uint32_t)(da0 >> 32), b_hi = (uint32_t)(db0 >> 32);
        const uint32_t a_lo0 = (uint32_t)da0 + (rows_s >> 4), b_lo0 = (uint32_t)db0 + (w_s >> 4);
        uint32_t r = 0, t_base = 0;                               // t_base: output rows issued so far (always even)
        tc::mbar_wait(w_full, 0);
        for (int lin = lin0; lin < lin1;) {
            const int y0 = lin % p.H;
            const int nrows = min(p.H - y0, lin1 - lin);
            lin += nrows;
            for (int i = 0; i <= nrows; ++i, ++r) {
                const uint32_t rs = r % C::RB;
                const bool has_new = i < nrows;                   // output rows 2i, 2i+1 are first touched by this input row
                const bool has_old = i > 0;                       // output row 2i-1 receives its ky = 0 tap
                const uint32_t tn = t_base + 2 * i;               // running index of output row 2i
                if (has_new) {
                    tc::mbar_wait(slot_empty + 8 * (tn % C::NSLOT), ((tn / C::NSLOT) & 1) ^ 1);
                    tc::mbar_wait(slot_empty + 8 * ((tn + 1) % C::NSLOT), (((tn + 1) / C::NSLOT) & 1) ^ 1);
                }
                tc::mbar_wait(row_full + 8 * rs, (r / C::RB) & 1);
                tc::tc_fence_after();
                if (elect_one()) {
                    const uint32_t a_lo = a_lo0 + rs * (C::SLOT_BYTES >> 4);
                    const uint32_t s_new = tn % C::NSLOT, s_old = (tn - 1) % C::NSLOT;     // s_new is 0 or 2: (2i, 2i+1) never wrap
                    // bank b <-> output pixel 4j+b: taps {A offset in 16 B units (even 0 | odd 4 | next even 8), kx}
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        const int ntap = (b & 1) ? 2 : 1;
#pragma unroll
                        for (int ti = 0; ti < 2; ++ti) {
                            if (ti >= ntap) continue;
                            const uint32_t aoff = b == 0 ? 0u : (b == 1 ? (ti == 0 ? 0u : 4u) : (b == 2 ? 4u : (ti == 0 ? 4u : 8u)));
                            const int kx = (b & 1) ? (ti == 0 ? 2 : 0) : 1;
#pragma unroll
                            for (int ks = 0; ks < 2; ++ks) {
                                const uint32_t al = a_lo + aoff + ks * 2;
                                const uint32_t bl = b_lo0 + kx * 96 * 4 + ks * 2;
                                const uint32_t d = tmem_base + b * (32 * C::NSLOT);
                                if (has_old) tc::umma_f16_split<true>(d + s_old * 32, al, a_hi, bl, b_hi, idesc32);                 // ky = 0
                                if (has_new) {
                                    if (ti == 0 && ks == 0) tc::umma_f16_split<false>(d + s_new * 32, al, a_hi, bl + 32 * 4, b_hi, idesc64);   // ky = 1 | 2
                                    else tc::umma_f16_split<true>(d + s_new * 32, al, a_hi, bl + 32 * 4, b_hi, idesc64);
                                }
                            }
                        }
                    }
                    tc::umma_commit(row_free + 8 * rs);
                    if (has_old) tc::umma_commit(slot_full + 8 * s_old);          // output row 2i-1 complete
                    if (has_new) tc::umma_commit(slot_full + 8 * s_new);          // output row 2i complete (ky = 1 only)
                }
                __syncwarp();
            }
            t_base += 2 * nrows;
        }
    } else {
        // =========================== epilogue ===========================
        const int q = warp & 3;                          // TMEM lane quarter
        const int half = (warp - 2) >> 2;                // 0: output pixels 4j, 4j+1 (banks 0, 1) | 1: 4j+2, 4j+3 (banks 2, 3)
        const bool issuer = half == 0 && lane == 0;
        const uint32_t stage_q = stage_s + q * 2 * C::OUT_TILE;
        const uint32_t mst = op_s + (warp - 2) * 2 * C::OP_TILE, ast = mst + C::OP_TILE;   // this warp's operand tiles
        const unsigned char* mrow = smem + (mst - smem_base) + lane * 128;
        const unsigned char* arow = smem + (ast - smem_base) + lane * 128;
        tc::named_bar_sync(5, 256);                      // bias_sm written (epilogue warps only)
        uint32_t t = 0;
        for (int lin = lin0; lin < lin1;) {
            const int col = lin / p.H, y0 = lin - col * p.H, y1 = min(p.H, y0 + (lin1 - lin));
            const int n = col / p.strips, sx = col - n * p.strips;
            lin += y1 - y0;
            const int jp = sx * 128 + q * 32;                                // first input pixel pair of this quarter
            const int vp = min(32, p.W / 2 - jp);                            // valid input pairs (may be <= 0)
            for (int R = 2 * y0; R < 2 * y1; ++R, ++t) {
                const uint32_t sl = t % C::NSLOT;
                if (OPS) {
                    __syncwarp();                        // every lane has read the previous row's tiles
                    // request k: lanes 8k'..8k'+7 copy the 128 B of lane s = 4k + (l >> 3), chunk l & 7; `add` may alias `out`: it is
                    // read here, before this CTA's store of the row
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        const int s = 4 * k + (lane >> 3), c = lane & 7;
                        const size_t off = (((size_t)n * Ho + R) * Wo + 4 * (jp + s) + 2 * half) * 32 + c * 8;
                        const uint32_t dst = s * 128 + ((c ^ (s & 7)) << 4);
                        if (p.mask) cp_async16(mst + dst, p.mask + off, s < vp);
                        if (p.add) cp_async16(ast + dst, p.add + off, s < vp);
                    }
                    cp_async_commit();
                }
                tc::mbar_wait(slot_full + 8 * sl, (t / C::NSLOT) & 1);
                tc::tc_fence_after();
                if (OPS) {
                    cp_async_wait_all();
                    __syncwarp();
                }
                const uint32_t buf = (t & 1) * C::OUT_TILE;
                unsigned char* srow = smem + (stage_q - smem_base) + buf + (2 * lane + half) * 128;
                const int swz = (2 * lane + half) & 7;
#pragma unroll
                for (int e = 0; e < 2; ++e) {                    // the two pixels of this thread, one accumulator bank each
                    uint32_t v[32];
                    tc::tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (2 * half + e) * (32 * C::NSLOT) + sl * 32, v);
                    if (e == 1) {
                        tc::tc_fence_before();
                        __syncwarp();
                        if (lane == 0) tc::mbar_arrive(slot_empty + 8 * sl);
                    }
                    float f[32];
#pragma unroll
                    for (int c = 0; c < 32; ++c) f[c] = __uint_as_float(v[c]) + bias_sm[c];
                    if (OPS && p.mask) {
#pragma unroll
                        for (int g = 0; g < 4; ++g) {
                            const uint32_t bits = positive_bits(*reinterpret_cast<const uint4*>(mrow + (((e * 4 + g) ^ (lane & 7)) << 4)));
#pragma unroll
                            for (int j = 0; j < 8; ++j) f[g * 8 + j] = (bits >> j) & 1u ? f[g * 8 + j] : 0.f;
                        }
                    }
                    if (OPS && p.add) {
#pragma unroll
                        for (int g = 0; g < 4; ++g) {
                            const uint4 av = *reinterpret_cast<const uint4*>(arow + (((e * 4 + g) ^ (lane & 7)) << 4));
                            const uint32_t* au = reinterpret_cast<const uint32_t*>(&av);
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const float2 a = unpack_bf162(au[j]);
                                f[g * 8 + j * 2] += a.x;
                                f[g * 8 + j * 2 + 1] += a.y;
                            }
                        }
                    }
                    if (p.relu_out) {
#pragma unroll
                        for (int c = 0; c < 32; ++c) f[c] = fmaxf(f[c], 0.f);
                    }
                    if (vp > 0) {
#pragma unroll
                        for (int g = 0; g < 4; ++g) {
                            uint4 ov;
                            ov.x = pack_bf162(f[g * 8 + 0], f[g * 8 + 1]); ov.y = pack_bf162(f[g * 8 + 2], f[g * 8 + 3]);
                            ov.z = pack_bf162(f[g * 8 + 4], f[g * 8 + 5]); ov.w = pack_bf162(f[g * 8 + 6], f[g * 8 + 7]);
                            *reinterpret_cast<uint4*>(srow + (((e * 4 + g) ^ swz) << 4)) = ov;
                        }
                    }
                }
                if (vp <= 0) continue;                   // whole quarter right of the image: both of its warps skip
                tc::fence_proxy_async();
                if (issuer) tc::bulk_store_wait_read_all();
                __syncwarp();
                tc::named_bar_sync(1 + q, 64);
                if (issuer) {
                    tc::tma_store_4d(&tmap_out, stage_q + buf, 0, 2 * jp, R, n);       // 64 output pairs; the map clips the right edge
                    tc::bulk_store_commit();
                }
            }
        }
        if (issuer) tc::bulk_store_wait_read_all();
    }

    tc::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc::tc_fence_after();
        tc::tmem_dealloc(tmem_base, 512);
    }
}

inline bool conv_tc_t2_supported(int N, int H, int W) { return N >= 1 && H >= 1 && W >= 2 && (W % 2) == 0; }

// in: [N, H, W, 32]; p.out (and p.mask / p.add): [N, 2H, 2W, 32]; p.N / p.H / p.W describe the INPUT
inline int launch_conv_tc_t2(const bf16* in, ConvTcParams p, cudaStream_t st) {
    static int sms = 0;
    if (!sms) {
        PTTA_CUDA(cudaFuncSetAttribute(conv3x3_tc_t2_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvTcT2Cfg<false>::SMEM));
        PTTA_CUDA(cudaFuncSetAttribute(conv3x3_tc_t2_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvTcT2Cfg<true>::SMEM));
        int dev = 0;
        PTTA_CUDA(cudaGetDevice(&dev));
        PTTA_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    }
    PTTA_CHECK(conv_tc_t2_supported(p.N, p.H, p.W), "conv3x3_tc_t2: input width %d must be even", p.W);
    PTTA_CHECK(!p.out2 && !p.add2 && !p.relu_in, "conv3x3_tc_t2: out2 / add2 / ReLU-on-load are not supported");
    p.strips = cdiv(p.W, 256);
    p.total_rows = p.N * p.strips * p.H;
    // input rows per CTA: each one costs two output rows of epilogue; one halo row per segment
    int best_rows = p.total_rows; long long best_cost = -1;
    for (int rows = 1; rows <= p.total_rows; ++rows) {
        const long long ctas = cdiv(p.total_rows, rows);
        const long long waves = (ctas + sms - 1) / sms;
        const long long cost = waves * (2 * rows + 1 + 4);
        if (best_cost < 0 || cost < best_cost) { best_cost = cost; best_rows = rows; }
        if (ctas <= 1) break;
    }
    p.rows_per_cta = best_rows;
    const int grid = cdiv(p.total_rows, p.rows_per_cta);
    const CUtensorMap* m = nullptr;
    PTTA_TRY(conv_tc_tmap(in, p.N, p.H, p.W, &m));
    const CUtensorMap map_in = *m;
    PTTA_TRY(conv_tc_tmap(p.out, p.N, 2 * p.H, 2 * p.W, &m, 64));
    const CUtensorMap map_out = *m;
    if (p.mask || p.add) launch_k(conv3x3_tc_t2_kernel<true>, grid, ConvTcT2Cfg<true>::THREADS, ConvTcT2Cfg<true>::SMEM, st, map_in, map_out, p);
    else launch_k(conv3x3_tc_t2_kernel<false>, grid, ConvTcT2Cfg<false>::THREADS, ConvTcT2Cfg<false>::SMEM, st, map_in, map_out, p);
    return check_launch("conv3x3_tc_t2");
}

}  // namespace ptta
