// 3x3 stride-1 32->32 NHWC bf16 convolution on the 5th-generation tensor cores (tcgen05.mma, accumulators in TMEM, operands
// staged by TMA, results stored by TMA) -- the layer shape that carries most of MSG-CHN's FLOPs and bytes
// (network_exp_msg_chn_adapt.py:166-311: every `conv(ReLU(x))` of the encoders / decoders, and their data gradients, which
// are the same convolution with flipped taps).  Design notes: the comment in front of conv3x3_tc_kernel and DESIGN.md section 3.
#pragma once
#include <cuda.h>
#include <vector>
#include "common.cuh"
#include "tc_ptx.cuh"
#include "conv_mma.cuh"
#include "small_kernels.cuh"   // up2_coord / up2_scale (bilinear x2, align_corners = True)

namespace ptta {

struct ConvTcParams {
    const bf16* w;       // 18 KB shared-memory image of the weights (pack_conv_weight_tc_kernel)
    const float* bias;   // [32] or null
    bf16* out;
    bf16* out2;          // optional second output: ReLU(out [+ add2]) (for consumers that have no ReLU-on-load), or null
    const bf16* add2;    // optional addend of out2 only (decoder sums s = ReLU(conv + skip)); mutually exclusive with `add`
    const bf16* mask;    // relu-derivative mask source (same shape as out) or null
    const bf16* add;     // out = add + mask * (conv + bias), or null
    int N, H, W;
    int relu_in;         // apply ReLU to the input while it sits in shared memory
    int relu_out;        // store ReLU(result) (producer-side activation for consumers that only read ReLU(x))
    int strips, segs_y, rows_per_seg, total_segs;      // stride-2 kernel: fixed row segments per strip
    int rows_per_cta, total_rows;                      // stride-1 kernel: contiguous range of the (image, strip, row) sequence per CTA
    const bf16* up2;     // optional: out = conv + bias + up2(half-resolution map [N][H/2][W/2][32]) (bilinear x2, align_corners = True): the
                         // cascade's `x = conv(.) + F.interpolate(pre_x)` (network_exp_msg_chn_adapt.py:172-186) without a pass of its own
    // 32 -> 1 channel form (conv3x3_tc_head_kernel): fp32 output plane, optional fp32 addend plane, scalar bias
    float* out_f32; const float* add_f32; float bias0;
};


// Shared-memory layout per instantiation (MASK / ADDS / UP2: the epilogue operands, see conv3x3_tc_body).  The plain kernel spends
// it all on eight input-row slots and the two output staging tiles; the operand instantiations give up input-row slots, and the
// mask (data-gradient) ones the out2 tile they never write, for the operand rings the producer fills by TMA.
template <bool MASK = false, bool ADDS = false, bool UP2 = false>
struct ConvTcCfg {
    static const int NOPS = (MASK ? 1 : 0) + (ADDS ? 1 : 0);     // full-resolution operand maps (mask, add / add2)
    static const bool OUT2 = !MASK;               // the out2 staging tile exists
    static const int RB = (NOPS == 0 && !UP2) || (MASK && !ADDS) ? 8 : (UP2 && ADDS ? 4 : 6);   // input-row slots in the shared-memory ring
    static const int NSLOT = 8;                   // output-row accumulator slots per pixel parity (2 x 8 x 32 columns = all 512)
    static const int BOXP = 130;                  // pixel PAIRS per staged row (128 + one halo pair each side)
    static const int ROW_BYTES = BOXP * 128;      // 16640: what one TMA box delivers
    static const int SLOT_BYTES = 17408;          // ROW_BYTES rounded up to the 1024 B swizzle-pattern alignment
    static const int W_BYTES = 9 * 32 * 64;       // 18432
    static const int OUT_TILE = 4096;             // one TMEM lane quarter's output row: 32 pixel pairs x 128 B (one TMA store box)
    static const int STAGE_BYTES = 4 * 2 * OUT_TILE;   // per output map: 4 quarters x double buffer
    static const int OP_BYTES = 128 * 128;        // one operand's row of a strip: 128 pixel pairs x 128 B (one SWIZZLE_128B box)
    static const int OPD = NOPS ? 2 : 0;          // operand ring: output rows in flight
    static const int UP_BOX = 130;                // half-resolution pixels per staged row: a strip's low-resolution span (<= 129) + 1
    static const int UP_BYTES = UP_BOX * 64;      // 8320 (SWIZZLE_64B box)
    static const int UP_SLOT = 9216;              // UP_BYTES rounded up to 1024 B
    static const int UPD = UP2 ? 4 : 0;           // up2 ring: half-resolution rows in flight (an output row reads two)
    static const int LAG = RB - 2;                // the producer stages output row y's operands right after input row y + LAG
    static const int BAR_BYTES = 1024;
    static const int SMEM = 1024 /*align slack*/ + RB * SLOT_BYTES + W_BYTES + (OUT2 ? 2 : 1) * STAGE_BYTES + OPD * NOPS * OP_BYTES +
                            UPD * UP_SLOT + BAR_BYTES;
    static const int THREADS = 320;               // warp 0 TMA producer | warp 1 MMA issuer | warps 2-9 epilogue (2 per TMEM lane quarter)
    static_assert(SMEM <= 232448, "conv3x3_tc: shared memory over the 227 KB a block can opt into");
    static_assert(!(MASK && UP2), "conv3x3_tc: mask and up2 are never used together");
};

// one bit per bf16 of a 16 B chunk: value > 0
__device__ __forceinline__ uint32_t positive_bits(const uint4& v) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    uint32_t b = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        b |= ((short)(w[j] & 0xffffu) > 0 ? 1u : 0u) << (2 * j);
        b |= ((int)w[j] >= 0x10000 ? 1u : 0u) << (2 * j + 1);
    }
    return b;
}

// bias / derivative mask / add / ReLU on one pixel's 32 accumulators -> four 16 B chunks of bf16
// mbits: bit c set = keep channel c (all ones without a mask); addp: this pixel's four staged `add` chunks or null
__device__ __forceinline__ void conv_tc_finish_pixel(const uint32_t (&v)[32], const float (&bias)[32], uint32_t mbits, const unsigned char* addrow,
                                                     int chunk0, int swz, int relu_out, uint4 (&ov)[4]) {
    float f[32];
#pragma unroll
    for (int c = 0; c < 32; ++c) f[c] = (mbits >> c) & 1u ? __uint_as_float(v[c]) + bias[c] : 0.f;
    if (addrow) {
#pragma unroll
        for (int g = 0; g < 4; ++g) {
            uint4 av = *reinterpret_cast<const uint4*>(addrow + (((chunk0 + g) ^ swz) << 4));
            const uint32_t* au = reinterpret_cast<const uint32_t*>(&av);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float2 a = unpack_bf162(au[j]);
                f[g * 8 + j * 2] += a.x;
                f[g * 8 + j * 2 + 1] += a.y;
            }
        }
    }
    if (relu_out) {
#pragma unroll
        for (int c = 0; c < 32; ++c) f[c] = fmaxf(f[c], 0.f);
    }
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        ov[g].x = pack_bf162(f[g * 8 + 0], f[g * 8 + 1]);
        ov[g].y = pack_bf162(f[g * 8 + 2], f[g * 8 + 3]);
        ov[g].z = pack_bf162(f[g * 8 + 4], f[g * 8 + 5]);
        ov[g].w = pack_bf162(f[g * 8 + 6], f[g * 8 + 7]);
    }
}

// [tap][cout][cin] bf16 (pack_conv_weight_kernel) -> the kernel's shared-memory weight image: row = kx*96 + (2-ky)*32 + cout,
// 64 B per row, 16 B chunks XOR-swizzled exactly as SWIZZLE_64B lays them out at a 512 B aligned base.  One bulk copy stages it.
__global__ void pack_conv_weight_tc_kernel(const bf16* __restrict__ pack, bf16* __restrict__ image) {
    PDL_SYNC();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 9 * 32 * 4) return;
    const int row = i >> 2, c = i & 3;
    const int kx = row / 96, rem = row - kx * 96;
    const int ky = 2 - rem / 32, co = rem & 31;
    uint4 v = *reinterpret_cast<const uint4*>(pack + (size_t)((ky * 3 + kx) * 32 + co) * 32 + c * 8);
    *reinterpret_cast<uint4*>(reinterpret_cast<unsigned char*>(image) + row * 64 + ((c ^ ((row >> 1) & 3)) << 4)) = v;
}

// Scatter-form implicit GEMM over PIXEL PAIRS.
//
// Shared-memory / TMA view of the NHWC bf16 input: [N][H][W/2][64] -- one 128 B row per pixel pair, SWIZZLE_128B, the layout
// TMA moves at full speed (64 B rows do not).  A strip is 128 pairs = 256 output pixels wide; a staged input row holds 130
// pairs (one halo pair each side, zero-filled by TMA outside the image = the convolution's padding).  The UMMA A operand is
// "128 rows of 128 B"; a K = 16 slice at byte offset 0/32 of a row is the EVEN pixel of each pair, at 64/96 the ODD pixel,
// and a descriptor may start at any pair row (the swizzle is a function of the shared-memory address).  Hence
//     even output pixel 2j   = W[kx=0] . odd(j-1) + W[kx=1] . even(j) + W[kx=2] . odd(j)
//     odd  output pixel 2j+1 = W[kx=0] . even(j)  + W[kx=1] . odd(j)  + W[kx=2] . even(j+1)
// with no wasted FLOPs, and the even / odd outputs of one lane are 128 contiguous bytes of the output row.
//
// Vertical taps: input row i of a segment (image row y0-1+i) contributes to output rows j = i-2, i-1, i with ky = 2, 1, 0.
// The three taps are stacked along N (weights pre-arranged as [kx][(2-ky)*32+cout][cin]), so 12 MMAs (2 parities x 3 kx x 2 K
// steps, M128 x N96 x K16) consume an input row exactly once and accumulate into three neighbouring 32-column TMEM slots of
// each parity bank; slot(t) = t mod 8 of the running output-row counter.  The FIRST MMA that touches an output row's slot
// (input row i = j, ky = 0, kx = 0, first K step) is issued on its own with accumulate = 0, so accumulator slots are never
// zeroed by hand; a slot is complete after input row j+2, is drained by the epilogue warps and reused 8 rows later.
//
// Roles: warp 0 TMA producer (one box per input row) | warp 1 MMA issuer (warp stays converged, elect.sync issues) |
// warps 2-9 epilogue, two per TMEM lane quarter (one takes the even-pixel accumulator bank, one the odd): tcgen05.ld ->
// bias / derivative mask / add / ReLU in registers -> bf16 -> the pixel's half of its 128 B pair row in a SWIZZLE_128B staging
// tile -> one TMA store per quarter row (32 pairs x 128 B; the tensor map clips the ragged right edge), double buffered.
//
// Epilogue operands come through shared memory, staged by the producer warp with TMA:
//   mask / add / add2: per output row one box of 128 pixel pairs of each map, in the same pair-row view and swizzle as the output
//   staging tile, into a ring of OPD output rows (zero-filled right of the image).  The thread's pixel sits at the address it
//   writes its output to, so the reads need no shuffles and hit no bank conflicts.  `add` may alias `out` (in-place accumulate):
//   a CTA's TMA load of a row completes before its epilogue stores that row, and no other CTA touches the row.
//   up2: the half-resolution rows the strip's output rows read (align_corners = True), 130 pixels from the strip's first source
//   column, in a ring of UPD rows keyed by half-resolution row: each is read from global memory once per segment.
// The producer stages output row y's operands after it issued input row y + LAG, so it can still run LAG rows ahead of the MMA.
// Every mbarrier has one arrival per phase except slot_empty, op_empty and up_empty (one per epilogue warp).
__device__ __forceinline__ void conv_tc_pixel(const uint32_t (&v)[32], const float (&bias)[32], const uint4* mk, const uint4* ad, int relu_out,
                                              uint4 (&ov)[4], const float* up = nullptr) {
    float f[32];
#pragma unroll
    for (int c = 0; c < 32; ++c) f[c] = __uint_as_float(v[c]) + bias[c];
    if (up) {
#pragma unroll
        for (int c = 0; c < 32; ++c) f[c] += up[c];
    }
    if (mk) {
#pragma unroll
        for (int g = 0; g < 4; ++g) {
            const uint32_t b = positive_bits(mk[g]);
#pragma unroll
            for (int j = 0; j < 8; ++j) f[g * 8 + j] = (b >> j) & 1u ? f[g * 8 + j] : 0.f;
        }
    }
    if (ad) {
#pragma unroll
        for (int g = 0; g < 4; ++g) {
            const uint32_t* au = reinterpret_cast<const uint32_t*>(&ad[g]);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float2 a = unpack_bf162(au[j]);
                f[g * 8 + j * 2] += a.x;
                f[g * 8 + j * 2 + 1] += a.y;
            }
        }
    }
    if (relu_out) {
#pragma unroll
        for (int c = 0; c < 32; ++c) f[c] = fmaxf(f[c], 0.f);
    }
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        ov[g].x = pack_bf162(f[g * 8 + 0], f[g * 8 + 1]);
        ov[g].y = pack_bf162(f[g * 8 + 2], f[g * 8 + 3]);
        ov[g].z = pack_bf162(f[g * 8 + 4], f[g * 8 + 5]);
        ov[g].w = pack_bf162(f[g * 8 + 6], f[g * 8 + 7]);
    }
}

namespace tc {
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                 ::"l"(map), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void bulk_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_store_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t threads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory"); }
}  // namespace tc

// NC = accumulator columns per output row and pixel parity: 32 = the 32 -> 32 convolution; 16 = the 32 -> 1 prediction-layer form
// (conv3x3_tc_head_kernel below: same producer and MMA schedule with N = 3 x 16, another epilogue)
// MASK / ADDS / UP2: which epilogue operands this instantiation handles (ADDS: `add` or `add2`).  They are template parameters because the
// kernel sits at its register cap (168 with 10 warps): every operand path compiled in costs the plain forward conv registers it never uses.
template <int NC, bool MASK, bool ADDS, bool UP2>
__device__ __forceinline__ void conv3x3_tc_body(const CUtensorMap& tmap_in, const CUtensorMap& tmap_out, const CUtensorMap& tmap_out2,
                                                const CUtensorMap& tmap_mask, const CUtensorMap& tmap_add, const CUtensorMap& tmap_up,
                                                const ConvTcParams& p) {
    typedef ConvTcCfg<MASK, ADDS, UP2> C;
    constexpr uint32_t W_BYTES_NC = 9 * NC * 64;
    extern __shared__ unsigned char smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    unsigned char* smem = smem_raw + (smem_base - smem_u32(smem_raw));
    const uint32_t rows_s = smem_base;                                   // RB row slots
    const uint32_t w_s = smem_base + C::RB * C::SLOT_BYTES;              // weights, SW64 canonical, row = kx*96 + (2-ky)*32 + cout
    const uint32_t stage_s = w_s + C::W_BYTES;                           // `out` staging: [quarter][2][32 pairs x 128 B], then `out2`
    const uint32_t op_s = stage_s + (C::OUT2 ? 2 : 1) * C::STAGE_BYTES;  // [OPD][mask | add][128 pairs x 128 B]
    const uint32_t up_s = op_s + C::OPD * C::NOPS * C::OP_BYTES;         // [UPD][130 half-resolution pixels x 64 B]
    const uint32_t bar_s = up_s + C::UPD * C::UP_SLOT;
    const uint32_t row_full = bar_s;                         // [RB]    TMA     -> MMA       (expect_tx + complete_tx)
    const uint32_t row_free = bar_s + 8 * C::RB;             // [RB]    MMA     -> producer  (tcgen05.commit)
    const uint32_t slot_full = bar_s + 16 * C::RB;           // [NSLOT] MMA     -> epilogue  (tcgen05.commit)
    const uint32_t slot_empty = slot_full + 8 * C::NSLOT;    // [NSLOT] epilogue -> MMA      (8 arrivals: one per epilogue warp)
    const uint32_t w_full = slot_empty + 8 * C::NSLOT;       //         bulk copy of the weight image landed
    const uint32_t tmem_slot = w_full + 8;                   // u32
    const uint32_t op_full = tmem_slot + 8;                  // [OPD]   TMA     -> epilogue  (expect_tx + complete_tx)
    const uint32_t op_empty = op_full + 8 * C::OPD;          // [OPD]   epilogue -> producer (8 arrivals)
    const uint32_t up_full = op_empty + 8 * C::OPD;          // [UPD]   TMA     -> epilogue
    const uint32_t up_empty = up_full + 8 * C::UPD;          // [UPD]   epilogue -> producer (8 arrivals)
    volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem + (tmem_slot - smem_base));

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int uh2 = p.H >> 1, uw2 = p.W >> 1;                // up2: half-resolution size

    // ---- one-time set-up: overlaps the tail of the previous kernel (programmatic dependent launch) --------------------
    if (warp == 0 && lane == 0) {
        tc::prefetch_tmap(&tmap_in);
        tc::prefetch_tmap(&tmap_out);
        tc::prefetch_tmap(&tmap_out2);
        if (MASK) tc::prefetch_tmap(&tmap_mask);
        if (ADDS) tc::prefetch_tmap(&tmap_add);
        if (UP2) tc::prefetch_tmap(&tmap_up);
        for (int i = 0; i < C::RB; ++i) {
            tc::mbar_init(row_full + 8 * i, 1);
            tc::mbar_init(row_free + 8 * i, 1);
        }
        for (int i = 0; i < C::NSLOT; ++i) {
            tc::mbar_init(slot_full + 8 * i, 1);
            tc::mbar_init(slot_empty + 8 * i, 8);
        }
        for (int i = 0; i < C::OPD; ++i) {
            tc::mbar_init(op_full + 8 * i, 1);
            tc::mbar_init(op_empty + 8 * i, 8);
        }
        for (int i = 0; i < C::UPD; ++i) {
            tc::mbar_init(up_full + 8 * i, 1);
            tc::mbar_init(up_empty + 8 * i, 8);
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

    // work: the (image, strip, row) sequence is cut into gridDim.x contiguous ranges, so every SM gets the same number of output
    // rows (+-1 halo pair per strip it touches) whatever H is; a range that crosses into the next strip is walked as two segments
    const int lin0 = min(blockIdx.x * p.rows_per_cta, p.total_rows), lin1 = min(lin0 + p.rows_per_cta, p.total_rows);

    if (warp == 0) {
        // =========================== TMA producer ===========================
        if (elect_one()) {
            tc::mbar_arrive_expect_tx(w_full, W_BYTES_NC);
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(w_s), "l"(p.w), "r"(W_BYTES_NC), "r"(w_full) : "memory");
        }
        __syncwarp();
        uint32_t r = 0, o = 0, u = 0;            // input rows, operand rows, half-resolution rows staged so far
        for (int lin = lin0; lin < lin1;) {
            const int col = lin / p.H, y0 = lin - col * p.H, y1 = min(p.H, y0 + (lin1 - lin));
            const int n = col / p.strips, sx = col - n * p.strips;
            int lx0 = 0, next_k = 0;             // up2: first source column of the strip, next half-resolution row to stage
            if (UP2) {
                int i1; float l0, l1;
                up2_coord(sx * 256, uw2, up2_scale(uw2), lx0, i1, l0, l1);
                up2_coord(y0, uh2, up2_scale(uh2), next_k, i1, l0, l1);
            }
            // everything the epilogue reads for output row y of this segment
            auto stage_operands = [&](int y) {
                if constexpr (MASK || ADDS) {
                    const uint32_t s = o % C::OPD;
                    tc::mbar_wait(op_empty + 8 * s, ((o / C::OPD) & 1) ^ 1);
                    if (elect_one()) {
                        const uint32_t dst = op_s + s * C::NOPS * C::OP_BYTES;
                        tc::mbar_arrive_expect_tx(op_full + 8 * s, C::NOPS * C::OP_BYTES);
                        if (MASK) tc::tma_load_4d(dst, &tmap_mask, op_full + 8 * s, 0, sx * 128, y, n);
                        if (ADDS) tc::tma_load_4d(dst + (MASK ? C::OP_BYTES : 0), &tmap_add, op_full + 8 * s, 0, sx * 128, y, n);
                    }
                    __syncwarp();
                    ++o;
                }
                if constexpr (UP2) {
                    int k0, k1; float l0, l1;
                    up2_coord(y, uh2, up2_scale(uh2), k0, k1, l0, l1);
                    for (; next_k <= k1; ++next_k, ++u) {
                        const uint32_t s = u % C::UPD;
                        tc::mbar_wait(up_empty + 8 * s, ((u / C::UPD) & 1) ^ 1);
                        if (elect_one()) {
                            tc::mbar_arrive_expect_tx(up_full + 8 * s, C::UP_BYTES);
                            tc::tma_load_4d(up_s + s * C::UP_SLOT, &tmap_up, up_full + 8 * s, 0, lx0, next_k, n);
                        }
                        __syncwarp();
                    }
                }
            };
            for (int yy = y0 - 1; yy <= y1; ++yy, ++r) {
                const uint32_t slot = r % C::RB;
                tc::mbar_wait(row_free + 8 * slot, ((r / C::RB) & 1) ^ 1);
                if (elect_one()) {
                    tc::mbar_arrive_expect_tx(row_full + 8 * slot, C::ROW_BYTES);
                    tc::tma_load_4d(rows_s + slot * C::SLOT_BYTES, &tmap_in, row_full + 8 * slot, 0, sx * 128 - 1, yy, n);
                }
                __syncwarp();
                if ((MASK || ADDS || UP2) && yy - C::LAG >= y0) stage_operands(yy - C::LAG);
            }
            if (MASK || ADDS || UP2)
                for (int y = max(y0, y1 + 1 - C::LAG); y < y1; ++y) stage_operands(y);
            lin += y1 - y0;
        }
    } else if (warp == 1) {
        // =========================== MMA issuer (converged warp, one elected lane issues) ===========================
        const uint32_t idesc32 = tc::make_idesc_bf16(128, NC), idesc64 = tc::make_idesc_bf16(128, 2 * NC), idesc96 = tc::make_idesc_bf16(128, 3 * NC);
        const uint64_t da0 = make_desc_sw128(0), db0 = tc::make_desc_sw64(0, 512, 0);
        const uint32_t a_hi = (uint32_t)(da0 >> 32), b_hi = (uint32_t)(db0 >> 32);
        const uint32_t a_lo0 = (uint32_t)da0 + (rows_s >> 4), b_lo0 = (uint32_t)db0 + (w_s >> 4);
        uint32_t r = 0, t_base = 0;
        tc::mbar_wait(w_full, 0);
        for (int lin = lin0; lin < lin1;) {
            const int y0 = lin % p.H;
            const int nrows = min(p.H - y0, lin1 - lin);
            lin += nrows;
            for (int i = 0; i < nrows + 2; ++i, ++r) {
                const uint32_t rs = r % C::RB;
                if (i < nrows) {                                   // first touch of the slot of output row i in this round
                    const uint32_t tn = t_base + i;
                    tc::mbar_wait(slot_empty + 8 * (tn % C::NSLOT), ((tn / C::NSLOT) & 1) ^ 1);
                }
                tc::mbar_wait(row_full + 8 * rs, (r / C::RB) & 1);
                tc::tc_fence_after();
                if (elect_one()) {
                    const uint32_t a_lo = a_lo0 + rs * (C::SLOT_BYTES >> 4);
                    // `first`: (kx, ks) == (0, 0).  There the row whose slot is touched for the first time (output row i, ky = 0) gets
                    // its own N = 32 MMA with accumulate = 0 and the older rows (ky = 2, 1) accumulate; all later MMAs of this input
                    // row accumulate into the whole stack.
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx) {
                        // 16 B units inside the slot: pair row = 8 units, odd pixel = +4, K step = +2
                        const uint32_t ae = kx == 0 ? 4u : (kx == 1 ? 8u : 12u);      // odd(j-1) | even(j) | odd(j)
                        const uint32_t ao = kx == 0 ? 8u : (kx == 1 ? 12u : 16u);     // even(j)  | odd(j)  | even(j+1)
#pragma unroll
                        for (int ks = 0; ks < 2; ++ks) {
                            const bool first = (kx | ks) == 0;
                            int j_lo = max(i - 2, 0), j_hi = min(i, nrows - 1);
                            const uint32_t b_tap = b_lo0 + kx * (3 * NC) * 4 + ks * 2;
                            if (first && i < nrows) {
                                const uint32_t s = (t_base + i) % C::NSLOT;
                                const uint32_t d_even = tmem_base + s * NC, d_odd = d_even + NC * C::NSLOT;
                                tc::umma_f16_split<false>(d_even, a_lo + ae, a_hi, b_tap + (2 * NC) * 4, b_hi, idesc32);
                                tc::umma_f16_split<false>(d_odd, a_lo + ao, a_hi, b_tap + (2 * NC) * 4, b_hi, idesc32);
                                j_hi = i - 1;
                            }
                            int cnt = j_hi - j_lo + 1;                          // 0..3 output rows accumulate this input row
                            int b_row = (2 - i + j_lo) * NC;                    // first stacked-weight row: ky = i - j_lo
                            uint32_t s0 = (t_base + j_lo) % C::NSLOT;
                            while (cnt > 0) {
                                const int c1 = min(cnt, C::NSLOT - (int)s0);    // contiguous TMEM slots before the ring wraps
                                const uint32_t idesc = c1 == 3 ? idesc96 : (c1 == 2 ? idesc64 : idesc32);
                                const uint32_t d_even = tmem_base + s0 * NC, d_odd = d_even + NC * C::NSLOT;
                                tc::umma_f16_split<true>(d_even, a_lo + ae + ks * 2, a_hi, b_tap + b_row * 4, b_hi, idesc);
                                tc::umma_f16_split<true>(d_odd, a_lo + ao + ks * 2, a_hi, b_tap + b_row * 4, b_hi, idesc);
                                cnt -= c1; b_row += c1 * NC; s0 = 0;
                            }
                        }
                    }
                    tc::umma_commit(row_free + 8 * rs);                                    // this input row is never read again
                    if (i >= 2) tc::umma_commit(slot_full + 8 * ((t_base + i - 2) % C::NSLOT));   // output row i-2 is complete
                }
                __syncwarp();
            }
            t_base += nrows;
        }
    } else if (NC == 16) {
        // =========================== epilogue, 32 -> 1 form ===========================
        // accumulator column 0 holds the dot product with the bf16 head of the fp32 weights, column 1 with their bf16 remainder
        // (pack_conv_weight_tc_head_kernel): their sum carries the weights to 16 mantissa bits, as the fp32 FMA kernel it replaces
        const int q = warp & 3;
        const int par = (warp - 2) >> 2;
        uint32_t t = 0;
        for (int lin = lin0; lin < lin1;) {
            const int col = lin / p.H, y0 = lin - col * p.H, y1 = min(p.H, y0 + (lin1 - lin));
            const int n = col / p.strips, sx = col - n * p.strips;
            lin += y1 - y0;
            const int xw = sx * 256 + q * 64;
            const int vp = min(32, (p.W - xw) / 2);
            const bool act = lane < vp;
            for (int y = y0; y < y1; ++y, ++t) {
                const uint32_t sl = t % C::NSLOT;
                const size_t idx = ((size_t)n * p.H + y) * p.W + xw + 2 * lane + par;
                float addv = p.bias0;
                if (p.add_f32 != nullptr && act) addv += p.add_f32[idx];
                tc::mbar_wait(slot_full + 8 * sl, (t / C::NSLOT) & 1);
                tc::tc_fence_after();
                uint32_t v0, v1;
                tmem_ld2(tmem_base + ((uint32_t)(q * 32) << 16) + par * NC * C::NSLOT + sl * NC, v0, v1);
                tc::tc_fence_before();
                __syncwarp();
                if (lane == 0) tc::mbar_arrive(slot_empty + 8 * sl);
                if (act) p.out_f32[idx] = (__uint_as_float(v0) + __uint_as_float(v1)) + addv;
            }
        }
    } else {
        // =========================== epilogue ===========================
        const int q = warp & 3;                          // TMEM lane quarter this warp may access
        const int par = (warp - 2) >> 2;                 // 0: even pixels (first accumulator bank), 1: odd pixels
        const bool issuer = par == 0 && lane == 0;       // issues this quarter's TMA stores
        const uint32_t stage_q = stage_s + q * 2 * C::OUT_TILE, stage2_q = stage_q + C::STAGE_BYTES;
        float bias[32];
#pragma unroll
        for (int c = 0; c < 32; ++c) bias[c] = p.bias ? __ldg(p.bias + c) : 0.f;
        uint32_t t = 0, ubase = 0;               // output rows done, half-resolution rows of earlier segments
        for (int lin = lin0; lin < lin1;) {
            const int col = lin / p.H, y0 = lin - col * p.H, y1 = min(p.H, y0 + (lin1 - lin));
            const int n = col / p.strips, sx = col - n * p.strips;
            lin += y1 - y0;
            const int xw = sx * 256 + q * 64;                                // first pixel of this quarter
            const int vp = min(32, (p.W - xw) / 2);                          // valid pixel pairs of this quarter (may be <= 0)
            const bool act = lane < vp;
            // bilinear x2 addend: this thread's column pair and weights are the same for every row of the segment; the staged
            // half-resolution rows start at the strip's first source column lx0 and run k_lo .. k_hi
            int ux0 = 0, ux1 = 0, lx0 = 0, k_lo = 0, k_hi = 0, rel = 0; float ulx0 = 0.f, ulx1 = 0.f;
            if (UP2) {
                int i1; float l0, l1;
                up2_coord(sx * 256, uw2, up2_scale(uw2), lx0, i1, l0, l1);
                up2_coord(y0, uh2, up2_scale(uh2), k_lo, i1, l0, l1);
                up2_coord(y1 - 1, uh2, up2_scale(uh2), i1, k_hi, l0, l1);
                rel = k_lo;
                if (act) {
                    up2_coord(xw + 2 * lane + par, uw2, up2_scale(uw2), ux0, ux1, ulx0, ulx1);
                    ux0 -= lx0; ux1 -= lx0;
                }
            }
            for (int y = y0; y < y1; ++y, ++t) {
                const uint32_t sl = t % C::NSLOT;
                float up[32];
                if constexpr (UP2) {
                    int uy0, uy1; float uly0, uly1;
                    up2_coord(y, uh2, up2_scale(uh2), uy0, uy1, uly0, uly1);
                    const uint32_t g0 = ubase + (uint32_t)(uy0 - k_lo), g1 = ubase + (uint32_t)(uy1 - k_lo);
                    tc::mbar_wait(up_full + 8 * (g0 % C::UPD), (g0 / C::UPD) & 1);
                    tc::mbar_wait(up_full + 8 * (g1 % C::UPD), (g1 / C::UPD) & 1);
                    if (act) {
                        // pixel x of a staged row: 64 B at x * 64, 16 B chunk g at ((g ^ ((x >> 1) & 3)) << 4) (SWIZZLE_64B)
                        const unsigned char* hr0 = smem + (up_s - smem_base) + (g0 % C::UPD) * C::UP_SLOT;
                        const unsigned char* hr1 = smem + (up_s - smem_base) + (g1 % C::UPD) * C::UP_SLOT;
                        const int sw0 = (ux0 >> 1) & 3, sw1 = (ux1 >> 1) & 3;
#pragma unroll
                        for (int g = 0; g < 4; ++g) {
                            const uint4 a00 = *reinterpret_cast<const uint4*>(hr0 + ux0 * 64 + ((g ^ sw0) << 4));
                            const uint4 a01 = *reinterpret_cast<const uint4*>(hr0 + ux1 * 64 + ((g ^ sw1) << 4));
                            const uint4 a10 = *reinterpret_cast<const uint4*>(hr1 + ux0 * 64 + ((g ^ sw0) << 4));
                            const uint4 a11 = *reinterpret_cast<const uint4*>(hr1 + ux1 * 64 + ((g ^ sw1) << 4));
                            const uint32_t *u00 = reinterpret_cast<const uint32_t*>(&a00), *u01 = reinterpret_cast<const uint32_t*>(&a01);
                            const uint32_t *u10 = reinterpret_cast<const uint32_t*>(&a10), *u11 = reinterpret_cast<const uint32_t*>(&a11);
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const float2 f00 = unpack_bf162(u00[j]), f01 = unpack_bf162(u01[j]), f10 = unpack_bf162(u10[j]), f11 = unpack_bf162(u11[j]);
                                up[g * 8 + j * 2] = uly0 * (ulx0 * f00.x + ulx1 * f01.x) + uly1 * (ulx0 * f10.x + ulx1 * f11.x);
                                up[g * 8 + j * 2 + 1] = uly0 * (ulx0 * f00.y + ulx1 * f01.y) + uly1 * (ulx0 * f10.y + ulx1 * f11.y);
                            }
                        }
                    } else {
#pragma unroll
                        for (int c = 0; c < 32; ++c) up[c] = 0.f;
                    }
                    // half-resolution rows no later output row of the segment reads go back to the producer
                    int keep = k_hi + 1;
                    if (y + 1 < y1) { int i1; float l0, l1; up2_coord(y + 1, uh2, up2_scale(uh2), keep, i1, l0, l1); }
                    __syncwarp();
                    for (; rel < keep; ++rel)
                        if (lane == 0) tc::mbar_arrive(up_empty + 8 * ((ubase + (uint32_t)(rel - k_lo)) % C::UPD));
                }
                tc::mbar_wait(slot_full + 8 * sl, (t / C::NSLOT) & 1);
                tc::tc_fence_after();
                uint32_t v[32];
                tc::tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + par * NC * C::NSLOT + sl * NC, v);
                tc::tc_fence_before();
                __syncwarp();
                if (lane == 0) tc::mbar_arrive(slot_empty + 8 * sl);
                uint4 mk[4], ad[4];
                if constexpr (MASK || ADDS) {            // this pixel's 64 B of the staged rows: where its output goes in the staging tile
                    const uint32_t os = t % C::OPD;
                    tc::mbar_wait(op_full + 8 * os, (t / C::OPD) & 1);
                    const unsigned char* orow = smem + (op_s - smem_base) + os * C::NOPS * C::OP_BYTES + (q * 32 + lane) * 128;
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        const int ch = ((par * 4 + g) ^ (lane & 7)) << 4;
                        if (MASK) mk[g] = *reinterpret_cast<const uint4*>(orow + ch);
                        if (ADDS) ad[g] = *reinterpret_cast<const uint4*>(orow + (MASK ? C::OP_BYTES : 0) + ch);
                    }
                    __syncwarp();
                    if (lane == 0) tc::mbar_arrive(op_empty + 8 * os);
                }
                if (vp <= 0) continue;                   // whole quarter right of the image: both of its warps skip
                uint4 ov[4];
                conv_tc_pixel(v, bias, MASK ? mk : nullptr, (ADDS && p.add) ? ad : nullptr, p.relu_out, ov, UP2 ? up : nullptr);
                const uint32_t buf = (t & 1) * C::OUT_TILE;
                unsigned char* srow = smem + (stage_q - smem_base) + buf + lane * 128;
#pragma unroll
                for (int g = 0; g < 4; ++g) *reinterpret_cast<uint4*>(srow + (((par * 4 + g) ^ (lane & 7)) << 4)) = ov[g];
                if (C::OUT2 && p.out2) {                 // out2 = ReLU(bf16(out) [+ add2])
                    unsigned char* srow2 = srow + C::STAGE_BYTES;
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        uint4 val = ov[g];
                        if (ADDS && p.add2) {
                            uint32_t* vu = reinterpret_cast<uint32_t*>(&val);
                            const uint32_t* au = reinterpret_cast<const uint32_t*>(&ad[g]);
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const float2 a = unpack_bf162(vu[j]), b = unpack_bf162(au[j]);
                                vu[j] = pack_bf162(a.x + b.x, a.y + b.y);
                            }
                        }
                        const bf162 z2 = __floats2bfloat162_rn(0.f, 0.f);
                        bf162* h2 = reinterpret_cast<bf162*>(&val);
#pragma unroll
                        for (int j = 0; j < 4; ++j) h2[j] = __hmax2(h2[j], z2);
                        *reinterpret_cast<uint4*>(srow2 + (((par * 4 + g) ^ (lane & 7)) << 4)) = val;
                    }
                }
                tc::fence_proxy_async();                 // generic-proxy writes -> visible to the TMA store
                if (issuer) tc::bulk_store_wait_read_all();      // the previous row's store (other buffer) has left shared memory
                __syncwarp();
                tc::named_bar_sync(1 + q, 64);           // both warps of the quarter have written their halves of the pair rows
                if (issuer) {
                    tc::tma_store_4d(&tmap_out, stage_q + buf, 0, xw >> 1, y, n);
                    if (C::OUT2 && p.out2) tc::tma_store_4d(&tmap_out2, stage2_q + buf, 0, xw >> 1, y, n);
                    tc::bulk_store_commit();
                }
            }
            if (UP2) ubase += (uint32_t)(k_hi - k_lo + 1);
        }
        if (issuer) tc::bulk_store_wait_read_all();      // shared memory may go once the stores have READ it; the grid's completion
                                                         // makes the writes visible (what CUTLASS's tma_store_wait does)
    }

    // ---- teardown -----------------------------------------------------------------------------------------
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc::tc_fence_after();
        tc::tmem_dealloc(tmem_base, 512);
    }
}

// tmap_mask / tmap_add: the mask and the add (or add2) map in the pair-row view with 128-pair boxes; tmap_up: the half-resolution
// map with UP_BOX-pixel boxes (each only read by the instantiation that uses it)
template <bool MASK, bool ADDS, bool UP2>
__global__ void __launch_bounds__(ConvTcCfg<>::THREADS, 1) conv3x3_tc_kernel(const __grid_constant__ CUtensorMap tmap_in,
                                                                             const __grid_constant__ CUtensorMap tmap_out,
                                                                             const __grid_constant__ CUtensorMap tmap_out2,
                                                                             const __grid_constant__ CUtensorMap tmap_mask,
                                                                             const __grid_constant__ CUtensorMap tmap_add,
                                                                             const __grid_constant__ CUtensorMap tmap_up, const ConvTcParams p) {
    conv3x3_tc_body<32, MASK, ADDS, UP2>(tmap_in, tmap_out, tmap_out2, tmap_mask, tmap_add, tmap_up, p);
}

// 32 -> 1 channel 3x3 s1 p1 convolution with an fp32 output plane: the prediction layer prdct.3 (network_exp_msg_chn_adapt.py:289)
// and, with flipped plane-1 weights, the data gradient of a two-plane stem with respect to its prediction input.  The layer reads
// 64 B and writes 4 B per pixel: it is bound by the read of the 32-channel map, which the tensor-core form streams through TMA exactly
// once (the CUDA-core form staged halo tiles and spent 288 shared-memory-fed FMAs per pixel: 22 us at 352x1216).
__global__ void __launch_bounds__(ConvTcCfg<>::THREADS, 1) conv3x3_tc_head_kernel(const __grid_constant__ CUtensorMap tmap_in, const ConvTcParams p) {
    conv3x3_tc_body<16, false, false, false>(tmap_in, tmap_in, tmap_in, tmap_in, tmap_in, tmap_in, p);
}

// fp32 [tap][cin] (tap = ky*3 + kx) -> the head kernel's weight image: row = kx*48 + (2-ky)*16 + c, 64 B per row (32 cin), SWIZZLE_64B
// chunk order; c = 0: bf16(w), c = 1: bf16(w - bf16(w)), c = 2..15: zero
__global__ void pack_conv_weight_tc_head_kernel(const float* __restrict__ w, bf16* __restrict__ image) {
    PDL_SYNC();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 9 * 16 * 4) return;
    const int row = i >> 2, c = i & 3;
    const int kx = row / 48, rem = row - kx * 48;
    const int ky = 2 - rem / 16, co = rem & 15;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (co < 2) {
        uint32_t* u = reinterpret_cast<uint32_t*>(&v);
        const float* src = w + (ky * 3 + kx) * 32 + c * 8;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float a = src[2 * j], b = src[2 * j + 1];
            const float ah = __bfloat162float(__float2bfloat16_rn(a)), bh = __bfloat162float(__float2bfloat16_rn(b));
            if (co == 1) { a -= ah; b -= bh; } else { a = ah; b = bh; }
            u[j] = pack_bf162(a, b);
        }
    }
    *reinterpret_cast<uint4*>(reinterpret_cast<unsigned char*>(image) + row * 64 + ((c ^ ((row >> 1) & 3)) << 4)) = v;
}

// ---- host side ----------------------------------------------------------------------------------------------
// NHWC bf16 [N,H,W,C] activation, box = {C, box_w, 1, 1}, SWIZZLE_64B (C = 32) / 128B (C = 64), zero fill outside
inline int make_tmap_nhwc(CUtensorMap* map, const void* ptr, int N, int H, int W, int Cc, int box_w) {
    PFN_encodeTiled enc = get_encode_tiled();
    PTTA_CHECK(enc != nullptr, "cuTensorMapEncodeTiled not available from the driver");
    cuuint64_t dims[4] = {(cuuint64_t)Cc, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
    cuuint64_t strides[3] = {(cuuint64_t)Cc * 2, (cuuint64_t)W * Cc * 2, (cuuint64_t)H * W * Cc * 2};
    cuuint32_t box[4] = {(cuuint32_t)Cc, (cuuint32_t)box_w, 1, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUtensorMapSwizzle sw = Cc * 2 == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B;
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(ptr), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    PTTA_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed with %d (N=%d H=%d W=%d C=%d box_w=%d)", (int)r, N, H, W, Cc, box_w);
    return 0;
}

// NHWC bf16 [N,H,W,32] activation viewed as [N][H][W/2][64]: box = {64, 130 pairs, 1, 1}, SWIZZLE_128B, zero fill outside
inline int make_tmap_pairs(CUtensorMap* map, const void* ptr, int N, int H, int W, int box_pairs = ConvTcCfg<>::BOXP) {
    PFN_encodeTiled enc = get_encode_tiled();
    PTTA_CHECK(enc != nullptr, "cuTensorMapEncodeTiled not available from the driver");
    cuuint64_t dims[4] = {64, (cuuint64_t)(W / 2), (cuuint64_t)H, (cuuint64_t)N};
    cuuint64_t strides[3] = {128, (cuuint64_t)W * 64, (cuuint64_t)H * W * 64};
    cuuint32_t box[4] = {64, (cuuint32_t)box_pairs, 1, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(ptr), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    PTTA_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed with %d (N=%d H=%d W=%d)", (int)r, N, H, W);
    return 0;
}

inline bool conv_tc_supported(int N, int H, int W) { return N >= 1 && H >= 1 && W >= 2 && (W % 2) == 0; }

// tensor maps are cached per (pointer, shape, box): the engine's arena addresses are fixed, so a step encodes nothing.
// pairs = true: the [N][H][W/2][64] pair-row view with `box` pairs per box; false: the plain NHWC view with `box` pixels (SWIZZLE_64B)
inline int conv_tc_tmap(const bf16* in, int N, int H, int W, const CUtensorMap** out, int box = ConvTcCfg<>::BOXP, bool pairs = true) {
    struct Entry { const void* ptr; int n, h, w, box; bool pairs; CUtensorMap map; };
    static thread_local std::vector<Entry> cache;
    for (const Entry& e : cache)
        if (e.ptr == in && e.n == N && e.h == H && e.w == W && e.box == box && e.pairs == pairs) { *out = &e.map; return 0; }
    if (cache.size() >= 1024) cache.clear();
    cache.reserve(1024);              // pointers into the cache are handed out: never reallocate
    Entry e; e.ptr = in; e.n = N; e.h = H; e.w = W; e.box = box; e.pairs = pairs;
    if (pairs) PTTA_TRY(make_tmap_pairs(&e.map, in, N, H, W, box));
    else PTTA_TRY(make_tmap_nhwc(&e.map, in, N, H, W, 32, box));
    cache.push_back(e);
    *out = &cache.back().map;
    return 0;
}

// work split shared by the stride-1 kernels: strips of 256 pixels, a contiguous range of (image, strip, row) per CTA
inline int conv_tc_split(ConvTcParams& p, int sms) {
    p.strips = cdiv(p.W, 256);
    p.total_rows = p.N * p.strips * p.H;
    // rows per CTA: minimise waves x (rows + halo + fixed cost) over the splits that fill the machine
    int best_rows = p.total_rows; long long best_cost = -1;
    for (int rows = 1; rows <= p.total_rows; ++rows) {
        const long long ctas = cdiv(p.total_rows, rows);
        const long long waves = (ctas + sms - 1) / sms;
        const long long cost = waves * (rows + 2 + 4);
        if (best_cost < 0 || cost < best_cost) { best_cost = cost; best_rows = rows; }
        if (ctas <= 1) break;
    }
    p.rows_per_cta = best_rows;
    return cdiv(p.total_rows, p.rows_per_cta);
}

// out_f32[n][y][x] = bias0 [+ add_f32[n][y][x]] + sum_taps in[n][y+ky-1][x+kx-1][:] . w[tap][:]   (p.w = image of pack_conv_weight_tc_head_kernel)
inline int launch_conv_tc_head(const bf16* in, ConvTcParams p, cudaStream_t st) {
    typedef ConvTcCfg<> C;
    static int sms = 0;
    if (!sms) {
        PTTA_CUDA(cudaFuncSetAttribute(conv3x3_tc_head_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM));
        int dev = 0;
        PTTA_CUDA(cudaGetDevice(&dev));
        PTTA_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    }
    PTTA_CHECK(conv_tc_supported(p.N, p.H, p.W), "conv3x3_tc_head: W=%d must be even", p.W);
    PTTA_CHECK(p.out_f32 != nullptr && p.w != nullptr, "conv3x3_tc_head: output / weight image missing");
    const int grid = conv_tc_split(p, sms);
    const CUtensorMap* m = nullptr;
    PTTA_TRY(conv_tc_tmap(in, p.N, p.H, p.W, &m));
    const CUtensorMap map_in = *m;
    launch_k(conv3x3_tc_head_kernel, grid, C::THREADS, C::SMEM, st, map_in, p);
    return check_launch("conv3x3_tc_head");
}

template <bool MASK, bool ADDS, bool UP2>
inline void launch_conv_tc_variant(int grid, cudaStream_t st, const CUtensorMap& map_in, const CUtensorMap& map_out, const CUtensorMap& map_out2,
                                   const CUtensorMap& map_mask, const CUtensorMap& map_add, const CUtensorMap& map_up, const ConvTcParams& p) {
    typedef ConvTcCfg<MASK, ADDS, UP2> C;
    launch_k(conv3x3_tc_kernel<MASK, ADDS, UP2>, grid, C::THREADS, C::SMEM, st, map_in, map_out, map_out2, map_mask, map_add, map_up, p);
}

inline int launch_conv_tc(const bf16* in, ConvTcParams p, cudaStream_t st) {
    static int sms = 0;
    if (!sms) {
        PTTA_CUDA(cudaFuncSetAttribute(conv3x3_tc_kernel<false, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvTcCfg<false, false, false>::SMEM));
        PTTA_CUDA(cudaFuncSetAttribute(conv3x3_tc_kernel<false, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvTcCfg<false, true, false>::SMEM));
        PTTA_CUDA(cudaFuncSetAttribute(conv3x3_tc_kernel<true, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvTcCfg<true, false, false>::SMEM));
        PTTA_CUDA(cudaFuncSetAttribute(conv3x3_tc_kernel<true, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvTcCfg<true, true, false>::SMEM));
        PTTA_CUDA(cudaFuncSetAttribute(conv3x3_tc_kernel<false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvTcCfg<false, false, true>::SMEM));
        PTTA_CUDA(cudaFuncSetAttribute(conv3x3_tc_kernel<false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvTcCfg<false, true, true>::SMEM));
        int dev = 0;
        PTTA_CUDA(cudaGetDevice(&dev));
        PTTA_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    }
    PTTA_CHECK(conv_tc_supported(p.N, p.H, p.W), "conv3x3_tc: W=%d must be even", p.W);
    PTTA_CHECK(!(p.up2 && p.mask), "conv3x3_tc: the upsampled addend and a derivative mask are never used together");
    PTTA_CHECK(!(p.out2 && p.mask), "conv3x3_tc: a derivative mask and the second output are never used together");
    PTTA_CHECK(!(p.add && p.add2), "conv3x3_tc: add and add2 are mutually exclusive");
    PTTA_CHECK(!p.relu_in, "conv3x3_tc: ReLU-on-load is not supported (producers store ReLU(x): relu_out)");
    PTTA_CHECK(!p.up2 || ((p.H & 1) == 0 && (p.W & 1) == 0), "conv3x3_tc: the x2-upsampled addend needs even H, W (got %dx%d)", p.H, p.W);
    const int grid = conv_tc_split(p, sms);
    // copies: the cache may be cleared by a later lookup, the kernel takes the maps by value
    const CUtensorMap* m = nullptr;
    PTTA_TRY(conv_tc_tmap(in, p.N, p.H, p.W, &m));
    const CUtensorMap map_in = *m;
    PTTA_TRY(conv_tc_tmap(p.out, p.N, p.H, p.W, &m, 32));
    const CUtensorMap map_out = *m;
    CUtensorMap map_out2 = map_out, map_mask = map_out, map_add = map_out, map_up = map_out;
    if (p.out2) { PTTA_TRY(conv_tc_tmap(p.out2, p.N, p.H, p.W, &m, 32)); map_out2 = *m; }
    const bf16* addsrc = p.add ? p.add : p.add2;
    const int opbox = ConvTcCfg<true>::OP_BYTES / 128;
    if (p.mask) { PTTA_TRY(conv_tc_tmap(p.mask, p.N, p.H, p.W, &m, opbox)); map_mask = *m; }
    if (addsrc) { PTTA_TRY(conv_tc_tmap(addsrc, p.N, p.H, p.W, &m, opbox)); map_add = *m; }
    if (p.up2) { PTTA_TRY(conv_tc_tmap(p.up2, p.N, p.H / 2, p.W / 2, &m, ConvTcCfg<false, false, true>::UP_BOX, false)); map_up = *m; }
    const bool mask = p.mask != nullptr, adds = addsrc != nullptr, up2 = p.up2 != nullptr;
    if (up2) {
        if (adds) launch_conv_tc_variant<false, true, true>(grid, st, map_in, map_out, map_out2, map_mask, map_add, map_up, p);
        else launch_conv_tc_variant<false, false, true>(grid, st, map_in, map_out, map_out2, map_mask, map_add, map_up, p);
    } else if (mask) {
        if (adds) launch_conv_tc_variant<true, true, false>(grid, st, map_in, map_out, map_out2, map_mask, map_add, map_up, p);
        else launch_conv_tc_variant<true, false, false>(grid, st, map_in, map_out, map_out2, map_mask, map_add, map_up, p);
    } else {
        if (adds) launch_conv_tc_variant<false, true, false>(grid, st, map_in, map_out, map_out2, map_mask, map_add, map_up, p);
        else launch_conv_tc_variant<false, false, false>(grid, st, map_in, map_out, map_out2, map_mask, map_add, map_up, p);
    }
    return check_launch("conv3x3_tc");
}

}  // namespace ptta
