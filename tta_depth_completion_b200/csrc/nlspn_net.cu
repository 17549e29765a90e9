// Second translation unit of libptta_b200.so: the general-channel tcgen05 convolution family and the channel-generic
// BatchNorm / activation kernels of the NLSPN network (SURVEY.md section 8 row a18), behind the C ABI of include/ptta_b200.h.
#include <cuda_runtime.h>
#include <string.h>
#include "common.cuh"
#include "conv_gen.cuh"
#include "nlspn_net.cuh"
#include "../../include/ptta_b200.h"

using namespace ptta;

extern "C" {

long long ptta_convg_packed_elems(int kind, int role, int cin0, int cin1, int cout, int has_short) {
    ConvGPlan pl;
    if (convg_make_plan(pl, kind, role, 1, 16, 16, cin0, cin1, cout, has_short)) return -1;
    return convg_packed_elems(pl);
}

int ptta_convg_pack(int kind, int role, const float* weight, const float* weight_short, int cin_w, int cout_w, int cin0, int cin1,
                    int cout, int has_short, int ident_from, void* packed, ptta_stream_t stream) {
    ConvGPlan pl;
    PTTA_TRY(convg_make_plan(pl, kind, role, 1, 16, 16, cin0, cin1, cout, has_short));
    PTTA_CHECK(weight && packed && (!has_short || weight_short), "convg_pack: null pointer");
    PTTA_CHECK(cin_w <= cin0 + cin1 && cout_w <= cout, "convg_pack: weight %d->%d larger than the stored %d->%d", cin_w, cout_w, cin0 + cin1, cout);
    return launch_convg_pack(pl, kind, role, weight, weight_short, cin_w, cout_w, ident_from, (bf16*)packed, (cudaStream_t)stream);
}

int ptta_convg_run(int kind, int role, const void* x0, const void* x1, const void* packed, const float* bias, void* out, int n, int h,
                   int w, int cin0, int cin1, int cout, int has_short, ptta_stream_t stream) {
    ConvGPlan pl;
    PTTA_TRY(convg_make_plan(pl, kind, role, n, h, w, cin0, cin1, cout, has_short));
    return launch_convg(pl, (const bf16*)x0, (const bf16*)x1, (const bf16*)packed, bias, (bf16*)out, (cudaStream_t)stream);
}

int ptta_convg_debug_set(int mask) {
#ifdef PTTA_EXPERIMENTS
    convg_multicast_flag() = (mask & 32) ? 1 : 0;
    PTTA_CUDA(cudaMemcpyToSymbol(g_convg_dbg, &mask, sizeof(int)));
    return 0;
#else
    // product build: the only switch is 32 (weight-tile multicast over 2-CTA clusters; results unchanged, tested).  The work-skipping
    // timing switches and the cycle stamps are compiled into the experiments build only
    PTTA_CHECK((mask & ~32) == 0, "convg_debug_set: mask %d needs the experiments build (-DPTTA_EXPERIMENTS); this library accepts 0 and 32", mask);
    convg_multicast_flag() = (mask & 32) ? 1 : 0;
    return 0;
#endif
}

int ptta_convg_debug_read_cta(unsigned long long* out_host, int n) {
#ifdef PTTA_EXPERIMENTS
    PTTA_CHECK(out_host && n > 0 && n <= 512, "convg_debug_read_cta: bad arguments");
    PTTA_CUDA(cudaDeviceSynchronize());
    PTTA_CUDA(cudaMemcpyFromSymbol(out_host, g_convg_cta, (size_t)n * sizeof(unsigned long long)));
    return 0;
#else
    (void)out_host; (void)n;
    PTTA_CHECK(false, "convg_debug_read_cta: experiments build only (-DPTTA_EXPERIMENTS)");
#endif
}

int ptta_convg_debug_read_ts(long long* out_host, int n) {
#ifdef PTTA_EXPERIMENTS
    PTTA_CHECK(out_host && n > 0 && n <= 64 * 16, "convg_debug_read_ts: bad arguments");
    PTTA_CUDA(cudaDeviceSynchronize());
    PTTA_CUDA(cudaMemcpyFromSymbol(out_host, g_convg_ts, (size_t)n * sizeof(long long)));
    return 0;
#else
    (void)out_host; (void)n;
    PTTA_CHECK(false, "convg_debug_read_ts: experiments build only (-DPTTA_EXPERIMENTS)");
#endif
}

int ptta_convg_run_thin(const void* x0, const void* x1, const void* packed, const float* bias, float* const* planes, const long long* nstrides,
                        const int* acts, int n_real, int n, int h, int w, int cin0, int cin1, ptta_stream_t stream) {
    ConvGPlan pl;
    PTTA_TRY(convg_make_plan(pl, CONVG_S1, 0, n, h, w, cin0, cin1, 16, 0));
    PTTA_CHECK(n_real >= 1 && n_real <= 16 && planes && nstrides && acts, "convg_run_thin: bad arguments");
    pl.p.thin_n = n_real;
    for (int c = 0; c < n_real; ++c) { pl.p.thin_ptr[c] = planes[c]; pl.p.thin_ns[c] = nstrides[c]; pl.p.thin_act[c] = acts[c]; }
    return launch_convg(pl, (const bf16*)x0, (const bf16*)x1, (const bf16*)packed, bias, nullptr, (cudaStream_t)stream);
}

int ptta_nl_stem(const float* image, const float* depth, const float* w_rgb, const float* b_rgb, const float* w_dep, const float* b_dep,
                 const float* scale, const float* shift, void* out, int n, int h, int w, ptta_stream_t stream) {
    PTTA_CHECK(depth && w_rgb && b_rgb && w_dep && b_dep && out, "nl_stem: null pointer");
    const long long total = (long long)n * h * w;
    launch_k(nl_stem_kernel, cdiv(total, 128), 128, 0, (cudaStream_t)stream, image, depth, w_rgb, b_rgb, w_dep, b_dep, scale, shift, (bf16*)out, n, h, w, n);
    return check_launch("nl_stem");
}

int ptta_nl_stem_pair(const float* image, const float* depth, const float* w_rgb, const float* b_rgb, const float* w_dep, const float* b_dep,
                      const float* scale, const float* shift, void* out, int n, int h, int w, ptta_stream_t stream) {
    PTTA_CHECK(image && depth && w_rgb && b_rgb && w_dep && b_dep && out, "nl_stem_pair: null pointer");
    const long long total = 2LL * n * h * w;
    launch_k(nl_stem_kernel, cdiv(total, 128), 128, 0, (cudaStream_t)stream, image, depth, w_rgb, b_rgb, w_dep, b_dep, scale, shift, (bf16*)out, 2 * n, h, w, n);
    return check_launch("nl_stem_pair");
}

int ptta_nl_reduce_blocks(long long rows, int c) {
    long long by_rows = (rows + 31) / 32;
    long long target = 592 / (c / 64 > 0 ? c / 64 : 1);
    if (target < 1) target = 1;
    long long b = by_rows < target ? by_rows : target;
    return (int)(b < 1 ? 1 : b);
}

int ptta_nl_bn_stats(const void* x, long long ldx, long long rows, int c, const float* gamma, const float* beta, float eps, float* partial,
                     float* mean, float* rstd, float* scale, float* shift, float* run_mean, float* run_var, long long* num_batches_tracked,
                     float momentum, ptta_stream_t stream) {
    PTTA_CHECK(x && gamma && beta && partial && mean && rstd && scale && shift && c % 64 == 0 && rows > 0, "nl_bn_stats: bad arguments");
    const int nblk = ptta_nl_reduce_blocks(rows, c);
    dim3 grid(nblk, c / 64);
    launch_k(chan_reduce_kernel<0>, grid, 256, 0, (cudaStream_t)stream, (const bf16*)x, ldx, nullptr, 0, nullptr, 0, nullptr, 0, nullptr, nullptr, rows, c, partial);
    PTTA_TRY(check_launch("nl_chan_stats"));
    launch_k(bn_finalize2_kernel, cdiv(c, 32), 1024, 0, (cudaStream_t)stream, partial, nblk, rows, c, gamma, beta, eps, mean, rstd, scale, shift, run_mean,
                                                                       run_var, num_batches_tracked, momentum, nullptr);
    return check_launch("nl_bn_finalize");
}

int ptta_nl_bn_stats_grouped(const void* x, long long ldx, long long rows_per_group, int groups, int c, const float* gamma, const float* beta,
                             float eps, float* partial, float* mean, float* rstd, float* scale, float* shift, ptta_stream_t stream) {
    PTTA_CHECK(x && gamma && beta && partial && mean && rstd && scale && shift && c % 64 == 0 && rows_per_group > 0 && groups >= 1 && groups <= 8,
               "nl_bn_stats_grouped: bad arguments");
    const int nblk = ptta_nl_reduce_blocks(rows_per_group, c);
    dim3 grid(nblk, c / 64, groups);
    launch_k(chan_reduce_kernel<0>, grid, 256, 0, (cudaStream_t)stream, (const bf16*)x, ldx, nullptr, 0, nullptr, 0, nullptr, 0, nullptr, nullptr, rows_per_group,
                                                                 c, partial);
    PTTA_TRY(check_launch("nl_chan_stats_grouped"));
    launch_k(bn_finalize2_kernel, dim3(cdiv(c, 32), groups), 1024, 0, (cudaStream_t)stream, partial, nblk, rows_per_group, c, gamma, beta, eps, mean, rstd, scale,
                                                                                    shift, nullptr, nullptr, nullptr, 0.f, nullptr);
    return check_launch("nl_bn_finalize_grouped");
}

int ptta_nl_col_sums(const void* x, long long ldx, long long rows, int c, float* partial, float* sums, ptta_stream_t stream) {
    PTTA_CHECK(x && partial && sums && c % 64 == 0 && rows > 0, "nl_col_sums: bad arguments");
    const int nblk = ptta_nl_reduce_blocks(rows, c);
    dim3 grid(nblk, c / 64);
    launch_k(chan_reduce_kernel<0>, grid, 256, 0, (cudaStream_t)stream, (const bf16*)x, ldx, nullptr, 0, nullptr, 0, nullptr, 0, nullptr, nullptr, rows, c, partial);
    PTTA_TRY(check_launch("nl_chan_stats"));
    launch_k(bn_finalize2_kernel, cdiv(c, 32), 1024, 0, (cudaStream_t)stream, partial, nblk, rows, c, nullptr, nullptr, 0.f, nullptr, nullptr, nullptr, nullptr,
                                                                       nullptr, nullptr, nullptr, 0.f, sums);
    return check_launch("nl_col_sums");
}

static int bn_act_launch(const void* x, const float* scale, const float* shift, const void* res, long long ldr, const float* rscale,
                         const float* rshift, void* y, long long rows, int c, int act, long long rows_per_group, ptta_stream_t stream);

int ptta_nl_bn_act(const void* x, const float* scale, const float* shift, const void* res, long long ldr, const float* rscale,
                   const float* rshift, void* y, long long rows, int c, int act, ptta_stream_t stream) {
    return bn_act_launch(x, scale, shift, res, ldr, rscale, rshift, y, rows, c, act, 0, stream);
}

int ptta_nl_bn_act_grouped(const void* x, const float* scale, const float* shift, const void* res, long long ldr, const float* rscale,
                           const float* rshift, void* y, long long rows_per_group, int groups, int c, int act, ptta_stream_t stream) {
    PTTA_CHECK(groups >= 1 && rows_per_group > 0, "nl_bn_act_grouped: bad arguments");
    return bn_act_launch(x, scale, shift, res, ldr, rscale, rshift, y, rows_per_group * groups, c, act, rows_per_group, stream);
}

static int bn_act_launch(const void* x, const float* scale, const float* shift, const void* res, long long ldr, const float* rscale,
                         const float* rshift, void* y, long long rows, int c, int act, long long rows_per_group, ptta_stream_t stream) {
    PTTA_CHECK(x && scale && shift && y && c % 64 == 0 && rows > 0 && (!rscale || (res && rshift)), "nl_bn_act: bad arguments");
    const long long total = (rows * (c / 8) + 1) / 2;
    launch_k(bn_act_kernel, cdiv(total, 256), 256, 0, (cudaStream_t)stream, (const bf16*)x, scale, shift, (const bf16*)res, ldr, rscale, rshift, (bf16*)y,
                                                                     rows, c, act, rows_per_group);
    return check_launch("nl_bn_act");
}

int ptta_nl_bn_backward(const void* dy_a, long long ld_a, const void* dy_b, long long ld_b, const void* y, int act, const void* x,
                        const float* mean, const float* rstd, const float* gamma, float* partial, float* dgamma, float* dbeta, float* coef,
                        void* dx, void* gskip, long long rows, int c, ptta_stream_t stream) {
    PTTA_CHECK(dy_a && x && mean && rstd && gamma && partial && coef && dx && c % 64 == 0 && rows > 0 && (!act || y), "nl_bn_backward: bad arguments");
    const int nblk = ptta_nl_reduce_blocks(rows, c);
    dim3 grid(nblk, c / 64);
    cudaStream_t st = (cudaStream_t)stream;
    launch_k(chan_reduce_kernel<1>, grid, 256, 0, st, (const bf16*)x, c, (const bf16*)dy_a, ld_a, (const bf16*)dy_b, ld_b, (const bf16*)y, act, mean, rstd,
                                               rows, c, partial);
    PTTA_TRY(check_launch("nl_bn_bwd_reduce"));
    launch_k(bn_bwd_finalize2_kernel, cdiv(c, 32), 1024, 0, st, partial, nblk, rows, c, gamma, rstd, dgamma, dbeta, coef, coef + c, coef + 2 * c);
    PTTA_TRY(check_launch("nl_bn_bwd_finalize"));
    const long long total = (rows * (c / 8) + 1) / 2;
    launch_k(bn_bwd_apply2_kernel, cdiv(total, 256), 256, 0, st, (const bf16*)dy_a, ld_a, (const bf16*)dy_b, ld_b, (const bf16*)y, act, (const bf16*)x, mean,
                                                          rstd, coef, coef + c, coef + 2 * c, (bf16*)dx, (bf16*)gskip, rows, c);
    return check_launch("nl_bn_bwd_apply");
}

// shared-model mode: the communicator must have every peer mapped, and one BatchNorm's sums must fit an exchange slot
static int comm_check(const ptta_comm* comm, int xid, int c, const char* what) {
    PTTA_CHECK(comm, "%s: null communicator", what);
    PTTA_CHECK(xid >= 0 && xid < PTTA_COMM_MAX_XID, "%s: exchange id %d outside [0, %d)", what, xid, PTTA_COMM_MAX_XID);
    PTTA_CHECK(2 * c <= PTTA_COMM_BN_DOUBLES, "%s: %d channels exceed the exchange slot (%d)", what, c, PTTA_COMM_BN_DOUBLES / 2);
    for (int r = 0; r < comm->dev.world; ++r) PTTA_CHECK(comm->dev.base[r] != nullptr, "%s: peer %d not opened (ptta_comm_open_peers)", what, r);
    return 0;
}

int ptta_nl_bn_stats_comm(const void* x, long long ldx, long long rows, int c, const float* gamma, const float* beta, float eps, float* partial,
                          float* mean, float* rstd, float* scale, float* shift, float* run_mean, float* run_var, long long* num_batches_tracked,
                          float momentum, ptta_comm* comm, int xid, ptta_stream_t stream) {
    PTTA_CHECK(x && gamma && beta && partial && mean && rstd && scale && shift && c % 64 == 0 && rows > 0, "nl_bn_stats_comm: bad arguments");
    PTTA_TRY(comm_check(comm, xid, c, "nl_bn_stats_comm"));
    const int nblk = ptta_nl_reduce_blocks(rows, c);
    dim3 grid(nblk, c / 64);
    launch_k(chan_reduce_kernel<0>, grid, 256, 0, (cudaStream_t)stream, (const bf16*)x, ldx, nullptr, 0, nullptr, 0, nullptr, 0, nullptr, nullptr, rows, c, partial);
    PTTA_TRY(check_launch("nl_chan_stats"));
    launch_k(bn_finalize2_sync_kernel, cdiv(c, 32), 1024, 0, (cudaStream_t)stream, partial, nblk, rows, c, gamma, beta, eps, mean, rstd, scale, shift, run_mean,
                                                                            run_var, num_batches_tracked, momentum, comm->dev, xid);
    return check_launch("nl_bn_finalize_sync");
}

int ptta_nl_bn_backward_comm(const void* dy_a, long long ld_a, const void* dy_b, long long ld_b, const void* y, int act, const void* x,
                             const float* mean, const float* rstd, const float* gamma, float* partial, float* dgamma, float* dbeta, float* coef,
                             void* dx, void* gskip, long long rows, int c, ptta_comm* comm, int xid, ptta_stream_t stream) {
    PTTA_CHECK(dy_a && x && mean && rstd && gamma && partial && coef && dx && c % 64 == 0 && rows > 0 && (!act || y), "nl_bn_backward_comm: bad arguments");
    PTTA_TRY(comm_check(comm, xid, c, "nl_bn_backward_comm"));
    const int nblk = ptta_nl_reduce_blocks(rows, c);
    dim3 grid(nblk, c / 64);
    cudaStream_t st = (cudaStream_t)stream;
    launch_k(chan_reduce_kernel<1>, grid, 256, 0, st, (const bf16*)x, c, (const bf16*)dy_a, ld_a, (const bf16*)dy_b, ld_b, (const bf16*)y, act, mean, rstd,
                                               rows, c, partial);
    PTTA_TRY(check_launch("nl_bn_bwd_reduce"));
    launch_k(bn_bwd_finalize2_sync_kernel, cdiv(c, 32), 1024, 0, st, partial, nblk, rows, c, gamma, rstd, dgamma, dbeta, coef, coef + c, coef + 2 * c,
                                                               comm->dev, xid);
    PTTA_TRY(check_launch("nl_bn_bwd_finalize_sync"));
    const long long total = (rows * (c / 8) + 1) / 2;
    launch_k(bn_bwd_apply2_kernel, cdiv(total, 256), 256, 0, st, (const bf16*)dy_a, ld_a, (const bf16*)dy_b, ld_b, (const bf16*)y, act, (const bf16*)x, mean,
                                                          rstd, coef, coef + c, coef + 2 * c, (bf16*)dx, (bf16*)gskip, rows, c);
    return check_launch("nl_bn_bwd_apply");
}

int ptta_nl_add3(const void* a, long long lda, const void* b, long long ldb, const void* c3, long long ldc, void* out, long long rows, int c,
                 ptta_stream_t stream) {
    PTTA_CHECK(a && b && out && c % 64 == 0 && rows > 0, "nl_add3: bad arguments");
    const long long total = rows * (c / 8);
    launch_k(add3_kernel, cdiv(total, 256), 256, 0, (cudaStream_t)stream, (const bf16*)a, lda, (const bf16*)b, ldb, (const bf16*)c3, ldc, (bf16*)out, rows, c);
    return check_launch("nl_add3");
}

int ptta_nl_clamp0(const float* y, float* out, long long n, ptta_stream_t stream) {
    launch_k(clamp0_kernel, cdiv(n, 256), 256, 0, (cudaStream_t)stream, y, out, n);
    return check_launch("nl_clamp0");
}

int ptta_nl_clamp(const float* x, float* out, float lo, float hi, long long n, ptta_stream_t stream) {
    launch_k(clamp_range_kernel, cdiv(n, 256), 256, 0, (cudaStream_t)stream, x, out, lo, hi, n);
    return check_launch("nl_clamp");
}

int ptta_nl_mask_pos(const float* g, const float* y, float* out, long long n, ptta_stream_t stream) {
    launch_k(mask_pos_kernel, cdiv(n, 256), 256, 0, (cudaStream_t)stream, g, y, out, n);
    return check_launch("nl_mask_pos");
}

int ptta_nl_thin_grad_pack(const float* g_pred, const float* pred_init, const float* g_guide, const float* g_conf, const float* conf, void* out,
                           int n, int h, int w, ptta_stream_t stream) {
    PTTA_CHECK(g_pred && pred_init && g_guide && g_conf && conf && out, "nl_thin_grad_pack: null pointer");
    const long long hw = (long long)h * w;
    launch_k(thin_grad_pack_kernel, cdiv(n * hw, 256), 256, 0, (cudaStream_t)stream, g_pred, pred_init, g_guide, g_conf, conf, (bf16*)out, n, hw);
    return check_launch("nl_thin_grad_pack");
}

int ptta_nl_conv8to24(const float* in, const float* weight, const float* bias, float* out, int n, int h, int w, int transposed, ptta_stream_t stream) {
    PTTA_CHECK(in && weight && out, "nl_conv8to24: null pointer");
    const long long total = (long long)n * h * w;
    if (transposed) launch_k(conv8to24_kernel<true>, cdiv(total, 128), 128, 0, (cudaStream_t)stream, in, weight, nullptr, out, n, h, w);
    else launch_k(conv8to24_kernel<false>, cdiv(total, 128), 128, 0, (cudaStream_t)stream, in, weight, bias, out, n, h, w);
    return check_launch("nl_conv8to24");
}

static int wgrad48_grid() {
    static int sms = 0;
    if (!sms) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) sms = 148;
    }
    return sms;
}

size_t ptta_nl_wgrad48_workspace_bytes(void) { return (size_t)wgrad48_grid() * 9 * 48 * 48 * sizeof(float); }

int ptta_nl_wgrad48(const void* x, const void* gout, float* dw, void* workspace, int n, int h, int w, ptta_stream_t stream) {
    PTTA_CHECK(x && gout && dw && workspace, "nl_wgrad48: null pointer");
    static bool attr = false;
    if (!attr) {
        PTTA_CUDA(cudaFuncSetAttribute(wgrad48_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, Wgrad48Cfg::SMEM));
        attr = true;
    }
    const int tiles = n * cdiv(h, 16) * cdiv(w, 16);
    const int grid = tiles < wgrad48_grid() ? tiles : wgrad48_grid();
    launch_k(wgrad48_kernel, grid, Wgrad48Cfg::THREADS, Wgrad48Cfg::SMEM, (cudaStream_t)stream, (const bf16*)x, (const bf16*)gout, (float*)workspace, n, h, w);
    PTTA_TRY(check_launch("nl_wgrad48"));
    launch_k(wgrad48_reduce_kernel, cdiv(9 * 48 * 48, 256), 256, 0, (cudaStream_t)stream, (const float*)workspace, dw, grid);
    return check_launch("nl_wgrad48_reduce");
}

size_t ptta_eval_metrics_workspace_bytes(void) { return 296 * 5 * sizeof(double); }

int ptta_eval_metrics(const float* output_depth, const float* ground_truth, long long n, float min_depth, float max_depth, void* workspace,
                      float* result5, ptta_stream_t stream) {
    PTTA_CHECK(output_depth && ground_truth && workspace && result5 && n > 0, "eval_metrics: bad arguments");
    int blocks = (int)(cdiv(n, 256) < 296 ? cdiv(n, 256) : 296);
    launch_k(eval_metrics_kernel, blocks, 256, 0, (cudaStream_t)stream, output_depth, ground_truth, n, min_depth, max_depth, (double*)workspace);
    PTTA_TRY(check_launch("eval_metrics"));
    launch_k(eval_metrics_finalize_kernel, 1, 256, 0, (cudaStream_t)stream, (const double*)workspace, blocks, result5);
    return check_launch("eval_metrics_finalize");
}

int ptta_input_stage(const void* image_u8_hwc, const void* depth_u16, float* image_nchw, float* depth, float* validity, int n, int h0, int w0,
                     int y0, int x0, int h, int w, float depth_multiplier, ptta_stream_t stream) {
    PTTA_CHECK(image_u8_hwc && depth_u16 && image_nchw && depth && validity, "input_stage: null pointer");
    PTTA_CHECK(n >= 1 && y0 >= 0 && x0 >= 0 && h >= 1 && w >= 1 && y0 + h <= h0 && x0 + w <= w0 && depth_multiplier > 0.f,
               "input_stage: crop %dx%d at (%d,%d) does not fit %dx%d", h, w, y0, x0, h0, w0);
    const long long total = (long long)n * h * w;
    launch_k(input_stage_kernel, cdiv(total, 256), 256, 0, (cudaStream_t)stream, (const unsigned char*)image_u8_hwc, (const unsigned short*)depth_u16, image_nchw,
                                                                          depth, validity, n, h0, w0, y0, x0, h, w, depth_multiplier);
    return check_launch("input_stage");
}

// host-only: the plan convg_make_plan builds for a layer, flattened into ints (CPU tests replay the implicit GEMM from it).
// header[16] = {n_items, n_classes, th, tw, tiles_y, tiles_x, n_tiles, BN, halo, b_resident, n_a, n_b, in_parity, out_parity, n_out, halo_rev},
// then per class {start, count, out_c, out_py}, then per item {c_inner, dx, dy, py, src, wsel, tap, k0}.  Returns the ints written, < 0 on error.
int ptta_convg_plan_describe(int kind, int role, int n, int h, int w, int cin0, int cin1, int cout, int has_short, int* out, int capacity) {
    ConvGPlan pl;
    if (convg_make_plan(pl, kind, role, n, h, w, cin0, cin1, cout, has_short)) return -1;
    const int need = 16 + 4 * 4 + 8 * pl.n_items;
    if (!out || capacity < need) { set_error("convg_plan_describe: need %d ints", need); return -need; }
    const ConvGParams& p = pl.p;
    const int hdr[16] = {pl.n_items, p.n_classes, p.th, p.tw, p.tiles_y, p.tiles_x, p.n_tiles, p.BN, p.halo, p.b_resident, p.n_a, p.n_b,
                         pl.in_parity, pl.out_parity, pl.n_out, p.halo_rev};
    int k = 0;
    for (int i = 0; i < 16; ++i) out[k++] = hdr[i];
    for (int c = 0; c < 4; ++c) { out[k++] = p.cls_start[c]; out[k++] = p.cls_count[c]; out[k++] = p.cls_out_c[c]; out[k++] = p.cls_out_py[c]; }
    for (int i = 0; i < pl.n_items; ++i) {
        const ConvGItem& it = p.items[i];
        int dx = it.dx, dy = (int)(short)(it.dyps & 0xffff);
        if (p.halo) {          // halo mode: the tap position is the descriptor offset into the 18x10 halo whose origin is (-1, -1)
            const int hpix = it.a_off16 / 8;
            dy = hpix / ConvGCfg::HALO_W - 1;
            dx = hpix % ConvGCfg::HALO_W - 1;
        }
        out[k++] = it.c_inner; out[k++] = dx; out[k++] = dy; out[k++] = (it.dyps >> 16) & 3; out[k++] = (it.dyps >> 20) & 1;
        out[k++] = (pl.pack[i].wsel_tap >> 8) & 1; out[k++] = pl.pack[i].wsel_tap & 255; out[k++] = pl.pack[i].k0;
    }
    return k;
}

}  // extern "C"
