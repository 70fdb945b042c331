// C ABI of libmelgan_b200.so (see include/melgan_b200.h for the contract of every entry point).
#include <new>
#include <stdlib.h>
#include <string.h>

#include "mg_common.cuh"

namespace mg {

// (error plumbing: mg_error.cu.  The first-generation fp32 SIMT generator is NOT part of this library: it builds into the
//  test-only libmelgan_b200_simt_test.so, csrc/testlib.)

static int *status_ptr(void *workspace, int B, int T) {
    return reinterpret_cast<int *>(reinterpret_cast<float *>(workspace) + ws_offset(6, (size_t)B, (size_t)T));
}

// mel_host / audio_host: optional pinned host buffers (the engine entry point); the copies ride on the batch slices' streams
// lengths: optional host array of per-item lengths (ragged batch), already validated
static int run_generator(const float *packed, const float *mel, float *audio, int B, int T, float *ws, cudaStream_t s,
                         cudaEvent_t *ev, const float *mel_host = nullptr, float *audio_host = nullptr, const int *lengths = nullptr) {
    int *st = status_ptr(ws, B, T);
    MG_CUDA_TRY(cudaMemsetAsync(st, 0, sizeof(int), s));
    return launch_generator_tc(packed, mel, audio, B, T, ws, st, s, ev, mel_host, audio_host, lengths);
}

static int check_lengths(const char *fn, const int *lengths, int B, int T) {
    if (!lengths) return set_error(MG_ERR_INVALID_ARGUMENT, "%s: lengths is NULL", fn);
    for (int i = 0; i < B; ++i)
        if (lengths[i] < 1 || lengths[i] > T)
            return set_error(MG_ERR_INVALID_ARGUMENT, "%s: lengths[%d] = %d is outside [1, T = %d]", fn, i, lengths[i], T);
    return MG_OK;
}

static int check_shape(const char *fn, int B, int T) {
    if (B < 1 || T < 1) return set_error(MG_ERR_INVALID_ARGUMENT, "%s: need B >= 1 and T >= 1 (got B=%d, T=%d)", fn, B, T);
    if ((long long)B * T > (1ll << 24)) return set_error(MG_ERR_INVALID_ARGUMENT, "%s: B*T = %lld too large", fn, (long long)B * T);
    return MG_OK;
}

// Parity-test entry points run ONE kernel synchronously with their own status word: launch, wait, report a timed-out pipeline.
template <class F>
static int run_one_kernel(const char *fn, cudaStream_t stream, F launch) {
    int *st = nullptr;
    MG_CUDA_TRY(cudaMalloc(&st, sizeof(int)));
    cudaMemsetAsync(st, 0, sizeof(int), stream);
    int rc = launch(st);
    int h = 0;
    if (rc == MG_OK) {
        cudaError_t e = cudaStreamSynchronize(stream);
        if (e != cudaSuccess) rc = set_error(MG_ERR_CUDA, "%s: %s", fn, cudaGetErrorString(e));
        else if (cudaMemcpy(&h, st, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess || h)
            rc = set_error(MG_ERR_CUDA, "%s: pipeline wait timed out (role code %d)", fn, h);
    }
    cudaFree(st);
    return rc;
}

}  // namespace mg

using namespace mg;

extern "C" {

int mg_abi_version(void) { return 2; }

const char *mg_last_error_string(void) { return error_buffer(); }

int mg_device_check(void) {
    int dev = 0;
    MG_CUDA_TRY(cudaGetDevice(&dev));
    cudaDeviceProp p;
    MG_CUDA_TRY(cudaGetDeviceProperties(&p, dev));
    if (p.major != 10)
        return set_error(MG_ERR_UNSUPPORTED_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a (B200) only",
                         dev, p.major, p.minor);
    return MG_OK;
}

size_t mg_gen_packed_bytes(void) { return packed_total_bytes(); }

int mg_gen_pack(const float *const *v, const float *const *g, const float *const *bias, void *packed, void *stream) {
    if (!v || !g || !bias || !packed) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_gen_pack: null argument");
    if ((uintptr_t)packed % 16) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_gen_pack: packed must be 16-byte aligned");
    return launch_pack(v, g, bias, (float *)packed, (cudaStream_t)stream);
}

size_t mg_gen_workspace_bytes(int B, int T) {
    if (B < 1 || T < 1) return 0;
    return ws_offset(6, (size_t)B, (size_t)T) * sizeof(float) + 256;  // + pipeline status word
}

int mg_gen_forward(const void *packed, const float *mel, float *audio, int B, int T, void *workspace,
                   size_t workspace_bytes, void *stream) {
    int rc = check_shape("mg_gen_forward", B, T);
    if (rc) return rc;
    if (!packed || !mel || !audio || !workspace) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_gen_forward: null argument");
    if (workspace_bytes < mg_gen_workspace_bytes(B, T))
        return set_error(MG_ERR_WORKSPACE_TOO_SMALL, "mg_gen_forward: workspace %zu < %zu bytes", workspace_bytes,
                         mg_gen_workspace_bytes(B, T));
    if ((uintptr_t)packed % 16 || (uintptr_t)workspace % 16)
        return set_error(MG_ERR_INVALID_ARGUMENT, "mg_gen_forward: packed/workspace must be 16-byte aligned");
    return run_generator((const float *)packed, mel, audio, B, T, (float *)workspace, (cudaStream_t)stream, nullptr);
}

int mg_gen_forward_varlen(const void *packed, const float *mel, float *audio, int B, int T, const int *lengths, void *workspace,
                          size_t workspace_bytes, void *stream) {
    int rc = check_shape("mg_gen_forward_varlen", B, T);
    if (rc) return rc;
    if (!packed || !mel || !audio || !workspace) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_gen_forward_varlen: null argument");
    if ((rc = check_lengths("mg_gen_forward_varlen", lengths, B, T))) return rc;
    if (workspace_bytes < mg_gen_workspace_bytes(B, T))
        return set_error(MG_ERR_WORKSPACE_TOO_SMALL, "mg_gen_forward_varlen: workspace %zu < %zu bytes", workspace_bytes,
                         mg_gen_workspace_bytes(B, T));
    if ((uintptr_t)packed % 16 || (uintptr_t)workspace % 16)
        return set_error(MG_ERR_INVALID_ARGUMENT, "mg_gen_forward_varlen: packed/workspace must be 16-byte aligned");
    return run_generator((const float *)packed, mel, audio, B, T, (float *)workspace, (cudaStream_t)stream, nullptr, nullptr,
                         nullptr, lengths);
}

int mg_gen_forward_timed(const void *packed, const float *mel, float *audio, int B, int T, void *workspace,
                         size_t workspace_bytes, void *stream, float *kernel_ms) {
    int rc = check_shape("mg_gen_forward_timed", B, T);
    if (rc) return rc;
    if (!packed || !mel || !audio || !workspace || !kernel_ms)
        return set_error(MG_ERR_INVALID_ARGUMENT, "mg_gen_forward_timed: null argument");
    if (workspace_bytes < mg_gen_workspace_bytes(B, T))
        return set_error(MG_ERR_WORKSPACE_TOO_SMALL, "mg_gen_forward_timed: workspace too small");
    const int n = mg_gen_forward_launches();  // events: one before each launch + one after the last
    cudaEvent_t ev[17];  // at most 12 kernels
    for (int i = 0; i <= n; ++i) MG_CUDA_TRY(cudaEventCreate(&ev[i]));
    rc = run_generator((const float *)packed, mel, audio, B, T, (float *)workspace, (cudaStream_t)stream, ev);
    if (rc == MG_OK) {
        cudaError_t e = cudaEventSynchronize(ev[n]);
        if (e != cudaSuccess) rc = set_error(MG_ERR_CUDA, "mg_gen_forward_timed: %s", cudaGetErrorString(e));
        for (int i = 0; i < n && rc == MG_OK; ++i)
            if (cudaEventElapsedTime(&kernel_ms[i], ev[i], ev[i + 1]) != cudaSuccess)
                rc = set_error(MG_ERR_CUDA, "mg_gen_forward_timed: cudaEventElapsedTime failed");
    }
    for (int i = 0; i <= n; ++i) cudaEventDestroy(ev[i]);
    return rc;
}

const char *mg_gen_kernel_name(int i) { return generator_tc_kernel_name(i); }

const char *mg_gen_kernel_config(int i, int T) { return generator_tc_kernel_config(i, T); }

int mg_gen_set_pipeline(int tail_mask) {
    if (tail_mask < -1 || tail_mask > 15) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_gen_set_pipeline: mask %d", tail_mask);
    generator_tc_set_tail(tail_mask);
    return MG_OK;
}

int mg_gen_stage_output(const void *workspace, int which, float *out, int B, int T, void *stream) {
    int rc = check_shape("mg_gen_stage_output", B, T);
    if (rc) return rc;
    if (which < 0 || which > 3 || !workspace || !out)
        return set_error(MG_ERR_INVALID_ARGUMENT, "mg_gen_stage_output: which must be 0..3 (the last stage is fused with conv_post)");
    if (which > 0 && generator_tc_tail() != 0)
        return set_error(MG_ERR_INVALID_ARGUMENT, "mg_gen_stage_output: ResBlock outputs are not materialised while the next stage's "
                         "ConvT is fused at their kernel's tail; select the unfused chain with mg_gen_set_pipeline(0) first");
    const size_t off = ws_offset(which, B, T), n = ws_offset(which + 1, B, T) - off;
    MG_CUDA_TRY(cudaMemcpyAsync(out, (const float *)workspace + off, n * sizeof(float), cudaMemcpyDeviceToDevice,
                                (cudaStream_t)stream));
    return MG_OK;
}

size_t mg_msd_grouped_backward_workspace_bytes(int layer, int Bt, int Lout) {
    if (layer < 1 || layer > 4 || Bt < 1 || Lout < 1) return 0;
    return grouped_bwd_workspace_bytes(layer, Bt, Lout);
}

int mg_msd_grouped_backward(const void *packed, int scale, int layer, const float *dz, const float *x, float *dx, float *dw,
                            float *db, void *workspace, size_t workspace_bytes, int Bt, int Lin, int Lout, void *stream) {
    if (!packed || !dz || scale < 0 || scale > 2 || layer < 1 || layer > 4 || Bt < 1 || Lin < 1 || Lout < 1)
        return set_error(MG_ERR_INVALID_ARGUMENT, "mg_msd_grouped_backward: bad argument");
    const DLayer d = d_layer(layer);
    if (Lout != (Lin + 2 * d.pad - d.k) / d.stride + 1)
        return set_error(MG_ERR_INVALID_ARGUMENT, "mg_msd_grouped_backward: Lout %d does not follow from Lin %d", Lout, Lin);
    if (dw && (!x || !db || !workspace || workspace_bytes < grouped_bwd_workspace_bytes(layer, Bt, Lout)))
        return set_error(MG_ERR_WORKSPACE_TOO_SMALL, "mg_msd_grouped_backward: dw needs x, db and a workspace of %zu bytes",
                         grouped_bwd_workspace_bytes(layer, Bt, Lout));
    const uint8_t *blob = reinterpret_cast<const uint8_t *>(packed) + (size_t)scale * d_blob_bytes();
    return launch_disc_grouped_backward(blob, layer, dz, x, dx, dw, db, (float *)workspace, Bt, Lin, Lout, (cudaStream_t)stream);
}

int mg_msd_post1_dgrad(const void *packed, int scale, const float *dz, float *dx, int Bt, int L, void *status_word, void *stream) {
    if (!packed || !dz || !dx || dz == dx || !status_word || scale < 0 || scale > 2 || Bt < 1 || L < 1)
        return set_error(MG_ERR_INVALID_ARGUMENT, "mg_msd_post1_dgrad: bad argument");
    const uint8_t *blob = reinterpret_cast<const uint8_t *>(packed) + (size_t)scale * d_blob_bytes();
    return launch_disc_post1_dgrad_tc(dz, dx, blob + d_tcT_start(), reinterpret_cast<const float *>(blob + d_zero_start()), Bt, L,
                                      (int *)status_word, (cudaStream_t)stream);
}

int mg_msd_post1_wgrad(const float *x, const float *dz, float *dw, float *db, int Bt, int L, void *status_word, void *stream) {
    if (!x || !dz || !dw || !db || !status_word || Bt < 1 || L < 1)
        return set_error(MG_ERR_INVALID_ARGUMENT, "mg_msd_post1_wgrad: bad argument");
    return launch_disc_post1_wgrad_tc(x, dz, dw, db, Bt, L, (int *)status_word, (cudaStream_t)stream);
}

size_t mg_msd_edge_backward_workspace_bytes(int layer, int Bt, int L) {
    return (layer == 0 && Bt > 0 && L > 0) ? edge_bwd_workspace_bytes(layer, Bt, L) : 0;
}

int mg_msd_edge_backward(const void *packed, int scale, int layer, const float *dz, const float *x, float *dx, float *dw, float *db,
                         void *workspace, size_t workspace_bytes, int Bt, int L, void *stream) {
    if (!packed || !dz || !x || !dw || !db || scale < 0 || scale > 2 || (layer != 0 && layer != 6) || Bt < 1 || L < 1)
        return set_error(MG_ERR_INVALID_ARGUMENT, "mg_msd_edge_backward: bad argument (layer is 0 = conv_pre or 6 = conv_post2)");
    if (layer == 0 && (!workspace || workspace_bytes < edge_bwd_workspace_bytes(0, Bt, L)))
        return set_error(MG_ERR_WORKSPACE_TOO_SMALL, "mg_msd_edge_backward: conv_pre needs a workspace of %zu bytes",
                         edge_bwd_workspace_bytes(0, Bt, L));
    const uint8_t *blob = reinterpret_cast<const uint8_t *>(packed) + (size_t)scale * d_blob_bytes();
    return launch_disc_edge_backward(blob, layer, dz, x, dx, dw, db, (float *)workspace, Bt, L, (cudaStream_t)stream);
}

size_t mg_msd_scale_backward_workspace_bytes(int Bt, int L0) {
    return (Bt > 0 && L0 > 0) ? disc_scale_backward_workspace_bytes(Bt, L0) : 0;
}

int mg_msd_scale_backward(const void *packed, int scale, const float *x0, const float *const *fmap, const float *const *gfmap,
                          float *gx0, float *const *dw, float *const *db, int *reached, void *workspace, size_t workspace_bytes,
                          int Bt, int L0, void *status_word, void *stream) {
    if (!packed || !x0 || !fmap || !gfmap || !dw || !db || !workspace || !status_word || scale < 0 || scale > 2 || Bt < 1 || L0 < 1)
        return set_error(MG_ERR_INVALID_ARGUMENT, "mg_msd_scale_backward: bad argument");
    for (int l = 0; l < kDiscLayers; ++l)
        if (!fmap[l]) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_msd_scale_backward: fmap[%d] is NULL", l);
    if (Bt > 65535) return set_error(MG_ERR_INVALID_ARGUMENT, "discriminator batch %d exceeds 65535", Bt);
    const uint8_t *blob = reinterpret_cast<const uint8_t *>(packed) + (size_t)scale * d_blob_bytes();
    return launch_disc_scale_backward(blob, x0, fmap, gfmap, gx0, dw, db, reached, workspace, workspace_bytes, Bt, L0,
                                      (int *)status_word, (cudaStream_t)stream);
}

int mg_lrelu_backward(const float *g1, const float *g2, const float *out, float *dz, long long n, void *stream) {
    return launch_lrelu_grad(g1, g2, out, dz, n, (cudaStream_t)stream);
}

int mg_msd_wn_backward(const float *const *v, const float *const *g, const float *const *dw, float *const *dv,
                       float *const *dg, void *stream) {
    if (!v || !g || !dw || !dv || !dg) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_msd_wn_backward: null argument");
    return launch_disc_wn_backward(v, g, dw, dv, dg, (cudaStream_t)stream);
}

int mg_adam_chunk(void) { return 4096; }

int mg_adam_step(float *const *p, const float *const *g, float *const *m, float *const *v, const long long *n,
                 const int *first, int count, int total_ctas, float lr, float beta1, float beta2, float eps,
                 float weight_decay, long long step, void *stream) {
    return launch_adam(p, g, m, v, n, first, count, total_ctas, lr, beta1, beta2, eps, weight_decay, step, (cudaStream_t)stream);
}

size_t mg_loss_workspace_bytes(const long long *n, int count) {
    if (!n || count < 1) return 0;
    return (size_t)loss_num_ctas(n, count) * sizeof(float);
}

int mg_loss_forward(const float *const *a, const float *const *b, const long long *n, const int *mode, int count,
                    float *out, void *workspace, size_t workspace_bytes, void *stream) {
    if (!out || !workspace) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_loss_forward: null argument");
    if (n && count >= 1 && workspace_bytes < mg_loss_workspace_bytes(n, count))
        return set_error(MG_ERR_WORKSPACE_TOO_SMALL, "mg_loss_forward: workspace too small");
    return launch_loss_forward(a, b, n, mode, count, out, (float *)workspace, (cudaStream_t)stream);
}

int mg_loss_backward(const float *const *a, const float *const *b, const long long *n, const int *mode, int count,
                     const float *grad_out, float *const *grad_a, float *const *grad_b, void *stream) {
    if (!grad_out) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_loss_backward: null grad_out");
    return launch_loss_backward(a, b, n, mode, count, grad_out, grad_a, grad_b, (cudaStream_t)stream);
}

int mg_gen_forward_launches(void) { return generator_tc_num_launches(); }

int mg_gen_forward_slices(int B, int T) { return (B >= 1 && T >= 1) ? generator_tc_slices(B, T) : 1; }

int mg_gen_check_status(const void *workspace, int B, int T, void *stream) {
    int rc = check_shape("mg_gen_check_status", B, T);
    if (rc) return rc;
    if (!workspace) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_gen_check_status: null workspace");
    MG_CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    int st = 0;
    MG_CUDA_TRY(cudaMemcpy(&st, status_ptr(const_cast<void *>(workspace), B, T), sizeof(int), cudaMemcpyDeviceToHost));
    if (st) return set_error(MG_ERR_CUDA, "tensor-core pipeline wait timed out (role code %d)", st);
    return MG_OK;
}

int mg_gen_convt(const void *packed, int stage, const float *x, float *y, int B, int Lin, void *stream) {
    if (!packed || !x || !y || x == y || stage < 0 || stage > 3 || B < 1 || Lin < 1)
        return set_error(MG_ERR_INVALID_ARGUMENT, "mg_gen_convt: bad argument");
    return run_one_kernel("mg_gen_convt", (cudaStream_t)stream, [&](int *st) {
        return launch_convt_tc(x, y, (const float *)packed, stage, B, Lin, st, (cudaStream_t)stream);
    });
}

int mg_gen_conv_pre(const void *packed, const float *mel, float *y, int B, int T, void *stream) {
    if (!packed || !mel || !y || B < 1 || T < 1) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_gen_conv_pre: bad argument");
    return run_one_kernel("mg_gen_conv_pre", (cudaStream_t)stream, [&](int *st) {
        return launch_gen_pre_tc(mel, y, (const float *)packed, B, T, st, (cudaStream_t)stream);
    });
}

int mg_gen_resblock_post(const void *packed, const float *x, float *audio, int B, int L, void *stream) {
    if (!packed || !x || !audio || B < 1 || L < 1) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_gen_resblock_post: bad argument");
    return run_one_kernel("mg_gen_resblock_post", (cudaStream_t)stream, [&](int *st) {
        return launch_resblock_tc(x, audio, (const float *)packed, 4, B, L, st, (cudaStream_t)stream);
    });
}

/* Diagnostic: runs one tensor-core ResBlock and returns clock64 stamps of one interior CTA in trace[0..127]
 * (host buffer): [0] start, [1] input loaded, per conv c: [2+3c] X handed to MMA warp, [3+3c] accumulator ready,
 * [4+3c] next X written, [20] output stored; MMA thread: [64+3c] X received, [65+3c] first weights landed,
 * [66+3c] last MMA issued. */
int mg_gen_resblock_trace(const void *packed, int stage, const float *x, float *y, int B, int L, long long *trace_host) {
    if (!packed || !x || !y || x == y || !trace_host || stage < 0 || stage > 3)
        return set_error(MG_ERR_INVALID_ARGUMENT, "mg_gen_resblock_trace: bad argument");
    int *st = nullptr;
    long long *tr = nullptr;
    MG_CUDA_TRY(cudaMalloc(&st, sizeof(int)));
    MG_CUDA_TRY(cudaMalloc(&tr, 128 * sizeof(long long)));
    cudaMemset(st, 0, sizeof(int));
    cudaMemset(tr, 0, 128 * sizeof(long long));
    int rc = launch_resblock_tc(x, y, (const float *)packed, stage, B, L, st, 0, tr);
    if (rc == MG_OK && cudaDeviceSynchronize() != cudaSuccess) rc = set_error(MG_ERR_CUDA, "mg_gen_resblock_trace: kernel failed");
    if (rc == MG_OK) cudaMemcpy(trace_host, tr, 128 * sizeof(long long), cudaMemcpyDeviceToHost);
    cudaFree(st);
    cudaFree(tr);
    return rc;
}

int mg_gen_resblock(const void *packed, int stage, const float *x, float *y, int B, int L, void *stream) {
    if (!packed || !x || !y || x == y || stage < 0 || stage > 3 || B < 1 || L < 1)
        return set_error(MG_ERR_INVALID_ARGUMENT, "mg_gen_resblock: bad argument");
    return run_one_kernel("mg_gen_resblock", (cudaStream_t)stream, [&](int *st) {
        return launch_resblock_tc(x, y, (const float *)packed, stage, B, L, st, (cudaStream_t)stream);
    });
}

int mg_gen_resup(const void *packed, int stage, const float *x, float *y, int B, int L, void *stream) {
    if (!packed || !x || !y || x == y || stage < 0 || stage > 2 || B < 1 || L < 1)
        return set_error(MG_ERR_INVALID_ARGUMENT, "mg_gen_resup: bad argument");
    return run_one_kernel("mg_gen_resup", (cudaStream_t)stream, [&](int *st) {
        return launch_resblock_tc(x, y, (const float *)packed, 20 + stage, B, L, st, (cudaStream_t)stream);
    });
}

int mg_gen_upres(const void *packed, int stage, const float *x, float *y, int B, int Lin, void *stream) {
    if (!packed || !x || !y || x == y || (stage != 2 && stage != 3) || B < 1 || Lin < 1)
        return set_error(MG_ERR_INVALID_ARGUMENT, "mg_gen_upres: bad argument");
    return run_one_kernel("mg_gen_upres", (cudaStream_t)stream, [&](int *st) {
        return launch_resblock_tc(x, y, (const float *)packed, 10 + stage, B, 2 * Lin, st, (cudaStream_t)stream);
    });
}

/* ------------------------------- multi-scale discriminator ------------------------------- */

size_t mg_msd_packed_bytes(void) { return msd_packed_bytes(); }

int mg_msd_pack(const float *const *v, const float *const *g, const float *const *bias, void *packed, void *stream) {
    if (!v || !g || !bias || !packed) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_msd_pack: null argument");
    if ((uintptr_t)packed % 256) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_msd_pack: packed must be 256-byte aligned");
    return launch_disc_pack(v, g, bias, packed, (cudaStream_t)stream);
}

int mg_msd_lengths(int L, int *lens) {
    if (L < 1 || !lens) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_msd_lengths: bad argument");
    msd_lengths(L, lens);
    for (int i = 0; i < 21; ++i)
        if (lens[i] < 1) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_msd_lengths: L = %d is too short for the discriminators", L);
    return MG_OK;
}

int mg_msd_forward(const void *packed, const float *y, int Bt, int L, float *const *fmaps, void *status_word, void *stream) {
    if (!packed || !y || !fmaps || !status_word || Bt < 1 || L < 1)
        return set_error(MG_ERR_INVALID_ARGUMENT, "mg_msd_forward: bad argument");
    int lens[21];
    int rc = mg_msd_lengths(L, lens);
    if (rc) return rc;
    for (int i = 0; i < 21; ++i)
        if (!fmaps[i]) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_msd_forward: null feature-map pointer %d", i);
    MG_CUDA_TRY(cudaMemsetAsync(status_word, 0, sizeof(int), (cudaStream_t)stream));
    return launch_msd_forward(packed, y, Bt, L, fmaps, (int *)status_word, (cudaStream_t)stream);
}

size_t mg_disc_packed_bytes(void) { return d_blob_bytes(); }

int mg_disc_pack(const float *const *v, const float *const *g, const float *const *bias, void *packed, void *stream) {
    if (!v || !g || !bias || !packed) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_disc_pack: null argument");
    if ((uintptr_t)packed % 256) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_disc_pack: packed must be 256-byte aligned");
    return launch_disc_pack(v, g, bias, packed, (cudaStream_t)stream, 1);
}

int mg_disc_forward(const void *packed, const float *x, int Bt, int L, float *const *fmaps, void *status_word, void *stream) {
    if (!packed || !x || !fmaps || !status_word || Bt < 1 || L < 1)
        return set_error(MG_ERR_INVALID_ARGUMENT, "mg_disc_forward: bad argument");
    int lens[21];
    msd_lengths(L, lens);
    for (int i = 0; i < 7; ++i) {
        if (lens[i] < 1) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_disc_forward: L = %d is too short", L);
        if (!fmaps[i]) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_disc_forward: null feature-map pointer %d", i);
    }
    MG_CUDA_TRY(cudaMemsetAsync(status_word, 0, sizeof(int), (cudaStream_t)stream));
    return launch_disc_forward(packed, x, Bt, L, fmaps, (int *)status_word, (cudaStream_t)stream);
}

int mg_msd_check_status(const void *status_word, void *stream) {
    if (!status_word) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_msd_check_status: null argument");
    MG_CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    int st = 0;
    MG_CUDA_TRY(cudaMemcpy(&st, status_word, sizeof(int), cudaMemcpyDeviceToHost));
    if (st) return set_error(MG_ERR_CUDA, "tensor-core pipeline wait timed out (role code %d)", st);
    return MG_OK;
}

/* ------------------------------- mel-spectrogram front end -------------------------------- */

size_t mg_mel_tables_bytes(void) { return mel_tables_bytes(); }

int mg_mel_tables_build(int sampling_rate, int n_mels, float fmin, float fmax, int norm, void *tables_host) {
    if (!tables_host) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_mel_tables_build: null buffer");
    return mel_tables_build(sampling_rate, n_mels, fmin, fmax, norm, reinterpret_cast<MelTables *>(tables_host));
}

int mg_mel_frames(int L) { return L < 1 ? 0 : mel_frames(L); }

int mg_mel_spectrogram(const void *tables, const float *audio, float *mel, int B, int L, void *stream) {
    if (!tables || !audio || !mel || B < 1 || L < 1) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_mel_spectrogram: bad argument");
    if ((uintptr_t)tables % 16) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_mel_spectrogram: tables must be 16-byte aligned");
    return launch_mel(tables, audio, mel, B, L, (cudaStream_t)stream);
}

/* ------------------------------- host-buffer engine ------------------------------------- */

struct mg_gen_engine {
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    float *packed = nullptr;
    float *raw = nullptr;  // device staging for raw v/g/bias
    float *mel = nullptr, *audio = nullptr, *ws = nullptr;
    float *pin_in = nullptr, *pin_out = nullptr;
    int *pin_status = nullptr;
    size_t cap_frames = 0;  // B*T capacity
    bool loaded = false;
    float last_ms = 0.f;
};

static void engine_free_io(mg_gen_engine *e) {
    cudaFree(e->mel); cudaFree(e->audio); cudaFree(e->ws);
    cudaFreeHost(e->pin_in); cudaFreeHost(e->pin_out);
    e->mel = e->audio = e->ws = e->pin_in = e->pin_out = nullptr;
    e->cap_frames = 0;
}

static int engine_reserve(mg_gen_engine *e, size_t frames) {
    if (frames <= e->cap_frames) return MG_OK;
    engine_free_io(e);
    MG_CUDA_TRY(cudaMalloc(&e->mel, frames * kMelBins * sizeof(float)));
    MG_CUDA_TRY(cudaMalloc(&e->audio, frames * 256 * sizeof(float)));
    MG_CUDA_TRY(cudaMalloc(&e->ws, mg_gen_workspace_bytes(1, (int)frames)));
    MG_CUDA_TRY(cudaMallocHost(&e->pin_in, frames * kMelBins * sizeof(float)));
    MG_CUDA_TRY(cudaMallocHost(&e->pin_out, frames * 256 * sizeof(float)));
    e->cap_frames = frames;
    return MG_OK;
}

int mg_gen_engine_create(mg_gen_engine **out, int max_B, int max_T) {
    if (!out) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_gen_engine_create: null out");
    int rc = check_shape("mg_gen_engine_create", max_B, max_T);
    if (rc) return rc;
    if ((rc = mg_device_check())) return rc;
    mg_gen_engine *e = new (std::nothrow) mg_gen_engine();
    if (!e) return set_error(MG_ERR_OUT_OF_MEMORY, "mg_gen_engine_create: host allocation failed");
    *out = e;
    MG_CUDA_TRY(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    MG_CUDA_TRY(cudaEventCreate(&e->ev0));
    MG_CUDA_TRY(cudaEventCreate(&e->ev1));
    MG_CUDA_TRY(cudaMalloc((void **)&e->packed, mg_gen_packed_bytes()));
    MG_CUDA_TRY(cudaMalloc(&e->raw, (packed_float_count() + 4353) * sizeof(float)));
    return engine_reserve(e, (size_t)max_B * max_T);
}

int mg_gen_engine_load_state(mg_gen_engine *e, const float *const *v, const float *const *g, const float *const *bias) {
    if (!e || !v || !g || !bias) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_gen_engine_load_state: null argument");
    const float *dv[kNumLayers], *dg[kNumLayers], *db[kNumLayers];
    float *p = e->raw;
    for (int l = 0; l < kNumLayers; ++l) {
        if (!v[l] || !g[l] || !bias[l]) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_gen_engine_load_state: null tensor, layer %d", l);
        const size_t nv = layer_weight_count(l), ng = layer_norm_rows(l), nb = layer_shape(l).cout;
        MG_CUDA_TRY(cudaMemcpyAsync(p, v[l], nv * sizeof(float), cudaMemcpyHostToDevice, e->stream)); dv[l] = p; p += nv;
        MG_CUDA_TRY(cudaMemcpyAsync(p, g[l], ng * sizeof(float), cudaMemcpyHostToDevice, e->stream)); dg[l] = p; p += ng;
        MG_CUDA_TRY(cudaMemcpyAsync(p, bias[l], nb * sizeof(float), cudaMemcpyHostToDevice, e->stream)); db[l] = p; p += nb;
    }
    int rc = launch_pack(dv, dg, db, e->packed, e->stream);
    if (rc) return rc;
    MG_CUDA_TRY(cudaStreamSynchronize(e->stream));
    e->loaded = true;
    return MG_OK;
}

static int engine_forward(mg_gen_engine *e, const float *mel_host, float *audio_host, int B, int T, const int *lengths) {
    int rc;
    if (!e->loaded) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_gen_engine_forward: no weights loaded");
    const size_t frames = (size_t)B * T;
    if ((rc = engine_reserve(e, frames))) return rc;
    const size_t nin = frames * kMelBins * sizeof(float), nout = frames * 256 * sizeof(float);
    cudaPointerAttributes at;
    const bool in_pinned = cudaPointerGetAttributes(&at, mel_host) == cudaSuccess && at.type == cudaMemoryTypeHost;
    const bool out_pinned = cudaPointerGetAttributes(&at, audio_host) == cudaSuccess && at.type == cudaMemoryTypeHost;
    cudaGetLastError();  // clear "invalid value" some drivers raise for pageable pointers
    const float *src = mel_host;
    if (!in_pinned) { memcpy(e->pin_in, mel_host, nin); src = e->pin_in; }
    if (!e->pin_status) MG_CUDA_TRY(cudaMallocHost(&e->pin_status, sizeof(int)));
    MG_CUDA_TRY(cudaEventRecord(e->ev0, e->stream));
    // upload, kernels and download are enqueued per batch slice (launch_generator_tc); one synchronisation at the end
    rc = run_generator(e->packed, e->mel, e->audio, B, T, e->ws, e->stream, nullptr, src, out_pinned ? audio_host : e->pin_out, lengths);
    if (rc) return rc;
    MG_CUDA_TRY(cudaEventRecord(e->ev1, e->stream));
    *e->pin_status = 0;
    MG_CUDA_TRY(cudaMemcpyAsync(e->pin_status, status_ptr(e->ws, B, T), sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    MG_CUDA_TRY(cudaStreamSynchronize(e->stream));
    if (!out_pinned) memcpy(audio_host, e->pin_out, nout);
    if (*e->pin_status)
        return set_error(MG_ERR_CUDA, "mg_gen_engine_forward: tensor-core pipeline wait timed out (code %d)", *e->pin_status);
    MG_CUDA_TRY(cudaEventElapsedTime(&e->last_ms, e->ev0, e->ev1));
    return MG_OK;
}

int mg_gen_engine_forward(mg_gen_engine *e, const float *mel_host, float *audio_host, int B, int T) {
    if (!e || !mel_host || !audio_host) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_gen_engine_forward: null argument");
    int rc = check_shape("mg_gen_engine_forward", B, T);
    if (rc) return rc;
    return engine_forward(e, mel_host, audio_host, B, T, nullptr);
}

int mg_gen_engine_forward_varlen(mg_gen_engine *e, const float *mel_host, float *audio_host, int B, int T, const int *lengths) {
    if (!e || !mel_host || !audio_host) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_gen_engine_forward_varlen: null argument");
    int rc = check_shape("mg_gen_engine_forward_varlen", B, T);
    if (rc) return rc;
    if ((rc = check_lengths("mg_gen_engine_forward_varlen", lengths, B, T))) return rc;
    return engine_forward(e, mel_host, audio_host, B, T, lengths);
}

int mg_gen_engine_last_kernel_ms(mg_gen_engine *e, float *ms) {
    if (!e || !ms) return set_error(MG_ERR_INVALID_ARGUMENT, "mg_gen_engine_last_kernel_ms: null argument");
    *ms = e->last_ms;
    return MG_OK;
}

void mg_gen_engine_destroy(mg_gen_engine *e) {
    if (!e) return;
    engine_free_io(e);
    cudaFree(e->packed); cudaFree(e->raw);
    if (e->pin_status) cudaFreeHost(e->pin_status);
    if (e->ev0) cudaEventDestroy(e->ev0);
    if (e->ev1) cudaEventDestroy(e->ev1);
    if (e->stream) cudaStreamDestroy(e->stream);
    delete e;
}

}  // extern "C"
