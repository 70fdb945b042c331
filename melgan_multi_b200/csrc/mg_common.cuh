// Shared helpers: error plumbing for the C ABI, cp.async wrappers, activation.
#pragma once
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#include <type_traits>

#include "../../include/melgan_b200.h"
#include "mg_layout.h"

namespace mg {

// thread-local error string (the only mutable global state of the library)
char *error_buffer();
int set_error(int code, const char *fmt, ...);

#define MG_CUDA_TRY(expr)                                                                     \
    do {                                                                                      \
        cudaError_t err__ = (expr);                                                           \
        if (err__ != cudaSuccess)                                                             \
            return ::mg::set_error(MG_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,               \
                                   cudaGetErrorString(err__), __FILE__, __LINE__);            \
    } while (0)

__device__ __forceinline__ float lrelu(float x) { return fmaxf(x, x * kSlope); }

__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gmem_src) {
    uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}

// Launch helper of the tensor-core kernels: optional thread-block cluster (x dimension) and programmatic dependent launch
// (mg_tc.cuh pdl_*; MG_PDL=0 in the environment turns the attribute off for A/B runs).
bool pdl_enabled();
template <class... KArgs, class... Args>
inline cudaError_t launch_ex(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, int cluster, bool pdl,
                             Args... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[2];
    int n = 0;
    if (cluster > 1) {
        attr[n].id = cudaLaunchAttributeClusterDimension;
        attr[n].val.clusterDim.x = cluster;
        attr[n].val.clusterDim.y = 1;
        attr[n].val.clusterDim.z = 1;
        ++n;
    }
    if (pdl && pdl_enabled()) {
        attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[n].val.programmaticStreamSerializationAllowed = 1;
        ++n;
    }
    cfg.attrs = attr;
    cfg.numAttrs = n;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// Per-item mel lengths of one ragged generator launch (mg_gen_forward_varlen).  Passed BY VALUE as a __grid_constant__ kernel
// parameter -- no device table, no copy, so the call stays asynchronous and graph-capturable.  Buffers keep the padded layout
// [item][C][mul * T]; only the first mul * (cum[b+1] - cum[b]) positions of item b are sequence.
//   cum[b]:   mel frames of the items before b (cum[n]: all of them)
//   first[b]: ResBlock launches: grid.x index (in super-tiles) of item b's first tile, first[n] = super-tiles in all
//   mul:      positions per mel frame at the kernel's input (1 conv_pre / up0, 8 res0, 64 res1, 64 up2, 128 res2, 256 res3)
// kVlMaxItems bounds the items of one launch: the struct (2 KB) stays far below the 32 KB kernel-parameter limit (parameter
// bytes are copied with every launch), and the launcher cuts a slice with more items into several launches.
constexpr int kVlMaxItems = 256;
struct VarLenTab {
    int n, mul;
    int cum[kVlMaxItems + 1];
    int first[kVlMaxItems + 1];
};
struct NoVarLen {};  // the uniform instantiations' (empty) parameter in the same place
template <bool VL>
using VarLenArg = typename std::conditional<VL, VarLenTab, NoVarLen>::type;

// the item that virtual row v (>= 0) belongs to when item b's rows start at  t.mul * t.cum[b] + pad * b;  t.n: past the last
__device__ __forceinline__ int vl_item_of_row(const VarLenTab &t, int pad, int v) {
    int lo = 0, hi = t.n;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (t.mul * t.cum[mid] + pad * mid <= v) lo = mid; else hi = mid - 1;
    }
    return lo;
}
// the item whose super-tiles [first[b], first[b+1]) contain grid index id (< first[n])
__device__ __forceinline__ int vl_item_of_tile(const VarLenTab &t, int id) {
    int lo = 0, hi = t.n - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (t.first[mid] <= id) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// ---- launches implemented in the .cu files ------------------------------------------------
int launch_pack(const float *const *v, const float *const *g, const float *const *bias, float *packed,
                cudaStream_t s);
// (test-only library, csrc/testlib) ev: nullptr, or 6 events recorded before each of the 5 launches and after the last one
int launch_generator_simt(const float *packed, const float *mel, float *audio, int B, int T, float *ws,
                          cudaStream_t s, cudaEvent_t *ev = nullptr);
int generator_simt_num_launches();
int generator_tc_num_launches();
int generator_tc_fused_up();  // bit 0: stage 2, bit 1: stage 3 run their stride-2 ConvT at the FRONT of the ResBlock kernel
int generator_tc_tail();      // bit i: stage i's ConvT runs at the TAIL of ResBlock i-1's kernel
void generator_tc_set_tail(int mask);
const char *generator_tc_kernel_name(int i);
const char *generator_tc_kernel_config(int i, int T);
const char *resblock_config_name(int stage, int L);
int generator_tc_slices(int B, int T);  // batch slices (concurrent kernel chains) one forward is cut into
int launch_generator_tc(const float *packed, const float *mel, float *audio, int B, int T, float *ws, int *status,
                        cudaStream_t s, cudaEvent_t *ev = nullptr, const float *mel_host = nullptr, float *audio_host = nullptr,
                        const int *lengths = nullptr);
int launch_gen_pre_tc_varlen(const float *mel, float *y, const float *packed, const VarLenTab &vt, int T, int *status, cudaStream_t s);
int launch_convt_tc_varlen(const float *x, float *y, const float *packed, int stage, const VarLenTab &vt, int T, int *status,
                           cudaStream_t s);
int launch_resblock_tc_varlen(const float *x, float *y, const float *packed, int code, const VarLenTab &vt, int T, int *status,
                              cudaStream_t s);
int launch_gen_pre_tc(const float *mel, float *y, const float *packed, int B, int T, int *status, cudaStream_t s);
int launch_disc_post1_tc(const float *x, float *y, const uint8_t *wtc, const float *bias, int Bt, int L, int *status,
                         cudaStream_t s);
int launch_disc_post1_dgrad_tc(const float *dz, float *dx, const uint8_t *wtcT, const float *zero_bias, int Bt, int L, int *status,
                               cudaStream_t s);
int launch_disc_post1_wgrad_tc(const float *x, const float *dz, float *dw, float *db, int Bt, int L, int *status, cudaStream_t s);
size_t disc_scale_backward_workspace_bytes(int Bt, int L0);
int launch_disc_scale_backward(const void *blob, const float *x0, const float *const *fmap, const float *const *gfmap, float *gx0,
                               float *const *dw, float *const *db, int *reached, void *workspace, size_t workspace_bytes, int Bt,
                               int L0, int *status, cudaStream_t st);
size_t edge_bwd_workspace_bytes(int l, int Bt, int L);
int launch_disc_edge_backward(const void *blob, int l, const float *dz, const float *x, float *dx, float *dw, float *db, float *ws,
                              int Bt, int L, cudaStream_t s);
int launch_disc_group_tc(const float *x, float *out, const uint8_t *wtc, const float *bias, int Bt, int Cin, int Cout,
                         int Lin, int Lout, int *status, cudaStream_t s);
int launch_disc_group4_tc(const float *x, float *out, const uint8_t *wtc, const float *bias, int Bt, int L, int *status,
                          cudaStream_t s);
int launch_disc_pack(const float *const *v, const float *const *g, const float *const *bias, void *packed, cudaStream_t s, int ndisc = 3);
int launch_disc_forward(const void *packed, const float *x, int Bt, int L, float *const *fmaps, int *status, cudaStream_t s);
void msd_lengths(int L, int *lens);
int launch_lrelu_grad(const float *g1, const float *g2, const float *out, float *dz, long long n, cudaStream_t s);
size_t grouped_bwd_workspace_bytes(int l, int Bt, int Lout);
int launch_disc_grouped_backward(const void *blob, int l, const float *dz, const float *x, float *dx, float *dw, float *db,
                                 float *ws, int Bt, int Lin, int Lout, cudaStream_t s);
int launch_disc_wn_backward(const float *const *v, const float *const *g, const float *const *dw, float *const *dv,
                            float *const *dg, cudaStream_t s);
int launch_adam(float *const *p, const float *const *g, float *const *m, float *const *v, const long long *n, const int *first,
                int count, int total_ctas, float lr, float b1, float b2, float eps, float wd, long long step, cudaStream_t s);
long long loss_num_ctas(const long long *n, int count);
int launch_loss_forward(const float *const *a, const float *const *b, const long long *n, const int *mode, int count, float *out,
                        float *partial, cudaStream_t s);
int launch_loss_backward(const float *const *a, const float *const *b, const long long *n, const int *mode, int count,
                         const float *gout, float *const *ga, float *const *gb, cudaStream_t s);
struct MelTables;
size_t mel_tables_bytes();
int mel_tables_build(int sr, int n_mels, float fmin, float fmax, int norm, MelTables *t);
int mel_frames(int L);
int launch_mel(const void *tables, const float *audio, float *mel, int B, int L, cudaStream_t s);
int launch_msd_forward(const void *packed, const float *y, int Bt, int L, float *const *fmaps, int *status, cudaStream_t s);
int launch_convt_tc(const float *x, float *y, const float *packed, int stage, int B, int Lin, int *status, cudaStream_t s);
int launch_resblock_tc(const float *x, float *y, const float *packed, int stage, int B, int L, int *status, cudaStream_t s,
                       long long *trace = nullptr);

}  // namespace mg
