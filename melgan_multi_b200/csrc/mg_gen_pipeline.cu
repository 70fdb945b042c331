// The generator's tensor-core pipeline: which kernels run, in what order, on which streams.
//   conv_pre -> 4 x [LeakyReLU -> ConvTranspose1d -> ResBlock] (-> LeakyReLU -> conv_post -> tanh), models.py:61-71,
// as 8 kernels per chain (mg_conv_tc.cu, mg_up_tc.cu, mg_res_tc.cu), the batch cut into concurrent slices.
#include <stdlib.h>

#include "mg_common.cuh"

namespace mg {

// Pipeline shape.  TAIL mask: bit i (i = 1..3) set = ConvTranspose of stage i runs at the TAIL of ResBlock i-1's kernel
// (mg_res_tc.cu, UPT): the chain is then  conv_pre, up0, res0+up1, res1+up2, res2+up3, res3+post  -- six kernels, no ResBlock
// output ever written to HBM.  Default: stages 1 and 3 (measured at config 2: res0+up1 and res2+up3 beat their two-kernel
// forms; res1+up2 does not -- the extra halo row a tail ConvT needs turns the 9 tiles of a 2048-position item into 10, i.e.
// 640 CTAs = 5 waves instead of 576 = 4).  MG_GEN_TAIL=<digits> ("123", "0" for none) / mg_gen_set_pipeline() override it.  Where stage 3's ConvT is not at res2's tail it runs at the FRONT of the last
// kernel (UPF, "up3+res3+post") unless MG_GEN_FUSE_UP says otherwise (bit 0: stage 2 front-fused, bit 1: stage 3).
static thread_local int g_tail_override = -1;
void generator_tc_set_tail(int mask) { g_tail_override = mask; }
int generator_tc_tail() {
    static const int env_mask = [] {
        const char *e = getenv("MG_GEN_TAIL");
        if (!e) return 0b1010;
        int m = 0;
        for (; *e; ++e) m |= (*e >= '1' && *e <= '3') ? 1 << (*e - '0') : 0;
        return m;
    }();
    return g_tail_override >= 0 ? (g_tail_override & 0b1110) : env_mask;
}
int generator_tc_fused_up() {
    static const int mask = [] {
        const char *e = getenv("MG_GEN_FUSE_UP");
        if (!e) return 2;
        int m = 0;
        for (; *e; ++e) m |= (*e == '2') ? 1 : (*e == '3') ? 2 : 0;
        return m;
    }();
    return mask;
}

// The chain as a list of steps (shared by the launcher, the launch counter and the kernel-name table).
struct ChainStep {
    const char *name;
    int kind;  // 0 conv_pre, 1 ConvT (arg = stage), 2 ResBlock kernel (arg = launch_resblock_tc code)
    int arg;
};
static int build_chain(ChainStep *st) {
    const int tail = generator_tc_tail(), front = generator_tc_fused_up();
    int n = 0;
    st[n++] = {"conv_pre", 0, 0};
    st[n++] = {"up0", 1, 0};
    if (tail & 2) st[n++] = {"res0+up1", 2, 20};
    else { st[n++] = {"res0", 2, 0}; st[n++] = {"up1", 1, 1}; }
    if (tail & 4) st[n++] = {"res1+up2", 2, 21};
    else if (front & 1) st[n++] = {"res1", 2, 1};
    else { st[n++] = {"res1", 2, 1}; st[n++] = {"up2", 1, 2}; }
    const bool front2 = !(tail & 4) && (front & 1);
    if (tail & 8) { st[n++] = {front2 ? "up2+res2+up3" : "res2+up3", 2, front2 ? -1 : 22}; st[n++] = {"res3+post", 2, 4}; }
    else if (front & 2) { st[n++] = {front2 ? "up2+res2" : "res2", 2, front2 ? 12 : 2}; st[n++] = {"up3+res3+post", 2, 14}; }
    else { st[n++] = {front2 ? "up2+res2" : "res2", 2, front2 ? 12 : 2}; st[n++] = {"up3", 1, 3}; st[n++] = {"res3+post", 2, 4}; }
    return n;
}
int generator_tc_num_launches() {
    ChainStep st[12];
    return build_chain(st);
}
const char *generator_tc_kernel_name(int i) {
    ChainStep st[12];
    const int n = build_chain(st);
    return (i >= 0 && i < n) ? st[i].name : "";
}

// template configuration of chain kernel i at T mel frames (what evidence files record; "" for non-ResBlock kernels)
const char *generator_tc_kernel_config(int i, int T) {
    ChainStep st[12];
    const int n = build_chain(st);
    if (i < 0 || i >= n || T < 1) return "";
    int len = T;
    for (int k = 0; k <= i; ++k) {
        if (st[k].kind == 1) len *= stage_stride(st[k].arg);
        else if (st[k].kind == 2) {
            const int a = st[k].arg;
            const int Lk = (a >= 12 && a <= 14) ? 2 * len : len;
            if (k == i) return resblock_config_name(a, Lk);
            len = a >= 20 ? Lk * stage_stride(a - 20 + 1) : Lk;
        }
    }
    return st[i].kind == 0 ? "conv_rows_tc_kernel<ConvCfg<80,512,7>>" : "convt_tc_kernel";
}

// Tensor-core pipeline of one contiguous slice of the batch.  a0: conv_pre output; a[0]: ResBlock-0 output (unfused chains);
// a[1], a[2], u: three buffers of 8192 T floats per item that the stages rotate through (a kernel never writes its input).
static int generator_tc_chain(const float *packed, const float *mel, float *audio, int B, int T, float *a0, float *const *a,
                              float *u, int *status, cudaStream_t s, cudaEvent_t *ev) {
    ChainStep st[12];
    const int n = build_chain(st);
    int rc;
    float *big[3] = {a[1], a[2], u};
    auto other = [&](const float *x, const float *y) -> float * {  // a rotation buffer that is neither x nor y
        for (float *b : big)
            if (b != x && b != y) return b;
        return nullptr;
    };
    const float *cur = mel;
    int len = T;  // length of `cur`
    for (int i = 0; i < n; ++i) {
        if (ev) MG_CUDA_TRY(cudaEventRecord(ev[i], s));
        const ChainStep &k = st[i];
        if (k.kind == 0) {
            if ((rc = launch_gen_pre_tc(cur, a0, packed, B, T, status, s))) return rc;
            cur = a0;
        } else if (k.kind == 1) {
            float *out = cur != u ? u : other(cur, nullptr);  // (unfused chain: ConvT outputs live in u, ResBlock i's in a[i])
            if ((rc = launch_convt_tc(cur, out, packed, k.arg, B, len, status, s))) return rc;
            cur = out;
            len *= stage_stride(k.arg);
        } else {
            if (k.arg < 0) return set_error(MG_ERR_INVALID_ARGUMENT, "generator pipeline: MG_GEN_FUSE_UP=2 cannot be combined with a tail-fused up3");
            const bool last = k.arg == 4 || k.arg == 14;
            const bool front = k.arg >= 12 && k.arg <= 14, tailf = k.arg >= 20;
            float *out = last ? audio : (k.arg <= 2 && cur != a[k.arg]) ? a[k.arg] : other(cur, nullptr);
            const int Lk = front ? 2 * len : len;  // the ResBlock's own length
            if ((rc = launch_resblock_tc(cur, out, packed, k.arg, B, Lk, status, s))) return rc;
            cur = out;
            len = tailf ? Lk * stage_stride(k.arg - 20 + 1) : Lk;
        }
    }
    if (ev) MG_CUDA_TRY(cudaEventRecord(ev[n], s));
    return MG_OK;
}

// The default chain on a ragged batch (vt: per-item lengths of this slice), whatever the A/B knobs above select: conv_pre -> a0,
// up0 -> u, res0+up1 -> a1, res1 -> a2, up2 -> u, res2+up3 -> a1, res3+post -> audio -- the buffers the uniform default chain uses.
static int generator_tc_chain_varlen(const float *packed, const float *mel, float *audio, const VarLenTab &vt, int T, float *a0,
                                     float *a1, float *a2, float *u, int *status, cudaStream_t s) {
    int rc;
    if ((rc = launch_gen_pre_tc_varlen(mel, a0, packed, vt, T, status, s))) return rc;
    if ((rc = launch_convt_tc_varlen(a0, u, packed, 0, vt, T, status, s))) return rc;
    if ((rc = launch_resblock_tc_varlen(u, a1, packed, 20, vt, T, status, s))) return rc;
    if ((rc = launch_resblock_tc_varlen(a1, a2, packed, 1, vt, T, status, s))) return rc;
    if ((rc = launch_convt_tc_varlen(a2, u, packed, 2, vt, T, status, s))) return rc;
    if ((rc = launch_resblock_tc_varlen(u, a1, packed, 22, vt, T, status, s))) return rc;
    return launch_resblock_tc_varlen(a1, audio, packed, 4, vt, T, status, s);
}

// Side streams for batch slices (forked from / joined into the caller's stream with events: the call stays asynchronous
// and stream-ordered for the caller).  Per host thread, like the rest of the library's state.
constexpr int kMaxDevices = 64;
struct SliceStreams {
    static constexpr int kMax = 8;
    cudaStream_t st[kMax - 1] = {};
    cudaEvent_t fork = nullptr, join[kMax - 1] = {};
    bool ready = false;
    int init() {
        if (ready) return MG_OK;
        for (int i = 0; i < kMax - 1; ++i) {
            MG_CUDA_TRY(cudaStreamCreateWithFlags(&st[i], cudaStreamNonBlocking));
            MG_CUDA_TRY(cudaEventCreateWithFlags(&join[i], cudaEventDisableTiming));
        }
        MG_CUDA_TRY(cudaEventCreateWithFlags(&fork, cudaEventDisableTiming));
        ready = true;
        return MG_OK;
    }
};

// Whole generator.  The batch items are independent and every kernel's grid is a whole number of tiles per item (or per
// 128 virtual rows), so the batch is cut into `slices` contiguous parts whose nine-kernel chains run on forked streams:
// the block scheduler fills the SMs one chain's partial last wave leaves idle (stage 0 at config 2 is 192 one-per-SM
// tiles on 148 SMs) with the other chain's tiles.  Same kernels, same per-item arithmetic: results are bit-identical
// to the single-chain order.  ev != nullptr (per-kernel timing) keeps everything on one stream.
int generator_tc_slices(int B, int T) {
    static const int forced = [] {  // MG_GEN_SLICES=n pins the slice count (experiments); default: chosen from the shape
        const char *e = getenv("MG_GEN_SLICES");
        const int v = e ? atoi(e) : 0;
        return v < 0 ? 0 : v > SliceStreams::kMax ? SliceStreams::kMax : v;
    }();
    // slicing pays while a slice still fills the machine: >= 512 mel frames per slice (stage-0 tiles ~ frames / 11)
    int slices = forced ? forced : 4;
    while (slices > 1 && ((!forced && (long long)B * T < 512ll * slices) || B < slices)) --slices;
    return slices;
}

// mel_host / audio_host (both or neither; pinned): the host-buffer entry point's copies, cut the same way -- each slice's
// stream uploads its mel slice before its chain and downloads its audio slice after it, so all but the last download
// overlap the other chains' kernels.
//
// lengths (host, B values in [1, T], checked by the caller): ragged batch -- the default chain with per-item lengths
// (generator_tc_chain_varlen).  Slices are then cut by cumulative mel frames instead of item counts (the same >= 512 frames per
// slice), and a slice with more than kVlMaxItems items runs as several launches in a row on its stream: each launch's
// tables travel as kernel parameters (VarLenTab), which bounds their size.
int launch_generator_tc(const float *packed, const float *mel, float *audio, int B, int T, float *ws, int *status,
                        cudaStream_t s, cudaEvent_t *ev, const float *mel_host, float *audio_host, const int *lengths) {
    long long frames = (long long)B * T;
    if (lengths) {
        frames = 0;
        for (int i = 0; i < B; ++i) frames += lengths[i];
    }
    int slices = ev ? 1 : generator_tc_slices(B, T);
    if (lengths && !ev) {  // the uniform rule on the frames that are really there
        slices = SliceStreams::kMax < 4 ? SliceStreams::kMax : 4;
        while (slices > 1 && (frames < 512ll * slices || B < slices)) --slices;
    }
    float *base[6];
    for (int i = 0; i < 6; ++i) base[i] = ws + ws_offset(i, B, T);
    const size_t per_item[6] = {(size_t)512 * T, (size_t)256 * 8 * T, (size_t)128 * 64 * T, (size_t)64 * 128 * T, 0, (size_t)8192 * T};
    const size_t mel_item = (size_t)kMelBins * T, audio_item = (size_t)256 * T;
    // one pool per (host thread, device): streams and events belong to the device that was current when they were created
    static thread_local SliceStreams pools[kMaxDevices];
    int dev = 0;
    MG_CUDA_TRY(cudaGetDevice(&dev));
    if (dev < 0 || dev >= kMaxDevices) return set_error(MG_ERR_INVALID_ARGUMENT, "launch_generator_tc: device ordinal %d", dev);
    SliceStreams &ss = pools[dev];
    int rc = MG_OK;
    if (slices > 1) {
        if ((rc = ss.init())) return rc;
        MG_CUDA_TRY(cudaEventRecord(ss.fork, s));
    }
    int forked = 0;  // side streams that wait on `fork` so far: all of them are joined back, also on the error path
    long long acc = 0;  // (ragged) mel frames of the items before b0
    for (int k = 0, b0 = 0; k < slices && rc == MG_OK; ++k) {
        int nb = B / slices + (k < B % slices);
        if (lengths) {  // items up to the k+1-th share of the frames (at least one; the last slice takes the rest)
            nb = 0;
            for (long long a = acc; b0 + nb < B && (k == slices - 1 || nb == 0 || a < frames * (k + 1) / slices); ++nb) a += lengths[b0 + nb];
            nb = nb < B - b0 - (slices - 1 - k) ? nb : B - b0 - (slices - 1 - k);  // every later slice keeps an item
            for (int i = 0; i < nb; ++i) acc += lengths[b0 + i];
        }
        cudaStream_t q = k == 0 ? s : ss.st[k - 1];
        auto slice = [&]() -> int {
            if (k > 0) {
                MG_CUDA_TRY(cudaStreamWaitEvent(q, ss.fork, 0));
                forked = k;
            }
            if (mel_host)
                MG_CUDA_TRY(cudaMemcpyAsync(const_cast<float *>(mel) + b0 * mel_item, mel_host + b0 * mel_item,
                                            nb * mel_item * sizeof(float), cudaMemcpyHostToDevice, q));
            float *a[3] = {base[1] + b0 * per_item[1], base[2] + b0 * per_item[2], base[3] + b0 * per_item[3]};
            int r = MG_OK;
            if (lengths) {
                static thread_local VarLenTab vt;  // (4 KB: not on the stack; copied into each launch's parameters)
                for (int c0 = 0; c0 < nb && r == MG_OK; c0 += kVlMaxItems) {  // launches of at most kVlMaxItems items
                    const int b = b0 + c0;
                    vt.n = nb - c0 < kVlMaxItems ? nb - c0 : kVlMaxItems;
                    vt.mul = 1;
                    vt.cum[0] = 0;
                    for (int i = 0; i < vt.n; ++i) vt.cum[i + 1] = vt.cum[i] + lengths[b + i];
                    r = generator_tc_chain_varlen(packed, mel + b * mel_item, audio + b * audio_item, vt, T, base[0] + b * per_item[0],
                                                  a[1] + c0 * per_item[2], a[2] + c0 * per_item[3], base[5] + b * per_item[5], status, q);
                }
            } else {
                r = generator_tc_chain(packed, mel + b0 * mel_item, audio + b0 * audio_item, nb, T, base[0] + b0 * per_item[0], a,
                                       base[5] + b0 * per_item[5], status, q, ev);
            }
            if (r) return r;
            if (audio_host)
                MG_CUDA_TRY(cudaMemcpyAsync(audio_host + b0 * audio_item, audio + b0 * audio_item, nb * audio_item * sizeof(float),
                                            cudaMemcpyDeviceToHost, q));
            return MG_OK;
        };
        rc = slice();
        b0 += nb;
    }
    for (int k = 1; k <= forked; ++k) {  // join (best effort after an error: the caller's stream must not outrun a forked one)
        cudaError_t e = cudaEventRecord(ss.join[k - 1], ss.st[k - 1]);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(s, ss.join[k - 1], 0);
        if (e != cudaSuccess && rc == MG_OK) rc = set_error(MG_ERR_CUDA, "launch_generator_tc: joining slice %d: %s", k, cudaGetErrorString(e));
    }
    return rc;
}

}  // namespace mg
