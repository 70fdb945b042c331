// Stride-1 "same" Conv1d with a dense channel contraction on the tensor cores (tcgen05 + TMEM, split-bf16).
//
// Used for   Generator.conv_pre      Conv1d(80 -> 512, k7, pad 3)                       models.py:46,62
//            Discriminator.conv_post1 Conv1d(1024 -> 1024, k5, pad 2) + LeakyReLU       models.py:84,96-97
//
// GEMM view: D[v, co] = sum_tap sum_pass X_pass[v + tap - PAD, :] * W_pass[tap][co, :]^T with M = 128 virtual positions
// (TMEM lane), N = 256 or 128 output channels, K = 16 per instruction.  Rows are VIRTUAL positions: the batch items are
// concatenated with PAD zero rows after each item (v = item*(L+PAD) + s), so every tap -- the same A buffer read
// `tap - PAD` rows further (row-linear operand layout, mg_tc.cuh) -- sees exactly the zero padding of the reference and
// short sequences (L = 17..128 in the discriminators, 32 in the generator) still fill the 128-row MMA.
// One CTA = 128 virtual positions x one group of N output channels; K = Cin is streamed: A slots (KCA channels, hi/lo
// split of x, optional LeakyReLU on the way in) are produced by the converter warps straight from the fp32 NCL input,
// B slots (one tap of 16 input channels: [hi, lo][k-panel][N][8] bf16 = 64 N bytes) arrive by 1-D bulk TMA.
#include "mg_common.cuh"
#include "mg_tc.cuh"

namespace mg {
using namespace tc;

template <int CIN_, int COUT_, int NTAP_, int KCA_, bool LRELU_OUT_, int MINB_ = 1, int N_ = 256, int CL_ = 1>
struct ConvCfg {
    // CL consecutive row tiles form a thread-block cluster: they stream the SAME weight slots (same output-channel group), so
    // the leader's bulk copies are multicast into every CTA's ring and L2 is read once per cluster instead of once per tile
    static constexpr int CL = CL_;
    static constexpr int MINB = MINB_;                      // CTAs per SM the shared-memory footprint is sized for
    static constexpr int CIN = CIN_, COUT = COUT_, NTAP = NTAP_, PAD = NTAP_ / 2, KCA = KCA_;
    static constexpr bool LRELU_OUT = LRELU_OUT_;
    static constexpr int N = N_;                            // output channels per CTA (= TMEM columns: 128 or 256)
    static constexpr int NCG = COUT / N;
    static constexpr int ROWS = 128;
    static constexpr int AROWS = ROWS + 2 * PAD + 2;        // row index i <-> virtual position r0 - PAD + i
    static constexpr int APITCH = AROWS * 16;
    static constexpr int ASLOT = 2 * (KCA / 8) * APITCH;    // [half][k-panel][AROWS][16 B]
    static constexpr int BSLOT = 2 * 2 * N * 16;            // [half][k-panel: 2][N][16 B]
    // B ring: a CTA streams CIN/16 * NTAP slots and each is consumed in 3 MMAs (192-381 cycles), far less than a bulk copy's
    // latency, so the ring depth (bytes in flight) sets the pace: 8 x 8 KB for the N = 128 tiles, 4 x 16 KB for N = 256
    static constexpr int NSA = (CIN == KCA) ? 1 : 2, NSB = (N_ == 128) ? 8 : 4;
    static constexpr int NCONV = 128;
    static constexpr int NT = NCONV + 64;
    static constexpr int SMEM_BYTES = NSA * ASLOT + NSB * BSLOT + (2 * NSA + 2 * NSB + 1) * 8 + 16;
    static_assert(CIN % KCA == 0 && KCA % 16 == 0 && COUT % N == 0, "shape");
    static_assert(MINB * (SMEM_BYTES + 1024) <= 228 * 1024 && MINB * N <= 512, "shared memory / TMEM budget");
};

// packed weights for this kernel: conv_tc_weight_index() in mg_layout.h

// VL (generator conv_pre only): ragged batch -- item b's rows start at vl.cum[b] + PAD * b, its length is cum[b+1] - cum[b],
// and L is the row stride of x / y (the padded length).  Uniform launches (VL = false) compile to the code without it.
template <class Cfg, bool VL = false>
__global__ void __launch_bounds__(Cfg::NT, Cfg::MINB)
conv_rows_tc_kernel(const float *__restrict__ x, float *__restrict__ y, const uint8_t *__restrict__ wtc,
                    const float *__restrict__ bias, int L, int B, int *__restrict__ status, const __grid_constant__ VarLenArg<VL> vl) {
    constexpr int CIN = Cfg::CIN, COUT = Cfg::COUT, NTAP = Cfg::NTAP, PAD = Cfg::PAD, KCA = Cfg::KCA, N = Cfg::N;
    constexpr int ROWS = Cfg::ROWS, APITCH = Cfg::APITCH, ASLOT = Cfg::ASLOT, BSLOT = Cfg::BSLOT;
    constexpr int NSA = Cfg::NSA, NSB = Cfg::NSB, NCONV = Cfg::NCONV;
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t *aring = smem, *bring = smem + NSA * ASLOT;
    uint64_t *fullA = reinterpret_cast<uint64_t *>(bring + NSB * BSLOT);
    uint64_t *emptyA = fullA + NSA, *fullB = emptyA + NSA, *emptyB = fullB + NSB, *done = emptyB + NSB;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(done + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int r0 = blockIdx.x * ROWS, cg = blockIdx.y;
    const int Lv = L + PAD;  // virtual rows per item: L positions + PAD zero rows

    if (warp == 0) tmem_alloc(tmem_slot, N);
    if (tid == 32) {
        for (int s = 0; s < NSA; ++s) { mbar_init(&fullA[s], NCONV); mbar_init(&emptyA[s], 1); }
        for (int s = 0; s < NSB; ++s) { mbar_init(&fullB[s], 1); mbar_init(&emptyB[s], Cfg::CL); }  // every CTA of the cluster frees a slot
        mbar_init(done, 1);
        fence_mbar_init();
    }
    tc_fence_before();
    __syncthreads();
    if constexpr (Cfg::CL > 1) cluster_sync();  // every CTA's barriers exist before a peer's copy or commit can land on them
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    constexpr uint16_t kClusterMask = (uint16_t)((1u << Cfg::CL) - 1);

    if (warp == NCONV / 32) {
        // ================= TMA producer: B slot = (16-channel chunk, tap) =================
        // (cluster: every CTA arms its own full barrier; only the leader copies, into all the CTAs' rings at once)
        if (lane == 0) {
            const uint8_t *src = wtc + (size_t)cg * (CIN / 16) * NTAP * BSLOT;
            const bool leader = Cfg::CL == 1 || cluster_ctarank() == 0;
            int s = 0, ph = 0;
            bool ok = true;
            for (int i = 0; i < (CIN / 16) * NTAP && ok; ++i) {
                if (!mbar_wait(&emptyB[s], ph ^ 1)) { ok = false; break; }
                mbar_arrive_expect_tx(&fullB[s], BSLOT);
                if constexpr (Cfg::CL > 1) {
                    if (leader) bulk_g2s_multicast(bring + s * BSLOT, src + (size_t)i * BSLOT, BSLOT, &fullB[s], kClusterMask);
                } else {
                    bulk_g2s(bring + s * BSLOT, src + (size_t)i * BSLOT, BSLOT, &fullB[s]);
                }
                if (++s == NSB) { s = 0; ph ^= 1; }
            }
            if (!ok) atomicExch(status, 22);
        }
    } else if (warp == NCONV / 32 + 1) {
        // ================= MMA issuer (warp-uniform loop, one elected lane issues) =================
        const uint32_t idesc = make_idesc_bf16(128, N);
        const uint64_t adesc_t = desc_template(APITCH, 128), bdesc_t = desc_template(N * 16, 128);
        const uint32_t aring_addr = smem_u32(aring), bring_addr = smem_u32(bring);
        int sa = 0, pha = 0, sb = 0, phb = 0;
        bool ok = true;
#pragma unroll 1
        for (int ca = 0; ca < CIN / KCA; ++ca) {
            ok &= mbar_wait(&fullA[sa], pha);
            tc_fence_after();
            const uint64_t abase = desc_at(adesc_t, aring_addr + sa * ASLOT);
#pragma unroll 1
            for (int j = 0; j < KCA / 16; ++j) {
#pragma unroll 1
                for (int tap = 0; tap < NTAP; ++tap) {
                    ok &= mbar_wait(&fullB[sb], phb);
                    tc_fence_after();
                    const uint64_t bbase = desc_at(bdesc_t, bring_addr + sb * BSLOT);
                    // A rows for this tap start at index `tap` (row i <-> v = r0 - PAD + i; the tap reads v + tap - PAD)
                    const uint64_t arow = abase + (uint64_t)tap + (uint64_t)(2 * j * (APITCH >> 4));
#pragma unroll
                    for (int pass = 0; pass < 3; ++pass) {
                        const uint64_t adesc = arow + (uint64_t)(((pass == 1) * (KCA / 8) * APITCH) >> 4);
                        const uint64_t bdesc = bbase + (uint64_t)(((pass == 2) * 2 * N * 16) >> 4);
                        const bool acc = !(ca == 0 && j == 0 && tap == 0 && pass == 0);
                        if (elect_one()) mma_bf16(tmem, adesc, bdesc, idesc, acc);
                    }
                    if (elect_one()) {
                        if constexpr (Cfg::CL > 1) mma_commit_multicast(&emptyB[sb], kClusterMask);
                        else mma_commit(&emptyB[sb]);
                    }
                    if (++sb == NSB) { sb = 0; phb ^= 1; }
                }
            }
            if (elect_one()) mma_commit(&emptyA[sa]);
            if (++sa == NSA) { sa = 0; pha ^= 1; }
        }
        if (elect_one()) mma_commit(done);
        if (!ok && lane == 0) atomicExch(status, 23);
    } else {
        // ================= converter warps: A slots = split(x), KCA channels of every row =================
        // Thread tid owns row tid of every slot and keeps the NEXT chunk's KCA loads in flight while it converts the
        // current one (the chain of dependent memory round trips, not the MMAs, bounds a CTA: 32 chunks at K = 1024);
        // the 2 PAD rows beyond the first NCONV are picked up by the first threads without prefetch.
        pdl_wait();  // x: the previous kernel's output
        int sa = 0, pha = 0;
        bool ok = true;
        constexpr int NCH = CIN / KCA;
        const int v0 = r0 - PAD + tid;
        int item0, s0;
        bool inr0;
        if constexpr (VL) {
            item0 = v0 >= 0 ? vl_item_of_row(vl, PAD, v0) : 0;
            s0 = v0 - (vl.cum[item0] + PAD * item0);
            inr0 = v0 >= 0 && item0 < vl.n && s0 < vl.cum[item0 + 1] - vl.cum[item0];
        } else {
            item0 = v0 >= 0 ? v0 / Lv : 0, s0 = v0 - item0 * Lv;
            inr0 = (v0 >= 0 && item0 < B && s0 < L);
        }
        const float *xrow = x + (size_t)(inr0 ? item0 : 0) * CIN * L + (inr0 ? s0 : 0);
        auto store_row = [&](uint8_t *slot, int i, const float *f) {
#pragma unroll
            for (int kp = 0; kp < KCA / 8; ++kp) {
                uint32_t h[4], l[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) split2_bf16(f[8 * kp + 2 * e], f[8 * kp + 2 * e + 1], h[e], l[e]);
                *reinterpret_cast<uint4 *>(slot + kp * APITCH + i * 16) = make_uint4(h[0], h[1], h[2], h[3]);
                *reinterpret_cast<uint4 *>(slot + (KCA / 8 + kp) * APITCH + i * 16) = make_uint4(l[0], l[1], l[2], l[3]);
            }
        };
        auto tail_rows = [&](uint8_t *slot, int ca) {
#pragma unroll 1
            for (int i = NCONV + tid; i < ROWS + 2 * PAD; i += NCONV) {
                const int v = r0 - PAD + i;
                int item, s;
                bool inr;
                if constexpr (VL) {
                    item = v >= 0 ? vl_item_of_row(vl, PAD, v) : 0;
                    s = v - (vl.cum[item] + PAD * item);
                    inr = v >= 0 && item < vl.n && s < vl.cum[item + 1] - vl.cum[item];
                } else {
                    item = v >= 0 ? v / Lv : 0, s = v - item * Lv;
                    inr = (v >= 0 && item < B && s < L);
                }
                const float *xp = x + ((size_t)(inr ? item : 0) * CIN + ca * KCA) * L + (inr ? s : 0);
                float f[KCA];
#pragma unroll
                for (int j = 0; j < KCA; ++j) f[j] = inr ? __ldg(xp + (size_t)j * L) : 0.f;
                store_row(slot, i, f);
            }
        };
        float fa[KCA], fb[KCA];  // chunk ca (even / odd) of this thread's row
#pragma unroll
        for (int j = 0; j < KCA; ++j) fa[j] = inr0 ? __ldg(xrow + (size_t)j * L) : 0.f;
#pragma unroll 1
        for (int ca = 0; ca < NCH; ca += 2) {
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int cc = ca + half;
                if (cc < NCH) {
                    float *cur = half ? fb : fa, *nxt = half ? fa : fb;
                    if (cc + 1 < NCH) {  // next chunk's loads go out before this chunk is converted
#pragma unroll
                        for (int j = 0; j < KCA; ++j) nxt[j] = inr0 ? __ldg(xrow + (size_t)((cc + 1) * KCA + j) * L) : 0.f;
                    }
                    if (ok && !mbar_wait(&emptyA[sa], pha ^ 1)) { ok = false; if (lane == 0) atomicExch(status, 24); }
                    uint8_t *slot = aring + sa * ASLOT;
                    store_row(slot, tid, cur);
                    tail_rows(slot, cc);
                    fence_proxy_async();
                    mbar_arrive(&fullA[sa]);
                    if (++sa == NSA) { sa = 0; pha ^= 1; }
                }
            }
        }
        // ================= epilogue: D[v, co] + bias (-> LeakyReLU) -> y[item][co][s] =================
        if (ok && !mbar_wait(done, 0)) { ok = false; if (lane == 0) atomicExch(status, 25); }
        tc_fence_after();
        pdl_trigger();  // MMAs done, only the output store is left: the next kernel of the chain may be scheduled
        const int q = warp & 3;
        const uint32_t lane_addr = tmem + ((uint32_t)(q * 32) << 16);
        const int v = r0 + q * 32 + lane;
        int item, s;
        bool row_ok;
        if constexpr (VL) {
            item = vl_item_of_row(vl, PAD, v);
            s = v - (vl.cum[item] + PAD * item);
            row_ok = item < vl.n && s < vl.cum[item + 1] - vl.cum[item];
        } else {
            item = v / Lv, s = v - item * Lv;
            row_ok = item < B && s < L;
        }
        float *yp = y + ((size_t)(row_ok ? item : 0) * COUT + cg * N) * L + (row_ok ? s : 0);
        const float *bp = bias + cg * N;
#pragma unroll 1
        for (int c0 = 0; c0 < N; c0 += 32) {
            uint32_t w[32];
            tmem_ld32(lane_addr + c0, w);
            tmem_ld_wait();
            if (row_ok) {
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    float o = __uint_as_float(w[j]) + __ldg(bp + c0 + j);
                    if (Cfg::LRELU_OUT) o = lrelu(o);
                    yp[(size_t)(c0 + j) * L] = o;
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, N);
    if constexpr (Cfg::CL > 1) cluster_sync();  // no CTA leaves while a peer may still multicast into its ring or barriers
}

// vt != nullptr: ragged launch (VL instantiation), B = vt->n items, L = the padded row stride
template <class Cfg, bool VL = false>
static int launch_conv_rows(const float *x, float *y, const uint8_t *wtc, const float *bias, int B, int L, int *status,
                            cudaStream_t s, const VarLenTab *vt = nullptr) {
    static bool configured = false;
    if (!configured) {
        MG_CUDA_TRY(cudaFuncSetAttribute(conv_rows_tc_kernel<Cfg, VL>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
        configured = true;
    }
    VarLenArg<VL> vl{};
    long long vrows = (long long)B * (L + Cfg::PAD);
    if constexpr (VL) {
        vl = *vt;
        vl.mul = 1;
        vrows = (long long)vl.cum[vl.n] + (long long)Cfg::PAD * vl.n;  // no rows for the padding frames
    }
    unsigned tiles = (unsigned)((vrows + Cfg::ROWS - 1) / Cfg::ROWS);
    tiles = (tiles + Cfg::CL - 1) / Cfg::CL * Cfg::CL;  // whole clusters (a tile past the last row converts zeros and stores nothing)
    MG_CUDA_TRY(launch_ex(conv_rows_tc_kernel<Cfg, VL>, dim3(tiles, Cfg::NCG), dim3(Cfg::NT), Cfg::SMEM_BYTES, s, Cfg::CL, true, x, y, wtc,
                          bias, L, B, status, vl));
    return MG_OK;
}

using PreCfg = ConvCfg<80, 512, 7, 80, false>;          // generator conv_pre
// discriminator conv_post1 (+ LeakyReLU): N = 128 per CTA (an N = 128 MMA is as efficient as an N = 256 one: 64 cycles of
// math = 64 cycles of operand reads), two CTAs per SM (the prefetching converter wants > 96 registers): the tiles of all three scales
// (264 + 136 + 40 CTAs at 8192 samples) are resident together and hide each other's conversion and ring stalls
// (CL = 2 -- the pair's weight slots multicast from one L2 read, frees by multicast commits -- is correct (the parity tests
//  pass) and measured neutral: 105 vs 102 us on scale 0.  The kernel is bound by SHARED-memory traffic, not L2: an N = 128 MMA
//  reads 8 KB of operands per 64 cycles = the whole 128 B/cycle, and the ring's bulk-copy writes (42 B/cycle) and the
//  converter's stores come on top.  The lever is cta_group::2, where each CTA of a pair holds half of B.)
using Post1Cfg = ConvCfg<1024, 1024, 5, 32, true, 2, kPost1NG, 1>;
using Post1DgradCfg = ConvCfg<1024, 1024, 5, 32, false, 2, kPost1NG, 1>;  // the same contraction on the transposed blob, no activation

// mel [B][80][T] -> y [B][512][T]   (Generator.conv_pre)
int launch_gen_pre_tc(const float *mel, float *y, const float *packed, int B, int T, int *status, cudaStream_t s) {
    const uint8_t *wtc = reinterpret_cast<const uint8_t *>(packed) + tc_region_start() + tc_pre_offset();
    return launch_conv_rows<PreCfg>(mel, y, wtc, packed + bias_offset(0), B, T, status, s);
}

// the same on a ragged batch: mel [vt->n][80][T], item b's first cum[b+1] - cum[b] frames (y: the same layout at 512 channels)
int launch_gen_pre_tc_varlen(const float *mel, float *y, const float *packed, const VarLenTab &vt, int T, int *status, cudaStream_t s) {
    const uint8_t *wtc = reinterpret_cast<const uint8_t *>(packed) + tc_region_start() + tc_pre_offset();
    return launch_conv_rows<PreCfg, true>(mel, y, wtc, packed + bias_offset(0), vt.n, T, status, s, &vt);
}

// x [Bt][1024][L] -> y [Bt][1024][L] = lrelu(conv_post1(x))   (Discriminator.conv_post1)
int launch_disc_post1_tc(const float *x, float *y, const uint8_t *wtc, const float *bias, int Bt, int L, int *status,
                         cudaStream_t s) {
    return launch_conv_rows<Post1Cfg>(x, y, wtc, bias, Bt, L, status, s);
}

// dz [Bt][1024][L] -> dx [Bt][1024][L]: data gradient of conv_post1 (autograd of models.py:96), wtcT = blob + d_tcT_start()
int launch_disc_post1_dgrad_tc(const float *dz, float *dx, const uint8_t *wtcT, const float *zero_bias, int Bt, int L, int *status,
                               cudaStream_t s) {
    return launch_conv_rows<Post1DgradCfg>(dz, dx, wtcT, zero_bias, Bt, L, status, s);
}

}  // namespace mg
