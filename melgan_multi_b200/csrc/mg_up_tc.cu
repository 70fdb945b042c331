// LeakyReLU -> ConvTranspose1d on the tensor cores (tcgen05 + TMEM, split-bf16).
//
// Reference: Generator.forward, models.py:64-65 -- x = ups[i](F.leaky_relu(x)); ConvTranspose1d(Cin, Cout, K=2S, stride S,
// padding S/2), models.py:48-51.
//
// A transposed conv with K = 2S is, per output phase phi = (t + pad) mod S, a 2-tap conv over the INPUT positions:
//     out[co][S*s + phi - pad] = sum_ci  x[ci][s] * W[ci][co][phi]  +  x[ci][s-1] * W[ci][co][phi + S]
// All S phases of a tap read the same activation rows, so they are stacked along the MMA N dimension:
//     D[s, phi*NG + co] (+)= X[s - tap, :] * Wstack_tap[phi*NG + co, :]^T,   M = 128 input positions (TMEM lane = s),
//     N = S*NG (256 for the stride-8 stages: the largest UMMA shape), K = 16 per instruction,
// i.e. 2 taps x 3 split-bf16 passes = 6 instructions per 16 input channels cover every phase.  The s-1 tap is the same
// A buffer read one row earlier (row-linear operand layout, mg_tc.cuh).  Because all S phases of a (row block, channel
// group) sit in TMEM together, the epilogue thread of input position s owns the S consecutive output samples
// [S*s - pad, S*s - pad + S) of each channel and stores them as contiguous, fully coalesced vectors.
//
// Rows are VIRTUAL input positions: the B batch items are concatenated with one zero row after each item
// (v = item*(Lin+1) + s, s in [0, Lin], row s = Lin is zero), so that x[-1] = x[Lin] = 0 falls out of the layout and short
// sequences (stage 0: Lin = 32) still fill 128-row blocks.
// One CTA = NB blocks of 128 virtual input positions x one group of NG output channels.  K (= Cin) is streamed: the A
// slots (KCA channels: LeakyReLU + hi/lo split of x) are produced in shared memory by the converter warps straight from
// the fp32 NCL input (all KCA loads of a row in flight at once), the B slots (16 channels: both taps, hi and lo, all
// phases) arrive by 1-D bulk TMA from the pre-packed blob (mg_layout.h).
// Warp roles: converter/epilogue warps, TMA producer, MMA issuer warps (one per row block).
#include "mg_common.cuh"
#include "mg_tc.cuh"

namespace mg {
using namespace tc;

template <int STAGE_>
struct UpCfg {
    static constexpr int STAGE = STAGE_;
    static constexpr int CIN = stage_cin(STAGE), COUT = stage_cout(STAGE), S = stage_stride(STAGE), PAD = stage_pad(STAGE);
    static constexpr int NG = up_ng(STAGE);
    static constexpr int NCG = COUT / NG;
    static constexpr int N = S * NG;                      // MMA N: every phase of the channel group
    static constexpr int NB = (S == 8) ? 1 : 2;          // 128-row blocks per CTA
    static constexpr int COLS = NB * N;                   // TMEM columns in use
    static constexpr int TCOLS = COLS <= 128 ? 128 : COLS <= 256 ? 256 : 512;
    // stride-8 stages: 32 KB B slots, so one CTA per SM with a deep ring and 64-channel A slots (one memory round trip
    // per 64 channels); stride-2 stages: small slots, two CTAs per SM hide each other's loads and stores.
    static constexpr int MINB = (S == 8) ? 1 : 2;
    // channels per A slot = channels fetched per memory round trip of a converter thread (measured: 16 -> 32 helps the
    // stride-2 stages; a single 64-channel slot for stage 3 loses the conversion/MMA overlap and is slower)
    static constexpr int KCA = (S == 8) ? 64 : 32;
    static constexpr int ROWS = 128 * NB;
    static constexpr int AROWS = ROWS + 8;                // row index i <-> virtual position r0 - 1 + i, i in [0, ROWS]
    static constexpr int APITCH = AROWS * 16;             // bytes between k-panels
    static constexpr int ASLOT = 2 * (KCA / 8) * APITCH;  // [half: hi, lo][k-panel][AROWS][16 B]
    static constexpr int BSLOT = up_slot_bytes(STAGE);    // [tap][half][k-panel: 2][N][16 B]
    static constexpr int NSA = (CIN == KCA) ? 1 : 2, NSB = (S == 8) ? 4 : (CIN >= 128 ? 2 : 3);
    static constexpr int NCHUNK = CIN / 16;               // B slots per tile
    static constexpr int NWG = NB >= 2 ? 2 : 1;
    static constexpr int NCONV = 128 * NWG;               // converter / epilogue threads
    static constexpr int NIW = NB;                        // MMA issuer warps (one per row block)
    static constexpr int NT = NCONV + 32 + 32 * NIW;
    static constexpr int SMEM_BYTES = NSA * ASLOT + NSB * BSLOT + (2 * NSA + 2 * NSB + 1) * 8 + 16;
    static_assert(N <= 256 && N % 16 == 0, "UMMA N");
    static_assert(MINB * TCOLS <= 512, "TMEM columns");
    static_assert(MINB * (SMEM_BYTES + 1024) <= 228 * 1024, "shared memory budget");
    static_assert(CIN % KCA == 0, "A slot");
};

// VL (ragged batch, mg_gen_forward_varlen): item b's rows start at vl.mul * vl.cum[b] + b and it has vl.mul * (cum[b+1] - cum[b])
// input positions; Lin is then the row stride of x (the padded length) and S * Lin that of y.  Uniform launches (VL = false)
// compile to the code without it.
template <class Cfg, bool VL = false>
__global__ void __launch_bounds__(Cfg::NT, Cfg::MINB)
convt_tc_kernel(const float *__restrict__ x, float *__restrict__ y, const float *__restrict__ packed, int Lin, int B,
                int *__restrict__ status, const __grid_constant__ VarLenArg<VL> vl) {
    constexpr int CIN = Cfg::CIN, COUT = Cfg::COUT, S = Cfg::S, PAD = Cfg::PAD, NG = Cfg::NG, NB = Cfg::NB, N = Cfg::N;
    constexpr int ROWS = Cfg::ROWS, APITCH = Cfg::APITCH, ASLOT = Cfg::ASLOT, BSLOT = Cfg::BSLOT, KCA = Cfg::KCA;
    constexpr int NSA = Cfg::NSA, NSB = Cfg::NSB, NCHUNK = Cfg::NCHUNK, NCONV = Cfg::NCONV, NWG = Cfg::NWG, NIW = Cfg::NIW;
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t *aring = smem, *bring = smem + NSA * ASLOT;
    uint64_t *fullA = reinterpret_cast<uint64_t *>(bring + NSB * BSLOT);
    uint64_t *emptyA = fullA + NSA, *fullB = emptyA + NSA, *emptyB = fullB + NSB, *done = emptyB + NSB;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(done + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int r0 = blockIdx.x * ROWS;  // first virtual row of the tile
    const int cg = blockIdx.y;
    const int Lout = Lin * S, Lv = Lin + 1;

    if (warp == 0) tmem_alloc(tmem_slot, Cfg::TCOLS);
    if (tid == 32) {
        for (int s = 0; s < NSA; ++s) { mbar_init(&fullA[s], NCONV); mbar_init(&emptyA[s], NIW); }
        for (int s = 0; s < NSB; ++s) { mbar_init(&fullB[s], 1); mbar_init(&emptyB[s], NIW); }
        mbar_init(done, NIW);
        fence_mbar_init();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp == NCONV / 32) {
        // ================= TMA producer: one B slot per 16 input channels =================
        if (lane == 0) {
            const uint8_t *src = reinterpret_cast<const uint8_t *>(packed) + tc_region_start() + tc_up_offset(Cfg::STAGE) +
                                 (size_t)cg * NCHUNK * BSLOT;
            int s = 0, ph = 0;
            bool ok = true;
            for (int i = 0; i < NCHUNK && ok; ++i) {
                if (!mbar_wait(&emptyB[s], ph ^ 1)) { ok = false; break; }
                mbar_arrive_expect_tx(&fullB[s], BSLOT);
                bulk_g2s(bring + s * BSLOT, src + (size_t)i * BSLOT, BSLOT, &fullB[s]);
                if (++s == NSB) { s = 0; ph ^= 1; }
            }
            if (!ok) atomicExch(status, 12);
        }
    } else if (warp > NCONV / 32) {
        // ================= MMA issuers: warp iw owns row block iw (warp-uniform loop, one elected lane issues) =========
        const int blk = warp - (NCONV / 32 + 1);
        const uint32_t idesc = make_idesc_bf16(128, N);
        const uint64_t adesc_t = desc_template(APITCH, 128), bdesc_t = desc_template(N * 16, 128);
        const uint32_t aring_addr = smem_u32(aring), bring_addr = smem_u32(bring);
        int sa = 0, pha = 0, sb = 0, phb = 0;
        bool ok = true;  // a timed-out wait only raises the status word: control flow stays uniform
#pragma unroll 1
        for (int ca = 0; ca < CIN / KCA; ++ca) {
            ok &= mbar_wait(&fullA[sa], pha);
            tc_fence_after();
            const uint64_t abase = desc_at(adesc_t, aring_addr + sa * ASLOT + (blk * 128) * 16);
#pragma unroll 1
            for (int j = 0; j < KCA / 16; ++j) {
                ok &= mbar_wait(&fullB[sb], phb);
                tc_fence_after();
                const uint64_t bbase = desc_at(bdesc_t, bring_addr + sb * BSLOT);
#pragma unroll
                for (int tap = 0; tap < 2; ++tap)
#pragma unroll
                    for (int pass = 0; pass < 3; ++pass) {
                        const int ahalf = (pass == 1), bhalf = (pass == 2);
                        const uint64_t bdesc = bbase + (uint64_t)((((tap * 2 + bhalf) * 2) * N * 16) >> 4);
                        const uint64_t adesc =
                            abase + (uint64_t)((ahalf * (KCA / 8) * APITCH + (1 - tap) * 16) >> 4) + (uint64_t)(2 * j * (APITCH >> 4));
                        const bool acc = !(ca == 0 && j == 0 && tap == 0 && pass == 0);
                        if (elect_one()) mma_bf16(tmem + blk * N, adesc, bdesc, idesc, acc);
                    }
                if (elect_one()) mma_commit(&emptyB[sb]);
                if (++sb == NSB) { sb = 0; phb ^= 1; }
            }
            if (elect_one()) mma_commit(&emptyA[sa]);
            if (++sa == NSA) { sa = 0; pha ^= 1; }
        }
        if (elect_one()) mma_commit(done);
        if (!ok && lane == 0) atomicExch(status, 13);
    } else {
        // ================= converter warps: A slots = split(lrelu(x)), KCA channels of every row =================
        pdl_wait();  // x: the previous kernel's output
        int sa = 0, pha = 0;
        bool ok = true;
#pragma unroll 1
        for (int ca = 0; ca < CIN / KCA; ++ca) {
            if (ok && !mbar_wait(&emptyA[sa], pha ^ 1)) { ok = false; if (lane == 0) atomicExch(status, 14); }
            uint8_t *slot = aring + sa * ASLOT;
#pragma unroll 1
            for (int i = tid; i <= ROWS; i += NCONV) {
                const int v = r0 - 1 + i;
                int item, s;
                bool inr;
                if constexpr (VL) {
                    item = v >= 0 ? vl_item_of_row(vl, 1, v) : 0;
                    s = v - (vl.mul * vl.cum[item] + item);
                    inr = v >= 0 && item < vl.n && s < vl.mul * (vl.cum[item + 1] - vl.cum[item]);
                } else {
                    item = v >= 0 ? v / Lv : 0, s = v - item * Lv;
                    inr = (v >= 0 && item < B && s < Lin);
                }
                const float *xp = x + ((size_t)(inr ? item : 0) * CIN + ca * KCA) * Lin + (inr ? s : 0);
                float f[KCA];
#pragma unroll
                for (int j = 0; j < KCA; ++j) f[j] = inr ? __ldg(xp + (size_t)j * Lin) : 0.f;  // all in flight together
#pragma unroll
                for (int kp = 0; kp < KCA / 8; ++kp) {
                    uint32_t h[4], l[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) split2_bf16(lrelu(f[8 * kp + 2 * e]), lrelu(f[8 * kp + 2 * e + 1]), h[e], l[e]);
                    *reinterpret_cast<uint4 *>(slot + kp * APITCH + i * 16) = make_uint4(h[0], h[1], h[2], h[3]);
                    *reinterpret_cast<uint4 *>(slot + (KCA / 8 + kp) * APITCH + i * 16) = make_uint4(l[0], l[1], l[2], l[3]);
                }
            }
            fence_proxy_async();
            mbar_arrive(&fullA[sa]);
            if (++sa == NSA) { sa = 0; pha ^= 1; }
        }
        // ================= epilogue: D[s, phi*NG + co] + bias -> out[co][S*s + phi - pad] =================
        if (ok && !mbar_wait(done, 0)) { ok = false; if (lane == 0) atomicExch(status, 15); }
        tc_fence_after();
        pdl_trigger();  // MMAs done, only the output store is left: the next kernel of the chain may be scheduled
        const int wg = warp >> 2, q = warp & 3;
        const uint32_t lane_addr = tmem + ((uint32_t)(q * 32) << 16);
        const float *bias = packed + bias_offset(1 + Cfg::STAGE) + cg * NG;
        for (int blk = wg; blk < NB; blk += NWG) {
            const int v = r0 + blk * 128 + q * 32 + lane;
            int item, s, Li = Lin;  // Li: this item's input length
            bool row_ok;
            if constexpr (VL) {
                item = vl_item_of_row(vl, 1, v);
                s = v - (vl.mul * vl.cum[item] + item);
                row_ok = item < vl.n;
                if (row_ok) Li = vl.mul * (vl.cum[item + 1] - vl.cum[item]);
            } else {
                item = v / Lv, s = v - item * Lv;
                row_ok = item < B;
            }
            const int t0 = S * s - PAD;  // first output sample owned by this input position
            float *yb = y + ((size_t)(row_ok ? item : 0) * COUT + cg * NG) * Lout;
            if (S == 8) {
                const bool lo_ok = row_ok && s >= 1, hi_ok = row_ok && s <= Li - 1;
#pragma unroll 1
                for (int j0 = 0; j0 < NG; j0 += 8) {
                    uint32_t w[8][8];
#pragma unroll
                    for (int phi = 0; phi < 8; ++phi) tmem_ld8(lane_addr + blk * N + phi * NG + j0, w[phi]);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float bj = __ldg(bias + j0 + j);
                        float *yp = yb + (size_t)(j0 + j) * Lout + t0;
                        if (lo_ok)
                            *reinterpret_cast<float4 *>(yp) = make_float4(__uint_as_float(w[0][j]) + bj, __uint_as_float(w[1][j]) + bj,
                                                                          __uint_as_float(w[2][j]) + bj, __uint_as_float(w[3][j]) + bj);
                        if (hi_ok)
                            *reinterpret_cast<float4 *>(yp + 4) = make_float4(__uint_as_float(w[4][j]) + bj, __uint_as_float(w[5][j]) + bj,
                                                                              __uint_as_float(w[6][j]) + bj, __uint_as_float(w[7][j]) + bj);
                    }
                }
            } else {  // S == 2: t0 = 2s - 1
                const bool lo_ok = row_ok && s >= 1, hi_ok = row_ok && s <= Li - 1;
#pragma unroll 1
                for (int j0 = 0; j0 < NG; j0 += 16) {
                    uint32_t v0[16], v1[16];
                    tmem_ld16(lane_addr + blk * N + j0, v0);
                    tmem_ld16(lane_addr + blk * N + NG + j0, v1);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        const float bj = __ldg(bias + j0 + j);
                        float *yp = yb + (size_t)(j0 + j) * Lout + t0;
                        if (lo_ok) yp[0] = __uint_as_float(v0[j]) + bj;
                        if (hi_ok) yp[1] = __uint_as_float(v1[j]) + bj;
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, Cfg::TCOLS);
}

// vt != nullptr: ragged launch (VL instantiation), vt->n items, Lin = the padded input row stride = mul * T
template <class Cfg, bool VL = false>
static int launch_convt(const float *x, float *y, const float *packed, int B, int Lin, int *status, cudaStream_t s,
                        const VarLenTab *vt = nullptr, int mul = 1) {
    static bool configured = false;
    if (!configured) {
        MG_CUDA_TRY(cudaFuncSetAttribute(convt_tc_kernel<Cfg, VL>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
        configured = true;
    }
    VarLenArg<VL> vl{};
    long long vrows = (long long)B * (Lin + 1);  // Lin + 1 rows per item: position s = Lin feeds the last `pad` outputs
    if constexpr (VL) {
        vl = *vt;
        vl.mul = mul;
        vrows = (long long)mul * vl.cum[vl.n] + vl.n;  // no rows for the padding positions
    }
    dim3 grid((unsigned)((vrows + Cfg::ROWS - 1) / Cfg::ROWS), Cfg::NCG);
    MG_CUDA_TRY(launch_ex(convt_tc_kernel<Cfg, VL>, grid, dim3(Cfg::NT), Cfg::SMEM_BYTES, s, 1, true, x, y, packed, Lin, B, status, vl));
    return MG_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// Variant for a stage whose whole activation tile fits in shared memory (stage 1: 129 rows x 256 channels, hi+lo =
// 136 KB): the A operand is converted ONCE per row tile and stays resident, and the CTA loops over the NCG output-channel
// groups with the accumulators double-buffered in TMEM (2 x 256 columns), so the epilogue (TMEM -> coalesced vector
// stores) of group g overlaps the MMAs of group g+1 and no activation is loaded or converted twice.
template <class Cfg>
__global__ void __launch_bounds__(192, 1)
convt_resident_tc_kernel(const float *__restrict__ x, float *__restrict__ y, const float *__restrict__ packed, int Lin, int B,
                         int *__restrict__ status) {
    constexpr int CIN = Cfg::CIN, COUT = Cfg::COUT, S = Cfg::S, PAD = Cfg::PAD, NG = Cfg::NG, N = Cfg::N, NCG = Cfg::NCG;
    constexpr int ROWS = 128, APITCH = Cfg::APITCH, BSLOT = Cfg::BSLOT, NCHUNK = Cfg::NCHUNK;
    constexpr int KPT = CIN / 8;                    // k-panels of the resident A
    constexpr int AHALF = KPT * APITCH;             // bytes of one of {hi, lo}
    constexpr int NSB = 2, NCONV = 128;
    static_assert(S == 8 && N == 256 && 2 * AHALF + NSB * BSLOT + 256 <= 227 * 1024, "resident ConvT shape");
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t *abuf = smem, *bring = smem + 2 * AHALF;
    uint64_t *fullA = reinterpret_cast<uint64_t *>(bring + NSB * BSLOT);  // [CIN/64]: a 64-channel slice of A is written
    uint64_t *fullB = fullA + CIN / 64, *emptyB = fullB + NSB, *done = emptyB + NSB, *tfree = done + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tfree + 2);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int r0 = blockIdx.x * ROWS;
    const int Lout = Lin * S, Lv = Lin + 1;

    if (warp == 0) tmem_alloc(tmem_slot, 512);
    if (tid == 32) {
        for (int s = 0; s < CIN / 64; ++s) mbar_init(&fullA[s], NCONV);
        for (int s = 0; s < NSB; ++s) { mbar_init(&fullB[s], 1); mbar_init(&emptyB[s], 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(&done[s], 1); mbar_init(&tfree[s], NCONV); }
        fence_mbar_init();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp == NCONV / 32) {
        // ================= TMA producer: B slots of every channel group, in consumption order =================
        if (lane == 0) {
            const uint8_t *src = reinterpret_cast<const uint8_t *>(packed) + tc_region_start() + tc_up_offset(Cfg::STAGE);
            int s = 0, ph = 0;
            bool ok = true;
            for (int i = 0; i < NCG * NCHUNK && ok; ++i) {  // blob order is [cg][chunk]: exactly this loop
                if (!mbar_wait(&emptyB[s], ph ^ 1)) { ok = false; break; }
                mbar_arrive_expect_tx(&fullB[s], BSLOT);
                bulk_g2s(bring + s * BSLOT, src + (size_t)i * BSLOT, BSLOT, &fullB[s]);
                if (++s == NSB) { s = 0; ph ^= 1; }
            }
            if (!ok) atomicExch(status, 32);
        }
    } else if (warp == NCONV / 32 + 1) {
        // ================= MMA issuer =================
        const uint32_t idesc = make_idesc_bf16(128, N);
        const uint64_t adesc_t = desc_template(APITCH, 128), bdesc_t = desc_template(N * 16, 128);
        const uint32_t a_addr = smem_u32(abuf), bring_addr = smem_u32(bring);
        int sb = 0, phb = 0;
        bool ok = true;
#pragma unroll 1
        for (int cg = 0; cg < NCG; ++cg) {
            const int buf = cg & 1, use = cg >> 1;
            if (use > 0) {  // the epilogue must have drained this accumulator buffer (group cg - 2)
                ok &= mbar_wait(&tfree[buf], (use - 1) & 1);
                tc_fence_after();
            }
#pragma unroll 1
            for (int ch = 0; ch < NCHUNK; ++ch) {
                if (cg == 0 && (ch & 3) == 0) {  // first pass only: wait for the 64-channel slice of A
                    ok &= mbar_wait(&fullA[ch >> 2], 0);
                    tc_fence_after();
                }
                ok &= mbar_wait(&fullB[sb], phb);
                tc_fence_after();
                const uint64_t bbase = desc_at(bdesc_t, bring_addr + sb * BSLOT);
                const uint64_t abase = desc_at(adesc_t, a_addr + 2 * ch * APITCH);
#pragma unroll
                for (int tap = 0; tap < 2; ++tap)
#pragma unroll
                    for (int pass = 0; pass < 3; ++pass) {
                        const uint64_t bdesc = bbase + (uint64_t)((((tap * 2 + (pass == 2)) * 2) * N * 16) >> 4);
                        const uint64_t adesc = abase + (uint64_t)((((pass == 1) ? AHALF : 0) + (1 - tap) * 16) >> 4);
                        const bool acc = !(ch == 0 && tap == 0 && pass == 0);
                        if (elect_one()) mma_bf16(tmem + buf * N, adesc, bdesc, idesc, acc);
                    }
                if (elect_one()) mma_commit(&emptyB[sb]);
                if (++sb == NSB) { sb = 0; phb ^= 1; }
            }
            if (elect_one()) mma_commit(&done[buf]);
        }
        if (!ok && lane == 0) atomicExch(status, 33);
    } else if (warp < NCONV / 32) {
        // ================= converter: the whole A tile, once =================
        pdl_wait();  // x: the previous kernel's output
#pragma unroll 1
        for (int ca = 0; ca < CIN / 64; ++ca) {
#pragma unroll 1
            for (int i = tid; i <= ROWS; i += NCONV) {
                const int v = r0 - 1 + i;
                const int item = v >= 0 ? v / Lv : 0, s = v - item * Lv;
                const bool inr = (v >= 0 && item < B && s < Lin);
                const float *xp = x + ((size_t)(inr ? item : 0) * CIN + ca * 64) * Lin + (inr ? s : 0);
                float f[64];
#pragma unroll
                for (int j = 0; j < 64; ++j) f[j] = inr ? __ldg(xp + (size_t)j * Lin) : 0.f;
#pragma unroll
                for (int kp = 0; kp < 8; ++kp) {
                    uint32_t h[4], l[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) split2_bf16(lrelu(f[8 * kp + 2 * e]), lrelu(f[8 * kp + 2 * e + 1]), h[e], l[e]);
                    *reinterpret_cast<uint4 *>(abuf + (ca * 8 + kp) * APITCH + i * 16) = make_uint4(h[0], h[1], h[2], h[3]);
                    *reinterpret_cast<uint4 *>(abuf + AHALF + (ca * 8 + kp) * APITCH + i * 16) = make_uint4(l[0], l[1], l[2], l[3]);
                }
            }
            fence_proxy_async();
            mbar_arrive(&fullA[ca]);
        }
        // ================= epilogue per channel group (overlaps the next group's MMAs) =================
        const int q = warp & 3;
        const uint32_t lane_addr = tmem + ((uint32_t)(q * 32) << 16);
        const int v = r0 + q * 32 + lane;
        const int item = v / Lv, s = v - item * Lv;
        const bool row_ok = item < B;
        const int t0 = S * s - PAD;
        const bool lo_ok = row_ok && s >= 1, hi_ok = row_ok && s <= Lin - 1;
        bool ok = true;
#pragma unroll 1
        for (int cg = 0; cg < NCG; ++cg) {
            const int buf = cg & 1, use = cg >> 1;
            if (ok && !mbar_wait(&done[buf], use & 1)) { ok = false; if (lane == 0) atomicExch(status, 35); }
            tc_fence_after();
            if (cg == NCG - 1) pdl_trigger();  // last channel group's MMAs done: the next kernel may be scheduled
            const float *bias = packed + bias_offset(1 + Cfg::STAGE) + cg * NG;
            float *yb = y + ((size_t)(row_ok ? item : 0) * COUT + cg * NG) * Lout;
#pragma unroll 1
            for (int j0 = 0; j0 < NG; j0 += 8) {
                uint32_t w[8][8];
#pragma unroll
                for (int phi = 0; phi < 8; ++phi) tmem_ld8(lane_addr + buf * N + phi * NG + j0, w[phi]);
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float bj = __ldg(bias + j0 + j);
                    float *yp = yb + (size_t)(j0 + j) * Lout + t0;
                    if (lo_ok)
                        *reinterpret_cast<float4 *>(yp) = make_float4(__uint_as_float(w[0][j]) + bj, __uint_as_float(w[1][j]) + bj,
                                                                      __uint_as_float(w[2][j]) + bj, __uint_as_float(w[3][j]) + bj);
                    if (hi_ok)
                        *reinterpret_cast<float4 *>(yp + 4) = make_float4(__uint_as_float(w[4][j]) + bj, __uint_as_float(w[5][j]) + bj,
                                                                          __uint_as_float(w[6][j]) + bj, __uint_as_float(w[7][j]) + bj);
                }
            }
            tc_fence_before();
            mbar_arrive(&tfree[buf]);  // accumulator buffer may be overwritten by group cg + 2
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512);
}

template <class Cfg>
static int launch_convt_resident(const float *x, float *y, const float *packed, int B, int Lin, int *status, cudaStream_t s) {
    constexpr int smem = 2 * (Cfg::CIN / 8) * Cfg::APITCH + 2 * Cfg::BSLOT + (Cfg::CIN / 64 + 2 * 2 + 4) * 8 + 16;
    static bool configured = false;
    if (!configured) {
        MG_CUDA_TRY(cudaFuncSetAttribute(convt_resident_tc_kernel<Cfg>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        configured = true;
    }
    const long long vrows = (long long)B * (Lin + 1);
    MG_CUDA_TRY(launch_ex(convt_resident_tc_kernel<Cfg>, dim3((unsigned)((vrows + 127) / 128)), dim3(192), smem, s, 1, true, x, y,
                          packed, Lin, B, status));
    return MG_OK;
}

// x [B][Cin][Lin] -> y [B][Cout][S*Lin], fp32 NCL, (Cin, Cout, S) of generator stage `stage`.
int launch_convt_tc(const float *x, float *y, const float *packed, int stage, int B, int Lin, int *status, cudaStream_t s) {
    switch (stage) {
        case 0: return launch_convt<UpCfg<0>>(x, y, packed, B, Lin, status, s);
        case 1: return launch_convt_resident<UpCfg<1>>(x, y, packed, B, Lin, status, s);
        case 2: return launch_convt<UpCfg<2>>(x, y, packed, B, Lin, status, s);
        case 3: return launch_convt<UpCfg<3>>(x, y, packed, B, Lin, status, s);
    }
    return set_error(MG_ERR_INVALID_ARGUMENT, "launch_convt_tc: stage %d", stage);
}

// The same on a ragged batch (the default chain's two stand-alone ConvTs, stages 0 and 2): x [vt.n][Cin][mul T], item b's
// first mul * (cum[b+1] - cum[b]) positions; y [vt.n][Cout][S mul T], the first S times as many.
int launch_convt_tc_varlen(const float *x, float *y, const float *packed, int stage, const VarLenTab &vt, int T, int *status,
                           cudaStream_t s) {
    switch (stage) {
        case 0: return launch_convt<UpCfg<0>, true>(x, y, packed, vt.n, T, status, s, &vt, 1);
        case 2: return launch_convt<UpCfg<2>, true>(x, y, packed, vt.n, 64 * T, status, s, &vt, 64);
    }
    return set_error(MG_ERR_INVALID_ARGUMENT, "launch_convt_tc_varlen: stage %d has no ragged form", stage);
}

}  // namespace mg
