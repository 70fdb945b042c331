// ResBlock on the 5th-gen tensor cores (tcgen05 + TMEM), split-bf16 (3 MMAs per product) for fp32-grade results.
//
// Reference semantics: ResBlock.forward, models.py:32-40 -- three times  x = c2(lrelu(c1(lrelu(x)))) + x  with
// c1 dilations 1/3/9 and c2 dilation 1, all k=3 "same" convs on C channels.
//
// One CTA owns P = 128*NBLK consecutive positions of one batch item (16-position halo per side, recomputed by
// the neighbours) and keeps the whole block on chip:
//   TMEM   per 128-position block: R  [128 lanes x C cols] fp32  residual stream  (lane = position)
//                                  D1 [128 lanes x C cols] fp32  c1 accumulator
//   smem   X  = lrelu(current conv input) as split-bf16 (hi, lo), "row-linear K-major" (mg_tc.cuh): row = position,
//               k-panels of 8 channels.  A conv tap at dilation d is the same buffer with the start address
//               moved by 16*d bytes -- there is no im2col and no per-tap restaging.
//   smem   ring of weight chunks (one (tap, K-slice) of [Cout x KC] hi+lo per chunk), filled by 1-D bulk TMA
//               copies from the pre-packed blob (mg_layout.h), released by tcgen05.commit.
// GEMM view of one conv: D[pos, co] (+)= sum_tap sum_pass X_pass[pos + (tap-1)*d, :] * W_pass[tap][co, :]^T with
// M = 128 positions, N = C, K = 16 per instruction; passes (xh,wh), (xl,wh), (xh,wl).
// c2 accumulates straight onto R, so the residual add costs nothing; conv biases are added when the accumulator
// is read back (b2 is carried in `pend`).  Positions outside [0, L) are written as zeros into X after every conv,
// which is the per-layer zero padding of the reference.
//
// Warp roles: NEPI/32 epilogue warps (TMEM -> registers -> bias/LeakyReLU/mask/split -> X), one TMA producer
// warp, NIW MMA issuer warps (each runs its loop warp-uniform and one elected lane issues tcgen05.mma for its blocks).
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include "mg_common.cuh"
#include "mg_tc.cuh"

namespace mg {
using namespace tc;

// C channels; NBLK 128-position blocks per CTA (a block needs 2C of the 512 TMEM columns); NSTAGE weight-ring slots;
// NWG epilogue warpgroups; MINB CTAs per SM.  With MINB = 2 (C <= 64: the per-CTA weight stream is small) one CTA's
// epilogue / tile load / store overlaps the other CTA's MMAs; C >= 128 needs the whole SM's shared memory for one tile.
// UPF (stride-2 stages): the stage's LeakyReLU -> ConvTranspose1d(2C -> C, k4, s2, p1) runs inside this kernel first, so
// the CTA reads the PREVIOUS stage's output [B][2C][L/2] and the ConvT output never goes to HBM.  TMEM lane m of a
// "ConvT block" owns the output pair (t = o + 2m, o + 2m + 1):
//     out[2s]     = x[s] W1 + x[s-1] W3        out[2s+1] = x[s+1] W0 + x[s] W2        (s = o/2 + m; taps of models.py:50-51)
// i.e. four MMAs chains of N = C over the 2C input channels, whose A operand is the same (input-position) buffer read at
// row offsets 1, 0, 2, 1 -- the even outputs accumulate in the D1 columns of output block 2cb, the odd ones in those of
// block 2cb + 1.  The pairs are then de-interleaved through shared memory (fp32, in the X region that is not in use
// yet) so that lane = output position can fill R, and from there on the kernel is the plain ResBlock.
// CL = 2 (C = 256): two CTAs of a thread-block cluster own the two halves of ONE 2P-position super-tile.  After every conv
// each CTA pushes its 16 boundary rows of X into the slack rows of its peer's X buffer through distributed shared memory,
// so the 16-row halo is only recomputed at the super-tile's outer edges (a stage-0 tile is one 128-row block: alone it would
// spend 32 of its 128 rows on halo, and at T = 32 an item of 256 positions would need three tiles = 1.5x over-compute; as a
// pair it is ONE super-tile without any halo, 128 CTAs = one wave).  The pair runs in lock step -- `done` counts the MMA
// commits of BOTH CTAs, so nobody overwrites rows a peer's MMAs may still read -- and streams the same weights: the leader's
// bulk copies are multicast into both rings, the ring slots freed by multicast commits.
// UPT = S (2 or 8): the NEXT stage's LeakyReLU -> ConvTranspose1d(C -> C/2, k = 2S, stride S) runs at the TAIL of this kernel
// (models.py:64-65 of the following loop iteration): after the sixth conv the epilogue writes X = split(lrelu(x)) exactly as
// it does between convs, and the ConvT is two more "taps" on that operand -- out[S s + phi - pad] = x[s] W[phi] + x[s-1] W[phi+S],
// all S phases stacked along N like mg_up_tc.cu (N = S * NG = C in every stage), accumulators in the TMEM columns the
// ResBlock no longer needs.  The kernel then stores the ConvT output [B][C/2][S L] instead of the ResBlock output: the
// ResBlock output never goes to HBM, and the separate ConvT kernel (its activation re-read, operand conversion and launch)
// disappears.  An input position s owns the outputs [S s - pad, S s - pad + S) and needs x[s - 1]: tiles overlap by one
// more row on the left (HL = HALO + 1).  Position L (x[L] = 0) would own the last `pad` outputs; giving it a row would cost a
// whole extra tile exactly where sequences are a multiple of the tile (stage 0 at T = 32: 256 positions = one CTA pair), so
// those pad * C/2 outputs -- dot products of x[L-1] with the tap-1 weights -- are computed in fp32 by the CTA that owns
// position L - 1 (fix-up at the end of the epilogue).
// TMA = true: the input tile arrives by tensor-map TMA (cp.async.bulk.tensor.3d) instead of per-thread strided loads: the
// producer streams [LCH channels][P positions] fp32 slabs of x through the (still idle) weight-ring slots, positions past
// the end of the sequence zero-filled by the copy engine; the epilogue warps turn each slab into R (TMEM) and
// X = split(lrelu(x)) as it lands.  Needs L % 4 == 0 (16-byte global strides); the launcher falls back otherwise.
// G2 = true: two CTAs with INDEPENDENT tiles (own halo, own input) form a cluster and run every MMA as one cta_group::2
// instruction of M = 256: each CTA keeps only HALF of every weight chunk in its ring (rows [rank*C/2, +C/2) of B), so an MMA
// reads 4 KB of A + N*16 B of B per SM instead of 4 KB + N*32 B -- the shared-memory bandwidth that the overlapped epilogue
// stores and the ring's writes compete for.  The leader CTA's issuer warps issue for both; the peer's epilogue warps arrive on
// the leader's xready barriers through DSMEM, the peer's (otherwise idle) issuer warp relays its ring's full barriers.
template <int C_, int NBLK_, int NSTAGE_, int NWG_, int MINB_, bool POST_ = false, bool UPF_ = false, int CL_ = 1, int UPT_ = 0,
          bool TMA_ = false, bool G2_ = false>
struct RbCfg {
    static constexpr bool G2 = G2_;
    static constexpr int CLUSTER = (CL_ > 1 || G2_) ? 2 : 1;  // CTAs per cluster (launch attribute)
    static constexpr bool TMA = TMA_;
    static constexpr int CL = CL_;
    static constexpr int UPT = UPT_;
    static constexpr bool UPF = UPF_;
    static constexpr int C = C_;
    static constexpr int NBLK = NBLK_, MINB = MINB_;
    static constexpr bool POST = POST_;  // fuse LeakyReLU -> conv_post -> tanh into the final epilogue (last stage)
    static constexpr int TCOLS = NBLK * 2 * C;  // TMEM columns (power of two: 256 or 512)
    static constexpr int P = 128 * NBLK;
    // zero rows either side of X (dilation-9 taps reach 9 rows out); 12 lets two C = 128 single-block CTAs share an SM
    static constexpr int SLACK = (C_ == 128 && NBLK_ == 1) ? 12 : 16;
    static constexpr int HALO = 16 + (POST ? 3 : 0);  // 1+1+3+1+9+1 (+3 for the fused k7 conv_post)
    // left halo: a fused tail ConvT also reads x[s - 1]; with tensor-map input the tile origin must stay a multiple of 4
    // positions (the copy engine wants 16-byte aligned box starts: an origin of 223 is an illegal instruction), so 4 rows
    static constexpr int HL = HALO + (UPT_ ? (TMA_ ? 4 : 1) : 0);
    static constexpr int PVALID = P - HALO - HL;
    static constexpr int ROWS = P + 2 * SLACK;
    static constexpr int XPITCH = ROWS * 16;  // bytes between k-panels
    static constexpr int KP = C / 8;
    static constexpr int XBYTES = KP * XPITCH;  // one of {hi, lo}
    static constexpr int KC = tc_kc(C);
    static constexpr int CHUNK = tc_chunk_bytes(C);
    static constexpr int HALF = CHUNK / 2;
    static constexpr int NCHUNK = tc_chunks_per_conv(C);
    static constexpr int KSL = C / KC;
    static constexpr int NSTAGE = NSTAGE_;
    // epilogue work split: NWG warpgroups; an item = (128-position block, CW-column part of its C columns)
    static constexpr int NWG = NWG_;
    static constexpr int PARTS = NBLK >= NWG ? 1 : NWG / NBLK;
    static constexpr int CW = C / PARTS;
    static constexpr int ITEMS = NBLK * PARTS;
    static constexpr int NEPI = 128 * NWG;
    static constexpr int NIW = NBLK >= 2 ? 2 : 1;  // MMA issuer warps (the MMAs are smem-bandwidth bound, not issue bound)
    static constexpr int NT = NEPI + 32 + 32 * NIW;
    // X is handed to the MMA warps in NH channel halves: the next conv starts on input channels [0, C/NH) while the
    // epilogue is still writing the rest (K-slice order of the weight chunks follows).  Each epilogue thread owns CW/NH
    // columns of every half.
    // (measured at config 2: C = 128 with 2 hand-offs -5 % per conv, with 4 another -2 % (209 -> 205 us); at C = 256 the early
    //  MMAs and the epilogue's stores fight for shared-memory bandwidth: 2 hand-offs are a wash, 4 cost 4 %, so that stage
    //  keeps the single hand-off.  -DMG_NH128 / -DMG_NH256 override for A/B builds, scripts/gpu_nh.sh)
#ifndef MG_NH128
#define MG_NH128 4
#endif
#ifndef MG_NH256
#define MG_NH256 1
#endif
    static constexpr int NH = (C == 128) ? MG_NH128 : (C == 256) ? MG_NH256 : 1;
    static constexpr int BND = SLACK;  // boundary rows pushed to the peer CTA (CL = 2); the widest tap reaches 9
    // xready arrivals: local epilogue threads + (pair) the peer's boundary threads / (G2, leader) one per epilogue warp of the peer
    static constexpr int XARRIVE = NEPI + (CL > 1 ? BND * PARTS : 0) + (G2_ ? NEPI / 32 : 0);
    static_assert(!G2_ || (CL_ == 1 && UPT_ == 0 && !UPF_ && !POST_ && C_ % 32 == 0), "cta_group::2: plain ResBlock tiles");
    static_assert(CL == 1 || (CL == 2 && !UPF_ && !POST_), "CTA pairs: plain ResBlock only");
    // tail ConvT: TNG output channels per group (mg_layout.h up_ng of the next stage), TN = MMA N, TNCG groups, ring slots of
    // TSLOT bytes (stride 8: one tap of a 16-channel chunk; stride 2: both taps), TNSLOT of them
    static constexpr int TNG = UPT == 8 ? 32 : C / 2, TN = (UPT ? UPT : 1) * TNG, TNCG = (C / 2) / TNG;
    static constexpr int TSLOT = UPT == 8 ? 16384 : 128 * UPT * TNG, TNSLOT = UPT ? TNCG * (C / 16) * (UPT == 8 ? 2 : 1) : 0;
    static_assert(UPT == 0 || ((UPT == 2 || UPT == 8) && TN == C && TSLOT <= CHUNK && !POST_ && !UPF_), "tail ConvT shape");
    static_assert(UPT != 8 || (NBLK == 1 && TCOLS == 512), "stride-8 tail ConvT double-buffers its accumulators in the 512 columns");
    // TMA input slabs: LCH channels x P positions x 4 B = one ring slot; unit = (128-row block, 8-channel k-panel) of a slab
    static constexpr int LCH = CHUNK / (P * 4), NSLAB = TMA ? C / (LCH > 0 ? LCH : 1) : 0, LUNITS = NBLK * (LCH / 8);
    static_assert(!TMA || (LCH >= 8 && LCH % 8 == 0 && LCH * P * 4 == CHUNK && LUNITS % NWG == 0 && !UPF_ && P <= 256 &&
                           (C / NH) % LCH == 0 && (CL == 1 || LUNITS == NWG)), "TMA input slabs");
    static constexpr int SMEM_BYTES = 2 * XBYTES + NSTAGE * CHUNK + 2 * C * 4 + (2 * NSTAGE + 1 + NH + 4 + 2 * NSTAGE + 1 + NSTAGE) * 8 + 16;
    static_assert(KSL % NH == 0 && (CW / NH) % 16 == 0 && (NH == 1 || ITEMS == NWG), "hand-off split");
    // fused ConvT: input rows s = o/2 - 1 .. o/2 + P/2 of 2C channels (2 KP k-panels), NCB blocks of 128 output pairs
    static constexpr int UROWS = P / 2 + 2, UPITCH = UROWS * 16, NCB = NBLK / 2, UKSL = 2 * C / KC, NUPCH = UPF ? 4 * UKSL : 0;
    static constexpr int SPITCH = P + 4;  // floats between channels of the fp32 staging buffer [C][P]
    static_assert(!UPF || (NBLK % 2 == 0 && NH == 1 && 2 * KP * UPITCH <= XBYTES && C * SPITCH * 4 <= 2 * XBYTES && C <= 64),
                  "fused ConvT must fit the X region");
    static_assert(MINB * (SMEM_BYTES + 1024) <= 228 * 1024, "shared memory budget");
    static_assert(MINB * TCOLS <= 512 && (TCOLS == 128 || TCOLS == 256 || TCOLS == 512), "TMEM budget");
    static_assert(XPITCH / 16 < 16384, "LBO field");
    static_assert(CW % 32 == 0 && ITEMS % NWG == 0, "epilogue split");
};

__device__ __forceinline__ void named_bar_sync(int id, int count) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory");
}

// split 16 consecutive channels of one position (already activated / masked) and store them into the two k-panels they span
__device__ __forceinline__ void store_x16(uint8_t *Xh, uint8_t *Xl, int xpitch, int c0, int xrow_bytes, const float *f) {
    uint32_t h[8], l[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) split2_bf16(f[2 * e], f[2 * e + 1], h[e], l[e]);
    uint8_t *ph = Xh + (c0 >> 3) * xpitch + xrow_bytes;
    uint8_t *pl = Xl + (c0 >> 3) * xpitch + xrow_bytes;
    *reinterpret_cast<uint4 *>(ph) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4 *>(ph + xpitch) = make_uint4(h[4], h[5], h[6], h[7]);
    *reinterpret_cast<uint4 *>(pl) = make_uint4(l[0], l[1], l[2], l[3]);
    *reinterpret_cast<uint4 *>(pl + xpitch) = make_uint4(l[4], l[5], l[6], l[7]);
}
// the same, plus (push: this row is one of the CTA's boundary rows) a copy into the peer CTA's X buffer at row offset
// peer_row_bytes; rxh / rxl: cluster addresses of the peer's Xh / Xl
__device__ __forceinline__ void store_x16_push(uint8_t *Xh, uint8_t *Xl, int xpitch, int c0, int xrow_bytes, const float *f,
                                               bool push, uint32_t rxh, uint32_t rxl, int peer_row_bytes) {
    uint32_t h[8], l[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) split2_bf16(f[2 * e], f[2 * e + 1], h[e], l[e]);
    const int poff = (c0 >> 3) * xpitch;
    uint8_t *ph = Xh + poff + xrow_bytes;
    uint8_t *pl = Xl + poff + xrow_bytes;
    *reinterpret_cast<uint4 *>(ph) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4 *>(ph + xpitch) = make_uint4(h[4], h[5], h[6], h[7]);
    *reinterpret_cast<uint4 *>(pl) = make_uint4(l[0], l[1], l[2], l[3]);
    *reinterpret_cast<uint4 *>(pl + xpitch) = make_uint4(l[4], l[5], l[6], l[7]);
    if (push) {
        const uint32_t o = (uint32_t)(poff + peer_row_bytes);
        st_cluster_v4(rxh + o, make_uint4(h[0], h[1], h[2], h[3]));
        st_cluster_v4(rxh + o + xpitch, make_uint4(h[4], h[5], h[6], h[7]));
        st_cluster_v4(rxl + o, make_uint4(l[0], l[1], l[2], l[3]));
        st_cluster_v4(rxl + o + xpitch, make_uint4(l[4], l[5], l[6], l[7]));
    }
}

// VL (ragged batch, mg_gen_forward_varlen): grid.x runs over the linearised (item, super-tile) list vl.first[] (grid.y = 1; both
// CTAs of a pair always belong to the same item), item b is vl.mul * (cum[b+1] - cum[b]) positions long and L_ is the row
// stride of x / y (the padded length).  Everything below uses the item's own length where it used L: s_hi, `interior`, the
// zero-padding masks, the tail ConvT's fix-up and conv_post's sequence end; tensor-map rows in [L, L_) are real memory and
// are masked as they land; res3+post writes the exact-zero audio past the item's end.  Uniform launches (VL = false)
// compile to the code without it.
template <class Cfg, bool VL = false>
__global__ void __launch_bounds__(Cfg::NT, Cfg::MINB)
resblock_tc_kernel(const float *__restrict__ x, float *__restrict__ y, const float *__restrict__ packed, int stage, int L_, int nB,
                   int *__restrict__ status, long long *__restrict__ trace, const __grid_constant__ CUtensorMap xmap,
                   const __grid_constant__ VarLenArg<VL> vl) {
    constexpr int C = Cfg::C, NBLK = Cfg::NBLK, P = Cfg::P, SLACK = Cfg::SLACK, HALO = Cfg::HALO;
    constexpr int XPITCH = Cfg::XPITCH, XBYTES = Cfg::XBYTES, KC = Cfg::KC, CHUNK = Cfg::CHUNK, NSTAGE = Cfg::NSTAGE;
    constexpr int NEPI = Cfg::NEPI, NWG = Cfg::NWG, PARTS = Cfg::PARTS, CW = Cfg::CW, ITEMS = Cfg::ITEMS, NIW = Cfg::NIW;
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t *Xh = smem, *Xl = smem + XBYTES, *ring = smem + 2 * XBYTES;
    float *pend = reinterpret_cast<float *>(ring + NSTAGE * CHUNK);  // sum of the c2 biases folded so far
    float *b1s = pend + C;                                            // bias of the c1 in flight
    uint64_t *full = reinterpret_cast<uint64_t *>(b1s + C);
    uint64_t *empty = full + NSTAGE;
    uint64_t *done = empty + NSTAGE;
    uint64_t *xready = done + 1;  // [NH]: X channels [h*C/NH, (h+1)*C/NH) of the next conv are written (all epilogue threads arrive)
    uint64_t *dup = xready + Cfg::NH;  // [2] tail ConvT (stride 8): accumulator buffer complete;  tfree[2]: drained by the epilogue
    uint64_t *tfree = dup + 2;
    uint64_t *lfull = tfree + 2;        // [NSTAGE] TMA input slab landed in ring slot s;  lempty[NSTAGE]: converted by every epilogue thread
    uint64_t *lempty = lfull + NSTAGE;
    uint64_t *rfree = lempty + NSTAGE;  // pair: both CTAs' input slabs are consumed, the leader may multicast weights into both rings
    uint64_t *pfull = rfree + 1;        // [NSTAGE] G2, leader: the PEER's half of ring slot s has landed (relayed by its issuer warp)
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(pfull + NSTAGE);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    int b = blockIdx.y;
    // Edge-aware tiling: a halo is only needed where the tile borders MORE sequence.  Tile 0 starts at position 0 (its
    // left edge is the real zero padding) and keeps P - HALO outputs; later tiles keep P - 2*HALO, and a tile that reaches
    // the end of the sequence keeps its right HALO rows too.  (L = 2048, P = 256: 9 tiles instead of 10.)
    // CL > 1: all of this at super-tile granularity (PS = CL * P rows), CTA `rank` of the cluster owning rows [rank * P, + P).
    constexpr int CL = Cfg::CL, PS = CL * P, HL = Cfg::HL, PVS = PS - HALO - HL;
    constexpr bool G2 = Cfg::G2;
    const int crank = Cfg::CLUSTER > 1 ? (int)cluster_ctarank() : 0;  // rank in the cluster (pair or G2)
    const int rank = CL > 1 ? crank : 0;                              // position inside a super-tile (pair only)
    int stile = (int)blockIdx.x / CL;
    bool phantom = false;
    if constexpr (G2) {
        // cta_group::2 pairs are formed over the linearised (item, tile) list (grid.y = 1), so that only an odd TOTAL leaves one
        // phantom tile: it sits past the last tile of the last item, reads zeros (or rows it ignores) and stores nothing
        const int nt = 1 + (L_ > PS ? (L_ - PS + PVS - 1) / PVS : 0), id = (int)blockIdx.x;
        b = id / nt;
        stile = id - b * nt;
        if (b >= nB) { b = nB - 1; stile = nt; phantom = true; }
    }
    int L = L_;         // length of item b
    const int LS = L_;  // row stride of x and y (positions per channel)
    if constexpr (VL) {
        static_assert(!G2 && !Cfg::UPF, "ragged launches: default-chain kernels only");
        b = vl_item_of_tile(vl, stile);
        stile -= vl.first[b];
        L = vl.mul * (vl.cum[b + 1] - vl.cum[b]);
    }
    const int os = stile == 0 ? 0 : (PS - HALO) + (stile - 1) * PVS - HL;  // position of super-tile row 0
    const int o = os + rank * P;                                            // position of tile-local p = 0
    const int Lc = L;  // (tail ConvT: position L would own the last `pad` outputs; they are x[L-1]-only and fixed up below)
    const int s_lo = stile == 0 ? 0 : HL;
    const int s_hi = (os + PS >= Lc) ? PS : PS - HALO;  // first super-tile row that is NOT a valid output
    const int p_lo = phantom ? 0 : min(max(s_lo - rank * P, 0), P), p_hi = phantom ? 0 : min(max(s_hi - rank * P, 0), P);
    const bool interior = (o >= 0 && o + P <= L);  // every row of the tile is a real position
    // CTA pair: my boundary rows (rank 0: the last BND rows, rank 1: the first BND) mirror into the peer's slack rows
    const uint32_t peer = (uint32_t)(crank ^ 1);
    const uint32_t rxh = CL > 1 ? mapa_shared(smem_u32(smem), peer) : 0u, rxl = rxh + XBYTES;
    uint32_t rxready[Cfg::NH];
    // consumption order of the six convs of ResBlock `stage`: c1[0], c2[0], c1[1], c2[1], c1[2], c2[2]
    const int l0 = 5 + 6 * stage;
    const uint8_t *tc_base = reinterpret_cast<const uint8_t *>(packed) + tc_region_start();

    if (warp == 0) {
        if constexpr (G2) tmem_alloc2(tmem_slot, Cfg::TCOLS); else tmem_alloc(tmem_slot, Cfg::TCOLS);
    }
    if (tid == 32) {
        for (int s = 0; s < NSTAGE; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], NIW * CL);  // every issuer warp (of every CTA of the pair) commits its own arrival
            mbar_init(&pfull[s], 1);
        }
        mbar_init(done, NIW * CL);
        for (int h = 0; h < Cfg::NH; ++h) mbar_init(&xready[h], Cfg::XARRIVE);
        for (int k = 0; k < 2; ++k) { mbar_init(&dup[k], NIW * CL); mbar_init(&tfree[k], NEPI); }
        for (int k = 0; k < NSTAGE; ++k) { mbar_init(&lfull[k], 1); mbar_init(&lempty[k], NEPI); }
        mbar_init(rfree, CL);
        fence_mbar_init();
    }
    for (int h = 0; h < Cfg::NH; ++h) rxready[h] = Cfg::CLUSTER > 1 ? mapa_shared(smem_u32(&xready[h]), peer) : 0u;
    // (fused ConvT: the X region first holds the ConvT operand and the staging buffer; its slack rows are zeroed later)
    for (int i = Cfg::UPF ? 1 << 30 : tid; i < 2 * Cfg::KP * 2 * SLACK; i += Cfg::NT) {  // zero the slack rows of Xh and Xl
        const int r = i % (2 * SLACK), kp = (i / (2 * SLACK)) % Cfg::KP, hl = i / (2 * SLACK * Cfg::KP);
        const int row = r < SLACK ? r : P + r;  // r in [SLACK, 2*SLACK) -> rows P+SLACK .. P+2*SLACK-1
        // (pair: the slack rows facing the peer are ITS boundary rows, written by it before every conv -- not zeroed here)
        if (CL == 1 || (r < SLACK ? rank == 0 : rank == CL - 1))
            *reinterpret_cast<uint4 *>((hl ? Xl : Xh) + kp * XPITCH + row * 16) = make_uint4(0, 0, 0, 0);
    }
    for (int i = tid; i < C; i += Cfg::NT) pend[i] = 0.f;
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    if constexpr (Cfg::CLUSTER > 1) cluster_sync();  // the peer's barriers exist before a copy, commit or arrival of mine can land on them
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    // optional timeline of one interior CTA (clock64 stamps; see mg_gen_resblock_trace)
    const bool tr = trace && blockIdx.y == 0 && blockIdx.x == (G2 ? 0u : gridDim.x > 1 ? 1u : 0u) && lane == 0 && (warp == 0 || warp == NEPI / 32 + 1);  // epilogue warp 0 and issuer 0
#define MG_TR(slot) do { if (tr) trace[slot] = clock64(); } while (0)
    // "channels h of the next conv's input are written": every epilogue thread arrives on its CTA's barrier -- except in the peer
    // CTA of a cta_group::2 pair, whose MMAs the LEADER issues: there one lane per warp arrives on the leader's barrier (DSMEM)
#define MG_XREADY_ARRIVE(h)                                              \
    do {                                                                 \
        if (G2 && crank == 1) {                                          \
            __syncwarp();                                                \
            if (lane == 0) mbar_arrive_cluster(rxready[h]);              \
        } else {                                                         \
            mbar_arrive(&xready[h]);                                     \
        }                                                                \
    } while (0)

    if (warp == NEPI / 32) {
        // ================= TMA producer: streams the 6 * NCHUNK weight chunks through the ring =================
        if (lane == 0) {
            int s = 0, ph = 0;
            bool ok = true;
            if constexpr (Cfg::TMA) {
                // ---- the input tile, LCH channels at a time, through the ring slots (weights follow once they are free again)
                tma_prefetch_desc(&xmap);
                pdl_wait();  // x is the previous kernel's output
                for (int k = 0; k < Cfg::NSLAB && ok; ++k) {
                    const int sl = k % NSTAGE;
                    if (k >= NSTAGE && !mbar_wait(&lempty[sl], ((k / NSTAGE) - 1) & 1)) { ok = false; break; }
                    mbar_arrive_expect_tx(&lfull[sl], CHUNK);
                    tma_load_3d(ring + sl * CHUNK, &xmap, o, k * Cfg::LCH, b, &lfull[sl]);
                }
                for (int k = Cfg::NSLAB > NSTAGE ? Cfg::NSLAB - NSTAGE : 0; k < Cfg::NSLAB && ok; ++k)  // every slot consumed
                    if (!mbar_wait(&lempty[k % NSTAGE], (k / NSTAGE) & 1)) ok = false;
                if constexpr (CL > 1) {  // ... in BOTH CTAs, before the leader's multicast copies land in both rings
                    mbar_arrive(rfree);
                    mbar_arrive_cluster(mapa_shared(smem_u32(rfree), peer));
                    if (ok && !mbar_wait_cluster(rfree, 0)) ok = false;
                }
            }
            if constexpr (Cfg::UPF) {  // the fused ConvT's 4 taps x 2 K-slices, in blob order
                const uint8_t *src = tc_base + tc_upf_offset(stage);
                for (int i = 0; i < Cfg::NUPCH && ok; ++i) {
                    if (!mbar_wait(&empty[s], ph ^ 1)) { ok = false; break; }
                    mbar_arrive_expect_tx(&full[s], CHUNK);
                    bulk_g2s(ring + s * CHUNK, src + (size_t)i * CHUNK, CHUNK, &full[s]);
                    if (++s == NSTAGE) { s = 0; ph ^= 1; }
                }
            }
            for (int conv = 0; conv < 6 && ok; ++conv) {
                const int layer = l0 + (conv >> 1) + 3 * (conv & 1);
                const uint8_t *src = tc_base + tc_res_offset(layer);
                // consumption order: channel half h outermost (hand-off order), then tap, then K-slice within the half;
                // the blob stores chunk (tap, ks) at index tap*KSL + ks
                for (int i = 0; i < Cfg::NCHUNK && ok; ++i) {
                    constexpr int KH = Cfg::KSL / Cfg::NH;
                    const int h = i / (3 * KH), tap = (i / KH) % 3, ks = h * KH + i % KH;
                    const int ch = tap * Cfg::KSL + ks;
                    if (!mbar_wait(&empty[s], ph ^ 1)) { ok = false; break; }  // (pair: free in BOTH CTAs, see the commits)
                    if constexpr (G2) {
                        // my half of the chunk: rows [crank*C/2, +C/2) of every (hi|lo, k-panel) piece, packed contiguously in the slot
                        constexpr int PIECE = (C / 2) * 16, NP = 2 * (KC / 8);
                        mbar_arrive_expect_tx(&full[s], CHUNK / 2);
#pragma unroll
                        for (int pc = 0; pc < NP; ++pc)
                            bulk_g2s(ring + s * CHUNK + pc * PIECE, src + (size_t)ch * CHUNK + (size_t)pc * C * 16 + (size_t)crank * PIECE,
                                     PIECE, &full[s]);
                        if (++s == NSTAGE) { s = 0; ph ^= 1; }
                        continue;
                    }
                    mbar_arrive_expect_tx(&full[s], CHUNK);
                    if constexpr (CL > 1) {  // every CTA arms its own barrier; the leader's copy lands in both rings
                        if (rank == 0)
                            bulk_g2s_multicast(ring + s * CHUNK, src + (size_t)ch * CHUNK, CHUNK, &full[s], (uint16_t)((1u << CL) - 1));
                    } else {
                        bulk_g2s(ring + s * CHUNK, src + (size_t)ch * CHUNK, CHUNK, &full[s]);
                    }
                    if (++s == NSTAGE) { s = 0; ph ^= 1; }
                }
            }
            if constexpr (Cfg::UPT != 0) {  // the tail ConvT's B slots, in blob order [group][16-channel chunk][tap]
                const uint8_t *src = tc_base + tc_up_offset(stage + 1);
                for (int i = 0; i < Cfg::TNSLOT && ok; ++i) {
                    if (!mbar_wait(&empty[s], ph ^ 1)) { ok = false; break; }
                    mbar_arrive_expect_tx(&full[s], Cfg::TSLOT);
                    if constexpr (CL > 1) {
                        if (rank == 0)
                            bulk_g2s_multicast(ring + s * CHUNK, src + (size_t)i * Cfg::TSLOT, Cfg::TSLOT, &full[s], (uint16_t)((1u << CL) - 1));
                    } else {
                        bulk_g2s(ring + s * CHUNK, src + (size_t)i * Cfg::TSLOT, Cfg::TSLOT, &full[s]);
                    }
                    if (++s == NSTAGE) { s = 0; ph ^= 1; }
                }
            }
            if (!ok) atomicExch(status, 2);
        }
    } else if (warp > NEPI / 32) {
        // ================= MMA issuers: NIW warps, issuer w owns the 128-position blocks w, w+NIW, ... =================
        // (each warp runs the loop warp-uniform and one elected lane issues; a single issuing thread sustains only
        //  one tcgen05.mma per ~50 cycles, which starves the pipe when N = C <= 64)
        const int iw = warp - (NEPI / 32 + 1);
        // cta_group::2: M = 256 (this CTA's 128 rows + the peer's), B rows per ring slot = C / 2 (the other half is the peer's)
        constexpr int BROWS = G2 ? C / 2 : C, BHALF = G2 ? Cfg::HALF / 2 : Cfg::HALF;
        const uint32_t idesc = make_idesc_bf16(G2 ? 256 : 128, C);
        const uint64_t adesc_t = desc_template(XPITCH, 128), bdesc_t = desc_template(BROWS * 16, 128);
        const uint32_t xh_addr = smem_u32(Xh), xl_addr = smem_u32(Xl), ring_addr = smem_u32(ring);
        int s = 0, ph = 0;
        bool ok = true;  // a timed-out wait only raises the status word: control flow stays warp-uniform
        if (G2 && crank == 1) {
            // ---- peer CTA of a cta_group::2 pair: the leader issues every MMA.  This warp only tells it when MY half of a ring slot
            // has landed (the leader cannot wait on another CTA's barrier): wait locally, arrive on the leader's pfull[s].
            if (iw == 0) {
                uint32_t rpfull[NSTAGE];
#pragma unroll
                for (int k = 0; k < NSTAGE; ++k) rpfull[k] = mapa_shared(smem_u32(&pfull[k]), 0);
#pragma unroll 1
                for (int i = 0; i < 6 * Cfg::NCHUNK; ++i) {
                    ok &= mbar_wait(&full[s], ph);
                    if (lane == 0) {
                        uint32_t a = rpfull[0];
#pragma unroll
                        for (int k = 1; k < NSTAGE; ++k) a = (s == k) ? rpfull[k] : a;
                        mbar_arrive_cluster(a);
                    }
                    __syncwarp();
                    if (++s == NSTAGE) { s = 0; ph ^= 1; }
                }
                if (!ok && lane == 0) atomicExch(status, 10);
            }
        } else {
        if constexpr (Cfg::UPF) {
            // ---- fused ConvT: chunk (tap k, K-slice ks); odd taps feed the even outputs (D1 of block 2cb), even taps the odd ones
            constexpr int UPITCH = Cfg::UPITCH, UKSL = Cfg::UKSL, NCB = Cfg::NCB;
            const uint64_t udesc_t = desc_template(UPITCH, 128);
            ok &= mbar_wait(&xready[0], 0);
            tc_fence_after();
#pragma unroll 1
            for (int ch = 0; ch < Cfg::NUPCH; ++ch) {
                const int k = ch / UKSL, ks = ch - k * UKSL;
                ok &= mbar_wait(&full[s], ph);
                tc_fence_after();
                const uint64_t bbase = desc_at(bdesc_t, ring_addr + s * CHUNK);
                const int rowoff = (k == 0) ? 2 : (k == 3) ? 0 : 1;  // A row i <-> input position o/2 - 1 + i
                const uint32_t arow = rowoff * 16 + ks * (KC / 8) * UPITCH;
                const uint64_t ah = desc_at(udesc_t, xh_addr + arow), al = desc_at(udesc_t, xl_addr + arow);
                const bool first = (k < 2 && ks == 0);
#pragma unroll
                for (int pass = 0; pass < 3; ++pass) {
#pragma unroll
                    for (int k16 = 0; k16 < KC / 16; ++k16) {
                        const uint64_t bdesc = bbase + (uint64_t)(((pass == 2 ? Cfg::HALF : 0) + 2 * k16 * (C * 16)) >> 4);
#pragma unroll
                        for (int bi = 0; bi < (NCB + NIW - 1) / NIW; ++bi) {
                            const int cb = iw + bi * NIW;
                            if (cb < NCB) {
                                const uint64_t adesc = (pass == 1 ? al : ah) + (uint64_t)((2 * k16 * UPITCH) >> 4) + (uint64_t)(cb * 128);
                                const uint32_t dc = (uint32_t)((2 * cb + ((k & 1) ? 0 : 1)) * 2 * C + C);
                                if (elect_one()) mma_bf16(tmem + dc, adesc, bdesc, idesc, !(first && pass == 0 && k16 == 0));
                            }
                        }
                    }
                }
                if (elect_one()) mma_commit(&empty[s]);
                if (++s == NSTAGE) { s = 0; ph ^= 1; }
            }
            if (elect_one()) mma_commit(done);
            __syncwarp();
        }
        constexpr int PH0 = Cfg::UPF ? 1 : 0;  // barrier phases consumed by the fused ConvT
#pragma unroll 1
        for (int conv = 0; conv < 6; ++conv) {
            const int dil = (conv & 1) ? 1 : (conv == 0 ? 1 : conv == 2 ? 3 : 9);
            const uint32_t dcol = (conv & 1) ? 0 : C;  // c1 -> D1, c2 -> R (accumulating onto the residual)
            const bool fresh = !(conv & 1);
#pragma unroll 1
            for (int ch = 0; ch < Cfg::NCHUNK; ++ch) {
                constexpr int KH = Cfg::KSL / Cfg::NH;
                const int h = ch / (3 * KH), tap = (ch / KH) % 3, ks = h * KH + ch % KH;
                if (ch % (3 * KH) == 0) {  // first chunk of channel half h: wait until the epilogue has written those channels of X
                    ok &= Cfg::CLUSTER > 1 ? mbar_wait_cluster(&xready[h], (conv + PH0) & 1) : mbar_wait(&xready[h], (conv + PH0) & 1);
                    tc_fence_after();
                    if (ch == 0 && iw == 0) MG_TR(64 + 3 * conv);
                }
                ok &= mbar_wait(&full[s], ph);
                if constexpr (G2) ok &= mbar_wait_cluster(&pfull[s], ph);  // the peer's half of the slot
                tc_fence_after();
                if (ch == 0 && iw == 0) MG_TR(65 + 3 * conv);
                // per-chunk base descriptors; every MMA below adds a compile-time constant to the address field
                const uint64_t bbase = desc_at(bdesc_t, ring_addr + s * CHUNK);
                const uint32_t arow = (SLACK + (tap - 1) * dil) * 16 + ks * (KC / 8) * XPITCH;
                const uint64_t ah = desc_at(adesc_t, xh_addr + arow), al = desc_at(adesc_t, xl_addr + arow);
#pragma unroll
                for (int pass = 0; pass < 3; ++pass) {
#pragma unroll
                    for (int k16 = 0; k16 < KC / 16; ++k16) {
                        const uint64_t bdesc = bbase + (uint64_t)(((pass == 2 ? BHALF : 0) + 2 * k16 * (BROWS * 16)) >> 4);
#pragma unroll
                        for (int bi = 0; bi < NBLK / NIW; ++bi) {
                            const int blk = iw + bi * NIW;
                            const uint64_t adesc = (pass == 1 ? al : ah) + (uint64_t)((2 * k16 * XPITCH) >> 4) + (uint64_t)(blk * 128);
                            const bool acc = !(fresh && ch == 0 && pass == 0 && k16 == 0);
                            if (elect_one()) {
                                if constexpr (G2) mma2_bf16(tmem + blk * 2 * C + dcol, adesc, bdesc, idesc, acc);
                                else mma_bf16(tmem + blk * 2 * C + dcol, adesc, bdesc, idesc, acc);
                            }
                        }
                    }
                }
                if (elect_one()) {  // ring slot free once these MMAs have read it
                    if constexpr (G2) mma2_commit(&empty[s], 3);  // ... in both CTAs
                    else if constexpr (CL > 1) mma_commit_multicast(&empty[s], (uint16_t)((1u << CL) - 1));
                    else mma_commit(&empty[s]);
                }
                if (++s == NSTAGE) { s = 0; ph ^= 1; }
            }
            if (elect_one()) {
                if constexpr (G2) mma2_commit(done, 3);  // both CTAs' epilogues
                else if constexpr (CL > 1) mma_commit_multicast(done, (uint16_t)((1u << CL) - 1));  // the peer's epilogue may write my slack rows
                else mma_commit(done);
            }
            if (iw == 0) MG_TR(66 + 3 * conv);
            if (!ok && lane == 0) atomicExch(status, 3);
            __syncwarp();
        }
        if constexpr (Cfg::UPT != 0) {
            // ---- tail ConvT: D[s, phi*TNG + co] (+)= X[s - tap, :] * Wstack_tap^T over the C channels of X = split(lrelu(x_out))
            constexpr int S = Cfg::UPT, TN = Cfg::TN;
            const uint64_t tbdesc_t = desc_template(TN * 16, 128);
            for (int h = 0; h < Cfg::NH; ++h)
                ok &= CL > 1 ? mbar_wait_cluster(&xready[h], (6 + PH0) & 1) : mbar_wait(&xready[h], (6 + PH0) & 1);
            tc_fence_after();
#pragma unroll 1
            for (int cg = 0; cg < Cfg::TNCG; ++cg) {
                const int buf = cg & 1;
                if (S == 8 && cg >= 2) {  // the epilogue must have drained this accumulator buffer (group cg - 2)
                    ok &= mbar_wait(&tfree[buf], ((cg >> 1) - 1) & 1);
                    tc_fence_after();
                }
#pragma unroll 1
                for (int ch = 0; ch < C / 16; ++ch) {
#pragma unroll 1
                    for (int ts = 0; ts < (S == 8 ? 2 : 1); ++ts) {  // stride 8: one ring slot per tap
                        ok &= mbar_wait(&full[s], ph);
                        tc_fence_after();
                        const uint64_t bbase = desc_at(tbdesc_t, ring_addr + s * CHUNK);
#pragma unroll
                        for (int tp = 0; tp < (S == 8 ? 1 : 2); ++tp) {
                            const int tap = S == 8 ? ts : tp;  // tap 0 reads x[s], tap 1 x[s - 1]: the same buffer one row earlier
#pragma unroll
                            for (int pass = 0; pass < 3; ++pass) {
                                const uint32_t boff = (uint32_t)((((S == 8 ? 0 : tp * 2) + (pass == 2 ? 1 : 0)) * 2) * TN * 16);
                                const uint64_t bdesc = bbase + (uint64_t)(boff >> 4);
#pragma unroll
                                for (int bi = 0; bi < NBLK / NIW; ++bi) {
                                    const int blk = iw + bi * NIW;
                                    const uint32_t arow = (uint32_t)((SLACK + blk * 128 - tap) * 16 + 2 * ch * XPITCH);
                                    const uint64_t adesc = desc_at(adesc_t, (pass == 1 ? xl_addr : xh_addr) + arow);
                                    const uint32_t dc = S == 8 ? (uint32_t)(buf * 256) : (uint32_t)(blk * 2 * C + C);
                                    if (elect_one()) mma_bf16(tmem + dc, adesc, bdesc, idesc, !(ch == 0 && tap == 0 && pass == 0));
                                }
                            }
                        }
                        if (elect_one()) {
                            if constexpr (CL > 1) mma_commit_multicast(&empty[s], (uint16_t)((1u << CL) - 1));
                            else mma_commit(&empty[s]);
                        }
                        if (++s == NSTAGE) { s = 0; ph ^= 1; }
                    }
                }
                if (elect_one()) {
                    uint64_t *bar = S == 8 ? &dup[buf] : done;
                    if constexpr (CL > 1) mma_commit_multicast(bar, (uint16_t)((1u << CL) - 1));
                    else mma_commit(bar);
                }
            }
            if (!ok && lane == 0) atomicExch(status, 7);
            __syncwarp();
        }
        }  // (leader / single-CTA issuer)
    } else {
        // ================= epilogue warps (16): lane = position, 4 warpgroups split blocks / column ranges =========
        const int wg = warp >> 2, q = warp & 3;
        const int row = q * 32 + lane;
        const uint32_t lane_addr = tmem + ((uint32_t)(q * 32) << 16);

        pdl_wait();  // x is the previous kernel's output (and y may still be read by it): every global access of this kernel is below
        if (warp == 0) MG_TR(0);
        constexpr int NH = Cfg::NH, CH = CW / NH;
        if constexpr (Cfg::UPF) {
            constexpr int UROWS = Cfg::UROWS, UPITCH = Cfg::UPITCH, SPITCH = Cfg::SPITCH, NCB = Cfg::NCB;
            const int Lin = L >> 1, s0 = (o >> 1) - 1;  // A row i <-> input position s0 + i (o is even)
            // ---- ConvT operand: A <- split(lrelu(x_in)), 2C channels of UROWS = P/2 + 2 input positions.  Every thread owns
            // one of the first P/2 rows (and 1 / HS of its channels); the two extra rows are 16-channel snippets of the first
            // threads, loaded in the same round trip as their main rows.
            constexpr int HS = NEPI / (P / 2), CPT = 2 * C / HS;  // threads per row, channels per thread
            static_assert(HS >= 1 && NEPI % (P / 2) == 0 && CPT % 32 == 0 && 2 * (2 * C / 16) <= NEPI, "ConvT operand split");
            {
                const int i = tid % (P / 2), cpart = (tid / (P / 2)) * CPT;
                const int sp = s0 + i;
                const bool inr = (sp >= 0 && sp < Lin);
                const float *xp = x + (size_t)b * 2 * C * Lin + (inr ? sp : 0);
                const bool extra = tid < 2 * (2 * C / 16);
                const int ei = P / 2 + tid / (2 * C / 16), ec0 = (tid % (2 * C / 16)) * 16, esp = s0 + ei;
                const bool einr = extra && esp >= 0 && esp < Lin;
                const float *exp_ = x + (size_t)b * 2 * C * Lin + (einr ? esp : 0);
                float fe[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) fe[j] = einr ? lrelu(__ldg(exp_ + (size_t)(ec0 + j) * Lin)) : 0.f;
#pragma unroll 1
                for (int c0 = cpart; c0 < cpart + CPT; c0 += 32) {
                    float f[32];
#pragma unroll
                    for (int j = 0; j < 32; ++j) f[j] = inr ? lrelu(__ldg(xp + (size_t)(c0 + j) * Lin)) : 0.f;  // all in flight together
                    store_x16(Xh, Xl, UPITCH, c0, i * 16, f);
                    store_x16(Xh, Xl, UPITCH, c0 + 16, i * 16, f + 16);
                }
                if (extra) store_x16(Xh, Xl, UPITCH, ec0, ei * 16, fe);
            }
            fence_proxy_async();
            mbar_arrive(&xready[0]);  // phase 0: the ConvT MMAs may start
            if (warp == 0) MG_TR(1);
            // ---- ConvT epilogue: lane m of ConvT block cb holds the output pair (256 cb + 2m, + 1) in the D1 columns of blocks
            // 2cb / 2cb + 1; + bias -> fp32 staging [c][p] (float2 per channel: consecutive lanes, consecutive 8 bytes)
            bool ok0 = mbar_wait(done, 0);
            if (!ok0 && lane == 0) atomicExch(status, 6);
            tc_fence_after();
            float *stg = reinterpret_cast<float *>(Xh);
            const float *ubias = packed + bias_offset(1 + stage);
            {
                constexpr int UITEMS = NCB * (NWG / NCB > 0 ? NWG / NCB : 1);  // (ConvT block, column part) items over the warpgroups
                constexpr int UPARTS = UITEMS / NCB, UCW = C / UPARTS;
                static_assert(UCW % 32 == 0 && UITEMS % NWG == 0, "ConvT epilogue split");
#pragma unroll 1
                for (int it = wg; it < UITEMS; it += NWG) {
                    const int cb = it / UPARTS, cbeg = (it % UPARTS) * UCW;
#pragma unroll 1
                    for (int c0 = cbeg; c0 < cbeg + UCW; c0 += 32) {
                        uint32_t ve[32], vo[32];
                        tmem_ld32(lane_addr + (2 * cb) * 2 * C + C + c0, ve);
                        tmem_ld32(lane_addr + (2 * cb + 1) * 2 * C + C + c0, vo);
                        tmem_ld_wait();
                        float *sp = stg + (size_t)c0 * SPITCH + 256 * cb + 2 * row;
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            const float bj = ubias[c0 + j];
                            *reinterpret_cast<float2 *>(sp + (size_t)j * SPITCH) =
                                make_float2(__uint_as_float(ve[j]) + bj, __uint_as_float(vo[j]) + bj);
                        }
                    }
                }
            }
            tc_fence_before();
            named_bar_sync(2, NEPI);
            tc_fence_after();
            // ---- R <- x (lane = output position); then X <- split(lrelu(x)) exactly like after a c2 (pend = 0)
            constexpr bool DIRECT = (ITEMS / NWG) * CW <= 64 && CW == 32;  // the thread's x values fit in registers: no TMEM round trip
            if constexpr (DIRECT) {
                float xv[ITEMS / NWG][32];
#pragma unroll
                for (int ii = 0; ii < ITEMS / NWG; ++ii) {
                    const int it = wg + ii * NWG, blk = it / PARTS, cbeg = (it % PARTS) * CW;
                    const float *sp = stg + 128 * blk + row;
#pragma unroll
                    for (int j = 0; j < 32; ++j) xv[ii][j] = sp[(size_t)(cbeg + j) * SPITCH];
                }
                named_bar_sync(2, NEPI);  // every staging read is done: the region becomes X
                for (int i = tid; i < 2 * Cfg::KP * 2 * SLACK; i += NEPI) {  // zero the slack rows of Xh and Xl
                    const int r = i % (2 * SLACK), kp = (i / (2 * SLACK)) % Cfg::KP, hl = i / (2 * SLACK * Cfg::KP);
                    const int xr = r < SLACK ? r : P + r;
                    *reinterpret_cast<uint4 *>((hl ? Xl : Xh) + kp * XPITCH + xr * 16) = make_uint4(0, 0, 0, 0);
                }
#pragma unroll
                for (int ii = 0; ii < ITEMS / NWG; ++ii) {
                    const int it = wg + ii * NWG, blk = it / PARTS, cbeg = (it % PARTS) * CW;
                    const int p = blk * 128 + row, t = o + p;
                    const bool inr = (t >= 0 && t < L);
                    uint32_t w[16];
                    float f[32];
#pragma unroll
                    for (int h16 = 0; h16 < 2; ++h16) {
#pragma unroll
                        for (int j = 0; j < 16; ++j) w[j] = __float_as_uint(xv[ii][16 * h16 + j]);
                        tmem_st16(lane_addr + blk * 2 * C + cbeg + 16 * h16, w);
                    }
#pragma unroll
                    for (int j = 0; j < 32; ++j) f[j] = inr ? lrelu(xv[ii][j]) : 0.f;
                    store_x16(Xh, Xl, XPITCH, cbeg, (p + SLACK) * 16, f);
                    store_x16(Xh, Xl, XPITCH, cbeg + 16, (p + SLACK) * 16, f + 16);
                }
                tmem_st_wait();
            } else {
#pragma unroll 1
            for (int it = wg; it < ITEMS; it += NWG) {
                const int blk = it / PARTS, cbeg = (it % PARTS) * CW;
                const float *sp = stg + 128 * blk + row;
#pragma unroll 1
                for (int c0 = cbeg; c0 < cbeg + CW; c0 += 16) {
                    uint32_t w[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) w[j] = __float_as_uint(sp[(size_t)(c0 + j) * SPITCH]);
                    tmem_st16(lane_addr + blk * 2 * C + c0, w);
                }
            }
            tmem_st_wait();
            named_bar_sync(2, NEPI);  // every staging read is done: the region becomes X
            for (int i = tid; i < 2 * Cfg::KP * 2 * SLACK; i += NEPI) {  // zero the slack rows of Xh and Xl
                const int r = i % (2 * SLACK), kp = (i / (2 * SLACK)) % Cfg::KP, hl = i / (2 * SLACK * Cfg::KP);
                const int xr = r < SLACK ? r : P + r;
                *reinterpret_cast<uint4 *>((hl ? Xl : Xh) + kp * XPITCH + xr * 16) = make_uint4(0, 0, 0, 0);
            }
#pragma unroll 1
            for (int it = wg; it < ITEMS; it += NWG) {
                const int blk = it / PARTS, cbeg = (it % PARTS) * CW;
                const int p = blk * 128 + row, t = o + p;
                const bool inr = (t >= 0 && t < L);
#pragma unroll 1
                for (int c0 = cbeg; c0 < cbeg + CW; c0 += 32) {
                    uint32_t v[32];
                    float f[32];
                    tmem_ld32(lane_addr + blk * 2 * C + c0, v);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 32; ++j) f[j] = inr ? lrelu(__uint_as_float(v[j])) : 0.f;
                    store_x16(Xh, Xl, XPITCH, c0, (p + SLACK) * 16, f);
                    store_x16(Xh, Xl, XPITCH, c0 + 16, (p + SLACK) * 16, f + 16);
                }
            }
            }
            fence_proxy_async();
            tc_fence_before();
            mbar_arrive(&xready[0]);  // phase 1: conv 0 may start
        } else if constexpr (Cfg::TMA) {
        // ---- the input tile arrives slab by slab (tensor-map TMA, see the producer): R <- x (fp32, exact), X <- split(lrelu(x)).
        // A slab is [LCH channels][P positions] fp32; warpgroup g converts the units (block, 8-channel panel) g, g + NWG, ...;
        // lane = position, so the eight reads of a unit are conflict-free and its two 16-byte X stores are the usual ones.
        constexpr int LCH = Cfg::LCH, LUNITS = Cfg::LUNITS;
        bool lok = true;
#pragma unroll 1
        for (int k = 0; k < Cfg::NSLAB; ++k) {
            const int sl = k % NSTAGE;
            if (lok && !mbar_wait(&lfull[sl], (k / NSTAGE) & 1)) { lok = false; if (lane == 0) atomicExch(status, 9); }
            const float *slab = reinterpret_cast<const float *>(ring + sl * CHUNK);
#pragma unroll
            for (int u = wg; u < LUNITS; u += NWG) {
                const int blk = u % NBLK, j = u / NBLK;
                const int p = blk * 128 + row, c0 = k * LCH + 8 * j;
                uint32_t w[8];
                float f[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    w[e] = __float_as_uint(slab[(8 * j + e) * P + p]);
                    f[e] = lrelu(__uint_as_float(w[e]));
                }
                if constexpr (VL) {  // the map spans the padded stride: rows past the item's end are memory, not zero fill
                    if (o + p >= L) {
#pragma unroll
                        for (int e = 0; e < 8; ++e) { w[e] = 0u; f[e] = 0.f; }
                    }
                }
                tmem_st8(lane_addr + blk * 2 * C + c0, w);
                uint32_t h[4], l[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) split2_bf16(f[2 * e], f[2 * e + 1], h[e], l[e]);
                const int poff = (c0 >> 3) * XPITCH;
                *reinterpret_cast<uint4 *>(Xh + poff + (p + SLACK) * 16) = make_uint4(h[0], h[1], h[2], h[3]);
                *reinterpret_cast<uint4 *>(Xl + poff + (p + SLACK) * 16) = make_uint4(l[0], l[1], l[2], l[3]);
                if constexpr (CL > 1) {
                    if (rank == 0 ? p >= P - Cfg::BND : p < Cfg::BND) {  // boundary row: mirror into the peer's slack rows
                        const uint32_t po = (uint32_t)(poff + (rank == 0 ? p - (P - Cfg::BND) : SLACK + P + p) * 16);
                        st_cluster_v4(rxh + po, make_uint4(h[0], h[1], h[2], h[3]));
                        st_cluster_v4(rxl + po, make_uint4(l[0], l[1], l[2], l[3]));
                    }
                }
            }
            mbar_arrive(&lempty[sl]);  // this thread is done reading the slot (every thread arrives for itself: its release covers
                                       // its own reads, which is also the form compute-sanitizer's racecheck can follow)
            if ((k + 1) * LCH % (C / NH) == 0) {      // a channel half (or everything) of conv 0's input is in place
                const int h = (k + 1) * LCH / (C / NH) - 1;
                tmem_st_wait();
                if constexpr (Cfg::CLUSTER > 1) fence_proxy_async_all(); else fence_proxy_async();
                tc_fence_before();
                MG_XREADY_ARRIVE(h);
                if constexpr (CL > 1) {  // (LUNITS == NWG: every thread converts exactly one unit per slab, so a boundary-row thread
                                         //  accounts for one of the BND * PARTS remote arrivals its peer's barrier expects)
                    if (rank == 0 ? row >= P - Cfg::BND : row < Cfg::BND) mbar_arrive_cluster(rxready[h]);
                }
            }
        }
        } else {
        // ---- load the input tile: R <- x (fp32, exact), X <- split(lrelu(x))
        // an item (blk, part) owns, in every channel half h, the CH = CW/NH columns  h*C/NH + part*CH .. + CH
        int nb0 = 0;  // boundary items this thread pushed to the peer (CL = 2)
#pragma unroll 1
        for (int it = wg; it < ITEMS; it += NWG) {
            const int blk = it / PARTS, part = it % PARTS;
            const int p = blk * 128 + row, t = o + p;
            const bool inr = (t >= 0 && t < L);
            const bool push = CL > 1 && (rank == 0 ? p >= P - Cfg::BND : p < Cfg::BND);
            const int prow = (rank == 0 ? p - (P - Cfg::BND) : SLACK + P + p) * 16;  // row offset in the peer's X buffer
            nb0 += push;
            const float *xp = x + (size_t)b * C * LS + (inr ? t : 0);
            // all CW loads of the item are issued before the first use: one memory round trip, not CW/16
            uint32_t v[CW];
#pragma unroll
            for (int j = 0; j < CW; ++j) {
                const int col = (j / CH) * (C / NH) + part * CH + j % CH;
                v[j] = inr ? __float_as_uint(__ldg(xp + (size_t)col * LS)) : 0u;
            }
#pragma unroll
            for (int c0 = 0; c0 < CW; c0 += 16) {
                const int col0 = (c0 / CH) * (C / NH) + part * CH + c0 % CH;
                uint32_t w[16];
                float f[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    w[j] = v[c0 + j];
                    f[j] = lrelu(__uint_as_float(v[c0 + j]));
                }
                tmem_st16(lane_addr + blk * 2 * C + col0, w);
                if constexpr (CL > 1) store_x16_push(Xh, Xl, XPITCH, col0, (p + SLACK) * 16, f, push, rxh, rxl, prow);
                else store_x16(Xh, Xl, XPITCH, col0, (p + SLACK) * 16, f);
            }
        }
        tmem_st_wait();
        if constexpr (Cfg::CLUSTER > 1) fence_proxy_async_all(); else fence_proxy_async();
        tc_fence_before();
        for (int h = 0; h < NH; ++h) {  // conv 0 may start (phase 0 of both halves)
            MG_XREADY_ARRIVE(h);
            for (int k = 0; k < nb0; ++k) mbar_arrive_cluster(rxready[h]);
        }
        }
        if (warp == 0) MG_TR(1);

        bool ok = true;
#pragma unroll 1
        for (int conv = 0; conv < 6; ++conv) {
            if (warp == 0) MG_TR(2 + 3 * conv);
            // X for this conv has been handed to the MMA warps through xready[] (by the load pass or the previous
            // iteration).  While the tensor core works: stage this conv's bias (c1: its own; c2: fold into pend).
            // (pend and b1s alternate between iterations, so a fast thread never overwrites what a slow one still reads.)
            const float *bias = packed + bias_offset(l0 + (conv >> 1) + 3 * (conv & 1));
            if (conv & 1) {
                for (int c = tid; c < C; c += NEPI) pend[c] += __ldg(bias + c);
            } else {
                for (int c = tid; c < C; c += NEPI) b1s[c] = __ldg(bias + c);
            }
            named_bar_sync(2, NEPI);
            if (ok && !mbar_wait(done, (conv + (Cfg::UPF ? 1 : 0)) & 1)) { ok = false; if (lane == 0) atomicExch(status, 4); }
            tc_fence_after();
            if (warp == 0) MG_TR(3 + 3 * conv);
            if (conv == 5 && Cfg::UPT == 0) {
                // all MMAs of this tile are done: the next kernel of the chain may be scheduled (its CTAs set up and prefetch
                // weights on SMs this grid has already vacated, then sit in pdl_wait() until this grid has completed).
                // Late on purpose: an early trigger parks waiting CTAs on SMs that other streams' kernels could be using.
                pdl_trigger();
                break;
            }
            // (tail ConvT: the sixth conv is followed by one more hand-off -- X = split(lrelu(R + pend)) is the ConvT's operand)
            const uint32_t scol = (conv & 1) ? 0 : C;  // next input comes from R (after c2) or D1 (after c1)
            const float *bsrc = (conv & 1) ? pend : b1s;
#pragma unroll 1
            for (int h = 0; h < NH; ++h) {
                int nb = 0;
#pragma unroll 1
                for (int it = wg; it < ITEMS; it += NWG) {
                    const int blk = it / PARTS, cbeg = h * (C / NH) + (it % PARTS) * CH;
                    const int p = blk * 128 + row, t = o + p;
                    const bool inr = (t >= 0 && t < L);
                    const bool push = CL > 1 && (rank == 0 ? p >= P - Cfg::BND : p < Cfg::BND);
                    const int prow = (rank == 0 ? p - (P - Cfg::BND) : SLACK + P + p) * 16;
                    nb += push;
                    constexpr int EW = CH >= 32 ? 32 : 16;  // columns per TMEM read
#pragma unroll 1
                    for (int c0 = cbeg; c0 < cbeg + CH; c0 += EW) {
                        uint32_t v[EW];
                        float f[EW];
                        if constexpr (EW == 32) tmem_ld32(lane_addr + blk * 2 * C + scol + c0, v);
                        else tmem_ld16(lane_addr + blk * 2 * C + scol + c0, v);
                        tmem_ld_wait();
                        if (interior) {  // whole tile inside [0, L): no zero-padding mask needed (CTA-uniform branch)
#pragma unroll
                            for (int j = 0; j < EW; ++j) f[j] = lrelu(__uint_as_float(v[j]) + bsrc[c0 + j]);
                        } else {
#pragma unroll
                            for (int j = 0; j < EW; ++j) f[j] = inr ? lrelu(__uint_as_float(v[j]) + bsrc[c0 + j]) : 0.f;
                        }
                        if (Cfg::UPT != 0 && conv == 5 && t == L - 1) {  // lrelu(x[L-1]) in fp32 for the fix-up (b1s is free now)
#pragma unroll
                            for (int j = 0; j < EW; ++j) b1s[c0 + j] = f[j];
                        }
#pragma unroll
                        for (int e0 = 0; e0 < EW; e0 += 16) {
                            if constexpr (CL > 1) store_x16_push(Xh, Xl, XPITCH, c0 + e0, (p + SLACK) * 16, f + e0, push, rxh, rxl, prow);
                            else store_x16(Xh, Xl, XPITCH, c0 + e0, (p + SLACK) * 16, f + e0);
                        }
                    }
                }
                // channels [h*C/NH, (h+1)*C/NH) of the next conv's input are in place: let its MMAs start on them
                if constexpr (Cfg::CLUSTER > 1) fence_proxy_async_all(); else fence_proxy_async();
                tc_fence_before();
                MG_XREADY_ARRIVE(h);
                for (int k = 0; k < nb; ++k) mbar_arrive_cluster(rxready[h]);  // my boundary rows are in the peer's slack rows
            }
            if (warp == 0) MG_TR(4 + 3 * conv);
        }
        if constexpr (Cfg::POST) {
            // ---- fused LeakyReLU -> conv_post (32 -> 1, k7, pad 3) -> tanh (models.py:67-69); y is audio [B][1][L].
            // Each position turns its 32 channels into the 7 per-tap partial sums q_k[p] = sum_ci w[ci][k] * lrelu(x[ci][p]),
            // parks them in shared memory (the X buffer is dead now), then audio[p] = tanh(b + sum_k q_k[p + k - 3]).
            static_assert(!Cfg::POST || (C == 32 && PARTS == 1), "conv_post fusion is for the 32-channel stage");
            float *Q = reinterpret_cast<float *>(Xh);      // [7][P]
            float *wpost = reinterpret_cast<float *>(Xl);  // [32][8]
            for (int i = tid; i < 32 * 8; i += NEPI)
                wpost[i] = (i & 7) < kPostK ? __ldg(packed + weight_offset(29) + (i >> 3) * kPostK + (i & 7)) : 0.f;
            named_bar_sync(2, NEPI);
#pragma unroll 1
            for (int it = wg; it < ITEMS; it += NWG) {
                const int p = it * 128 + row, t = o + p;
                const bool inr = (t >= 0 && t < L);
                uint32_t v[32];
                tmem_ld32(lane_addr + it * 2 * C, v);
                tmem_ld_wait();
                float q[kPostK];
#pragma unroll
                for (int k = 0; k < kPostK; ++k) q[k] = 0.f;
#pragma unroll
                for (int ci = 0; ci < 32; ++ci) {
                    const float a = inr ? lrelu(__uint_as_float(v[ci]) + pend[ci]) : 0.f;
                    const float4 w0 = *reinterpret_cast<const float4 *>(wpost + ci * 8);
                    const float4 w1 = *reinterpret_cast<const float4 *>(wpost + ci * 8 + 4);
                    q[0] = fmaf(w0.x, a, q[0]); q[1] = fmaf(w0.y, a, q[1]); q[2] = fmaf(w0.z, a, q[2]); q[3] = fmaf(w0.w, a, q[3]);
                    q[4] = fmaf(w1.x, a, q[4]); q[5] = fmaf(w1.y, a, q[5]); q[6] = fmaf(w1.z, a, q[6]);
                }
#pragma unroll
                for (int k = 0; k < kPostK; ++k) Q[k * P + p] = q[k];
            }
            named_bar_sync(2, NEPI);
            const float bpost = __ldg(packed + bias_offset(29));
#pragma unroll 1
            for (int it = wg; it < ITEMS; it += NWG) {
                const int p = it * 128 + row, t = o + p;
                if (p >= p_lo && p < p_hi && t < L) {
                    float acc = bpost;
#pragma unroll
                    for (int k = 0; k < kPostK; ++k) {
                        const int pp = p + k - 3;  // outside the tile only where it is outside the sequence too (zero padding)
                        if (pp >= 0 && pp < P) acc += Q[k * P + pp];
                    }
                    y[(size_t)b * LS + t] = tanhf(acc);
                }
            }
            if constexpr (VL) {  // audio past the item's end is exactly zero (written by the item's last tile)
                if (os + PS >= L)
                    for (int t = L + tid; t < LS; t += NEPI) y[(size_t)b * LS + t] = 0.f;
            }
        } else if constexpr (Cfg::UPT != 0) {
            // ---- tail ConvT epilogue: the thread of input position s stores the S outputs [S s - pad, S s - pad + S) of its channels
            constexpr int S = Cfg::UPT, TNG = Cfg::TNG, PADT = S / 2, COT = C / 2;
            const int Lout = S * LS;  // row stride of y
            const float *tbias = packed + bias_offset(1 + stage + 1);
            // ---- fix-up (first: it only needs b1s[], so it runs while the tensor core works on the ConvT): out[co][S L - pad + j] = bias + sum_ci lrelu(x[ci][L-1]) * W[ci][co][j + S], j < pad (the outputs position
            // L would own: x[L] = 0 leaves only the x[L-1] tap), by the CTA whose owned rows include position L - 1.  fp32 FFMA
            // on the fp32 copy of the ConvT weights ([Cin][Cout][S][2], mg_layout.h): pad * C/2 dot products of length C.
            {
                const int pl = L - 1 - o;  // tile-local row of position L - 1
                if (pl >= p_lo && pl < p_hi) {  // CTA-uniform
                    named_bar_sync(2, NEPI);     // every thread's b1s[] contribution (written during the last hand-off) is visible
                    const float *wf = packed + weight_offset(1 + stage + 1);
                    for (int i = tid; i < PADT * COT; i += NEPI) {
                        const int co = i / PADT, j = i - co * PADT;
                        const float *wp = wf + ((size_t)co * S + j) * 2 + 1;  // + ci * COT * S * 2
                        float acc0 = 0.f, acc1 = 0.f, acc2 = 0.f, acc3 = 0.f;
#pragma unroll 1
                        for (int c0 = 0; c0 < C; c0 += 32) {  // 32 weights in flight per round trip
                            float wv[32];
#pragma unroll
                            for (int k = 0; k < 32; ++k) wv[k] = __ldg(wp + (size_t)(c0 + k) * COT * S * 2);
#pragma unroll
                            for (int k = 0; k < 32; k += 4) {
                                acc0 = fmaf(b1s[c0 + k], wv[k], acc0);
                                acc1 = fmaf(b1s[c0 + k + 1], wv[k + 1], acc1);
                                acc2 = fmaf(b1s[c0 + k + 2], wv[k + 2], acc2);
                                acc3 = fmaf(b1s[c0 + k + 3], wv[k + 3], acc3);
                            }
                        }
                        y[((size_t)b * COT + co) * Lout + (size_t)S * L - PADT + j] = (acc0 + acc1) + (acc2 + acc3) + __ldg(tbias + co);
                    }
                }
            }
            if constexpr (S == 2) {
                if (ok && !mbar_wait(done, (6 + (Cfg::UPF ? 1 : 0)) & 1)) { ok = false; if (lane == 0) atomicExch(status, 8); }
                tc_fence_after();
                pdl_trigger();
                constexpr int COI = TNG / PARTS;  // output channels per item
                static_assert(COI % 16 == 0, "tail ConvT epilogue split");
#pragma unroll 1
                for (int it = wg; it < ITEMS; it += NWG) {
                    const int blk = it / PARTS, jbeg = (it % PARTS) * COI;
                    const int p = blk * 128 + row, sg = o + p;  // sg: global input position
                    const bool own = (p >= p_lo && p < p_hi && sg < L);
                    const bool lo_ok = own && sg >= 1, hi_ok = own;
                    float *yb = y + (size_t)b * COT * Lout + (own ? 2 * sg - PADT : 0);
#pragma unroll 1
                    for (int j0 = jbeg; j0 < jbeg + COI; j0 += 16) {
                        uint32_t v0[16], v1[16];
                        tmem_ld16(lane_addr + blk * 2 * C + C + j0, v0);
                        tmem_ld16(lane_addr + blk * 2 * C + C + TNG + j0, v1);
                        tmem_ld_wait();
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const float bj = __ldg(tbias + j0 + j);
                            float *yp = yb + (size_t)(j0 + j) * Lout;
                            if (lo_ok) yp[0] = __uint_as_float(v0[j]) + bj;
                            if (hi_ok) yp[1] = __uint_as_float(v1[j]) + bj;
                        }
                    }
                }
            } else {
                static_assert(S == 2 || (NBLK == 1 && PARTS * 8 == TNG), "stride-8 tail: each warpgroup stores 8 channels of a group");
                const int p = row, sg = o + p;
                const bool own = (p >= p_lo && p < p_hi && sg < L);
                const bool lo_ok = own && sg >= 1, hi_ok = own;
#pragma unroll 1
                for (int cg = 0; cg < Cfg::TNCG; ++cg) {
                    const int buf = cg & 1;
                    if (ok && !mbar_wait(&dup[buf], (cg >> 1) & 1)) { ok = false; if (lane == 0) atomicExch(status, 8); }
                    tc_fence_after();
                    if (cg == Cfg::TNCG - 1) pdl_trigger();
                    const int j0 = wg * 8;  // this warpgroup's 8 channels of the group
                    uint32_t w[8][8];
#pragma unroll
                    for (int phi = 0; phi < 8; ++phi) tmem_ld8(lane_addr + buf * 256 + phi * TNG + j0, w[phi]);
                    tmem_ld_wait();
                    tc_fence_before();
                    mbar_arrive(&tfree[buf]);  // values are in registers: the buffer may be overwritten by group cg + 2
                    float *yb = y + ((size_t)b * COT + cg * TNG + j0) * Lout + (own ? 8 * sg - PADT : 0);
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float bj = __ldg(tbias + cg * TNG + j0 + j);
                        float *yp = yb + (size_t)j * Lout;
                        if (lo_ok)
                            *reinterpret_cast<float4 *>(yp) = make_float4(__uint_as_float(w[0][j]) + bj, __uint_as_float(w[1][j]) + bj,
                                                                          __uint_as_float(w[2][j]) + bj, __uint_as_float(w[3][j]) + bj);
                        if (hi_ok)
                            *reinterpret_cast<float4 *>(yp + 4) = make_float4(__uint_as_float(w[4][j]) + bj, __uint_as_float(w[5][j]) + bj,
                                                                              __uint_as_float(w[6][j]) + bj, __uint_as_float(w[7][j]) + bj);
                    }
                }
            }
        } else {
        // ---- store the valid part of R + pend
#pragma unroll 1
        for (int it = wg; it < ITEMS; it += NWG) {
            const int blk = it / PARTS, cbeg = (it % PARTS) * CW;
            const int p = blk * 128 + row, t = o + p;
            const bool valid = (p >= p_lo && p < p_hi && t < L);
            float *yp = y + (size_t)b * C * LS + (valid ? t : 0);
#pragma unroll 1
            for (int c0 = cbeg; c0 < cbeg + CW; c0 += 32) {
                uint32_t v[32];
                tmem_ld32(lane_addr + blk * 2 * C + c0, v);
                tmem_ld_wait();
                if (valid) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) yp[(size_t)(c0 + j) * LS] = __uint_as_float(v[j]) + pend[c0 + j];
                }
            }
        }
        }
        if (warp == 0) MG_TR(20);
    }
#undef MG_TR
#undef MG_XREADY_ARRIVE
    tc_fence_before();
    __syncthreads();
    if constexpr (G2) cluster_sync();  // both CTAs are done with the pair's tensor memory
    if (warp == 0) {
        if constexpr (G2) tmem_dealloc2(tmem, Cfg::TCOLS); else tmem_dealloc(tmem, Cfg::TCOLS);
    }
    if constexpr (CL > 1) cluster_sync();  // nobody leaves while the peer may still multicast into its ring or arrive on its barriers
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (the library does not link libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess)
            p = nullptr;
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}
static bool tma_disabled() {
    static const bool off = [] { const char *e = getenv("MG_RES_TMA"); return e && e[0] == '0'; }();
    return off;
}
// can x [B][C][L] fp32 be described by a tensor map? (16-byte aligned base and row stride)
static bool tma_input_ok(const float *x, int L) {
    return !tma_disabled() && (L % 4) == 0 && ((uintptr_t)x % 16) == 0 && encode_tiled_fn() != nullptr;
}
// x as a 3-D tensor (L, C, B) with boxes of (P positions, LCH channels, 1 item); out-of-bounds positions read as zero
static int make_input_map(CUtensorMap *m, const float *x, int B, int C, int L, int P, int LCH) {
    const cuuint64_t dims[3] = {(cuuint64_t)L, (cuuint64_t)C, (cuuint64_t)B};
    const cuuint64_t strides[2] = {(cuuint64_t)L * 4, (cuuint64_t)L * C * 4};
    const cuuint32_t box[3] = {(cuuint32_t)P, (cuuint32_t)LCH, 1}, estr[3] = {1, 1, 1};
    const CUresult r = encode_tiled_fn()(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float *>(x), dims, strides, box, estr,
                                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_error(MG_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) for [%d][%d][%d]", (int)r, B, C, L);
    return MG_OK;
}

// vt != nullptr: ragged launch (VL instantiation), vt->n items, L = the padded row stride = mul * T
template <class Cfg, bool VL = false>
static int launch_resblock(const float *x, float *y, const float *packed, int stage, int B, int L, int *status,
                           long long *trace, cudaStream_t s, const VarLenTab *vt = nullptr, int mul = 1) {
    static bool configured = false;
    if (!configured) {
        MG_CUDA_TRY(cudaFuncSetAttribute(resblock_tc_kernel<Cfg, VL>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
        configured = true;
    }
    constexpr int PS = Cfg::CL * Cfg::P, PVS = PS - Cfg::HALO - Cfg::HL;  // edge-aware tiling in super-tiles of CL tiles, see the kernel
    const int Lc = L;
    const int ntiles = 1 + (Lc > PS ? (Lc - PS + PVS - 1) / PVS : 0);
    CUtensorMap xmap;
    memset(&xmap, 0, sizeof(xmap));
    if constexpr (Cfg::TMA) {
        int rc = make_input_map(&xmap, x, B, Cfg::C, L, Cfg::P, Cfg::LCH);
        if (rc) return rc;
    }
    // (G2: the (item, tile) list pairs up along x; an odd total gets one phantom tile, see the kernel)
    dim3 grid = Cfg::G2 ? dim3((unsigned)(((long long)ntiles * B + 1) / 2 * 2), 1) : dim3(ntiles * Cfg::CL, B);
    VarLenArg<VL> vl{};
    if constexpr (VL) {  // the (item, super-tile) list: each item gets exactly the tiles a launch of its own length would
        vl = *vt;
        vl.mul = mul;
        int acc = 0;
        for (int i = 0; i < vl.n; ++i) {
            const int Li = mul * (vl.cum[i + 1] - vl.cum[i]);
            vl.first[i] = acc;
            acc += 1 + (Li > PS ? (Li - PS + PVS - 1) / PVS : 0);
        }
        vl.first[vl.n] = acc;
        grid = dim3((unsigned)acc * Cfg::CL, 1);
    }
    MG_CUDA_TRY(launch_ex(resblock_tc_kernel<Cfg, VL>, grid, dim3(Cfg::NT), Cfg::SMEM_BYTES, s, Cfg::CLUSTER, true, x, y,
                          packed, stage, L, B, status, trace, xmap, vl));
    return MG_OK;
}

template <class Cfg>
static const char *cfg_name() {
    static char buf[96];
    snprintf(buf, sizeof(buf), "resblock_tc_kernel<RbCfg<%d,%d,%d,%d,%d,%d,%d,%d,%d,%d,%d>>/NH%d", Cfg::C, Cfg::NBLK, Cfg::NSTAGE, Cfg::NWG,
             Cfg::MINB, (int)Cfg::POST, (int)Cfg::UPF, Cfg::CL, Cfg::UPT, (int)Cfg::TMA, (int)Cfg::G2, Cfg::NH);
    return buf;
}

// x, y: [B][C][L] fp32 NCL with C = 256 >> stage; status: device int, set non-zero if a pipeline wait timed out.
int launch_resblock_tc(const float *x, float *y, const float *packed, int stage, int B, int L, int *status, cudaStream_t s,
                       long long *trace) {
    const bool tma = tma_input_ok(x, L);  // input tile by tensor-map TMA (needs 16-byte aligned rows), else per-thread loads
    switch (stage) {
        //                                       C  NBLK NSTAGE NWG MINB
        // (C = 256 is paced by its 4-slot weight ring -- 3 slots: 204 us, 4: 184 us -- but a fifth 16 KB slot only fits if the
        //  bias staging goes: reading the biases from global memory in the epilogue instead cost far more (264 us; at 231 KB of
        //  shared memory there is no L1 left for them))
        // L > 128: CTA pairs sharing a 256-position super-tile (no halo between the two; multicast weights).  MG_RES0_PAIR=0: A/B.
        case 0: {
            static const bool pair = [] { const char *e = getenv("MG_RES0_PAIR"); return !(e && e[0] == '0'); }();
            if (pair && L > 128)
                return tma ? launch_resblock<RbCfg<256, 1, 4, 4, 1, false, false, 2, 0, true>>(x, y, packed, stage, B, L, status, trace, s)
                           : launch_resblock<RbCfg<256, 1, 4, 4, 1, false, false, 2>>(x, y, packed, stage, B, L, status, trace, s);
            return tma ? launch_resblock<RbCfg<256, 1, 4, 4, 1, false, false, 1, 0, true>>(x, y, packed, stage, B, L, status, trace, s)
                       : launch_resblock<RbCfg<256, 1, 4, 4, 1>>(x, y, packed, stage, B, L, status, trace, s);
        }
        // (C = 128 as two single-block CTAs per SM, RbCfg<128, 1, 2, 2, 2>: measured 244 us vs 213 us at config 2 -- the
        //  25 % halo recompute and the two-slot weight rings cost more than the overlap buys)
        case 1: {
            // cta_group::2 pairs of tiles (RbCfg<..., G2>): built, parity-green, and SLOWER at config 2 -- 257 us vs 197 us: the
            // M = 256 MMAs issue at ~78 cycles instead of 64-69 and the epilogue that overlaps them takes 6.5 k cycles instead of
            // 3.8 k (phase trace in DESIGN.md section 5) -- so it is opt-in: MG_RES1_G2=1
            static const bool g2 = [] { const char *e = getenv("MG_RES1_G2"); return e && e[0] == '1'; }();
            if (g2 && tma && (long long)B * (1 + (L > 256 ? (L - 256 + 223) / 224 : 0)) >= 2)
                return launch_resblock<RbCfg<128, 2, 4, 4, 1, false, false, 1, 0, true, true>>(x, y, packed, stage, B, L, status, trace, s);
            return tma ? launch_resblock<RbCfg<128, 2, 4, 4, 1, false, false, 1, 0, true>>(x, y, packed, stage, B, L, status, trace, s)
                       : launch_resblock<RbCfg<128, 2, 4, 4, 1>>(x, y, packed, stage, B, L, status, trace, s);
        }
        // (3 CTAs/SM with half-size tiles was measured slower for C = 64 / 32: the extra halo recompute outweighs the overlap)
        case 2:
            return tma ? launch_resblock<RbCfg<64, 2, 2, 2, 2, false, false, 1, 0, true>>(x, y, packed, stage, B, L, status, trace, s)
                       : launch_resblock<RbCfg<64, 2, 2, 2, 2>>(x, y, packed, stage, B, L, status, trace, s);
        // (C = 32 with the two A = hi(x) passes merged into one N = 64 MMA against [w hi | w lo] -- 4C TMEM columns per
        //  block, so NBLK = 2: measured 184 us vs 142 us; this stage is bound by its epilogue, which then reads twice the
        //  accumulator columns, not by the A-operand re-reads the merge saves)
        case 3: return launch_resblock<RbCfg<32, 4, 4, 2, 2>>(x, y, packed, stage, B, L, status, trace, s);
        // stage 4 = ResBlock 3 with LeakyReLU -> conv_post -> tanh fused: y is the audio [B][1][L]
        case 4: return launch_resblock<RbCfg<32, 4, 4, 2, 2, true>>(x, y, packed, 3, B, L, status, trace, s);
        // 12 / 13 / 14 = stages 2 / 3 / 3+post with the stage's stride-2 ConvT fused in: x is the PREVIOUS stage's output
        // [B][2C][L/2] (L stays the output length)
        // 20 / 21 / 22 = ResBlock 0 / 1 / 2 with the NEXT stage's LeakyReLU -> ConvT at its tail: y is [B][C/2][S L]
        case 20:
            if (L > 128)
                return tma ? launch_resblock<RbCfg<256, 1, 4, 4, 1, false, false, 2, 8, true>>(x, y, packed, 0, B, L, status, trace, s)
                           : launch_resblock<RbCfg<256, 1, 4, 4, 1, false, false, 2, 8>>(x, y, packed, 0, B, L, status, trace, s);
            return tma ? launch_resblock<RbCfg<256, 1, 4, 4, 1, false, false, 1, 8, true>>(x, y, packed, 0, B, L, status, trace, s)
                       : launch_resblock<RbCfg<256, 1, 4, 4, 1, false, false, 1, 8>>(x, y, packed, 0, B, L, status, trace, s);
        case 21:
            return tma ? launch_resblock<RbCfg<128, 2, 4, 4, 1, false, false, 1, 2, true>>(x, y, packed, 1, B, L, status, trace, s)
                       : launch_resblock<RbCfg<128, 2, 4, 4, 1, false, false, 1, 2>>(x, y, packed, 1, B, L, status, trace, s);
        case 22:
            return tma ? launch_resblock<RbCfg<64, 2, 2, 2, 2, false, false, 1, 2, true>>(x, y, packed, 2, B, L, status, trace, s)
                       : launch_resblock<RbCfg<64, 2, 2, 2, 2, false, false, 1, 2>>(x, y, packed, 2, B, L, status, trace, s);
        case 12: return launch_resblock<RbCfg<64, 2, 2, 2, 2, false, true>>(x, y, packed, 2, B, L, status, trace, s);
        case 13: return launch_resblock<RbCfg<32, 4, 4, 2, 2, false, true>>(x, y, packed, 3, B, L, status, trace, s);
        case 14: return launch_resblock<RbCfg<32, 4, 4, 2, 2, true, true>>(x, y, packed, 3, B, L, status, trace, s);
    }
    return set_error(MG_ERR_INVALID_ARGUMENT, "launch_resblock_tc: stage %d", stage);
}

// The default chain's four ResBlock kernels on a ragged batch: code 20 (res0+up1), 1 (res1), 22 (res2+up3), 4 (res3+post), the
// configurations launch_resblock_tc picks for a uniform batch.  x [vt.n][C][mul T] with mul = 8 / 64 / 128 / 256, item b's first
// mul * (cum[b+1] - cum[b]) positions.  Stage 0 runs CTA pairs if the LONGEST item would (a pair is bit-identical to the single
// tile on a short item: the same products in the same K order; the second CTA just owns positions past the item's end).
int launch_resblock_tc_varlen(const float *x, float *y, const float *packed, int code, const VarLenTab &vt, int T, int *status,
                              cudaStream_t s) {
    int maxlen = 0;
    for (int i = 0; i < vt.n; ++i) maxlen = vt.cum[i + 1] - vt.cum[i] > maxlen ? vt.cum[i + 1] - vt.cum[i] : maxlen;
    const int mul = code == 20 ? 8 : code == 1 ? 64 : code == 22 ? 128 : 256, LS = mul * T;
    const bool tma = tma_input_ok(x, LS);
    switch (code) {
        case 20:
            if (8 * maxlen > 128)
                return tma ? launch_resblock<RbCfg<256, 1, 4, 4, 1, false, false, 2, 8, true>, true>(x, y, packed, 0, vt.n, LS, status, nullptr, s, &vt, mul)
                           : launch_resblock<RbCfg<256, 1, 4, 4, 1, false, false, 2, 8>, true>(x, y, packed, 0, vt.n, LS, status, nullptr, s, &vt, mul);
            return tma ? launch_resblock<RbCfg<256, 1, 4, 4, 1, false, false, 1, 8, true>, true>(x, y, packed, 0, vt.n, LS, status, nullptr, s, &vt, mul)
                       : launch_resblock<RbCfg<256, 1, 4, 4, 1, false, false, 1, 8>, true>(x, y, packed, 0, vt.n, LS, status, nullptr, s, &vt, mul);
        case 1:
            return tma ? launch_resblock<RbCfg<128, 2, 4, 4, 1, false, false, 1, 0, true>, true>(x, y, packed, 1, vt.n, LS, status, nullptr, s, &vt, mul)
                       : launch_resblock<RbCfg<128, 2, 4, 4, 1>, true>(x, y, packed, 1, vt.n, LS, status, nullptr, s, &vt, mul);
        case 22:
            return tma ? launch_resblock<RbCfg<64, 2, 2, 2, 2, false, false, 1, 2, true>, true>(x, y, packed, 2, vt.n, LS, status, nullptr, s, &vt, mul)
                       : launch_resblock<RbCfg<64, 2, 2, 2, 2, false, false, 1, 2>, true>(x, y, packed, 2, vt.n, LS, status, nullptr, s, &vt, mul);
        case 4: return launch_resblock<RbCfg<32, 4, 4, 2, 2, true>, true>(x, y, packed, 3, vt.n, LS, status, nullptr, s, &vt, mul);
    }
    return set_error(MG_ERR_INVALID_ARGUMENT, "launch_resblock_tc_varlen: code %d is not a default-chain ResBlock kernel", code);
}

// the configuration launch_resblock_tc picks for (stage code, L) with a 16-byte aligned input: evidence files (ncu captures) record
// it, bench.py refuses a capture whose configuration is not the one this build runs
const char *resblock_config_name(int stage, int L) {
    const bool tma = !tma_disabled() && (L % 4) == 0 && encode_tiled_fn() != nullptr;
    switch (stage) {
        case 0: {
            static const bool pair = [] { const char *e = getenv("MG_RES0_PAIR"); return !(e && e[0] == '0'); }();
            if (pair && L > 128)
                return tma ? cfg_name<RbCfg<256, 1, 4, 4, 1, false, false, 2, 0, true>>()
                           : cfg_name<RbCfg<256, 1, 4, 4, 1, false, false, 2>>();
            return tma ? cfg_name<RbCfg<256, 1, 4, 4, 1, false, false, 1, 0, true>>()
                       : cfg_name<RbCfg<256, 1, 4, 4, 1>>();
        }
        case 1: {
            const char *e = getenv("MG_RES1_G2");
            if (e && e[0] == '1' && tma) return cfg_name<RbCfg<128, 2, 4, 4, 1, false, false, 1, 0, true, true>>();
            return tma ? cfg_name<RbCfg<128, 2, 4, 4, 1, false, false, 1, 0, true>>()
                       : cfg_name<RbCfg<128, 2, 4, 4, 1>>();
        }
        case 2:
            return tma ? cfg_name<RbCfg<64, 2, 2, 2, 2, false, false, 1, 0, true>>()
                       : cfg_name<RbCfg<64, 2, 2, 2, 2>>();
        case 3: return cfg_name<RbCfg<32, 4, 4, 2, 2>>();
        case 4: return cfg_name<RbCfg<32, 4, 4, 2, 2, true>>();
        case 20:
            if (L > 128)
                return tma ? cfg_name<RbCfg<256, 1, 4, 4, 1, false, false, 2, 8, true>>()
                           : cfg_name<RbCfg<256, 1, 4, 4, 1, false, false, 2, 8>>();
            return tma ? cfg_name<RbCfg<256, 1, 4, 4, 1, false, false, 1, 8, true>>()
                       : cfg_name<RbCfg<256, 1, 4, 4, 1, false, false, 1, 8>>();
        case 21:
            return tma ? cfg_name<RbCfg<128, 2, 4, 4, 1, false, false, 1, 2, true>>()
                       : cfg_name<RbCfg<128, 2, 4, 4, 1, false, false, 1, 2>>();
        case 22:
            return tma ? cfg_name<RbCfg<64, 2, 2, 2, 2, false, false, 1, 2, true>>()
                       : cfg_name<RbCfg<64, 2, 2, 2, 2, false, false, 1, 2>>();
        case 12: return cfg_name<RbCfg<64, 2, 2, 2, 2, false, true>>();
        case 13: return cfg_name<RbCfg<32, 4, 4, 2, 2, false, true>>();
        case 14: return cfg_name<RbCfg<32, 4, 4, 2, 2, true, true>>();
    }
    return "";
}

}  // namespace mg
