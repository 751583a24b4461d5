// preproc_bsw.cuh — banded store-warp kernel: frames that do not fit shared memory whole (240x320), compile-time geometry.
//
// The phases are those of preproc_fast.cuh (P1 strip walk, P2 non-maximum suppression, P3 hysteresis, P4 output), the frame goes
// through them in bands of R rows like k_preprocess_banded, and two store warps own the output phase like k_preprocess_sw.  What
// is new is how the ten compute warps are ordered against each other: there is NO CTA-wide barrier inside a frame's bands.
//
//  * A warp owns a column block of 32 pixels (8 strips x 4 row segments of R/4 rows) in both walks, so the non-maximum suppression
//    of a band depends only on the magnitudes of the warp's own block and of the blocks left and right of it: after its strip walk a
//    warp arrives on its own mbarrier (two per warp, by band parity) and waits for its two neighbours' barriers, nobody else's.  A
//    waiting warp sleeps in the barrier unit (try_wait with a suspend hint) instead of spinning on issue slots the other warps need.
//  * The magnitude rows of a band live in one of two buffers (band parity).  A warp that writes buffer q for band b + 2 has passed
//    the suppression of band b + 1, which needed its neighbours' strip walks of band b + 1, which they run after their suppression of
//    band b: the forward barriers alone make the reuse safe, and a neighbour can never be two phases ahead on one barrier.
//  * The suppression lags the strip walk by one row (band b decides rows R b - 1 .. R b + R - 2), so it never needs a magnitude row
//    of a later band and no halo row is computed twice; the two rows it needs from the band before are the last two window rows of
//    the same warp's bottom segment: they cross the band boundary through a 48-byte slot per lane.  Row H - 1 is decided by one
//    extra step after the last band.
//  * The band's pixel rows arrive by one bulk copy; the last warp to finish the strip walk of a band (a shared-memory counter)
//    issues the copy of the next band, the others are already in the suppression.
//  * The colour-mask rows live in a ring of NB + 2 band slots (a band's rows are final after its strip walk and are only read slab by
//    slab by the store warps): the store warps arrive on a slot's barrier when its slab is written and a strip walk waits for the slot it
//    is about to reuse, so the first bands of a frame never wait for the store warps to get going.  The edge plane is double-buffered
//    by frame parity, the candidate plane is handed back by a "hysteresis finished" barrier.
//  * NSW store warps per CTA: two at 240x320 (two CTAs per SM), one at 120x160 (five compute warps, four CTAs per SM).
//  * One named barrier per frame among the compute warps (before the hysteresis, whose row bands cut across the column blocks).
//  * Frames come on demand (draw_frames, preproc_fast.cuh): the store warps draw frame j + 2 while the compute warps finish frame j and
//    publish it in the frame ring before their "hysteresis finished" arrival of frame j, which the compute warps wait for in band 0 of
//    frame j + 1, ahead of the last band, where the last warp out issues the copy of frame j + 2's first band.
#pragma once
#include "preproc_fast.cuh"

namespace trs {

template <int H, int W, int R, int NR, int NSW = 2>
struct BswLayout {
    static_assert(W % 32 == 0 && H % R == 0 && R % 12 == 0, "column blocks of 32 pixels, whole bands, four segments of a multiple of 3 rows");
    static constexpr int NCW = W / 32;                                 // compute warps = column blocks
    static constexpr int NB = H / R;                                   // bands per frame
    static constexpr int SEG = R / 4;
    static constexpr int ROWB = W * 3;
    static constexpr int MS2 = (W + 4) * 2;                            // bytes per magnitude row
    static constexpr int PRB = W / 8;                                  // plane bytes per row
    static constexpr int PLANE = (((H + 2) * (W / 32) * 4) + 15) & ~15;
    static constexpr int NSLOT = NB + 2;                               // colour-mask ring: band slots of R rows
    static constexpr int SLOTB = R * PRB;
    static constexpr int MASKP = NSLOT * SLOTB;                        // ring bytes per colour range
    static constexpr int PIX = 16 + (R + 2) * ROWB + 16;
    static constexpr int MAG = (((2 * R + 1) * MS2 + 16) + 15) & ~15;   // two buffers of R rows + the row the look-ahead fetch touches
    static constexpr int STASH_ROW = 24, STASH_LANE = 2 * STASH_ROW;
    static constexpr int OFF_PIX = 0;
    static constexpr int OFF_MAG = OFF_PIX + PIX;
    static constexpr int OFF_MASK = OFF_MAG + MAG;
    static constexpr int OFF_CAND = OFF_MASK + NR * MASKP;
    static constexpr int OFF_EDGE = OFF_CAND + PLANE;                  // two planes
    static constexpr int OFF_STASH = OFF_EDGE + 2 * PLANE;             // NCW x 8 lanes x 2 rows, then one zero row
    static constexpr int OFF_SDIV = (OFF_STASH + NCW * 8 * STASH_LANE + STASH_ROW + 15) & ~15;
    static constexpr int OFF_HUE = OFF_SDIV + 1024;
    static constexpr int OFF_BAR = OFF_HUE + 1024;                     // mbarriers: pixels, hysteresis finished, 2 per compute warp, 1 per mask slot
    static constexpr int NBAR = 2 + 2 * NCW + NSLOT;
    static constexpr int OFF_SYNC = OFF_BAR + 8 * NBAR;                // strip-walk counter, then the frame ring (FRAME_RING u32)
    static constexpr int OFF_RED = (OFF_SYNC + 16 + 4 * FRAME_RING + 15) & ~15;
    static constexpr int OFF_LUT = OFF_RED + 32 + 128;                 // brightness / contrast table (static, or rebuilt per frame)
    static constexpr int TOTAL = OFF_LUT + 256;
    static constexpr int THREADS = 32 * (NCW + NSW);
};

__device__ __forceinline__ uint32_t atom_inc_acq_rel(uint32_t a)
{
    uint32_t old;
    asm volatile("atom.acq_rel.cta.shared.add.u32 %0, [%1], 1;" : "=r"(old) : "r"(a) : "memory");
    return old;
}

// =========================================================================================================
// P2 for one band, lagging the strip walk by a row: every lane decides SEG rows starting at r0 (the band's rows shifted up by one).
// The first two window rows come from a_up / a_ce (per lane: magnitude rows of this band, or the slot the bottom segment filled a
// band earlier, or the zero row at the top of the frame); slot != 0: leave the last two window rows there for the next band;
// tail: decide one more row with zeros below it (the frame's last row, after the last band), stored by the tail lanes only.
// =========================================================================================================
template <int SEG>
__device__ __forceinline__ void p2_nms_lagged(const FastParams& P, const Dims& Dm, uint32_t a_mag, uint32_t a_cand, uint32_t a_edge, const SmemMap& S, int strip,
                                              bool store_lane, int r0, uint32_t a_up, uint32_t a_ce, uint32_t slot, bool tail, bool tail_lane)
{
    static_assert(SEG % 3 == 0, "whole trips only");
    const int prb = Dm.w >> 3, MS2 = Dm.mag_stride * 2;
    const uint32_t mbase = a_mag + 2 * (4 + 4 * strip);
    struct Row { uint32_t p01, p23, l01, m12, r23, raw01, raw23; };
    struct Raw { uint2 c; uint32_t ml, mr; };
    auto fetch_at = [&](uint32_t rp) {
        Raw q;
        q.c = lds64(rp); q.ml = lds16(rp - 2); q.mr = lds16(rp + 8);
        return q;
    };
    auto unpack_row = [&](const Raw& q) {
        Row r;
        r.raw01 = q.c.x; r.raw23 = q.c.y;
        r.p01 = q.c.x & 0x07ff07ffu; r.p23 = q.c.y & 0x07ff07ffu;
        r.l01 = prmt(q.ml & 0x7ffu, r.p01, 0x5410);
        r.m12 = prmt(r.p01, r.p23, 0x5432);
        r.r23 = prmt(r.p23, q.mr & 0x7ffu, 0x5432);
        return r;
    };
    Raw ahead;
    uint32_t cp = a_cand + (strip >> 1) + r0 * prb, ep = a_edge + (strip >> 1) + r0 * prb;      // plane bytes of the row being decided
    uint32_t ap = mbase + (r0 + 3) * MS2;                                                     // row fetched ahead: r0 + 2 + k at step k
    auto nms_step = [&](bool store, const Row& up, const Row& ce, Row& dn) {
        dn = unpack_row(ahead);
        ahead = fetch_at(ap); ap += MS2;
        uint32_t cm[2], sm[2];
#pragma unroll
        for (int pr = 0; pr < 2; ++pr) {
            const uint32_t C = pr ? ce.p23 : ce.p01;
            const uint32_t raw = pr ? ce.raw23 : ce.raw01;
            const uint32_t L = pr ? ce.m12 : ce.l01, Rr = pr ? ce.r23 : ce.m12;
            const uint32_t U = pr ? up.p23 : up.p01, Dw = pr ? dn.p23 : dn.p01;
            const uint32_t UL = pr ? up.m12 : up.l01, DR = pr ? dn.r23 : dn.m12;
            const uint32_t UR = pr ? up.r23 : up.m12, DL = pr ? dn.m12 : dn.l01;
            const uint32_t b0 = prmt_sx(raw << 4, 0, 0xbb99), b1 = prmt_sx(raw << 3, 0, 0xbb99);
            const uint32_t na = bsel(b1, bsel(b0, UR, UL), bsel(b0, U, L));
            const uint32_t nb = bsel(b1, bsel(b0, DL, DR), bsel(b0, Dw, Rr)) + (b1 & 0x00010001u);
            cm[pr] = hgt_mask(C, na) & hge_mask(C, nb) & hgt_mask(C, P.low2);
            sm[pr] = cm[pr] & hgt_mask(C, P.high2);
        }
        const uint32_t top = nibble_pair_top(prmt(cm[0], cm[1], 0x6420), prmt(sm[0], sm[1], 0x6420));
        const uint32_t other = __shfl_down_sync(0xffffffffu, top, 1);
        uint32_t bc, bs;
        merge_nibble_pairs(top, other, bc, bs);
        sts8_if(store, cp, bc);
        sts8_if(store, ep, bs);
        cp += prb; ep += prb;
    };
    Row ra = unpack_row(fetch_at(a_up)), rb = unpack_row(fetch_at(a_ce)), rc;
    ahead = fetch_at(mbase + (r0 + 2) * MS2);                    // row r0 + 1
#pragma unroll 1
    for (int k = 0; k < SEG; k += 3) {
        nms_step(store_lane, ra, rb, rc);
        nms_step(store_lane, rb, rc, ra);
        nms_step(store_lane, rc, ra, rb);
    }
    if (slot) {                                                  // window rows (ra, rb) = the first two of the segment below
        sts16(slot + 8 - 2, ra.l01 & 0xffffu); sts64(slot + 8, make_uint2(ra.raw01, ra.raw23)); sts16(slot + 8 + 8, ra.r23 >> 16);
        sts16(slot + 24 + 8 - 2, rb.l01 & 0xffffu); sts64(slot + 24 + 8, make_uint2(rb.raw01, rb.raw23)); sts16(slot + 24 + 8 + 8, rb.r23 >> 16);
    }
    if (tail) {
        ahead.c = make_uint2(0u, 0u); ahead.ml = 0; ahead.mr = 0;
        nms_step(store_lane && tail_lane, ra, rb, rc);
    }
}

// =========================================================================================================
// the kernel: NCW compute warps + 2 store warps, two CTAs per SM
// =========================================================================================================
// LUT: a brightness / contrast table that is not the identity.  The strip walk applies it to the pixel words as it loads them (the column-block
// warps have no common moment at which the band's rows could be rewritten in place).  The dynamic table of a frame is built at the top of the
// frame from exact channel sums over rows 40..118 (img_preprocessing.py:88), read from global memory by the compute warps (the bands read those
// rows again, from L2); the sums of two consecutive frames alternate between two sets of accumulators, so two barriers among the compute
// warps per frame are enough.
template <int NR, int F0, int F1, int H, int W, int R, int NSW = 2, int MAXREG = SW_MAXREG, bool LUT = false, bool LIST = false>
__global__ void __maxnreg__(MAXREG) k_preprocess_bsw(const __grid_constant__ FastParams P, const FrameList fl = {})
{
    using L = BswLayout<H, W, R, NR, NSW>;
    extern __shared__ __align__(16) uint8_t smem[];
    const PreKParams& p = P.k;
    int n_list = 0;
    const int* list = nullptr;
    if constexpr (LIST) {                                          // (the frame ring holds positions in the list, the loads map them to frames)
        plist_open(fl, list, n_list);
        if ((int)blockIdx.x >= n_list) return;
    }
    uint32_t sb = smem_u32(smem);
    asm volatile("" : "+r"(sb));
    constexpr int NCW = L::NCW, NC = 32 * NCW, NS = 32 * NSW, NT = NC + NS, NB = L::NB, SEG = L::SEG, ww = W / 32, NSLOT = L::NSLOT;
    constexpr uint32_t frame_bytes = (uint32_t)H * W * 3;
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);       // (tells the compiler the role branch below is warp-uniform)
    SmemMap S;
    S.pix[0] = S.pix[1] = sb + L::OFF_PIX + 16;
    S.mag[0] = S.mag[1] = sb + L::OFF_MAG;
    S.mask = sb + L::OFF_MASK;                                     // slot 0 of the ring of range 0
    S.cand = sb + L::OFF_CAND + ww * 4;
    S.edge = sb + L::OFF_EDGE + ww * 4;
    S.edge2 = S.edge + L::PLANE;
    S.sdiv = sb + L::OFF_SDIV; S.hue = sb + L::OFF_HUE; S.lut = sb + L::OFF_LUT; S.bar = sb + L::OFF_BAR; S.red = sb + L::OFF_RED;
    // mbarriers: [0] pixels of a band landed, [1] hysteresis of a frame finished, [2 + 2 w + q] strip walk of warp w for a band of parity q,
    // [2 + 2 NCW + s] the slab in mask slot s is written
    const uint32_t bar_pix = S.bar, bar_p3 = S.bar + 8, bar_p1 = S.bar + 16, bar_slot = bar_p1 + 16 * NCW;
    const uint32_t a_cnt = sb + L::OFF_SYNC, a_ring = a_cnt + 16;
    const uint32_t a_stash = sb + L::OFF_STASH, a_zero = a_stash + NCW * 8 * L::STASH_LANE;
    Dims Dm;
    Dm.h = H; Dm.w = W; Dm.mag_stride = W + 4; Dm.plane_bytes = L::MASKP;      // (the walks use plane_bytes for the stride between colour ranges only)
    const uint32_t n = (uint32_t)(LIST ? n_list : p.n);
    static_assert(NB >= 2, "the last band reads the next frame after band 0's wait for the hysteresis of the frame before");

    uint32_t ticket = 0;
    if (tid == NC) ticket = draw_frames(p);                        // frame 1, in flight during the set-up
    init_tables<NR, F0, F1>(p, S, tid, NT);
    stats_zero(S, tid);
    for (int i = tid; i < 2 * R + 2; i += NT) {                   // the zero left of pixel 0 (element 3) and right of pixel W - 1 (element 0 of the next row)
        sts16(S.mag[0] + i * L::MS2, 0);
        if (i < 2 * R + 1) sts16(S.mag[0] + i * L::MS2 + 6, 0);
    }
    zero_plane_pads(S, H * ww, ww, tid, NT);
    if (tid == 0) sts32(a_cnt, 0);
    if (tid < 6) sts32(S.red + 4 * tid, 0);                        // ROI sums: three u32 per frame parity
    for (int i = tid; i < L::STASH_ROW / 4; i += NT) sts32(a_zero + 4 * i, 0);
    if (tid < L::NBAR) mbar_init(S.bar + 8 * tid, tid >= 2 + 2 * NCW ? (uint32_t)NSW : 1u);      // a slot's barrier takes every store warp
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    if (tid == NC) { sts32(a_ring, blockIdx.x); sts32(a_ring + 4, ticket); }
    __syncthreads();

    // pixel rows of band b: [max(R b - 1, 0), min(R b + R + 1, H))
    auto issue_band = [&](size_t f, int b) {
        const int p0 = max(b * R - 1, 0), p1 = min(b * R + R + 1, H);
        issue_frame_load(S.pix[0], p.in + f * frame_bytes + (size_t)p0 * L::ROWB, (uint32_t)(p1 - p0) * L::ROWB, bar_pix);
    };

    if (warp < NCW) {
        // ------------------------------------------------ compute warps -----------------------------------------------
        const int seg = lane >> 3;
        StripMap M;
        M.strip = 8 * warp + (lane & 7);
        M.ok = true;
        M.store_lane = !(lane & 1);
        const uint32_t my_slot = a_stash + (uint32_t)(warp * 8 + (lane & 7)) * L::STASH_LANE;
        const uint32_t my_bar = bar_p1 + 16 * warp;
        if (tid == 0 && blockIdx.x < n) issue_band(plist_frame<LIST>(list, blockIdx.x), 0);
        uint32_t gb = 0;                                          // bands finished by this warp since the kernel started
        int slot = 0;                                             // gb % NSLOT: the mask slot of the band
        uint32_t round = 0;                                       // gb / NSLOT: how often the slot has been used before
        // the CTA's frame k (k >= 2) is published before the store warps' arrival on bar_p3 for frame k - 2, which every compute thread
        // waits for in band 0 of frame k - 1; it is read in the last band of frame k - 1 (the last warp out) and at the top of iteration k.
        // Frames 0 and 1: set-up barrier.
#pragma unroll 1
        for (int j = 0;; ++j) {
            const uint32_t fj = ring_frame(a_ring, j);
            if (fj >= n) break;
            const uint32_t f = plist_frame<LIST>(list, fj);
            const uint32_t a_edge = (j & 1) ? S.edge2 : S.edge;
            if (LUT && p.dynamic) {
                constexpr int Y0 = H < 40 ? H : 40, Y1 = H < 119 ? H : 119, NTRI = (Y1 - Y0) * L::ROWB / 12;      // groups of four pixels = three words
                const uint32_t* roi = reinterpret_cast<const uint32_t*>(p.in + (size_t)f * frame_bytes + (size_t)Y0 * L::ROWB);
                uint32_t c0 = 0, c1 = 0, c2 = 0;
#pragma unroll 4
                for (int i = tid; i < NTRI; i += NC) {
                    const uint32_t w0 = __ldg(roi + 3 * i), w1 = __ldg(roi + 3 * i + 1), w2 = __ldg(roi + 3 * i + 2);      // R G B R | G B R G | B R G B
                    c0 = __dp4a(w2, 0x00000100u, __dp4a(w1, 0x00010000u, __dp4a(w0, 0x01000001u, c0)));
                    c1 = __dp4a(w2, 0x00010000u, __dp4a(w1, 0x01000001u, __dp4a(w0, 0x00000100u, c1)));
                    c2 = __dp4a(w2, 0x01000001u, __dp4a(w1, 0x00000100u, __dp4a(w0, 0x00010000u, c2)));
                }
                for (int o = 16; o; o >>= 1) {
                    c0 += __shfl_xor_sync(0xffffffffu, c0, o);
                    c1 += __shfl_xor_sync(0xffffffffu, c1, o);
                    c2 += __shfl_xor_sync(0xffffffffu, c2, o);
                }
                const uint32_t a_sum = S.red + 12 * (uint32_t)(j & 1);
                if (lane == 0) {
                    asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(a_sum), "r"(c0) : "memory");
                    asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(a_sum + 4), "r"(c1) : "memory");
                    asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(a_sum + 8), "r"(c2) : "memory");
                }
                bar_sync(3, NC);
                const uint32_t s0 = lds32(a_sum), s1 = lds32(a_sum + 4), s2 = lds32(a_sum + 8);
                const float fdelta = (float)brightness_delta(s0, s1, s2, (double)((Y1 - Y0) * W), p.baseline);
                for (int i = tid; i < 256; i += NC) sts8(S.lut + i, adjust_entry(i, true, fdelta, p.foff, p.fratio));
                if (tid == 0) {
                    const uint32_t a_next = S.red + 12 * (uint32_t)((j + 1) & 1);      // (last touched a frame ago, before that frame's hysteresis barrier)
                    sts32(a_next, 0); sts32(a_next + 4, 0); sts32(a_next + 8, 0);
                    if (p.stats) stat_add_one(S, 9, (unsigned long long)s0 + s1 + s2);
                }
                bar_sync(3, NC);
            }
#pragma unroll 1
            for (int b = 0; b < NB; ++b, ++gb) {
                if (round) mbar_wait(bar_slot + 8 * slot, (round - 1) & 1u);      // the store warps have written the slab that sat in this slot
                mbar_wait(bar_pix, gb & 1u);
                M.r0 = R * b + SEG * seg;
                M.r1 = M.r0 + SEG;
                const uint32_t a_pix = S.pix[0] - (uint32_t)(max(R * b - 1, 0) * L::ROWB);               // virtual address of image row 0
                const uint32_t a_mag = S.mag[0] + (uint32_t)((b & 1) * R * L::MS2) - (uint32_t)((R * b + 1) * L::MS2);      // ... of magnitude row -1
                const uint32_t a_mask = S.mask + (uint32_t)(slot * L::SLOTB) - (uint32_t)(R * b * L::PRB);           // ... of mask row 0
                p1_strip_walk<NR, true, F0, F1, false, SEG, LUT>(P, Dm, a_pix, a_mag, a_mask, S, M, SEG);
                __syncwarp();
                if (lane == 0) {
                    mbar_arrive(my_bar + 8 * (gb & 1u));
                    if (atom_inc_acq_rel(a_cnt) == (uint32_t)NCW * (gb + 1) - 1) {      // the last warp out: the band's pixels are dead
                        if (b + 1 < NB) issue_band(f, b + 1);
                        else if (const uint32_t fn = ring_frame(a_ring, j + 1); fn < n) issue_band(plist_frame<LIST>(list, fn), 0);
                    }
                }
                // the neighbours' magnitudes of this band (barrier gb & 1 of a warp is in its phase gb >> 1)
                if (warp > 0) mbar_wait(my_bar - 16 + 8 * (gb & 1u), (gb >> 1) & 1u);
                if (warp + 1 < NCW) mbar_wait(my_bar + 16 + 8 * (gb & 1u), (gb >> 1) & 1u);
                if (b == 0 && j > 0) mbar_wait(bar_p3, (uint32_t)(j - 1) & 1u);         // the candidate plane of the frame before is dead
                // first decided row of this lane; its two window rows: this band's magnitudes, the slot of the band before, or zeros
                const int n0 = R * b - 1 + SEG * seg;
                const uint32_t mrow = a_mag + 2 * (4 + 4 * M.strip) + (uint32_t)(n0 * L::MS2);           // magnitude row n0 - 1
                const uint32_t a_up = seg ? mrow : (b ? my_slot + 8 : a_zero + 8);
                const uint32_t a_ce = seg ? mrow + L::MS2 : (b ? my_slot + 24 + 8 : a_zero + 8);
                p2_nms_lagged<SEG>(P, Dm, a_mag, S.cand, a_edge, S, M.strip, M.store_lane, n0, a_up, a_ce, seg == 3 ? my_slot : 0u, b == NB - 1, seg == 3);
                __syncwarp();                                     // the slot is read by other lanes of this warp in the next band
                if (++slot == NSLOT) { slot = 0; ++round; }
            }
            bar_sync(1, NC);                                      // the hysteresis bands cut across the column blocks
            if (p.stats) count_strong_band(S, a_edge, H, ww, lane, warp, NCW);
            p3_relax_band(S.cand, a_edge, H, ww, lane, warp, NCW);
            bar_arrive(2, NT);                                    // planes of frame j are final: the store warps take them from here
        }
    } else {
        // ------------------------------------------------ store warps -------------------------------------------------
        const int st = tid - NC;
        Dims Ds = Dm;
        Ds.h = R;
        int slot = 0;
        // slot j was written by thread NC two frames ago, before a barrier of both store warps
#pragma unroll 1
        for (int j = 0;; ++j) {
            const uint32_t fj = ring_frame(a_ring, j);
            if (fj >= n) break;
            const uint32_t f = plist_frame<LIST>(list, fj);
            if (st == 0) ticket = draw_frames(p);                 // frame j + 2: published after this frame's hysteresis
            const uint32_t a_edge = (j & 1) ? S.edge2 : S.edge;
            bar_sync(2, NT);
            int sw = 0;                                           // growth across the compute warps' row bands (usually one checking pass)
            if (bar_or(4, NS, p3_check_band_boundaries(S.cand, a_edge, H, ww, (H + NCW - 1) / NCW, st, NS)))
                sw = p3_hysteresis(S.cand, a_edge, H, ww, st, NS, [](int c) { return bar_or(4, 32 * NSW, c); });
            if (p.stats) {
                if (st == 0) stat_add_one(S, 8, (unsigned long long)sw + 1);
                count_planes<0, true>(p, S, S.cand, a_edge, 0u, 0, H * ww, st, NS);
                bar_sync(4, NS);
            }
            if (st == 0) {                                        // (the barriers above order both store warps' reads of the candidate plane)
                sts32(a_ring + 4 * (uint32_t)((j + 2) % FRAME_RING), ticket);      // (slot of frame j - 2: every reader is past it)
                mbar_arrive(bar_p3);
            }
            uint8_t* gu8 = p.out_u8 ? p.out_u8 + (size_t)f * frame_bytes : nullptr;
            float* gf32 = p.out_f32 ? p.out_f32 + (size_t)f * frame_bytes : nullptr;
#pragma unroll 1
            for (int b = 0; b < NB; ++b) {
                // the slab's sources: rows R b .. of the frame's edge plane, the band's slot of the mask ring
                uint32_t ps[3];
                plane_sources(p, a_edge + (uint32_t)(b * R * L::PRB), S.mask + (uint32_t)(slot * L::SLOTB), L::MASKP, ps);
                const size_t so = (size_t)b * R * L::ROWB;
                p4_output(P, Ds, ps, 0u, gu8 ? gu8 + so : nullptr, gf32 ? gf32 + so : nullptr, st, NS);
                if (p.stats) {
                    uint32_t n_mask[NR > 0 ? NR : 1] = {0};
                    for (int i = st; i < L::SLOTB / 4; i += NS)
#pragma unroll
                        for (int k = 0; k < NR; ++k) n_mask[k] += __popc(lds32(S.mask + (uint32_t)(slot * L::SLOTB + k * L::MASKP + 4 * i)));
#pragma unroll
                    for (int k = 0; k < NR; ++k) stat_add(S, 1 + p.range_stat[k], n_mask[k]);
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_slot + 8 * slot);
                if (++slot == NSLOT) slot = 0;
            }
        }
        if (p.stats) {
            bar_sync(4, NS);
            stats_flush(p, S, st);
        }
    }
}

}  // namespace trs
