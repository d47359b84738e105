// s1 step A: pileup count tensor [L][18] + per-position flags, straight from flat packed reads.
//
// Replaces `samtools mpileup` (make_predict_data.sh:117,151) + TensorMaker::make_tensor
// (tensor_maker.cpp:61-249) + the candidate gate of create_pileup_tensor (main.cpp:196) using the event
// formulation of SURVEY.md appendix A.8.  No text, no per-base atomics:
//
//   read_scan_kernel   one warp per read: reference end, (ref,query) checkpoints every 32 CIGAR ops,
//                      first/last read index per position tile.
//   pileup_tile_kernel persistent CTAs, one position tile (kTile bp) at a time in shared memory:
//       - one warp per overlapping read, ONE LANE PER CIGAR OP (warp scan gives each op its ref/query start)
//       - an aligned run (M/=/X) costs two run-boundary increments (depth by prefix sum later) plus a
//         bit-parallel 2-bit XOR against the reference tile, 16 bases per word: only MISMATCHES touch a
//         counter (matches are implied: the reference channel is -(A+C+G+T), tensor_maker.cpp:230-246)
//       - a deletion costs two boundary increments ('*'/'#' depth) plus one indel event
//       - indel events are chained per position (exact grouping for I1/D1 by length / sequence identity)
//       - epilogue: prefix sums -> 18 channels + AF gate (IEEE double, tensor_maker.cpp:195-228)
//         -> rows staged in shared memory -> coalesced 16-byte stores of the int32 [kTile][18] block.
#include <type_traits>
#include "common.cuh"

namespace nsnp {
namespace {

constexpr int kCkShift = 5;                 // checkpoint every 32 ops
constexpr int kReadList = 1024;             // overlapping reads handled per round
constexpr int kTileShift = 10, kTile = 1 << kTileShift;     // position tile of pileup_tile_kernel (bp)

struct Event {                               // 16 bytes, lives in the per-CTA global slab (L2 resident)
    uint32_t next;                           // previous event anchored at the same position (chain)
    uint32_t info;                           // len | class << 8     class: 0 I, 1 i, 2 D, 3 d
    uint64_t seq;                            // absolute base index of the inserted sequence
};

struct Workspace {
    int32_t* rend;        // [n_reads]
    int32_t* ck_ref;      // [n_slots]
    int32_t* ck_q;        // [n_slots]
    int32_t* tile_lo;     // [n_tiles]
    int32_t* tile_hi;     // [n_tiles]
    int32_t* counters;    // [16]  0: tile ticket, 1: depth-cap fast check (max buffered reads), 2: reads dropped by the cap
    int32_t* cap_end;     // [n_reads] exclusive end of every passing read (INT32_MIN: filtered)
    int32_t* cap_heap;    // [n_reads] min-heap of the slow path
    Event*   slabs;       // [n_ctas][slab_cap]
    int64_t  slab_cap;
    // target intervals (nsnp_pileup_counts_targets); tile_list == nullptr: every tile of the region, in ticket order
    int32_t* targets;     // [2 * n_targets] copied from the host
    int32_t* tile_diff;   // [n_tiles + 1] boundary deltas of the listed tile ranges
    int32_t* tile_list;   // [n_tiles] ascending tile indices, count in counters[6]
};

// CIGAR words: BAM's u32 (len << 4 | op), or the same values as u16 when every length is below 4096 (nsnp_reads.cigar_bits = 16:
// halves the bytes a host decoder ships per op)
__device__ __forceinline__ uint32_t ld_cigar(const nsnp_reads_t& rd, int64_t i) {
    return rd.cigar_bits == 16 ? (uint32_t)__ldg(reinterpret_cast<const uint16_t*>(rd.cigar) + i) : __ldg(rd.cigar + i);
}

__device__ __forceinline__ bool op_ref(int op) { return op == 0 || op == 2 || op == 3 || op == 7 || op == 8; }
__device__ __forceinline__ bool op_query(int op) { return op == 0 || op == 1 || op == 4 || op == 7 || op == 8; }

__device__ __forceinline__ int warp_incl_scan(int v) {
    const int l = lane_id();
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const int t = __shfl_up_sync(0xffffffffu, v, d); if (l >= d) v += t; }
    return v;
}

// 16 two-bit bases starting at base index i of a packed array of 32-bit words
__device__ __forceinline__ uint32_t bases16(const uint32_t* __restrict__ w, int64_t i) {
    const int64_t k = i >> 4;
    return __funnelshift_r(w[k], w[k + 1], (int)(i & 15) * 2);
}
__device__ __forceinline__ uint32_t bases16_g(const uint32_t* __restrict__ w, int64_t i) {
    const int64_t k = i >> 4;
    return __funnelshift_r(__ldg(w + k), __ldg(w + k + 1), (int)(i & 15) * 2);
}
// 16 one-bit flags starting at bit index i
__device__ __forceinline__ uint32_t bits16_g(const uint32_t* __restrict__ w, int64_t i) {
    const int64_t k = i >> 5;
    return __funnelshift_r(__ldg(w + k), __ldg(w + k + 1), (int)(i & 31)) & 0xFFFFu;
}
__device__ __forceinline__ uint32_t spread16(uint32_t x) {     // bit j -> bit 2j
    x = (x | (x << 8)) & 0x00FF00FFu; x = (x | (x << 4)) & 0x0F0F0F0Fu;
    x = (x | (x << 2)) & 0x33333333u; x = (x | (x << 1)) & 0x55555555u;
    return x;
}

// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) read_scan_kernel(nsnp_reads_t rd, nsnp_params_t prm, int64_t region_start,
                                                        int64_t region_end, Workspace ws, int32_t* status)
{
    const int lane = lane_id();
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp0; r < rd.n_reads; r += nwarps) {
        const int32_t pos = rd.pos[r];
        const uint32_t flag = rd.flag[r];
        const bool pass = !(flag & 4u) && !(flag & prm.excl_flags) && (int)rd.mapq[r] >= prm.min_mapq;   // appendix B.1
        if (!pass) { if (lane == 0) { ws.rend[r] = INT32_MIN; ws.cap_end[r] = INT32_MIN; } continue; }          // never overlaps any tile
        const int64_t c0 = rd.cigar_off[r], c1 = rd.cigar_off[r + 1];
        const int64_t slot0 = (c0 >> kCkShift) + r;
        int32_t R = pos, Q = 0;
        uint32_t bad = 0u, carry_i = 0u, carry_d = 0u;                            // carry: the previous chunk's last op was I / D
        // kUnroll chunks of 32 ops per iteration: the loads are independent, so a long read (thousands of ops: the
        // critical path of this kernel) keeps kUnroll loads in flight instead of one
        constexpr int kUnroll = 8;
        for (int64_t k = c0; k < c1; k += 32 * kUnroll) {
            uint32_t cg[kUnroll];
#pragma unroll
            for (int j = 0; j < kUnroll; ++j) cg[j] = (k + 32 * j + lane < c1) ? ld_cigar(rd, k + 32 * j + lane) : 6u;   // 6 = pad
            const int64_t s = slot0 + ((k - c0) >> kCkShift);
#pragma unroll
            for (int j = 0; j < kUnroll; ++j) {
                const int op = cg[j] & 15, len = cg[j] >> 4;
                const int rl = op_ref(op) ? len : 0, ql = op_query(op) ? len : 0;
                // canonical CIGARs only: adjacent I I / D D must arrive merged (htslib reports them as ONE indel) and
                // pads inside insertions are not modelled -- refuse loudly instead of counting something else.
                // Three votes and a few warp-uniform bit operations per 32 ops (pad lanes carry op 6 but lie beyond c1).
                {
                    const int64_t nv = c1 - (k + 32 * j);
                    const uint32_t vm = nv >= 32 ? 0xffffffffu : nv > 0 ? (1u << nv) - 1u : 0u;
                    const uint32_t mi = __ballot_sync(0xffffffffu, op == 1), md = __ballot_sync(0xffffffffu, op == 2);
                    const uint32_t mp = __ballot_sync(0xffffffffu, op == 6) & vm;
                    bad |= mp | (mi & ((mi << 1) | carry_i)) | (md & ((md << 1) | carry_d));
                    carry_i = mi >> 31; carry_d = md >> 31;
                }
                if (lane == j && k + 32 * j < c1) { ws.ck_ref[s + j] = R; ws.ck_q[s + j] = Q; }
                R += __reduce_add_sync(0xffffffffu, rl);
                Q += __reduce_add_sync(0xffffffffu, ql);
            }
        }
        if (lane == 0) {
            ws.rend[r] = R;
            ws.cap_end[r] = max(R, pos + 1);                                      // bam_endpos: at least pos + 1
            atomicMax(&ws.counters[4], max(R, pos + 1) - pos);                    // longest reference span of the call
        }
        if (bad && lane == 0) dev_fail(status, DEV_E_CIGAR, (int)r);
        // tiles this read overlaps
        const int64_t a = pos > region_start ? pos : region_start;
        const int64_t b = R < region_end ? R : region_end;
        if (a < b) {
            const int t0 = (int)((a - region_start) >> kTileShift), t1 = (int)((b - 1 - region_start) >> kTileShift);
            for (int t = t0 + lane; t <= t1; t += 32) { atomicMin(&ws.tile_lo[t], (int)r); atomicMax(&ws.tile_hi[t], (int)r + 1); }
        }
    }
}


// ------------------------------------------------------------------------------------------------
// htslib streaming depth cap (`samtools mpileup --max-depth 144`, make_predict_data.sh:117; SURVEY appendix B.3).
// The pileup engine refuses a read at push time iff it is already assembling the read's own start column (an earlier
// passing read starts there too) and its node pool holds more than max_depth nodes: every pushed read whose exclusive
// end is >= that column, plus two bookkeeping nodes.  The rule is sequential in file order, so it runs in three steps:
//   read_scan_kernel   exclusive end of every passing read, longest reference span
//   cap_kernel         upper bound of the pool size seen by any read if nothing were dropped (sampled, then exact): when
//                      it never exceeds the cap (every 10-60x data set) nothing is dropped; otherwise one thread replays
//                      the push order with a min-heap of ends and marks dropped reads as filtered.
// Exact for the read set of one call; across region shards it is exact as long as no read of the lead-in window before
// the region is itself affected by the cap (SURVEY 8e caveat).
// counters: [1] sampled bound, [3] exact bound, [4] longest reference span (read_scan), [2] reads dropped.
// alive(b) = earlier passing reads with end >= pos[b]; alive(b) <= alive(b - 1) + 1, so counting every kCapStride-th read
// bounds all of them: the full per-read count only runs when that bound is not conclusive.
constexpr int kCapStride = 16;
// one warp per read: the lanes share the backward scan
__device__ __forceinline__ int cap_alive(const nsnp_reads_t& rd, const Workspace& ws, int64_t b, int limit) {
    const int lane = lane_id();
    const int32_t P = rd.pos[b];
    const int32_t far = P - ws.counters[4];                     // no read starting before this can reach P
    int cnt = 0;
    for (int64_t r0 = b - 1; r0 >= 0 && cnt < limit; r0 -= 32) {
        const int64_t r = r0 - lane;
        const bool in = r >= 0 && rd.pos[r] >= far;
        cnt += __popc(__ballot_sync(0xffffffffu, in && ws.cap_end[r] >= P));
        if (!__all_sync(0xffffffffu, in)) break;
    }
    return cnt;
}
// One launch: every warp counts one sampled read; the last block to finish looks at the bound and -- only when it is not
// conclusive -- counts every read exactly and, if the pool can really fill, replays the push order on one thread.
__global__ void __launch_bounds__(256) cap_kernel(nsnp_reads_t rd, Workspace ws, int max_depth)
{
    __shared__ int last;
    const int lane = lane_id();
    {
        const int64_t b = (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) * kCapStride;
        if (b < rd.n_reads) {
            const int cnt = cap_alive(rd, ws, b, max_depth);                  // the sampled bound holds for any read index
            if (cnt > 0 && lane == 0) atomicMax(&ws.counters[1], cnt);
        }
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(&ws.counters[5], 1) == (int)gridDim.x - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    if (*(volatile int32_t*)&ws.counters[1] + kCapStride + 2 <= max_depth) return;     // the pool never fills: nothing is dropped
    for (int64_t b = threadIdx.x >> 5; b < rd.n_reads; b += blockDim.x >> 5) {          // exact bound (rare: > ~125x deep data)
        if (ws.cap_end[b] == INT32_MIN) continue;
        const int cnt = cap_alive(rd, ws, b, max_depth);
        if (cnt > 0 && lane == 0) atomicMax(&ws.counters[3], cnt);
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x != 0 || *(volatile int32_t*)&ws.counters[3] + 2 <= max_depth) return;
    int32_t* h = ws.cap_heap;
    int hn = 0, dropped = 0;
    int64_t last_pos = -1;
    for (int64_t i = 0; i < rd.n_reads; ++i) {
        const int32_t e = ws.cap_end[i];
        if (e == INT32_MIN) continue;
        const int32_t P = rd.pos[i];
        while (hn && h[0] < P) {                                // columns < P are done: their reads left the pool
            const int32_t v = h[--hn];
            int k = 0;
            for (;;) { int c = 2 * k + 1; if (c >= hn) break; if (c + 1 < hn && h[c + 1] < h[c]) ++c; if (h[c] >= v) break; h[k] = h[c]; k = c; }
            if (hn) h[k] = v;
        }
        if (last_pos == P && hn + 2 > max_depth) { ws.rend[i] = INT32_MIN; ++dropped; continue; }
        int k = hn++;
        while (k > 0 && h[(k - 1) >> 1] > e) { h[k] = h[(k - 1) >> 1]; k = (k - 1) >> 1; }
        h[k] = e;
        last_pos = P;
    }
    ws.counters[2] = dropped;
}

// ------------------------------------------------------------------------------------------------
constexpr int kGateTab = 256;            // AF-gate thresholds are tabulated for depths below this

constexpr uint32_t kBias = 0x40004000u; // packed signed boundary deltas: each u16 half carries +0x4000
constexpr int kMaxOverlap = 16383;       // reads overlapping one tile (keeps the biased halves inside [1, 0x7FFF])
constexpr uint32_t kNoEvent = 0xFFFFFFFFu;

struct TileSmem {
    // --- cleared to zero per tile (contiguous) ---
    uint32_t base[4][kTile];          // mismatch counters, u16 pairs: [strand*2 + (b>>1)][p], half = b&1
    uint32_t nn[kTile];               // read-N bases: fwd | rev << 16
    uint32_t cnt4[kTile];             // indel events per class (I i D d), one byte each (exact while <= 255 reads overlap)
    uint32_t dfast[kTile];            // deletions of length 1 / 2 per strand, one byte each: D1 D2 d1 d2
    uint32_t ifast[2][kTile];         // 1-base insertions per strand, one byte per inserted base: A C G T
    // --- cleared to kBias ---
    uint32_t ms[kTile];               // read-span boundary deltas (fwd | rev << 16, biased); after the scan: aligned depth
    uint32_t ds[kTile];               // deletion-span boundary deltas;                      after the scan: '*' / '#' depth
    // --- cleared to kNoEvent ---
    uint32_t head[kTile];             // chain heads of the indel events that have no fast counter
    uint32_t ref2[kTile / 16 + 2];    // 2-bit reference tile
    uint32_t refx[kTile / 16 + 2];    // 01 at non-ACGT reference positions (forces a "mismatch" event)
    uint32_t skipcov[kTile / 32];     // positions inside a reference skip (N op)
    int32_t  thr_snp[kGateTab], thr_indel[kGateTab];   // smallest count c with (double)c / den >= min_af
    int32_t  rlist[kTile];                              // >= kReadList; reused as per-warp walk lists (kTile / warps each)
    int32_t  warp_tot[kTile / 128][4];
    int32_t  n_rlist, next_task, n_events, tile, ref_has_x, sub_end;
};

struct ReadMeta { int32_t rpos; int32_t rend; int32_t strand; int64_t c0, c1, sbase; };
__device__ __forceinline__ ReadMeta load_meta(const nsnp_reads_t& rd, const Workspace& ws, int r) {
    ReadMeta m;
    m.rpos = __ldg(rd.pos + r); m.rend = ws.rend[r]; m.c0 = __ldg(rd.cigar_off + r); m.c1 = __ldg(rd.cigar_off + r + 1);
    m.sbase = __ldg(rd.seq_off + r); m.strand = (__ldg(rd.flag + r) >> 4) & 1;
    return m;
}

// ------------------------------------------------------------------------------------------------
// The per-read walk: TWO consecutive CIGAR ops per lane (64 ops per warp iteration, one packed scan for both), 32-bit
// read-relative sequence coordinates, and per-lane comparison loops with rolling word registers instead of a flattened
// word list (its scan + binary search + four broadcasts cost more than the lanes it saved: ONT aligned runs average 14
// bases, i.e. one or two 16-base words).  Runs longer than kSelfWords words -- HiFi-like reads -- finish
// warp-cooperatively, one word per lane.  In strictly alternating CIGARs (M indel M indel ...) each of the two slots is
// type-uniform across the warp, so the aligned-run code and the indel code run without divergence.
// All coordinates are 32-bit: contig positions are int32 (BAM), query offsets are < 2^31; only the absolute base index
// of the packed sequence array needs 64 bits (added last).
// kEvOnly: the re-walk of a tile whose indel events overflowed the slab (see pileup_tile_kernel): only the chained events
// anchored in [elo, ehi) are recorded, no counter is touched.  The first walk passes elo = ts, ehi = te.
constexpr uint32_t kRefOps = 0x18Du;        // M D N = X consume the reference   (bits 0 2 3 7 8)
constexpr uint32_t kQryOps = 0x193u;        // M I S = X consume the query       (bits 0 1 4 7 8)
constexpr uint32_t kAlnOps = 0x181u;        // M = X are aligned runs
constexpr int kSelfWords = 8;

__device__ __forceinline__ void count_mismatches(TileSmem& sm, uint32_t* __restrict__ bs, const uint32_t* __restrict__ nmr,
                                                 uint32_t sw, uint32_t rw, uint32_t xw, int pw, int qb, int m, bool ref_has_x, uint32_t sinc)
{
    uint32_t x = sw ^ rw;
    uint32_t mm = (x | (x >> 1)) & 0x55555555u;
    if (ref_has_x) mm |= xw;
    if (m < 16) mm &= (1u << (2 * m)) - 1u;
    if (nmr) {
        uint32_t nb = bits16_g(nmr, qb);
        if (m < 16) nb &= (1u << m) - 1u;
        if (nb) {
            mm &= ~spread16(nb);
            while (nb) { const int q = __ffs(nb) - 1; nb &= nb - 1; atomicAdd(&sm.nn[pw + q], sinc); }
        }
    }
    while (mm) {
        const int j2 = __ffs(mm) - 1; mm &= mm - 1;
        const uint32_t bcode = (sw >> j2) & 3u;
        atomicAdd(bs + (bcode >> 1) * kTile + pw + (j2 >> 1), 1u << (16 * (bcode & 1u)));
    }
}

template <bool kEvOnly>
__device__ __forceinline__ void process_read2(TileSmem& sm, const nsnp_reads_t& rd, const Workspace& ws, Event* slab,
                                              int r, const ReadMeta& meta, int ts, int te, int elo, int ehi, bool deep, int32_t* status)
{
    const int lane = lane_id();
    const int rpos = meta.rpos;
    const int strand = meta.strand;
    const uint32_t sinc = 1u << (16 * strand);
    const int n_ops = (int)(meta.c1 - meta.c0);
    const int nchunks = (n_ops + 31) >> kCkShift;
    const bool ref_has_x = sm.ref_has_x != 0;                       // tile-uniform
    const int32_t* ckr = ws.ck_ref + ((meta.c0 >> kCkShift) + r);
    const int32_t* ckq = ws.ck_q + ((meta.c0 >> kCkShift) + r);
    if (!kEvOnly && lane == 0) atomicAdd(&sm.ms[max(rpos - ts, 0)], sinc);
    if (!kEvOnly && lane == 1 && meta.rend < te) atomicSub(&sm.ms[meta.rend - ts], sinc);
    int lo = 0, hi = nchunks;
    if (rpos < elo) {
        while (hi - lo > 1) {
            const int step = (hi - lo + 31) >> 5;
            const int c = lo + lane * step;
            const bool le = c < hi && __ldg(ckr + c) <= elo;
            const int cnt = __popc(__ballot_sync(0xffffffffu, le));
            lo = lo + (cnt - 1) * step;
            hi = min(hi, lo + step);
        }
    }
    const int chunk = lo;
    int R = __ldg(ckr + chunk), Q = __ldg(ckq + chunk);
    // read-relative sequence addressing: word pointer of the read's first base + a small offset, everything else 32-bit
    const int sb_lo = (int)(meta.sbase & 15);
    const uint32_t* seqr = reinterpret_cast<const uint32_t*>(rd.seq2) + (meta.sbase >> 4);
    const int nb_lo = (int)(meta.sbase & 31);
    const uint32_t* nmr = rd.nmask ? reinterpret_cast<const uint32_t*>(rd.nmask) + (meta.sbase >> 5) : nullptr;
    uint32_t* bs = &sm.base[strand * 2][0];

    int64_t cgp = meta.c0 + ((int64_t)chunk << kCkShift);
    int left = n_ops - (chunk << kCkShift);
    uint32_t nx0 = 2 * lane < left ? ld_cigar(rd, cgp + 2 * lane) : 6u;
    uint32_t nx1 = 2 * lane + 1 < left ? ld_cigar(rd, cgp + 2 * lane + 1) : 6u;
    for (; left > 0 && R <= ehi; left -= 64, cgp += 64) {
        const uint32_t cgv[2] = {nx0, nx1};
        nx0 = (64 + 2 * lane < left) ? ld_cigar(rd, cgp + 64 + 2 * lane) : 6u;
        nx1 = (65 + 2 * lane < left) ? ld_cigar(rd, cgp + 65 + 2 * lane) : 6u;
        const int op0 = cgv[0] & 15, len0 = cgv[0] >> 4, op1 = cgv[1] & 15, len1 = cgv[1] >> 4;
        const int rl0 = ((kRefOps >> op0) & 1u) ? len0 : 0, ql0 = ((kQryOps >> op0) & 1u) ? len0 : 0;
        const int rl1 = ((kRefOps >> op1) & 1u) ? len1 : 0, ql1 = ((kQryOps >> op1) & 1u) ? len1 : 0;
        const int rl = rl0 + rl1, ql = ql0 + ql1;
        int ri, qi;
        if (!__any_sync(0xffffffffu, (len0 | len1) >= 1024)) {          // 64 lengths below 1024: both prefix sums fit 16 bits
            const int pk = warp_incl_scan(rl | (ql << 16));
            ri = pk & 0xFFFF; qi = (int)((uint32_t)pk >> 16);
        } else {
            ri = warp_incl_scan(rl); qi = warp_incl_scan(ql);
        }
        const int rsv[2] = {R + ri - rl, R + ri - rl + rl0};
        const int qsv[2] = {Q + qi - ql, Q + qi - ql + ql0};
        R += __shfl_sync(0xffffffffu, ri, 31);
        Q += __shfl_sync(0xffffffffu, qi, 31);

#pragma unroll
        for (int s = 0; s < 2; ++s) {
            const int op = cgv[s] & 15, len = cgv[s] >> 4, rs = rsv[s], qs = qsv[s];
            const int a = max(rs, ts), b = min(rs + len, te);                 // clipped reference span
            // ---- aligned run: bit-parallel mismatch detection, this lane's own run, 16 bases per step ----
            const int n = (!kEvOnly && ((kAlnOps >> op) & 1u) && a < b) ? (b - a) : 0;
            const int pa = a - ts;
            const int qa = qs + (a - rs) + sb_lo;                            // offset (bases) from the read's first seq word
            if (n > 0) {
                const uint32_t* sp = seqr + (qa >> 4);
                const uint32_t* rp = sm.ref2 + (pa >> 4);
                const uint32_t* xp = sm.refx + (pa >> 4);
                const int ssh = (qa & 15) * 2, rsh = (pa & 15) * 2;
                uint32_t s_lo = __ldg(sp), r_lo = rp[0], x_lo = ref_has_x ? xp[0] : 0u;
                const int ne = min(n, 16 * kSelfWords);
                for (int o = 0; o < ne; o += 16) {
                    ++sp; ++rp; ++xp;
                    const uint32_t s_hi = __ldg(sp), r_hi = rp[0], x_hi = ref_has_x ? xp[0] : 0u;
                    count_mismatches(sm, bs, nmr, __funnelshift_r(s_lo, s_hi, ssh), __funnelshift_r(r_lo, r_hi, rsh),
                                        __funnelshift_r(x_lo, x_hi, rsh), pa + o, qa + o - sb_lo + nb_lo, n - o, ref_has_x, sinc);
                    s_lo = s_hi; r_lo = r_hi; x_lo = x_hi;
                }
            }
            // long runs: the remaining words one per lane
            for (uint32_t lm = __ballot_sync(0xffffffffu, n > 16 * kSelfWords); lm; lm &= lm - 1) {
                const int j = __ffs(lm) - 1;
                const int pa_j = __shfl_sync(0xffffffffu, pa, j), n_j = __shfl_sync(0xffffffffu, n, j), qa_j = __shfl_sync(0xffffffffu, qa, j);
                for (int o = 16 * (kSelfWords + lane); o < n_j; o += 16 * 32) {
                    const int pw = pa_j + o, qw = qa_j + o;
                    count_mismatches(sm, bs, nmr, bases16_g(seqr, qw), bases16(sm.ref2, pw), ref_has_x ? bases16(sm.refx, pw) : 0u,
                                        pw, qw - sb_lo + nb_lo, n_j - o, ref_has_x, sinc);
                }
            }
            // ---- indel event anchored at the preceding reference position (appendix A.8 iii/iv) ----
            const bool isins = op == 1, isdel = op == 2;
            if (isins || isdel) {
                const int anchor = rs - 1;
                const bool ev = len <= NSNP_MAX_INDEL && rs > rpos && anchor >= elo && anchor < ehi;
                const bool fastdel = ev && isdel && len <= 2 && !deep;
                if (!kEvOnly && isdel && a < b && !fastdel) {
                    atomicAdd(&sm.ds[a - ts], sinc);
                    if (b < te) atomicSub(&sm.ds[b - ts], sinc);
                }
                if (ev) {
                    const int cls = (isdel ? 2 : 0) + strand;
                    const int ap = anchor - ts;
                    // deep tiles count chained events per position in the whole word (the classes come from the chain walk)
                    if (!kEvOnly) atomicAdd(&sm.cnt4[ap], deep ? 1u : 1u << (8 * cls));
                    bool chain = true;
                    if (fastdel) {
                        if (!kEvOnly) atomicAdd(&sm.dfast[ap], 1u << (8 * (2 * strand + len - 1)));
                        chain = false;
                    } else if (isins && len == 1 && !deep) {                  // 1-base insertion: fast counter unless the base is N
                        const int qi1 = qs + sb_lo;
                        const uint32_t iword = __ldg(seqr + (qi1 >> 4));
                        const int qn = qs + nb_lo;
                        const uint32_t inbit = nmr ? (__ldg(nmr + (qn >> 5)) >> (qn & 31)) & 1u : 0u;
                        if (!inbit) {
                            if (!kEvOnly) atomicAdd(&sm.ifast[strand][ap], 1u << (8 * ((iword >> (2 * (qi1 & 15))) & 3u)));
                            chain = false;
                        }
                    }
                    if (chain) {
                        const int e = atomicAdd(&sm.n_events, 1);
                        if (e < ws.slab_cap) {
                            Event evr;
                            evr.next = atomicExch(&sm.head[ap], (uint32_t)e);
                            evr.info = (uint32_t)len | ((uint32_t)cls << 8);
                            evr.seq = (uint64_t)(meta.sbase + qs);
                            slab[e] = evr;
                        } else if (kEvOnly) {
                            dev_fail(status, DEV_E_INDEL_SLAB, sm.tile);
                        }
                    }
                }
            } else if (!kEvOnly && op == 3 && a < b) {                                    // reference skip: covered, nothing counted
                atomicSub(&sm.ms[a - ts], sinc);
                if (b < te) atomicAdd(&sm.ms[b - ts], sinc);
                for (int p = a; p < b; ++p) atomicOr(&sm.skipcov[(p - ts) >> 5], 1u << ((p - ts) & 31));
            }
        }
    }
}

__device__ __forceinline__ bool same_insert(const uint32_t* seqw, const uint32_t* nmw, uint64_t g1, uint64_t g2, int len) {
    for (int o = 0; o < len; o += 16) {
        const int m = min(16, len - o);
        uint32_t x = bases16_g(seqw, (int64_t)g1 + o) ^ bases16_g(seqw, (int64_t)g2 + o);
        if (nmw) {
            uint32_t n1 = bits16_g(nmw, (int64_t)g1 + o), n2 = bits16_g(nmw, (int64_t)g2 + o);
            if (m < 16) { n1 &= (1u << m) - 1u; n2 &= (1u << m) - 1u; }
            if (n1 != n2) return false;
            x &= ~(spread16(n1) * 3u);
        }
        if (m < 16) x &= (1u << (2 * m)) - 1u;
        if (x) return false;
    }
    return true;
}

__device__ __forceinline__ int min_count_for_af(double af, int den) {
    if (!(af == af)) return INT32_MAX;                      // NaN threshold: the comparison is never true
    if (af <= 0.0) return 0;
    const double x = af * den;
    if (x > 2.0e9) return INT32_MAX;
    int c = (int)ceil(x);
    while (c > 0 && (double)(c - 1) / den >= af) --c;
    while ((double)c / den < af) ++c;
    return c;
}

__global__ void __launch_bounds__(kTile / 4, 4096 / kTile) pileup_tile_kernel(nsnp_reads_t rd, nsnp_params_t prm, const uint8_t* __restrict__ ref,
                                                               int64_t region_start, int64_t region_len, int n_tiles,
                                                               Workspace ws, int32_t* __restrict__ counts,
                                                               uint8_t* __restrict__ flags, int32_t* status)
{
    constexpr int kThreads = kTile / 4, kWarps = kThreads / 32;   // one thread packs 4 reference bases
    static_assert(kTile >= kReadList, "read list");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    TileSmem& sm = *reinterpret_cast<TileSmem*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    Event* slab = ws.slabs + (int64_t)blockIdx.x * ws.slab_cap;
    const uint32_t* seqw = reinterpret_cast<const uint32_t*>(rd.seq2);
    const uint32_t* nmw = reinterpret_cast<const uint32_t*>(rd.nmask);

    // AF gate as integer thresholds: thr[den] = smallest count c with (double)c / den >= min_af, evaluated with the
    // same IEEE double division as tensor_maker.cpp:213,218 -- the comparison result is identical, the divide is
    // done once per CTA instead of ~6 times per position
    for (int d = tid; d < kGateTab; d += kThreads) {
        const int den = d ? d : 1;                          // tensor_maker.cpp:195
        sm.thr_snp[d] = min_count_for_af(prm.snp_min_af, den);
        sm.thr_indel[d] = min_count_for_af(prm.indel_min_af, den);
    }

    for (;;) {
        __syncthreads();                                    // previous tile fully written, smem reusable
        if (tid == 0) {
            const int k = atomicAdd(&ws.counters[0], 1);
            sm.tile = ws.tile_list == nullptr ? k : k < *(volatile int32_t*)&ws.counters[6] ? ws.tile_list[k] : n_tiles;
        }
        __syncthreads();
        const int tile = sm.tile;
        if (tile >= n_tiles) break;
        const int ts = (int)region_start + tile * kTile;                      // contig coordinates are int32 (checked by the host)
        const int te = (int)min((int64_t)ts + kTile, region_start + region_len);
        const int tn = te - ts;

        // ---- clear counters, stage the reference tile ----
        {
            uint4* z = reinterpret_cast<uint4*>(&sm.base[0][0]);
            for (int i = tid; i < 9 * kTile / 4; i += kThreads) z[i] = make_uint4(0u, 0u, 0u, 0u);    // base, nn, cnt4, dfast, ifast
            uint4* zb = reinterpret_cast<uint4*>(&sm.ms[0]);
            for (int i = tid; i < 2 * kTile / 4; i += kThreads) zb[i] = make_uint4(kBias, kBias, kBias, kBias);   // ms, ds
            uint4* zh = reinterpret_cast<uint4*>(&sm.head[0]);
            for (int i = tid; i < kTile / 4; i += kThreads) zh[i] = make_uint4(kNoEvent, kNoEvent, kNoEvent, kNoEvent);
            for (int i = tid; i < kTile / 32; i += kThreads) sm.skipcov[i] = 0u;
            if (tid == 0) { sm.n_events = 0; }
            // 4 reference bases per thread -> one byte of the 2-bit tile and of the non-ACGT mask
            uint32_t r2 = 0, rx = 0;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int pp = tid * 4 + j;
                const uint8_t ch = pp < tn ? ref[(int64_t)ts + pp] : (uint8_t)'N';
                const int cd = nt4(ch);
                if (cd < 4) r2 |= (uint32_t)cd << (2 * j); else rx |= 1u << (2 * j);
            }
            reinterpret_cast<uint8_t*>(sm.ref2)[tid] = (uint8_t)r2;
            reinterpret_cast<uint8_t*>(sm.refx)[tid] = (uint8_t)rx;
            if (tid < 8) { reinterpret_cast<uint8_t*>(sm.ref2)[kTile / 4 + tid] = 0; reinterpret_cast<uint8_t*>(sm.refx)[kTile / 4 + tid] = 0x55; }
            const int any_x = __syncthreads_or(rx != 0u && tid * 4 < tn);
            if (tid == 0) sm.ref_has_x = any_x;
        }
        __syncthreads();

        // ---- accumulate: reads [lo, hi) that overlap the tile, one warp per read ----
        const int rlo = ws.tile_lo[tile], rhi = ws.tile_hi[tile];
        int n_overlap = 0;                                  // reads that really overlap the tile (block-uniform)
        // byte counters (class totals, fast indel groups) are exact while <= 255 reads overlap the tile.  The overlap
        // count is known before any read is processed only when the candidates fit one round; otherwise assume deep:
        // then every indel event is chained and counted by the walk (16-bit results).
        bool deep = rhi - rlo > kReadList;
        // one walk over the reads that overlap [elo, ehi): the whole tile first; events-only re-walks of anchor sub-ranges
        // (kEv) when the tile's chained indel events overflowed the slab
        auto walk = [&](const int elo, const int ehi, auto ev_tag) {
            constexpr bool kEv = decltype(ev_tag)::value;
            for (int rb = rlo; rb < rhi; rb += kReadList) {
                __syncthreads();
                if (tid == 0) { sm.n_rlist = 0; sm.next_task = 0; }
                __syncthreads();
                for (int r = rb + tid; r < min(rhi, rb + kReadList); r += kThreads) {
                    // overlap test; a read that merely starts at ehi has no anchor inside the window
                    if (rd.pos[r] < ehi && ws.rend[r] > elo) sm.rlist[atomicAdd(&sm.n_rlist, 1)] = r;
                }
                __syncthreads();
                const int nr = sm.n_rlist;
                if (!kEv) { n_overlap += nr; deep = deep || nr > 255; }
                // dynamic read -> warp assignment; the NEXT read's metadata is fetched before the current one is processed
                auto grab = [&]() { int t = 0; if (lane == 0) t = atomicAdd(&sm.next_task, 1); return __shfl_sync(0xffffffffu, t, 0); };
                int t = grab();
                ReadMeta meta = {};
                int r = 0;
                if (t < nr) { r = sm.rlist[t]; meta = load_meta(rd, ws, r); }
                while (t < nr) {
                    const int tn = grab();
                    ReadMeta mnext = {};
                    int rn = 0;
                    if (tn < nr) { rn = sm.rlist[tn]; mnext = load_meta(rd, ws, rn); }
                    process_read2<kEv>(sm, rd, ws, slab, r, meta, ts, te, elo, ehi, deep, status);
                    t = tn; r = rn; meta = mnext;
                }
            }
        };
        walk(ts, te, std::false_type{});
        __syncthreads();
        if (tid == 0 && n_overlap > kMaxOverlap) dev_fail(status, DEV_E_DEPTH, (int)(ts & 0x7fffffff));

        // ---- prefix sums: biased boundary deltas -> depths (fwd | rev << 16 stays valid: depths are <= kMaxOverlap) ----
        {
            constexpr int K = kTile / kThreads;
            constexpr int kB = (int)(kBias & 0xFFFFu);
            int s0 = 0, s1 = 0, s2 = 0, s3 = 0;          // read span fwd, span rev, del fwd, del rev
#pragma unroll
            for (int j = 0; j < K; ++j) {
                const int p = tid * K + j;
                const uint32_t a = sm.ms[p], c = sm.ds[p];
                s0 += (int)(a & 0xFFFF) - kB; s1 += (int)(a >> 16) - kB;
                s2 += (int)(c & 0xFFFF) - kB; s3 += (int)(c >> 16) - kB;
            }
            const int i0 = warp_incl_scan(s0), i1 = warp_incl_scan(s1), i2 = warp_incl_scan(s2), i3 = warp_incl_scan(s3);
            if (lane == 31) { sm.warp_tot[warp][0] = i0; sm.warp_tot[warp][1] = i1; sm.warp_tot[warp][2] = i2; sm.warp_tot[warp][3] = i3; }
            __syncthreads();
            int e0 = i0 - s0, e1 = i1 - s1, e2 = i2 - s2, e3 = i3 - s3;
            for (int w = 0; w < warp; ++w) { e0 += sm.warp_tot[w][0]; e1 += sm.warp_tot[w][1]; e2 += sm.warp_tot[w][2]; e3 += sm.warp_tot[w][3]; }
#pragma unroll
            for (int j = 0; j < K; ++j) {
                const int p = tid * K + j;
                const uint32_t a = sm.ms[p], c = sm.ds[p];
                e0 += (int)(a & 0xFFFF) - kB; e1 += (int)(a >> 16) - kB;
                e2 += (int)(c & 0xFFFF) - kB; e3 += (int)(c >> 16) - kB;
                // deletions covered by the fast counters: 1-base anchored at p-1, 2-base anchored at p-1 or p-2
                const uint32_t f1 = p >= 1 ? sm.dfast[p - 1] : 0u, f2 = p >= 2 ? sm.dfast[p - 2] : 0u;
                const int d2 = e2 + (int)(f1 & 0xFF) + (int)((f1 >> 8) & 0xFF) + (int)((f2 >> 8) & 0xFF);
                const int d3 = e3 + (int)((f1 >> 16) & 0xFF) + (int)(f1 >> 24) + (int)(f2 >> 24);
                sm.ms[p] = (uint32_t)(e0 - d2) | ((uint32_t)(e1 - d3) << 16);        // aligned depth = span - deletions
                sm.ds[p] = (uint32_t)d2 | ((uint32_t)d3 << 16);
            }
        }
        __syncthreads();

        // ---- indel channels.  Totals come from the class byte counters; the multiplicity of the most frequent identical
        //      indel (I1/D1) is the larger of the fast group counters and the largest group among the chained events.
        //      The chain is walked only where a class holds >= 2 chained events (or the tile is deep).  Every warp owns
        //      the positions {warp*32 + lane + 256*k}: it first COMPACTS the positions that need a walk into a list
        //      (ballot ranks), then walks them one per lane, so the walk runs with full lanes and the channel epilogue
        //      below stays straight-line and convergent.  Results per position (u16 pairs):
        //      cnt4 <- tot I | i << 16,  head <- tot D | d << 16,  dfast <- max I | i << 16,  ifast[0] <- max D | d << 16.
        //      Positions [plo, phi) only: all of them, or one anchor sub-range of an overflowed tile. ----
        auto indel_channels = [&](const int plo, const int phi) {
            // per-class (I i D d) sum and maximum of the fast group counters, as bytes of one word each
            auto fast_stats = [](uint32_t dfv, uint32_t if0, uint32_t if1, uint32_t& fsum, uint32_t& fmax) {
                auto sum4 = [](uint32_t x) { const uint32_t t = (x & 0x00FF00FFu) + ((x >> 8) & 0x00FF00FFu); return (t + (t >> 16)) & 0x3FFu; };
                auto max4 = [](uint32_t x) { const uint32_t t = __vmaxu4(x, x >> 16); return max(t & 0xFFu, (t >> 8) & 0xFFu); };
                const uint32_t d0 = dfv & 0xFFu, d1 = (dfv >> 8) & 0xFFu, d2 = (dfv >> 16) & 0xFFu, d3 = dfv >> 24;
                fsum = sum4(if0) | (sum4(if1) << 8) | ((d0 + d1) << 16) | ((d2 + d3) << 24);      // each <= 255 when not deep
                fmax = max4(if0) | (max4(if1) << 8) | (max(d0, d1) << 16) | (max(d2, d3) << 24);
            };
            int32_t* wl = sm.rlist + warp * (kTile / kWarps);      // the read list is dead here: 128 slots per warp
            int nlist = 0;
            for (int sb = warp * 32; sb < kTile; sb += kThreads) {
                const int p = sb + lane;
                const uint32_t c4 = sm.cnt4[p];                    // zero beyond tn
                uint32_t fsum, fmax;
                fast_stats(sm.dfast[p], sm.ifast[0][p], sm.ifast[1][p], fsum, fmax);
                const uint32_t oth = __vsub4(c4, fsum);            // chained events per class
                const bool inr = p >= plo && p < phi;
                const bool need = inr && p < tn && (deep ? sm.head[p] != kNoEvent : ((oth + 0x7E7E7E7Eu) & 0x80808080u) != 0u);   // some byte >= 2
                const uint32_t bal = __ballot_sync(0xffffffffu, need);
                if (need) wl[nlist + __popc(bal & ((1u << lane) - 1u))] = p;
                else if (inr) {
                    const uint32_t mx = __vmaxu4(fmax, oth);       // a class with <= 1 chained event: that event is its own group
                    sm.cnt4[p] = (c4 & 0xFFu) | ((c4 & 0xFF00u) << 8); sm.head[p] = ((c4 >> 16) & 0xFFu) | ((c4 >> 24) << 16);
                    sm.dfast[p] = (mx & 0xFFu) | ((mx & 0xFF00u) << 8); sm.ifast[0][p] = ((mx >> 16) & 0xFFu) | ((mx >> 24) << 16);
                }
                nlist += __popc(bal);
            }
            __syncwarp();
            for (int i = lane; i < nlist; i += 32) {
                const int p = wl[i];
                // pass 1 over the chain: totals per class and how many events equal the FIRST event seen of their
                // class.  All equal -> multiplicity = total; a class of two unequal events -> 1.  Only a class with
                // >= 3 events that are not all identical needs the quadratic pass below (rare).
                int tt[4] = {0, 0, 0, 0}, same[4] = {0, 0, 0, 0};
                uint32_t finfo[4] = {0, 0, 0, 0};
                uint64_t fseq[4] = {0, 0, 0, 0};
                for (uint32_t e = sm.head[p]; e != kNoEvent;) {
                    const uint4 raw = __ldcg(reinterpret_cast<const uint4*>(slab + e));
                    const int cls = (raw.y >> 8) & 3, len = raw.y & 0xFF;
                    const uint64_t g = (uint64_t)raw.z | ((uint64_t)raw.w << 32);
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        if (cls == c) {
                            if (tt[c] == 0) { finfo[c] = raw.y & 0x3FF; fseq[c] = g; }
                            else if ((raw.y & 0x3FF) == finfo[c] && (c >= 2 || same_insert(seqw, nmw, g, fseq[c], len))) ++same[c];
                            ++tt[c];
                        }
                    }
                    e = raw.x;
                }
                int mxs[4]; uint32_t need_full = 0;
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    if (tt[c] <= 1 || same[c] == tt[c] - 1) mxs[c] = tt[c];
                    else if (tt[c] == 2) mxs[c] = 1;
                    else { mxs[c] = 0; need_full |= 1u << c; }
                }
                if (need_full) {
                    for (uint32_t e = sm.head[p]; e != kNoEvent;) {
                        const uint4 raw = __ldcg(reinterpret_cast<const uint4*>(slab + e));
                        const int cls = (raw.y >> 8) & 3, len = raw.y & 0xFF;
                        if ((need_full >> cls) & 1u) {
                            const uint64_t g = (uint64_t)raw.z | ((uint64_t)raw.w << 32);
                            // multiplicity = this event + identical events further down the chain: the group member
                            // nearest the head sees the whole group
                            int mult = 1;
                            for (uint32_t f = raw.x; f != kNoEvent;) {
                                const uint4 o = __ldcg(reinterpret_cast<const uint4*>(slab + f));
                                if ((o.y & 0x3FF) == (raw.y & 0x3FF) &&
                                    (cls >= 2 || same_insert(seqw, nmw, g, (uint64_t)o.z | ((uint64_t)o.w << 32), len))) ++mult;
                                f = o.x;
                            }
#pragma unroll
                            for (int c = 0; c < 4; ++c) if (cls == c) mxs[c] = max(mxs[c], mult);
                        }
                        e = raw.x;
                    }
                }
                if (!deep) {                                        // totals from the byte counters, groups: fast vs chained
                    const uint32_t c4 = sm.cnt4[p];
                    uint32_t fsum, fmax;
                    fast_stats(sm.dfast[p], sm.ifast[0][p], sm.ifast[1][p], fsum, fmax);
#pragma unroll
                    for (int c = 0; c < 4; ++c) { tt[c] = (c4 >> (8 * c)) & 0xFF; mxs[c] = max(mxs[c], (int)((fmax >> (8 * c)) & 0xFF)); }
                }
                sm.cnt4[p] = (uint32_t)tt[0] | ((uint32_t)tt[1] << 16); sm.head[p] = (uint32_t)tt[2] | ((uint32_t)tt[3] << 16);
                sm.dfast[p] = (uint32_t)mxs[0] | ((uint32_t)mxs[1] << 16); sm.ifast[0][p] = (uint32_t)mxs[2] | ((uint32_t)mxs[3] << 16);
            }
            __syncwarp();
        };
        if (sm.n_events <= ws.slab_cap) {
            indel_channels(0, kTile);
        } else {
            // The slab held only the first slab_cap chained events of this tile (the rest were not linked).  Re-walk the
            // reads once per anchor sub-range whose events fit the slab, each time rebuilding the chains of that range
            // and reducing them.  cnt4 bounds the chained events per position: in a deep tile it counts exactly them, else
            // its byte sum counts every event.  One position holds at most two events per read (an insertion and a
            // deletion after it), so with <= kMaxOverlap reads a single position always fits.  Tiles that fit never get here.
            for (int i = tid; i < kTile; i += kThreads) sm.head[i] = kNoEvent;
            for (int alo = 0; alo < tn;) {
                __syncthreads();                            // heads reset / previous sub-range reduced, read list free
                if (tid == 0) {
                    int64_t acc = 0;
                    int p = alo;
                    for (; p < tn; ++p) {
                        const uint32_t c4 = sm.cnt4[p];
                        const int64_t w = deep ? (int64_t)c4 : (int64_t)((c4 & 0xFFu) + ((c4 >> 8) & 0xFFu) + ((c4 >> 16) & 0xFFu) + (c4 >> 24));
                        if (acc + w > ws.slab_cap && p > alo) break;
                        acc += w;
                    }
                    sm.sub_end = p;
                    sm.n_events = 0;
                }
                __syncthreads();
                const int ahi = sm.sub_end;
                walk(ts + alo, ts + ahi, std::true_type{});
                __syncthreads();
                indel_channels(alo, ahi);
                alo = ahi;
            }
        }

        // ---- epilogue: 18 channels + gate per position, rows stored straight from registers.  Warp-private positions:
        //      no block-wide barrier. ----
        for (int sb = warp * 32; sb < tn; sb += kThreads) {
            const int p = sb + lane;
            if (p < tn) {
                const uint32_t t01 = sm.cnt4[p], t23 = sm.head[p], m01 = sm.dfast[p], m23 = sm.ifast[0][p];
                const int tot0 = t01 & 0xFFFF, tot1 = t01 >> 16, tot2 = t23 & 0xFFFF, tot3 = t23 >> 16;
                const int mx0 = m01 & 0xFFFF, mx1 = m01 >> 16, mx2 = m23 & 0xFFFF, mx3 = m23 >> 16;
                const uint32_t md = sm.ms[p], dd = sm.ds[p], nnv = sm.nn[p];
                const int mf = (int)(md & 0xFFFF) - (int)(nnv & 0xFFFF), mr = (int)(md >> 16) - (int)(nnv >> 16);
                const int df = (int)(dd & 0xFFFF), dr = (int)(dd >> 16);
                int cf[4], cr[4];
                { const uint32_t w0 = sm.base[0][p], w1 = sm.base[1][p], w2 = sm.base[2][p], w3 = sm.base[3][p];
                  cf[0] = w0 & 0xFFFF; cf[1] = w0 >> 16; cf[2] = w1 & 0xFFFF; cf[3] = w1 >> 16;
                  cr[0] = w2 & 0xFFFF; cr[1] = w2 >> 16; cr[2] = w3 & 0xFFFF; cr[3] = w3 >> 16; }
                const uint32_t rsh = 2u * (p & 15);
                const int chr = (sm.ref2[p >> 4] >> rsh) & 3;                        // non-ACGT packs as 0: evc_base_from -> 'A'
                const bool ref_acgt = ((sm.refx[p >> 4] >> rsh) & 1u) == 0u;
                // merged-strand tallies (tensor_maker.cpp:124,168-171): the reference base's own count is implied
                const int allb = mf + mr;
                int tb[4];
#pragma unroll
                for (int b = 0; b < 4; ++b) tb[b] = b == chr ? 0 : cf[b] + cr[b];
                const int refcnt = allb - (tb[0] + tb[1] + tb[2] + tb[3]);
                const int tI = tot0 + tot1, tD = tot2 + tot3;
                const int depth = allb + df + dr;
                // pass_af (tensor_maker.cpp:195-228,248): top allele (stable order A<C<D<G<I<T on ties) differs from the
                // reference, or a non-reference allele / indel class reaches its minimum frequency.  Branch-free on purpose:
                // short-circuit logic here split the warp for the rest of the loop body.
                // top != ref  <=>  some non-ref entry beats the ref count, or ties it while sorting before it
                const int key_ref = (0x5310 >> (4 * chr)) & 15;                      // A C G T -> 0 1 3 5 (D = 2, I = 4)
                auto beats = [&](int v, int key) -> bool { return (v > 0) & ((v > refcnt) | ((v == refcnt) & (key < key_ref))); };
                const bool top_other = beats(tb[0], 0) | beats(tb[1], 1) | beats(tb[2], 3) | beats(tb[3], 5) | beats(tD, 2) | beats(tI, 4);
                const int mxb = max(max(tb[0], tb[1]), max(tb[2], tb[3]));
                const int mxi = max(tI, tD);
                const int dgt = min(depth, kGateTab - 1);
                bool af_pass = ((mxb > 0) & (mxb >= sm.thr_snp[dgt])) | ((mxi > 0) & (mxi >= sm.thr_indel[dgt]));
                if (depth >= kGateTab)                                                  // beyond the table: the divide itself
                    af_pass = (mxb > 0 && 1.0 * mxb / depth >= prm.snp_min_af) || (mxi > 0 && 1.0 * mxi / depth >= prm.indel_min_af);
                const bool pass = top_other | af_pass;
                const bool covered = ((int)(md & 0xFFFF) + (int)(md >> 16) + df + dr > 0) | (((sm.skipcov[p >> 5] >> (p & 31)) & 1u) != 0u);
                const bool gate = covered & ref_acgt & pass & (depth >= prm.min_coverage);      // main.cpp:196
                flags[((int64_t)ts - region_start) + p] = (uint8_t)((covered ? NSNP_F_COVERED : 0) | (gate ? NSNP_F_GATE : 0));
                // the row is 72 contiguous bytes at 72*p: four 16-byte vector stores plus one 8-byte store.  Rows of odd
                // positions start 8 bytes off a 16-byte boundary, so the 8-byte piece goes first there and last otherwise;
                // the values are selected, not branched on (lane parity is loop-invariant: a branch gets unswitched and
                // the two half-warps then run the whole loop separately).  Neighbouring lanes complete each other's sectors.
                const int v0 = chr == 0 ? -mf : cf[0], v1 = chr == 1 ? -mf : cf[1], v2 = chr == 2 ? -mf : cf[2], v3 = chr == 3 ? -mf : cf[3];
                const int v9 = chr == 0 ? -mr : cr[0], v10 = chr == 1 ? -mr : cr[1], v11 = chr == 2 ? -mr : cr[2], v12 = chr == 3 ? -mr : cr[3];
                const int r[18] = {v0, v1, v2, v3, tot0, mx0, tot2, mx2, df, v9, v10, v11, v12, tot1, mx1, tot3, mx3, dr};
                int32_t* orow = counts + (((int64_t)ts - region_start) + p) * 18;
                const bool odd = (p & 1) != 0;
                int4* o16 = reinterpret_cast<int4*>(orow + (odd ? 2 : 0));
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    st_stream(o16 + q, make_int4(odd ? r[4 * q + 2] : r[4 * q], odd ? r[4 * q + 3] : r[4 * q + 1],
                                                 odd ? r[4 * q + 4] : r[4 * q + 2], odd ? r[4 * q + 5] : r[4 * q + 3]));
                st_stream(reinterpret_cast<int2*>(orow + (odd ? 0 : 16)), make_int2(odd ? r[0] : r[16], odd ? r[1] : r[17]));
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Tile list of a targeted call: the tiles holding any position of [start - 16, end + 16) of some interval, ascending.
// One block, no per-interval launch: boundary deltas per interval (tile ranges of neighbouring intervals may overlap),
// then a running sum and an ordered compaction over the tiles.  Count -> counters[6].
__global__ void __launch_bounds__(1024) tile_list_kernel(Workspace ws, int n_iv, int64_t region_start, int64_t region_len,
                                                         int n_tiles)
{
    __shared__ int wtot[2][32];
    __shared__ int carry[2];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i <= n_tiles; i += 1024) ws.tile_diff[i] = 0;
    if (tid < 2) carry[tid] = 0;
    __syncthreads();
    for (int k = tid; k < n_iv; k += 1024) {
        const int64_t a = max((int64_t)ws.targets[2 * k] - NSNP_FLANK, region_start) - region_start;
        const int64_t b = min((int64_t)ws.targets[2 * k + 1] + NSNP_FLANK, region_start + region_len) - region_start;
        if (a < b) { atomicAdd(&ws.tile_diff[a >> kTileShift], 1); atomicSub(&ws.tile_diff[((b - 1) >> kTileShift) + 1], 1); }
    }
    __syncthreads();
    for (int base = 0; base < n_tiles; base += 1024) {
        const int i = base + tid;
        const int d = i < n_tiles ? ws.tile_diff[i] : 0;
        const int di = warp_incl_scan(d);
        if (lane == 31) wtot[0][warp] = di;
        __syncthreads();
        int run = carry[0] + di;
        for (int w = 0; w < warp; ++w) run += wtot[0][w];
        const bool listed = i < n_tiles && run > 0;
        const uint32_t bal = __ballot_sync(0xffffffffu, listed);
        if (lane == 0) wtot[1][warp] = __popc(bal);
        __syncthreads();
        int off = carry[1] + __popc(bal & ((1u << lane) - 1u));
        for (int w = 0; w < warp; ++w) off += wtot[1][w];
        if (listed) ws.tile_list[off] = i;
        __syncthreads();
        if (tid == 1023) { carry[0] = run; carry[1] = off + (listed ? 1 : 0); }
        __syncthreads();
    }
    if (tid == 0) ws.counters[6] = carry[1];
}

}  // namespace
}  // namespace nsnp

using namespace nsnp;

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
static constexpr int kMaxCtas = kNumSMs * 4;
static constexpr int64_t kSlabCapMax = 32768;

// n_targets < 0: no target areas (the layout of nsnp_pileup_counts)
static void carve(void* base, int64_t n_reads, int64_t n_cigar, int64_t region_len, Workspace* w, size_t* total,
                  int64_t n_targets = -1) {
    const int64_t n_slots = (n_cigar >> kCkShift) + n_reads + 2;
    const int64_t n_tiles = (region_len + kTile - 1) >> kTileShift;
    int64_t cap = n_cigar < kSlabCapMax ? n_cigar : kSlabCapMax; if (cap < 64) cap = 64;
    size_t off = 0;
    auto take = [&](size_t bytes) { void* p = base ? (char*)base + off : nullptr; off += align_up(bytes, 256); return p; };
    w->rend = (int32_t*)take((size_t)(n_reads + 1) * 4);
    w->ck_ref = (int32_t*)take((size_t)n_slots * 4);
    w->ck_q = (int32_t*)take((size_t)n_slots * 4);
    w->tile_lo = (int32_t*)take((size_t)(n_tiles + 1) * 4);
    w->tile_hi = (int32_t*)take((size_t)(n_tiles + 1) * 4);
    w->counters = (int32_t*)take(64);
    w->cap_end = (int32_t*)take((size_t)(n_reads + 1) * 4);
    w->cap_heap = (int32_t*)take((size_t)(n_reads + 1) * 4);
    w->slabs = (Event*)take((size_t)kMaxCtas * (size_t)cap * sizeof(Event));
    w->slab_cap = cap;
    w->targets = w->tile_diff = w->tile_list = nullptr;
    if (n_targets >= 0) {
        w->targets = (int32_t*)take((size_t)(2 * n_targets + 2) * 4);
        w->tile_diff = (int32_t*)take((size_t)(n_tiles + 1) * 4);
        w->tile_list = (int32_t*)take((size_t)(n_tiles + 1) * 4);
    }
    *total = off;
}

// targets == nullptr && n_targets < 0: the whole region (nsnp_pileup_counts)
static int pileup_counts(const nsnp_reads_t* reads, const uint8_t* ref_dev, int64_t contig_len, int64_t region_start,
                         int64_t region_len, const int32_t* targets, int64_t n_targets, const nsnp_params_t* params,
                         int32_t* counts_dev, uint8_t* flags_dev, void* workspace_dev, size_t workspace_bytes,
                         int32_t* status_dev, void* stream_)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!reads || !params || !ref_dev || !counts_dev || !flags_dev || !status_dev || !workspace_dev)
        return set_error(NSNP_E_INVALID, "nsnp_pileup_counts: null argument");
    if (region_start < 0 || region_len < 0 || region_start + region_len > contig_len)
        return set_error(NSNP_E_INVALID, "nsnp_pileup_counts: region [%lld,+%lld) outside contig of %lld",
                         (long long)region_start, (long long)region_len, (long long)contig_len);
    if (reads->n_reads < 0 || (reads->n_reads > 0 && (!reads->pos || !reads->flag || !reads->mapq || !reads->cigar_off || !reads->cigar || !reads->seq_off || !reads->seq2)))
        return set_error(NSNP_E_INVALID, "nsnp_pileup_counts: incomplete read arrays");
    if (reads->cigar_bits != 0 && reads->cigar_bits != 16 && reads->cigar_bits != 32)
        return set_error(NSNP_E_INVALID, "nsnp_pileup_counts: cigar_bits must be 32 (or 0) or 16");
    if (((uintptr_t)reads->seq2 & 3) || ((uintptr_t)reads->nmask & 3) || ((uintptr_t)counts_dev & 15))
        return set_error(NSNP_E_INVALID, "nsnp_pileup_counts: seq2/nmask must be 4-byte and counts 16-byte aligned");
    if (reads->n_reads > 0x7fffffff - 1) return set_error(NSNP_E_UNSUPPORTED, "more than 2^31 reads in one call");
    if (contig_len > 0x7fffffff - 4096) return set_error(NSNP_E_UNSUPPORTED, "contig longer than 2^31 - 4096 (BAM positions are int32)");
    if (n_targets >= 0) {
        if (int e = check_targets("nsnp_pileup_counts_targets", targets, n_targets, region_start, region_start + region_len)) return e;
    }
    if (nsnp_device_count() == 0) return set_error(NSNP_E_NO_DEVICE, "no CUDA device (there is no CPU fallback)");
    if (region_len == 0) return NSNP_OK;

    Workspace w; size_t need = 0;
    carve(workspace_dev, reads->n_reads, reads->n_cigar, region_len, &w, &need, n_targets);
    if (need > workspace_bytes) return set_error(NSNP_E_WORKSPACE, "pileup workspace: need %zu bytes, have %zu", need, workspace_bytes);
    const int n_tiles = (int)((region_len + kTile - 1) >> kTileShift);

    cudaMemsetAsync(w.tile_lo, 0x7f, (size_t)(n_tiles + 1) * 4, stream);
    cudaMemsetAsync(w.tile_hi, 0, (size_t)(n_tiles + 1) * 4, stream);
    cudaMemsetAsync(w.counters, 0, 64, stream);
    if (n_targets >= 0) {
        // unlisted tiles: flags zero, count rows left unwritten (nothing reads them)
        cudaMemsetAsync(flags_dev, 0, (size_t)region_len, stream);
        if (n_targets > 0)
            cudaMemcpyAsync(w.targets, targets, (size_t)n_targets * 8, cudaMemcpyHostToDevice, stream);
        tile_list_kernel<<<1, 1024, 0, stream>>>(w, (int)n_targets, region_start, region_len, n_tiles);
        if (int e = cuda_status("tile_list_kernel")) return e;
    }
    if (reads->n_reads > 0) {
        const int64_t warps = reads->n_reads;
        int blocks = (int)((warps + 7) / 8); if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
        ProfScope prof(NSNP_PROF_READ_SCAN, stream);
        read_scan_kernel<<<blocks, 256, 0, stream>>>(*reads, *params, region_start, region_start + region_len, w, status_dev);
        if (int e = cuda_status("read_scan_kernel")) return e;
        if (params->max_depth > 0) {
            cap_kernel<<<(int)((reads->n_reads / kCapStride + 8) / 8), 256, 0, stream>>>(*reads, w, params->max_depth);
            if (int e = cuda_status("depth cap kernels")) return e;
        }
    }
    {
        constexpr size_t smem = sizeof(TileSmem);
        constexpr int threads = kTile / 4;
        static bool attr_done = false;
        if (!attr_done) {
            if (cudaFuncSetAttribute(pileup_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
                return cuda_status("cudaFuncSetAttribute(pileup_tile_kernel)");
            attr_done = true;
        }
        int occ = 1;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, pileup_tile_kernel, threads, smem);
        if (occ < 1) occ = 1; if (occ > 4) occ = 4;
        int grid = kNumSMs * occ; if (grid > n_tiles) grid = n_tiles; if (grid > kMaxCtas) grid = kMaxCtas;
        ProfScope prof(NSNP_PROF_PILEUP_TILE, stream);
        pileup_tile_kernel<<<grid, threads, smem, stream>>>(*reads, *params, ref_dev, region_start, region_len, n_tiles, w,
                                                            counts_dev, flags_dev, status_dev);
        if (int e = cuda_status("pileup_tile_kernel")) return e;
    }
    return NSNP_OK;
}

extern "C" {

size_t nsnp_pileup_workspace_bytes(int64_t n_reads, int64_t n_cigar, int64_t region_len) {
    Workspace w; size_t total = 0;
    carve(nullptr, n_reads < 0 ? 0 : n_reads, n_cigar < 0 ? 0 : n_cigar, region_len < 0 ? 0 : region_len, &w, &total);
    return total;
}

int nsnp_pileup_counts(const nsnp_reads_t* reads, const uint8_t* ref_dev, int64_t contig_len, int64_t region_start,
                       int64_t region_len, const nsnp_params_t* params, int32_t* counts_dev, uint8_t* flags_dev,
                       void* workspace_dev, size_t workspace_bytes, int32_t* status_dev, void* stream)
{
    return pileup_counts(reads, ref_dev, contig_len, region_start, region_len, nullptr, -1, params, counts_dev, flags_dev,
                         workspace_dev, workspace_bytes, status_dev, stream);
}

size_t nsnp_pileup_targets_workspace_bytes(int64_t n_reads, int64_t n_cigar, int64_t region_len, int64_t n_targets) {
    Workspace w; size_t total = 0;
    carve(nullptr, n_reads < 0 ? 0 : n_reads, n_cigar < 0 ? 0 : n_cigar, region_len < 0 ? 0 : region_len, &w, &total,
          n_targets < 0 ? 0 : n_targets);
    return total;
}

int nsnp_pileup_counts_targets(const nsnp_reads_t* reads, const uint8_t* ref_dev, int64_t contig_len, int64_t region_start,
                               int64_t region_len, const int32_t* targets, int64_t n_targets, const nsnp_params_t* params,
                               int32_t* counts_dev, uint8_t* flags_dev, void* workspace_dev, size_t workspace_bytes,
                               int32_t* status_dev, void* stream)
{
    if (n_targets < 0) return set_error(NSNP_E_INVALID, "nsnp_pileup_counts_targets: negative interval count");
    return pileup_counts(reads, ref_dev, contig_len, region_start, region_len, targets, n_targets, params, counts_dev, flags_dev,
                         workspace_dev, workspace_bytes, status_dev, stream);
}

}  // extern "C"
