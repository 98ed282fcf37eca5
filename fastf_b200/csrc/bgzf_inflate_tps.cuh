// K1 (v3) -- BGZF / raw-DEFLATE inflate, "thread per stream".
//
// The lock-step kernel (bgzf_inflate.cuh) spends a whole warp on one serial Huffman chain: every lane repeats the same
// ~50 instructions per symbol, and ncu shows it bound by instruction issue (77 % of issue slots, 1 % of DRAM).  This kernel
// removes the redundancy by splitting the work by role inside one persistent CTA per SM:
//
//   decoder warps  (7 warps x 32 lanes)  lane = one BGZF block ("stream").  Pure scalar Huffman decoding out of that stream's
//                                        own shared-memory tables; emits 4-byte TOKENS (up to three literals | match(len, dist)
//                                        | end) into the stream's 64-token shared-memory ring.  No global stores, no warp
//                                        collectives.  One ROUND of a lane = up to three literal tokens (decoded without inner
//                                        branches) plus the match that ends the literal run: the divergent paths of a warp
//                                        execute one after the other and some lane always needs each of them, so every lane
//                                        walks through both.
//                                        A match whose source lies more than 512 bytes back is prefetched into L2 on the spot.
//   service warps  (25 warps, lock step) own 9 consecutive streams each; one poll pass looks at all of them (lane k reads the
//                                        k-th stream's control block, a ballot picks the streams with work).  (a) LZ77: take up
//                                        to 32 tokens of one stream, prefix-sum their output lengths, store the literals and
//                                        copy the matches with all 32 lanes (the source loads of several matches, or of several
//                                        pieces of a long one, are issued before any is stored so the L2 round trips overlap).
//                                        (b) stream set-up: fetch the next BGZF block from a global counter, parse deflate block
//                                        headers, copy stored blocks, build the Huffman tables warp-parallel -- decoders never
//                                        run that code.  Streams whose decoder waits are served first in a pass, and the next
//                                        deflate block of a BGZF block is set up while the previous one's tokens still drain.
//
// Tables per stream: 8-bit literal/length table and 6-bit distance table with 16-bit entries (code length, kind, symbol) in shared
// memory; a code longer than the table takes one lookup in the stream's second-level table in global memory (L2), with the
// canonical walk (range limits and symbol list in L2) as the fallback when the second level does not fit (never on the synthetic
// 10x BAM); length/distance base+extra bits sit in a CTA-wide table.  224 streams x 952 B + the set-up scratch fill the SM's shared
// memory (229 536 of 232 448 bytes).
// What bounds it (profiles/r02_inflate_ab.md, r05_inflate_ab.md): a latency machine -- throughput = independent Huffman chains per SM
// / per-symbol latency.  With 224 streams the LZ77 side co-limits: with a 32-token ring a third of the decoders' lane-rounds found
// it full (the service warps 97 % busy, 5 700 cycles per batch of 22 tokens); the 64-token ring lets every visit take a full 32
// tokens and cuts that share to an eighth.  DRAM traffic is 5x the algorithmic bytes (the windows of 33 152 resident streams do not
// fit the L2) but at 12 % of the bandwidth it is not the limit.
#pragma once
#include "bgzf_inflate.cuh"

// Shape and table sizes (round 2, measured on B200 with scripts/gpu_inflate_ab.sh on images of exactly two rounds of each shape's
// own stream count; profiles/r02_inflate_ab.md).  The kernel is bound by the number of independent Huffman chains an SM keeps
// going: a stream decodes a symbol every ~1000 cycles whatever the shape, so throughput follows the stream count, which shared
// memory limits.  8-bit literal/length and 6-bit distance tables with a 32-token ring fit 224 streams per SM (7 full decoder
// warps + 25 service warps = 1024 threads): 179-183 GB/s algorithmic against 156 GB/s for the round-1 shape (128 streams, 9/7-bit
// tables, 16 lanes x 8 warps + 24).  16-lane decoder warps at 224 streams leave too few service warps (138 GB/s); 256 streams need
// a 16-token ring that starves the decoders (147 GB/s).  Moving the canonical walk's limits to global scratch pays for a 64-token
// ring at 224 streams: 193 -> 205 GB/s, 207 with three literal tokens per round (profiles/r05_inflate_ab.md).
#ifndef FASTF_TPS_LBITS
#define FASTF_TPS_LBITS 8
#endif
#ifndef FASTF_TPS_DBITS
#define FASTF_TPS_DBITS 6
#endif
// kernel shape (template parameters L = decoding lanes per decoder warp, SVC = service warps): FASTF_TPS_STREAMS streams per CTA,
// FASTF_TPS_STREAMS / L decoder warps
#ifndef FASTF_TPS_STREAMS
#define FASTF_TPS_STREAMS 224
#endif
#define FASTF_TPS_THREADS_OF(L, SVC) ((FASTF_TPS_STREAMS / (L) + (SVC)) * 32)
// the shape the host launches (and the emulator tests)
#ifndef FASTF_TPS_LANES
#define FASTF_TPS_LANES 32
#endif
#ifndef FASTF_TPS_SVC_WARPS
#define FASTF_TPS_SVC_WARPS 25
#endif
#ifndef FASTF_TPS_MAX_SVC
#define FASTF_TPS_MAX_SVC FASTF_TPS_SVC_WARPS
#endif
// Second-level tables (FASTF_TPS_SUBTABLES): a code longer than the primary table is resolved by ONE more look-up instead of the
// canonical walk (~45 instructions that every lane of the warp sits through whenever one lane meets such a code -- with 32 streams
// per warp that is nearly every round).  The primary entry of a long prefix names a sub-table (offset / 8, index bits); sub-tables
// live in the stream's global scratch (L2) next to the sorted symbol lists.  A code whose sub-tables would not fit keeps the walk.
#ifndef FASTF_TPS_SUBTABLES
#define FASTF_TPS_SUBTABLES 1
#endif
#define FASTF_TPS_LITSUB_U16 1016u   // capacity of the literal/length sub-tables (7-bit offset field x 8)
#define FASTF_TPS_DISTSUB_U16 512u
// Per stream in GLOBAL scratch: symbols sorted by code length (288 lit/len + 32 dist), read only for codes longer than the tables,
// then the two sub-table areas, then the canonical walk's range limits / index offsets (literal/length table, then distance table).
#if FASTF_TPS_SUBTABLES
#define FASTF_TPS_WALK_AT (320 + 1024 + 512)
#else
#define FASTF_TPS_WALK_AT 320
#endif
#define FASTF_TPS_SORTED_U16 (FASTF_TPS_WALK_AT + FASTF_TPS_WALK_U16(FASTF_TPS_LBITS) + FASTF_TPS_WALK_U16(FASTF_TPS_DBITS))
#define FASTF_TPS_THREADS FASTF_TPS_THREADS_OF(FASTF_TPS_LANES, FASTF_TPS_SVC_WARPS)
#ifndef FASTF_TPS_RING
#define FASTF_TPS_RING 64u
#endif
#ifndef FASTF_TPS_TRIPLES
#define FASTF_TPS_TRIPLES 3           // literal tokens (three literals each) a decoder round may produce in front of a match
#endif
#ifndef FASTF_TPS_BATCH_MIN
#define FASTF_TPS_BATCH_MIN (FASTF_TPS_RING >= 64u ? 32u : FASTF_TPS_RING / 2u)       // tokens that make a stream worth a visit of its service warp
#endif
#ifndef FASTF_TPS_BRANCHFREE
#define FASTF_TPS_BRANCHFREE 1      // 1: literal triples without inner branches (+4 % at 224 streams, +7 % on the decoders alone); 2: also the bit-buffer refills
#endif
#ifndef FASTF_TPS_PREFETCH2
#define FASTF_TPS_PREFETCH2 0
#endif
#ifndef FASTF_TPS_FAR_LEN
#define FASTF_TPS_FAR_LEN 32u         // longest match handled in the far group (32 or 64: one or two bytes per lane)
#endif
#ifndef FASTF_TPS_SLOW_UNROLL
#define FASTF_TPS_SLOW_UNROLL 1      // long non-overlapping matches: four pieces' loads in flight (+1 %)
#endif
#ifndef FASTF_TPS_FAR
#define FASTF_TPS_FAR 4              // far matches whose source loads are in flight together
#endif

// 16-bit table entry: bits 0-3 code length (0 = longer than the table), bits 4-5 kind, bits 8-15 payload.  A slot whose code is
// longer than the table holds FASTF_T16_LONG (length 0, kind BAD), so that "literal resolved by the table" is the single test
// (e & 0x30) == 0, and a literal byte moves into its token with one masked OR (e & 0xff00).
#define FASTF_T16_LIT 0u     // payload = literal byte / code-length symbol
#define FASTF_T16_SYM 1u     // payload = length symbol - 257, or distance symbol
#define FASTF_T16_EOB 2u
#define FASTF_T16_BAD 3u
#define FASTF_T16_LONG (FASTF_T16_BAD << 4)
#define FASTF_T16_IS_TABLE_LIT(e) (((e) & 0x30u) == 0u)
// tokens
#define FASTF_TOK_LIT 0u             // bits 0-23 up to three literal bytes (first in bits 0-7), bits 24-25 their number
#define FASTF_TOK_MATCH (1u << 30)   // bits 0-8 length, bits 9-24 distance
#define FASTF_TOK_END (2u << 30)     // bits 0-15 status bits of the decoder
// stream states
enum { FASTF_TPS_NEXT = 0, FASTF_TPS_RUN = 1, FASTF_TPS_BUILD = 2, FASTF_TPS_DONE = 3 };

// Codes longer than a primary table of TBITS bits have 15 - TBITS possible lengths; per length the decoder needs a range limit and
// an index offset (fastf_tps_build).  Limits sit in [0, OFFS), offsets in [OFFS, 2 OFFS), OFFS = 8 or 12 (vector loads).
#define FASTF_TPS_WALK_OFFS(TBITS) ((15 - (TBITS)) <= 8 ? 8 : 12)
#define FASTF_TPS_WALK_U16(TBITS) (2 * FASTF_TPS_WALK_OFFS(TBITS))   // per table in the stream's global scratch (a multiple of 4: vector loads)
// The walk's limits live in global scratch, not in the stream structure: the hot path resolves long codes through the sub-tables,
// so the walk is rare, and its 80 bytes per stream pay for the 64-token ring at 224 streams.
// Lane i of a decoder warp (and lane k of a polling service warp) works on stream i: the same field of consecutive streams must
// not fall into the same shared-memory bank.  The structure is 8-byte aligned and its size = 8 (mod 16) bytes, i.e. a bank step
// of 2 between streams (an exact multiple of 128 bytes would put every lane on one bank).
struct FastfTpsStream {
    u16 lit[1 << FASTF_TPS_LBITS];
    u16 dist[1 << FASTF_TPS_DBITS];
    alignas(8) u32 ring[FASTF_TPS_RING];
    // control block (volatile accesses; every hand-over is fenced)
    u32 state, wr, rd, last;         // state, wr, rd: polled as ctl[0..2] by the service warps
    u32 bitpos_lo, bitpos_hi;        // absolute bit offset of the next unread bit inside `comp`
    u32 pos, isize;                  // decoder's output position / block size
    u32 blk, opos;                   // service side: block index, bytes written
    u32 inend_lo, inend_hi;          // absolute bit offset of the end of the payload
    u32 obase_lo, obase_hi;          // offset of the block in the inflated buffer
};

// scratch of one service warp while it sets a stream up
struct FastfTpsSvc {
    struct { u8 lens[320]; u16 scratch[32]; u8 submax[256]; } setup;   // code lengths of the block being set up; first[16], start[16] of the table being built; longest code per table prefix
};
struct FastfTpsShared {
    u32 lenK[32], distK[32];         // base << 8 | extra bits
    u8 cl_order[20];
    alignas(16) FastfTpsSvc svc[FASTF_TPS_MAX_SVC];
};
// largest dynamic shared memory a block may opt in to on sm_100 (227 KB): the shape must fit it at compile time, not at launch
#define FASTF_TPS_SMEM_MAX 232448u
#define FASTF_TPS_SMEM_BYTES (sizeof(FastfTpsStream) * FASTF_TPS_STREAMS + sizeof(FastfTpsShared))
static_assert(sizeof(FastfTpsStream) % 16 == 8, "stream size must be 8 (mod 16) bytes: bank step of 2 between the streams of a warp");
static_assert(FASTF_TPS_SMEM_BYTES <= FASTF_TPS_SMEM_MAX, "streams + set-up scratch exceed the shared memory of an SM");


// Hand-over between warps of the CTA goes through shared memory only.  One thread's shared-memory stores are performed in
// program order and so are another thread's volatile loads, so publishing "data, then counter" needs no MEMBAR on the hot
// path -- a real fence would also wait for the decoder's outstanding global prefetch.  The compiler must not reorder, though.
#ifdef FASTF_EMU
#define FASTF_SMEM_ORDER() ((void)0)
#else
#define FASTF_SMEM_ORDER() __asm__ __volatile__("" ::: "memory")
#endif
// FASTF_TPS_PROF: where the lane-rounds of the decoders and the cycles of the service warps go (debug builds only; read with
// fastf_debug_tps_prof).  [0] decoder lane-rounds decoded, [1] skipped with a full ring, [2] skipped waiting for set-up,
// [3] service passes, [4] passes without work, [5] cycles in copies, [6] cycles in set-up, [7] cycles in passes without work,
// [8] batches, [9] tokens, [10] total service cycles, [11] codes longer than the primary table, [12] of them resolved by the
// canonical walk (their sub-tables did not fit).
// Set-up in time: [13] of [2] the rounds that wait for a new BGZF block (NEXT, launch start included; the rest wait for the next
// deflate block of the same BGZF block, BUILD), [14] / [15] decoder cycles waiting for BUILD / NEXT (summed over lanes, from the
// hand-over or the launch start to RUN; the last wait, for DONE, is not counted), [16] decoder cycles from the launch to DONE
// (summed over lanes), [17] BGZF blocks fetched, [18] deflate block headers parsed, [19] set-up cycles in table builds (the rest of
// [6] is block fetch, headers, code-length decode and stored copies), [20] / [21] cycles from a BUILD hand-over to the start of its
// set-up and their number, [22] / [23] the same for NEXT hand-overs (END token), [24] set-ups started while tokens were pending,
// [25] of them left for later (stored block or error: set up again once the ring is empty)
#ifndef FASTF_TPS_PROF
#define FASTF_TPS_PROF 0
#endif
#define FASTF_TPS_PROF_N 32
#if FASTF_TPS_PROF
__device__ unsigned long long g_fastf_tps_prof[FASTF_TPS_PROF_N];
// clock64 of each stream's last hand-over (0 = none yet in this launch); grids of up to 1024 CTAs
__device__ unsigned long long g_fastf_tps_handover[1024 * FASTF_TPS_STREAMS];
#define FASTF_PROF(x) x
// time from a stream's hand-over to the start of its set-up: slot [at] cycles, [at + 1] count
__device__ __forceinline__ void fastf_tps_prof_handover(u32 sidx, u32 at)
{
    unsigned long long &h = g_fastf_tps_handover[blockIdx.x * FASTF_TPS_STREAMS + sidx];
    if (h) { atomicAdd(&g_fastf_tps_prof[at], (unsigned long long)(clock64() - (long long)h)); atomicAdd(&g_fastf_tps_prof[at + 1], 1ull); h = 0; }
}
#else
#define FASTF_PROF(x)
#endif
// control-block words polled in a loop: a 32-bit shared-memory address the compiler cannot re-derive (it would rebuild it from the
// thread index in every pass), read with volatile shared loads
#ifdef FASTF_EMU
typedef const u32 *fastf_ctl_ptr;
static inline fastf_ctl_ptr fastf_ctl_of(const u32 *p) { return p; }
static inline u32 fastf_ctl_ld(fastf_ctl_ptr p, u32 word) { return *(const volatile u32 *)(p + word); }
#else
typedef u32 fastf_ctl_ptr;
__device__ __forceinline__ fastf_ctl_ptr fastf_ctl_of(const u32 *p)
{
    u32 a = (u32)__cvta_generic_to_shared(p);
    asm volatile("" : "+r"(a));
    return a;
}
__device__ __forceinline__ u32 fastf_ctl_ld(fastf_ctl_ptr a, u32 word)
{
    u32 v;
    asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(v) : "r"(a + 4u * word) : "memory");
    return v;
}
#endif
// the sorted-symbol lists live in global memory, are rewritten for every deflate block by a service warp and read by another warp
// of the same CTA: read them through L2 (ld.cg), never through a possibly stale L1 line
#ifdef FASTF_EMU
__device__ __forceinline__ u32 fastf_ld_sorted(const u16 *p) { return *p; }
#else
#ifndef FASTF_TPS_SORTED_L1
#define FASTF_TPS_SORTED_L1 0
#endif
#if FASTF_TPS_SORTED_L1
__device__ __forceinline__ u32 fastf_ld_sorted(const u16 *p) { return *p; }
#else
__device__ __forceinline__ u32 fastf_ld_sorted(const u16 *p) { return __ldcg(p); }
#endif
#endif
// the walk's limits / offsets: rewritten for every deflate block by a service warp, so always read through L2 (8-byte vectors)
#ifdef FASTF_EMU
__device__ __forceinline__ uint2 fastf_ld_walk2(const u16 *p) { return *reinterpret_cast<const uint2 *>(p); }
__device__ __forceinline__ u32 fastf_ld_walk(const u16 *p) { return *p; }
#else
__device__ __forceinline__ uint2 fastf_ld_walk2(const u16 *p) { return __ldcg(reinterpret_cast<const uint2 *>(p)); }
__device__ __forceinline__ u32 fastf_ld_walk(const u16 *p) { return __ldcg(p); }
#endif
// A decoder knows the source of a match thousands of cycles before the stream's service warp copies it: it asks the L2 for the line
// right away (the windows of all resident streams are far larger than the L2, so a distant source is usually a DRAM access).
#ifndef FASTF_TPS_PREFETCH_SRC
#define FASTF_TPS_PREFETCH_SRC 512u   // smallest distance worth a prefetch (0 = never); +2 % at 224 streams
#endif
#ifdef FASTF_EMU
__device__ __forceinline__ void fastf_prefetch_l2(const void *) {}
#else
__device__ __forceinline__ void fastf_prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
#endif
#ifndef FASTF_TPS_NOCOPY
#define FASTF_TPS_NOCOPY 0            // measurement builds only: 1 = service warps skip the match copies, 2 = they store nothing at all
#endif
__device__ __forceinline__ u32 fastf_ldv(const u32 *p) { return *(const volatile u32 *)p; }
__device__ __forceinline__ void fastf_stv(u32 *p, u32 v) { *(volatile u32 *)p = v; }

__device__ __forceinline__ u32 fastf_make16(u32 alpha, u32 sym)
{
    if (alpha == FASTF_ALPHA_PLAIN) return (FASTF_T16_LIT << 4) | (sym << 8);
    if (alpha == FASTF_ALPHA_LITLEN) {
        if (sym < 256) return (FASTF_T16_LIT << 4) | (sym << 8);
        if (sym == 256) return FASTF_T16_EOB << 4;
        if (sym > 285) return FASTF_T16_BAD << 4;
        return (FASTF_T16_SYM << 4) | ((sym - 257) << 8);
    }
    if (sym >= 30) return FASTF_T16_BAD << 4;
    return (FASTF_T16_SYM << 4) | (sym << 8);
}

// lanes of a chunk whose code length is l, from the four ballots of the lengths' bits
__device__ __forceinline__ u32 fastf_tps_len_peers(u32 l, u32 b0, u32 b1, u32 b2, u32 b3)
{
    return ((l & 1u) ? b0 : ~b0) & ((l & 2u) ? b1 : ~b1) & ((l & 4u) ? b2 : ~b2) & ((l & 8u) ? b3 : ~b3);
}

// Cooperative (32 lanes, lock step) construction of one 16-bit decode table.  Returns non-zero for an invalid code (over-subscribed,
// or incomplete with more than one code).  No lane walks the symbols alone: symbol 32 c + k sits in lane k of chunk c, and four
// ballots over the bits of the chunk's code lengths give every lane the lanes that share its length.  Lane l (1..15) counts the
// codes of length l; a scan over those 15 lanes gives first[l] (first canonical code of length l) and start[l] (index of its first
// symbol in sorted[]); a symbol's canonical code is then first[l] + the codes of length l in earlier chunks + its rank among its
// peers, and its lane fills its table slots (and those of its sub-table) straight from registers.
// first[16], start[16]: shared scratch, for the sub-table layout.  lb: the stream's walk limits / offsets in global scratch (null for
// the code-length table, whose codes all fit the table).
__device__ __forceinline__ u32 fastf_tps_build(u32 alpha, const u8 *lens, u32 n, u16 *lb, u16 *sorted, u16 *lut, u32 tbits, u16 *first, u16 *start, u32 lane,
                                               u16 *sub = nullptr, u32 sub_cap = 0, u8 *submax = nullptr)
{
    for (u32 i = lane; i < (1u << tbits); i += 32) lut[i] = FASTF_T16_LONG;
    const u32 nch = (n + 31u) >> 5, ml = lane & 15u, lt = (1u << lane) - 1u;
    u32 cnt = 0;
    for (u32 c = 0; c < nch; c++) {
        const u32 s = (c << 5) + lane, l = s < n ? lens[s] : 0u;
        const u32 b0 = __ballot_sync(FASTF_FULL_MASK, l & 1u), b1 = __ballot_sync(FASTF_FULL_MASK, l & 2u);
        const u32 b2 = __ballot_sync(FASTF_FULL_MASK, l & 4u), b3 = __ballot_sync(FASTF_FULL_MASK, l & 8u);
        cnt += (u32)__popc(fastf_tps_len_peers(ml, b0, b1, b2, b3));
    }
    if (lane == 0 || lane >= 16) cnt = 0;   // length 0: symbol not used
    // Inclusive scans over the lengths of the symbol count and of the Kraft sum: a code of length l takes 2^(15-l) of the 2^15
    // 15-bit codes.  The code over-subscribes iff that sum exceeds 2^15 (a deficit, once negative, stays negative from one length to
    // the next), and is incomplete iff it falls short.  first[l] = sum over k < l of cnt[k] << (l - k): the exclusive Kraft sum at
    // l, shifted down (exactly: every term is a multiple of 2^(15-l+1)).
    const u32 kw = cnt << (15u - ml);
    u32 ns = cnt, ks = kw;
#pragma unroll
    for (int o = 1; o < 16; o <<= 1) {
        const u32 a = __shfl_up_sync(FASTF_FULL_MASK, ns, o), k = __shfl_up_sync(FASTF_FULL_MASK, ks, o);
        if ((int)lane >= o) { ns += a; ks += k; }
    }
    const u32 used = __shfl_sync(FASTF_FULL_MASK, ns, 15), kraft = __shfl_sync(FASTF_FULL_MASK, ks, 15);
    if (kraft > 32768u || (kraft < 32768u && used > 1u)) return 1;
    const u32 st = ns - cnt, fc = (ks - kw) >> (15u - ml);
    if (lane < 16) { first[lane] = (u16)fc; start[lane] = (u16)st; }
    // For the codes longer than the table the decoder needs, per length l = tbits+1+k: the left-aligned (15-bit) end of the length's
    // code range (ranges of a canonical code follow one another in length order) and start[l] - first[l], the offset that turns a
    // code into its index in sorted[].  Limits go to lb[0, OFFS), offsets behind them.
    if (lb) {
        const u32 offs_at = FASTF_TPS_WALK_OFFS(tbits), l = tbits + 1u + lane, src = l <= 15u ? l : 15u;
        const u32 f = __shfl_sync(FASTF_FULL_MASK, fc, (int)src), c = __shfl_sync(FASTF_FULL_MASK, cnt, (int)src), s0 = __shfl_sync(FASTF_FULL_MASK, st, (int)src);
        if (lane < offs_at) {
            lb[lane] = l <= 15u ? (u16)((f + c) << (15u - l)) : (u16)0xffff;
            lb[offs_at + lane] = l <= 15u ? (u16)(s0 - f) : (u16)0;
        }
    }
    const u32 long_from = __shfl_sync(FASTF_FULL_MASK, st, (int)tbits + 1);
    __syncwarp();
    bool subs = false;
#if FASTF_TPS_SUBTABLES
    const u32 nidx = 1u << tbits;
    if (sub && long_from < used) {
        // (1) per table index j (the code's first tbits bits, in stream order): the longest code that starts with them.  The canonical
        // codes of length l are [first[l], first[l] + cnt[l]); the ones with the (MSB-first) prefix q are q << (l - tbits) ... .
        // The primary entry has 3 bits for the sub-table's index bits: a prefix with codes more than 7 bits longer than the table (a
        // distance code of 14 or 15 bits) gets no sub-table, its codes take the walk.
        for (u32 j = lane; j < nidx; j += 32) {
            const u32 q = __brev(j) >> (32 - tbits);
            u32 mx = 0;
            for (u32 l = tbits + 1; l <= 15; l++) {
                const u32 c = (l < 15 ? (u32)start[l + 1] : used) - (u32)start[l];
                const u32 lo = q << (l - tbits), hi = (q + 1u) << (l - tbits);
                if (c && (u32)first[l] < hi && (u32)first[l] + c > lo) mx = l;
            }
            submax[j] = (u8)(mx && mx - tbits <= 7u ? mx - tbits : 0u);
        }
        __syncwarp();
        // (2) sub-table offsets: sizes 2^bits padded to 8 entries, exclusive prefix sum over the indices (lane k owns a contiguous run)
        const u32 per = (nidx + 31u) / 32u, j0 = lane * per;
        u32 mine = 0;
        for (u32 j = j0; j < j0 + per && j < nidx; j++) { const u32 b = submax[j]; mine += b ? (b < 3u ? 8u : (1u << b)) : 0u; }
        u32 inc = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const u32 t = __shfl_up_sync(FASTF_FULL_MASK, inc, o); if ((int)lane >= o) inc += t; }
        const u32 total = __shfl_sync(FASTF_FULL_MASK, inc, 31);
        subs = total <= sub_cap;
        if (subs) {
            u32 at = inc - mine;
            for (u32 j = j0; j < j0 + per && j < nidx; j++) {
                const u32 b = submax[j];
                if (b) { lut[j] = (u16)(FASTF_T16_LONG | (b << 6) | ((at >> 3) << 9)); at += b < 3u ? 8u : (1u << b); }
            }
        }
        __syncwarp();
    }
#endif
    // (3) every symbol: its place in sorted[], its primary-table slots, or (a long code) its slots of its prefix's sub-table.
    // Lane l carries the code and the sorted[] index of the next symbol of length l.
    u32 nf = fc, nsrt = st;
    for (u32 c = 0; c < nch; c++) {
        const u32 s = (c << 5) + lane, l = s < n ? lens[s] : 0u;
        const u32 b0 = __ballot_sync(FASTF_FULL_MASK, l & 1u), b1 = __ballot_sync(FASTF_FULL_MASK, l & 2u);
        const u32 b2 = __ballot_sync(FASTF_FULL_MASK, l & 4u), b3 = __ballot_sync(FASTF_FULL_MASK, l & 8u);
        const u32 rank = (u32)__popc(fastf_tps_len_peers(l, b0, b1, b2, b3) & lt);
        const u32 code = __shfl_sync(FASTF_FULL_MASK, nf, (int)l) + rank, idx = __shfl_sync(FASTF_FULL_MASK, nsrt, (int)l) + rank;
        const u32 here = (u32)__popc(fastf_tps_len_peers(ml, b0, b1, b2, b3));
        nf += here; nsrt += here;
        if (l) {
            sorted[idx] = (u16)s;
            const u32 rev = __brev(code) >> (32 - l);
            const u16 e = (u16)(fastf_make16(alpha, s) | l);
            if (l <= tbits) {
                for (u32 j = rev; j < (1u << tbits); j += (1u << l)) lut[j] = e;
            }
#if FASTF_TPS_SUBTABLES
            else if (subs) {
                const u32 pe = lut[rev & (nidx - 1u)];
                const u32 b = (pe >> 6) & 7u, at = (pe >> 9) << 3;
                if (b) for (u32 k = rev >> tbits; k < (1u << b); k += 1u << (l - tbits)) sub[at + k] = e;
            }
#endif
        }
    }
    __syncwarp();
    return 0;
}

// entry of a code longer than the primary table: through its sub-table when the primary entry names one, else by the canonical walk
template <int TBITS>
__device__ __forceinline__ u32 fastf_tps_long(u32 e, u64 buf, const u16 *lb, const u16 *sorted, const u16 *sub, u32 alpha);

// lock-step lookup used by the service warp while it reads the code-length code (7-bit table in the literal table's storage;
// code-length codes are at most 7 bits long, so every valid one is resolved by the table)
__device__ __forceinline__ u32 fastf_tps_decode16(const FastfBitReader<32> &br, const u16 *lut, u32 tbits)
{
    return lut[(u32)br.buf & ((1u << tbits) - 1u)];
}

// ------------------------------------------------------------------------------------------------------------------
// service side
// ------------------------------------------------------------------------------------------------------------------
struct FastfTpsArgs {
    const u8 *comp;
    u64 comp_total;
    const u64 *in_off;
    const u32 *in_len;
    const u64 *out_off;
    const u32 *isize;
    u32 nblocks;
    u8 *out;
    u32 *status;
    u32 *next_block;   // global work counter (zeroed before the launch)
    u16 *sorted;       // gridDim.x * FASTF_TPS_STREAMS * FASTF_TPS_SORTED_U16 entries of scratch
};

// Parse deflate block headers of stream S from its current bit position until a Huffman block is ready for the decoder
// (state RUN) or the BGZF block is finished / broken (status written, state NEXT).  Stored blocks are copied here.
// pending: the previous deflate block's tokens are still in the ring (a BUILD hand-over set up before the ring drains, so that the
// decoder does not wait for the copies).  Then only the tables and the bit position change: the copy side keeps reading the ring
// in FIFO order at S.opos, the decoder goes on at S.pos.  A stored block or an error then leaves everything as it was and
// returns non-zero: the stream stays in BUILD and is set up again from the same bit position once the ring is empty.
__device__ __forceinline__ u32 fastf_tps_setup(const FastfTpsArgs &A, FastfTpsStream &S, u16 *lit_sorted, FastfTpsShared &G, u32 sw, u32 lane, bool pending)
{
    u16 *dist_sorted = lit_sorted + 288;
    const u32 b = S.blk;
    u8 *out = A.out + (((u64)S.obase_hi << 32) | S.obase_lo);
    const u64 in_end = ((u64)S.inend_hi << 32) | S.inend_lo;
    u64 bitpos = ((u64)S.bitpos_hi << 32) | S.bitpos_lo;
    u32 opos = S.pos, err = 0;
    u8 *lens = G.svc[sw].setup.lens;
    u16 *first = G.svc[sw].setup.scratch, *start = G.svc[sw].setup.scratch + 16;
    u16 *lit_walk = lit_sorted + FASTF_TPS_WALK_AT, *dist_walk = lit_walk + FASTF_TPS_WALK_U16(FASTF_TPS_LBITS);
    for (;;) {
        if (bitpos + 3 > in_end) { err |= FASTF_ST_IN_OVERRUN; break; }
        FastfBitReader<32> br;
        br.init(A.comp, A.comp_total, bitpos >> 3, FASTF_FULL_MASK, lane);
        br.drop((u32)(bitpos & 7u));
        const u64 origin = (bitpos >> 3) * 8ull;   // bits consumed are counted from here
        br.refill();
        const u32 last = br.take(1);
        const u32 btype = br.take(2);
        FASTF_PROF(if (lane == 0) atomicAdd(&g_fastf_tps_prof[18], 1ull);)
        if (btype == 3) { err |= FASTF_ST_BAD_BTYPE; break; }
        if (btype == 0) {
            if (pending) return 1;
            br.drop(br.nbits & 7u);
            br.refill();
            const u32 len = br.take(16);
            br.refill();
            const u32 nlen = br.take(16);
            if ((len ^ nlen) != 0xffffu) { err |= FASTF_ST_BAD_STORED; break; }
            if (opos + len > S.isize) { err |= FASTF_ST_OUT_OVERFLOW; break; }
            const u64 consumed = (u64)br.widx * 32u - br.nbits - br.skip_bits;
            const u64 src = (origin + consumed) >> 3;
            if ((src + len) * 8ull > in_end) { err |= FASTF_ST_BAD_STORED; break; }
            for (u32 i = lane; i < len; i += 32) out[opos + i] = A.comp[src + i];
            opos += len;
            bitpos = (src + len) * 8ull;
            if (last) break;   // block complete
            continue;
        }
        u32 hlit = 288, hdist = 32;
        if (btype == 1) {
            for (u32 i = lane; i < 288; i += 32) lens[i] = (u8)(i < 144 ? 8 : (i < 256 ? 9 : (i < 280 ? 7 : 8)));
            if (lane < 32) lens[288 + lane] = 5;
            __syncwarp();
        } else {
            br.refill();
            hlit = br.take(5) + 257;
            hdist = br.take(5) + 1;
            const u32 hclen = br.take(4) + 4;
            if (hlit > 286 || hdist > 30) { err |= FASTF_ST_BAD_CODELENS; break; }
            if (lane < 19) lens[lane] = 0;
            __syncwarp();
            for (u32 i = 0; i < hclen; i++) {
                br.refill();
                const u32 v = br.take(3);
                if (lane == 0) lens[G.cl_order[i]] = (u8)v;
            }
            __syncwarp();
            FASTF_PROF(const long long p_tb = clock64();)
            const u32 clbad = fastf_tps_build(FASTF_ALPHA_PLAIN, lens, 19, nullptr, dist_sorted, S.lit, 7, first, start, lane);
            FASTF_PROF(if (lane == 0) atomicAdd(&g_fastf_tps_prof[19], (u64)(clock64() - p_tb));)
            if (clbad) { err |= FASTF_ST_BAD_CODELENS; break; }
            const u32 n = hlit + hdist;
            u32 i = 0, prev = 0;
            while (i < n) {
                br.refill();
                const u32 e = fastf_tps_decode16(br, S.lit, 7);
                if ((e & 15u) == 0) { err |= FASTF_ST_BAD_CODELENS; break; }
                br.drop(e & 15u);
                const u32 sym = e >> 8;
                u32 rep, val;
                if (sym < 16) { rep = 1; val = sym; prev = sym; }
                else if (sym == 16) { if (i == 0) { err |= FASTF_ST_BAD_CODELENS; break; } rep = 3 + br.take(2); val = prev; }
                else if (sym == 17) { rep = 3 + br.take(3); val = 0; prev = 0; }
                else { rep = 11 + br.take(7); val = 0; prev = 0; }
                if (i + rep > n) { err |= FASTF_ST_BAD_CODELENS; break; }
                for (u32 k = lane; k < rep; k += 32) lens[i + k] = (u8)val;
                i += rep;
            }
            if (err) break;
            __syncwarp();
            if (lens[256] == 0) { err |= FASTF_ST_BAD_CODELENS; break; }
        }
        FASTF_PROF(const long long p_tb = clock64();)
        // the distance lengths sit behind the literal/length ones in `lens`; the literal table's storage was the code-length table
#if FASTF_TPS_SUBTABLES
        if (fastf_tps_build(FASTF_ALPHA_LITLEN, lens, hlit, lit_walk, lit_sorted, S.lit, FASTF_TPS_LBITS, first, start, lane, lit_sorted + 320, FASTF_TPS_LITSUB_U16, G.svc[sw].setup.submax)) { err |= FASTF_ST_BAD_CODELENS; break; }
        if (fastf_tps_build(FASTF_ALPHA_DIST, lens + hlit, hdist, dist_walk, dist_sorted, S.dist, FASTF_TPS_DBITS, first, start, lane, lit_sorted + 320 + 1024, FASTF_TPS_DISTSUB_U16, G.svc[sw].setup.submax)) { err |= FASTF_ST_BAD_CODELENS; break; }
#else
        if (fastf_tps_build(FASTF_ALPHA_LITLEN, lens, hlit, lit_walk, lit_sorted, S.lit, FASTF_TPS_LBITS, first, start, lane)) { err |= FASTF_ST_BAD_CODELENS; break; }
        if (fastf_tps_build(FASTF_ALPHA_DIST, lens + hlit, hdist, dist_walk, dist_sorted, S.dist, FASTF_TPS_DBITS, first, start, lane)) { err |= FASTF_ST_BAD_CODELENS; break; }
#endif
        FASTF_PROF(if (lane == 0) atomicAdd(&g_fastf_tps_prof[19], (u64)(clock64() - p_tb));)
        const u64 consumed = (u64)br.widx * 32u - br.nbits - br.skip_bits;
        bitpos = origin + consumed;
        if (lane == 0) {
            S.bitpos_lo = (u32)bitpos; S.bitpos_hi = (u32)(bitpos >> 32);
            S.last = last; S.pos = opos;
            if (!pending) S.opos = opos;
            __threadfence_block();
            fastf_stv(&S.state, FASTF_TPS_RUN);
        }
        __syncwarp();
        return 0;
    }
    if (pending) return 1;
    // the BGZF block ended inside this routine (stored-only block, or an error)
    if (!err && opos != S.isize) err |= FASTF_ST_SIZE_MISMATCH;
    if (lane == 0) {
        A.status[b] = err;
        S.opos = opos;
        __threadfence_block();
        fastf_stv(&S.state, FASTF_TPS_NEXT);
    }
    __syncwarp();
    return 0;
}

// LZ77 resolution of up to 32 tokens of one stream by a whole warp.  Returns the number of tokens consumed.
__device__ __forceinline__ u32 fastf_tps_copy(const FastfTpsArgs &A, FastfTpsStream &S, u32 rd, u32 n, u32 lane)
{
    u8 *out = A.out + (((u64)S.obase_hi << 32) | S.obase_lo);
    const u32 opos = S.opos;
    u32 tok = (lane < n) ? fastf_ldv(&S.ring[(rd + lane) & (FASTF_TPS_RING - 1u)]) : FASTF_TOK_END;
    // an END token closes the batch (nothing follows it until the stream is set up again)
    const u32 endm = __ballot_sync(FASTF_FULL_MASK, lane < n && (tok >> 30) == 2u);
    u32 ntok = n;
    if (endm) ntok = (u32)__ffs((int)endm) - 1u;
    const bool is_lit = lane < ntok && (tok >> 30) == 0u;
    const bool is_match = lane < ntok && (tok >> 30) == 1u;
    const u32 mylen = is_lit ? ((tok >> 24) & 3u) : (is_match ? (tok & 511u) : 0u);
    // exclusive prefix sum of the output lengths
    u32 inc = mylen;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        u32 t = __shfl_up_sync(FASTF_FULL_MASK, inc, o);
        if ((int)lane >= o) inc += t;
    }
    const u32 off = inc - mylen;
    const u32 total = __shfl_sync(FASTF_FULL_MASK, inc, 31);
    if (is_lit && FASTF_TPS_NOCOPY < 2) {
        out[opos + off] = (u8)tok;
        if (mylen > 1u) out[opos + off + 1u] = (u8)(tok >> 8);
        if (mylen > 2u) out[opos + off + 2u] = (u8)(tok >> 16);
    }
    // Matches.  "Far" ones -- short (<= 32 bytes), non-overlapping (dist >= len) and reading only bytes written before this
    // batch -- depend on nothing in the batch: the source loads of up to FASTF_TPS_FAR of them are issued back to back (one L2
    // round trip for all), then stored.  The rest (long, overlapping, or reading this batch's own output) goes afterwards,
    // one at a time in token order behind a __syncwarp.  A far match never reads what a later-handled one writes, and the
    // bytes a slow match reads lie before its own position, so handling the far ones first preserves the result.
    // (Synthetic 10x BAM: a batch of 32 tokens holds ~10 matches of 12 bytes on average, 9 % longer than 32, 14 % closer than 200.)
    u32 farm, slowm;
    {
        const u32 len = tok & 511u, dist = (tok >> 9) & 0xffffu;
        const bool far = is_match && len <= FASTF_TPS_FAR_LEN && off + len <= dist;   // source ends before the batch starts (implies dist >= len)
        farm = __ballot_sync(FASTF_FULL_MASK, far);
        slowm = __ballot_sync(FASTF_FULL_MASK, is_match && !far);
        if (FASTF_TPS_NOCOPY) farm = slowm = 0;
    }
    __syncwarp();
    while (farm) {
        u32 dpos[FASTF_TPS_FAR], dlen[FASTF_TPS_FAR], dbyte[FASTF_TPS_FAR];
#pragma unroll
        for (int u = 0; u < FASTF_TPS_FAR; u++) {
            dlen[u] = 0; dpos[u] = 0; dbyte[u] = 0;
            if (farm) {
                const u32 m = (u32)__ffs((int)farm) - 1u;
                farm &= farm - 1u;
                const u32 t = __shfl_sync(FASTF_FULL_MASK, tok, (int)m);
                const u32 o = __shfl_sync(FASTF_FULL_MASK, off, (int)m);
                const u32 len = t & 511u, dist = (t >> 9) & 0xffffu;
                dpos[u] = opos + o; dlen[u] = len;
                if (lane < len) dbyte[u] = out[opos + o - dist + lane];
#if FASTF_TPS_FAR_LEN > 32
                if (lane + 32u < len) dbyte[u] |= (u32)out[opos + o - dist + lane + 32u] << 8;
#endif
            }
        }
#pragma unroll
        for (int u = 0; u < FASTF_TPS_FAR; u++) {
            if (lane < dlen[u]) out[dpos[u] + lane] = (u8)dbyte[u];
#if FASTF_TPS_FAR_LEN > 32
            if (lane + 32u < dlen[u]) out[dpos[u] + lane + 32u] = (u8)(dbyte[u] >> 8);
#endif
        }
    }
    while (slowm) {
        const u32 m = (u32)__ffs((int)slowm) - 1u;
        slowm &= slowm - 1u;
        const u32 t = __shfl_sync(FASTF_FULL_MASK, tok, (int)m);
        const u32 o = __shfl_sync(FASTF_FULL_MASK, off, (int)m);
        const u32 len = t & 511u, dist = (t >> 9) & 0xffffu;
        const u32 dst = opos + o;
        __syncwarp();   // everything stored so far in this batch is ordered before these loads
        const u8 *src = out + dst - dist;
        if (dist >= len) {
#if FASTF_TPS_SLOW_UNROLL
            // the source does not overlap the destination: the loads of four 32-byte pieces are issued before any store (a long match
            // costs one round trip, not one per piece -- matches longer than 32 bytes hold a quarter of the output of BAM data)
            for (u32 k = 0; k < len; k += 128) {
                u32 v[4];
#pragma unroll
                for (int u = 0; u < 4; u++) { const u32 j = k + 32u * (u32)u + lane; v[u] = j < len ? src[j] : 0u; }
#pragma unroll
                for (int u = 0; u < 4; u++) { const u32 j = k + 32u * (u32)u + lane; if (j < len) out[dst + j] = (u8)v[u]; }
            }
#else
            for (u32 k = 0; k < len; k += 32) {
                const u32 j = k + lane;
                if (j < len) out[dst + j] = src[j];
            }
#endif
        } else {
            // overlapping copy: the pattern src[0..dist) repeats; j % dist by a reciprocal multiply (exact for j < 258)
            const u32 rcp = (u32)(1048576.0f * __frcp_rn((float)dist)) + 2u;
            for (u32 k = 0; k < len; k += 32) {
                const u32 j = k + lane;
                if (j < len) {
                    const u32 q = (j * rcp) >> 20;
                    u32 r = j - q * dist;
                    if (r >= dist) r += dist;   // q overshoots by at most one
                    out[dst + j] = src[r];
                }
            }
        }
    }
    u32 consumed = ntok;
    u32 new_opos = opos + total;
    if (endm) {
        // END: the decoder's verdict plus the size check; the stream goes back to set-up
        const u32 e = __shfl_sync(FASTF_FULL_MASK, tok, (int)ntok) & 0xffffu;
        if (lane == 0) A.status[S.blk] = e | ((e == 0 && new_opos != S.isize) ? (u32)FASTF_ST_SIZE_MISMATCH : 0u);
        consumed = ntok + 1;
    }
    __syncwarp();   // the stores of this batch are ordered before the next batch's loads
    if (lane == 0) {
        S.opos = new_opos;
        FASTF_SMEM_ORDER();
        fastf_stv(&S.rd, rd + consumed);
    }
    __syncwarp();
    return consumed;
}


// ------------------------------------------------------------------------------------------------------------------
// decoder side (one thread = one stream)
// ------------------------------------------------------------------------------------------------------------------
struct FastfTpsReader {
    const u32 *words;   // the 32-bit word of `comp` that holds the first bit handed to init()
    u64 base_bits;      // its absolute bit offset inside comp (streams may sit anywhere in a buffer of many GB)
    u32 max_words;
    u32 widx;           // words [0, widx) (relative to `words`) are in buf or consumed; nextw = word widx, nextw2 = word widx + 1
    u32 nextw, nextw2;  // two words of prefetch: a second refill right behind the first (length + distance of a match) must not
    u64 buf;            // wait for a load that was only just issued
    u32 nbits;
    __device__ __forceinline__ u32 ldw(u32 i) const { return i < max_words ? __ldg(words + i) : 0u; }
    __device__ __forceinline__ void init(const u8 *comp, u64 comp_total, u64 bitpos)
    {
        const u64 w0 = bitpos >> 5;
        const u32 sh = (u32)(bitpos & 31u);
        words = (const u32 *)comp + w0;
        base_bits = w0 << 5;
        const u64 total_words = comp_total >> 2;
        const u64 left = total_words > w0 ? total_words - w0 : 0;
        max_words = left > 0xffffffffull ? 0xffffffffu : (u32)left;
        buf = (u64)(ldw(0) >> sh);
        nbits = 32u - sh;
        widx = 1;
        nextw = ldw(1);
        nextw2 = FASTF_TPS_PREFETCH2 ? ldw(2) : 0u;
        refill();
    }
    __device__ __forceinline__ void refill()
    {
#if FASTF_TPS_BRANCHFREE >= 2 && !FASTF_TPS_PREFETCH2
        // straight-line form: in a warp of 32 streams some lane refills at nearly every refill point, so nobody gains from jumping
        // over the block, and the branch costs its resolution.  Only the load of the next word stays predicated.
        const bool take_w = nbits <= 32u;
        buf |= take_w ? ((u64)nextw << nbits) : 0ull;
        nbits += take_w ? 32u : 0u;
        widx += take_w ? 1u : 0u;
        if (take_w) nextw = ldw(widx);
#else
        if (nbits <= 32u) {
            buf |= (u64)nextw << nbits;
            nbits += 32u;
            widx++;
#if FASTF_TPS_PREFETCH2
            nextw = nextw2;
            nextw2 = ldw(widx + 1u);
#else
            nextw = ldw(widx);
#endif
        }
#endif
    }
    __device__ __forceinline__ u32 take(u32 n) { u32 v = (u32)buf & ((1u << n) - 1u); buf >>= n; nbits -= n; return v; }
    __device__ __forceinline__ void drop(u32 n) { buf >>= n; nbits -= n; }
    __device__ __forceinline__ u64 bitpos() const { return base_bits + (u64)widx * 32u - nbits; }
};

// Entry of a code longer than the primary table.  lb = the stream's limit / offset array written by fastf_tps_build (global
// scratch): the code's length is TBITS + 1 + the number of length ranges that end at or below the next 15 stream bits.
template <int TBITS>
__device__ __forceinline__ u32 fastf_tps_walk(u64 buf, const u16 *lb, const u16 *sorted, u32 alpha)
{
    constexpr int NL = 15 - TBITS, OFFS = FASTF_TPS_WALK_OFFS(TBITS);
    const u32 code15 = __brev((u32)buf) >> 17;   // the next 15 stream bits, first bit most significant
    const uint2 La = fastf_ld_walk2(lb), Lb = fastf_ld_walk2(lb + 4);
    u32 w[6] = {La.x, La.y, Lb.x, Lb.y, 0xffffffffu, 0xffffffffu};
    if (NL > 8) {
        const uint2 L2 = fastf_ld_walk2(lb + 8);
        w[4] = L2.x; w[5] = L2.y;
    }
    u32 k = 0;
#pragma unroll
    for (int i = 0; i < NL; i++) k += code15 >= ((i & 1) ? (w[i >> 1] >> 16) : (w[i >> 1] & 0xffffu));
    if (k >= (u32)NL) return FASTF_T16_BAD << 4;
    const u32 len = (u32)TBITS + 1u + k;
    const u32 idx = ((code15 >> (15u - len)) + fastf_ld_walk(lb + OFFS + k)) & 0xffffu;
    return fastf_make16(alpha, fastf_ld_sorted(sorted + idx)) | len;
}

template <int TBITS>
__device__ __forceinline__ u32 fastf_tps_long(u32 e, u64 buf, const u16 *lb, const u16 *sorted, const u16 *sub, u32 alpha)
{
#if FASTF_TPS_SUBTABLES
    const u32 b = (e >> 6) & 7u;
    if (b) return fastf_ld_sorted(sub + ((e >> 9) << 3) + ((u32)(buf >> TBITS) & ((1u << b) - 1u)));
#endif
    return fastf_tps_walk<TBITS>(buf, lb, sorted, alpha);
}

template <int L, int SVC>
__global__ void __launch_bounds__(FASTF_TPS_THREADS_OF(L, SVC), 1) fastf_bgzf_inflate_tps_kernel(FastfTpsArgs A)
{
    FASTF_DYN_SMEM(smem);
    FastfTpsStream *streams = reinterpret_cast<FastfTpsStream *>(smem);
    FastfTpsShared &G = *reinterpret_cast<FastfTpsShared *>(smem + sizeof(FastfTpsStream) * FASTF_TPS_STREAMS);
    const u32 warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    u16 *sorted_base = A.sorted + (size_t)blockIdx.x * FASTF_TPS_STREAMS * FASTF_TPS_SORTED_U16;
    // CTA-wide constants and stream control blocks
    if (threadIdx.x < 32) {
        G.lenK[lane] = ((u32)FASTF_LEN_BASE[lane] << 8) | FASTF_LEN_EXTRA[lane];
        G.distK[lane] = ((u32)FASTF_DIST_BASE[lane] << 8) | FASTF_DIST_EXTRA[lane];
        if (lane < 20) G.cl_order[lane] = FASTF_CL_ORDER[lane];
    }
    if (threadIdx.x < FASTF_TPS_STREAMS) {
        FastfTpsStream &S = streams[threadIdx.x];
        S.state = FASTF_TPS_NEXT; S.wr = 0; S.rd = 0; S.last = 0; S.pos = 0; S.isize = 0; S.opos = 0; S.blk = 0;
        FASTF_PROF(g_fastf_tps_handover[blockIdx.x * FASTF_TPS_STREAMS + threadIdx.x] = 0;)
    }
    __syncthreads();

    // The SM's warp arbiter favours higher warp ids; the two decoder warps carry the critical path, so they take the LAST two
    // warp slots of the CTA and the (mostly polling) service warps the lower ones.
    if (warp >= (u32)SVC) {
        // ---------------- decoder: lane = stream ----------------
        if (lane >= (u32)L) return;
        const u32 sidx = (warp - (u32)SVC) * (u32)L + lane;
        FastfTpsStream &S = streams[sidx];
        const u16 *lit_sorted = sorted_base + (size_t)sidx * FASTF_TPS_SORTED_U16, *dist_sorted = lit_sorted + 288;
        FastfTpsReader br;
        bool have = false;
        u32 wr = 0, rd_cache = 0, pos = 0, isize = 0, last = 0;
        u64 in_end = 0;
        const u8 *obase = A.out;
        FASTF_PROF(u32 p_dec = 0; u32 p_full = 0; u32 p_wait = 0; u32 p_long = 0; u32 p_walk = 0; u32 p_waitn = 0; bool p_next = true;
                   u64 p_cbuild = 0; u64 p_cnext = 0; const long long p_t00 = clock64(); long long p_tw = p_t00;)
        for (;;) {
            if (!have) {
                const u32 st = fastf_ldv(&S.state);
                if (st == FASTF_TPS_DONE) break;
                if (st != FASTF_TPS_RUN) { FASTF_PROF(p_wait++; p_waitn += p_next;) fastf_spin_poll(); continue; }
                FASTF_PROF(if (p_next) p_cnext += (u64)(clock64() - p_tw); else p_cbuild += (u64)(clock64() - p_tw);)
                __threadfence_block();
                br.init(A.comp, A.comp_total, ((u64)S.bitpos_hi << 32) | S.bitpos_lo);
                pos = S.pos; isize = S.isize; last = S.last;
                in_end = ((u64)S.inend_hi << 32) | S.inend_lo;
                if (FASTF_TPS_PREFETCH_SRC) obase = A.out + (((u64)S.obase_hi << 32) | S.obase_lo);
                wr = S.wr;
                have = true;
            }
            // a round stores up to FASTF_TPS_TRIPLES + 1 tokens
            if (wr - rd_cache > FASTF_TPS_RING - (FASTF_TPS_TRIPLES + 1u)) {
                rd_cache = fastf_ldv(&S.rd);
                if (wr - rd_cache > FASTF_TPS_RING - (FASTF_TPS_TRIPLES + 1u)) { FASTF_PROF(p_full++;) fastf_stv(&S.wr, wr); fastf_spin_poll(); continue; }
            }
            FASTF_PROF(p_dec++;)
            // ---- one round: up to FASTF_TPS_TRIPLES literal tokens (three literals each) and the match behind them ----
            // Both the literal and the match path of a warp run in every round anyway (some lane always needs each), so a lane
            // walks through both: literals first, then the match that ends the literal run.  Only the first symbol of a round may
            // have a code longer than the primary table (canonical walk); behind it `e` is always a PEEK of the primary table
            // ((e & 63) in 1..15 <=> literal inside the table) that the next step consumes or leaves to the next round.
            // Bit budget: a refill leaves >= 33 bits; 15 + 9 + 9 for the first triple, 27 for each further one, 9 + 5 for a length.
            br.refill();
            u32 e = S.lit[(u32)br.buf & ((1u << FASTF_TPS_LBITS) - 1u)];
            if ((e & 15u) == 0) {
                FASTF_PROF(p_long++; p_walk += ((e >> 6) & 7u) == 0u;)
                e = fastf_tps_long<FASTF_TPS_LBITS>(e, br.buf, lit_sorted + FASTF_TPS_WALK_AT, lit_sorted, lit_sorted + 320, FASTF_ALPHA_LITLEN);
            }
            u32 kind = (e >> 4) & 3u;
            u32 err = 0;
            const u32 wr0 = wr;
            bool end_stream = false, end_block = false;
#if FASTF_TPS_BRANCHFREE
            // The literal run without inner branches: with 32 streams per warp some lane takes every path of a branchy triple in
            // nearly every round, so all lanes walk the longest chain anyway and only pay for resolving the branches.  Every lane does
            // the three look-ups of a triple; a lane whose run has ended drops zero bits and looks the same entry up again.
            if (kind == FASTF_T16_LIT) {
                bool act = true;
#pragma unroll
                for (int triple = 0; triple < FASTF_TPS_TRIPLES; triple++) {
                    br.drop(act ? (e & 15u) : 0u);
                    u32 tok = e >> 8;
                    const u32 e1 = S.lit[(u32)br.buf & ((1u << FASTF_TPS_LBITS) - 1u)];
                    const bool l1 = act && FASTF_T16_IS_TABLE_LIT(e1);
                    br.drop(l1 ? (e1 & 15u) : 0u);
                    tok |= l1 ? (e1 & 0xff00u) : 0u;
                    const u32 e2 = S.lit[(u32)br.buf & ((1u << FASTF_TPS_LBITS) - 1u)];
                    const bool l2 = l1 && FASTF_T16_IS_TABLE_LIT(e2);
                    br.drop(l2 ? (e2 & 15u) : 0u);
                    tok |= l2 ? ((e2 & 0xff00u) << 8) : 0u;
                    const u32 cnt = 1u + (u32)l1 + (u32)l2;
                    br.refill();
                    const u32 e3 = S.lit[(u32)br.buf & ((1u << FASTF_TPS_LBITS) - 1u)];
                    if (act) {
                        if (pos + cnt > isize) { err = FASTF_ST_OUT_OVERFLOW; }   // never hand out bytes beyond the block
                        else {
                            fastf_stv(&S.ring[wr & (FASTF_TPS_RING - 1u)], tok | (cnt << 24));
                            wr++;
                            pos += cnt;
                        }
                        e = e3;
                    }
                    act = act && !err && l2 && FASTF_T16_IS_TABLE_LIT(e3);
                }
                kind = (((e >> 4) & 3u) == FASTF_T16_SYM && !err) ? (u32)FASTF_T16_SYM : 4u;
                if (kind == FASTF_T16_SYM) br.refill();
            }
#else
            if (kind == FASTF_T16_LIT) {
#pragma unroll
                for (int triple = 0; triple < FASTF_TPS_TRIPLES; triple++) {
                    br.drop(e & 15u);
                    u32 tok = e >> 8, cnt = 1;
                    e = S.lit[(u32)br.buf & ((1u << FASTF_TPS_LBITS) - 1u)];
                    if (FASTF_T16_IS_TABLE_LIT(e)) {
                        br.drop(e & 15u);
                        tok |= e & 0xff00u;
                        cnt = 2;
                        e = S.lit[(u32)br.buf & ((1u << FASTF_TPS_LBITS) - 1u)];
                        if (FASTF_T16_IS_TABLE_LIT(e)) {
                            br.drop(e & 15u);
                            tok |= (e & 0xff00u) << 8;
                            cnt = 3;
                            br.refill();
                            e = S.lit[(u32)br.buf & ((1u << FASTF_TPS_LBITS) - 1u)];
                        }
                    }
                    if (pos + cnt > isize) { err = FASTF_ST_OUT_OVERFLOW; break; }   // never hand out bytes beyond the block
                    fastf_stv(&S.ring[wr & (FASTF_TPS_RING - 1u)], tok | (cnt << 24));
                    wr++;
                    pos += cnt;
                    if (cnt < 3u || !FASTF_T16_IS_TABLE_LIT(e)) break;
                }
                // what follows the literals: a length code inside the table joins this round, anything else waits for the next
                kind = (((e >> 4) & 3u) == FASTF_T16_SYM && !err) ? (u32)FASTF_T16_SYM : 4u;
                if (kind == FASTF_T16_SYM) br.refill();
            }
#endif
            if (kind == FASTF_T16_SYM) {
                br.drop(e & 15u);
                const u32 K = G.lenK[e >> 8];
                const u32 len = (K >> 8) + br.take(K & 255u);
                br.refill();
                u32 d = S.dist[(u32)br.buf & ((1u << FASTF_TPS_DBITS) - 1u)];
                if ((d & 15u) == 0) {
                    FASTF_PROF(p_long++; p_walk += ((d >> 6) & 7u) == 0u;)
                    d = fastf_tps_long<FASTF_TPS_DBITS>(d, br.buf, lit_sorted + FASTF_TPS_WALK_AT + FASTF_TPS_WALK_U16(FASTF_TPS_LBITS), dist_sorted, lit_sorted + 320 + 1024, FASTF_ALPHA_DIST);
                }
                if (((d >> 4) & 3u) != FASTF_T16_SYM) err = FASTF_ST_BAD_SYMBOL;
                else {
                    br.drop(d & 15u);
                    const u32 K2 = G.distK[d >> 8];
                    const u32 dist = (K2 >> 8) + br.take(K2 & 255u);
                    if (dist > pos) err = FASTF_ST_BAD_DISTANCE;
                    else if (pos + len > isize) err = FASTF_ST_OUT_OVERFLOW;
                    else {
                        fastf_stv(&S.ring[wr & (FASTF_TPS_RING - 1u)], FASTF_TOK_MATCH | len | (dist << 9));
                        if (FASTF_TPS_PREFETCH_SRC && dist >= FASTF_TPS_PREFETCH_SRC) fastf_prefetch_l2(obase + pos - dist);
                        wr++;
                        pos += len;
                    }
                }
            } else if (kind == FASTF_T16_EOB) {
                br.drop(e & 15u);
                end_block = true;
                if (last) end_stream = true;
            } else if (kind == FASTF_T16_BAD) {
                err = FASTF_ST_BAD_SYMBOL;
            }
            if (err) { end_stream = true; end_block = true; }
            if (!end_block) {
                if ((wr ^ wr0) & ~7u) { FASTF_SMEM_ORDER(); fastf_stv(&S.wr, wr); }   // publish whenever a multiple of 8 is crossed
                continue;
            }
            // ---- end of a deflate block: hand the stream to its service warp ----
            const u64 bp = br.bitpos();
            if (end_stream) {
                if (!err && bp > in_end) err = FASTF_ST_IN_OVERRUN;
                if (!err && pos != isize) err = FASTF_ST_SIZE_MISMATCH;
                S.ring[wr & (FASTF_TPS_RING - 1u)] = FASTF_TOK_END | err;
                wr++;
            }
            S.bitpos_lo = (u32)bp; S.bitpos_hi = (u32)(bp >> 32);
            S.pos = pos;
            FASTF_PROF(p_next = end_stream; p_tw = clock64(); g_fastf_tps_handover[blockIdx.x * FASTF_TPS_STREAMS + sidx] = (u64)p_tw;)
            __threadfence_block();
            fastf_stv(&S.wr, wr);
            __threadfence_block();
            fastf_stv(&S.state, end_stream ? (u32)FASTF_TPS_NEXT : (u32)FASTF_TPS_BUILD);
            have = false;
        }
#if FASTF_TPS_PROF
        atomicAdd(&g_fastf_tps_prof[0], (unsigned long long)p_dec); atomicAdd(&g_fastf_tps_prof[1], (unsigned long long)p_full); atomicAdd(&g_fastf_tps_prof[2], (unsigned long long)p_wait);
        atomicAdd(&g_fastf_tps_prof[11], (unsigned long long)p_long); atomicAdd(&g_fastf_tps_prof[12], (unsigned long long)p_walk);
        atomicAdd(&g_fastf_tps_prof[13], (unsigned long long)p_waitn); atomicAdd(&g_fastf_tps_prof[14], p_cbuild); atomicAdd(&g_fastf_tps_prof[15], p_cnext);
        atomicAdd(&g_fastf_tps_prof[16], (u64)(clock64() - p_t00));
#endif
    } else {
        // ---------------- service: lock-step warp, owns the streams sw, sw + SVC, sw + 2 SVC, ... ----------------
        // One poll pass costs a handful of instructions: lane k looks at the control block of the k-th stream of this warp, a
        // ballot collects the streams that need something, and only those are visited.  (A pass that walked the streams one
        // after the other was half of all instructions the SM issued.)
        const u32 sw = warp;
        constexpr u32 NPER = (FASTF_TPS_STREAMS + SVC - 1) / SVC;
        static_assert(NPER <= 32, "one lane per owned stream");
        // a service warp owns NPER consecutive streams: lane k polls stream sw * NPER + k (neighbouring structures, distinct banks)
        constexpr u32 Q = FASTF_TPS_STREAMS / SVC, R = FASTF_TPS_STREAMS % SVC;
        const u32 first_sidx = sw * Q + (sw < R ? sw : R), n_mine = Q + (sw < R ? 1u : 0u);
        const u32 my_sidx = first_sidx + lane;
        const bool mine = lane < n_mine;
        // The poll pass is the hottest loop of the service side (one pass per batch on average), so it is written to stay at a
        // dozen instructions: the address of the control block is made opaque to the compiler (it recomputed it from the thread
        // index in every pass otherwise), and the states are numbered so that "needs service" is one test -- NEXT and BUILD (even)
        // always do, RUN and DONE (odd) only with a batch of tokens waiting (DONE never has one).
        static_assert((FASTF_TPS_NEXT & 1) == 0 && (FASTF_TPS_BUILD & 1) == 0 && (FASTF_TPS_RUN & 1) == 1 && (FASTF_TPS_DONE & 1) == 1, "state parity");
        const fastf_ctl_ptr ctl = fastf_ctl_of(&streams[mine ? my_sidx : first_sidx].state);
        FASTF_PROF(u64 p_pass = 0; u64 p_empty = 0; u64 p_ccopy = 0; u64 p_csetup = 0; u64 p_cempty = 0; u64 p_batches = 0; u64 p_tokens = 0; const long long p_t00 = clock64();)
        for (;;) {
            FASTF_PROF(const long long p_t0 = clock64(); p_pass++;)
            const u32 st = fastf_ctl_ld(ctl, 0);  // volatile shared-memory reads stay in program order: once the state says the
            const u32 wr = fastf_ctl_ld(ctl, 1);  // decoder handed the stream over, wr is final
            const u32 rd = fastf_ctl_ld(ctl, 2);
            const u32 avail = wr - rd;
            const bool need = mine && (((st & 1u) == 0) || avail >= FASTF_TPS_BATCH_MIN);
            u32 m = __ballot_sync(FASTF_FULL_MASK, need);
            if (!m) {
                if (__ballot_sync(FASTF_FULL_MASK, mine && st != FASTF_TPS_DONE) == 0) break;
                fastf_spin_pause();   // nothing to copy or set up: leave the issue slots to the decoders
                FASTF_PROF(p_empty++; p_cempty += (u64)(clock64() - p_t0);)
                continue;
            }
            // Streams whose decoder waits (set-up, or the drain of an ended BGZF block) go first: a stream with a partly full ring
            // still decodes.  A BUILD hand-over is set up at once, its tokens stay in the ring; a NEXT hand-over drains first, because
            // the copy side still reads the old block's blk / isize / obase.
            u32 rest = m & ~__ballot_sync(FASTF_FULL_MASK, mine && (st & 1u) == 0);
            m &= ~rest;
            const u32 work = st == FASTF_TPS_BUILD ? 3u : (avail ? 1u : 2u);
            while (m | rest) {
                if (!m) { m = rest; rest = 0; }
                const u32 k = (u32)__ffs((int)m) - 1u;
                m &= m - 1u;
                const u32 w = __shfl_sync(FASTF_FULL_MASK, work, (int)k);
                const u32 krd = __shfl_sync(FASTF_FULL_MASK, rd, (int)k);
                const u32 kav = __shfl_sync(FASTF_FULL_MASK, avail, (int)k);
                const u32 sidx = first_sidx + k;
                FastfTpsStream &S = streams[sidx];
                u16 *ssorted = sorted_base + (size_t)sidx * FASTF_TPS_SORTED_U16;
                FASTF_PROF(const long long p_t1 = clock64();)
                if (w == 1) {
                    FASTF_PROF(p_batches++; p_tokens += kav < 32u ? kav : 32u;)
                    fastf_tps_copy(A, S, krd, kav < 32u ? kav : 32u, lane);
                } else if (w == 2) {
                    // fetch the next BGZF block for this stream
                    FASTF_PROF(if (lane == 0) fastf_tps_prof_handover(sidx, 22);)
                    u32 b = 0;
                    if (lane == 0) b = atomicAdd(A.next_block, 1u);
                    b = __shfl_sync(FASTF_FULL_MASK, b, 0);
                    if (b >= A.nblocks) {
                        if (lane == 0) fastf_stv(&S.state, FASTF_TPS_DONE);
                        __syncwarp();
                    } else {
                        if (lane == 0) {
                            const u64 bp = A.in_off[b] * 8ull, be = (A.in_off[b] + A.in_len[b]) * 8ull, ob = A.out_off[b];
                            S.blk = b; S.isize = A.isize[b]; S.opos = 0; S.pos = 0;
                            S.bitpos_lo = (u32)bp; S.bitpos_hi = (u32)(bp >> 32);
                            S.inend_lo = (u32)be; S.inend_hi = (u32)(be >> 32);
                            S.obase_lo = (u32)ob; S.obase_hi = (u32)(ob >> 32);
                        }
                        FASTF_PROF(if (lane == 0) atomicAdd(&g_fastf_tps_prof[17], 1ull);)
                        __syncwarp();
                        fastf_tps_setup(A, S, ssorted, G, sw, lane, false);
                    }
                } else {
                    FASTF_PROF(if (lane == 0) fastf_tps_prof_handover(sidx, 20);)
                    const u32 later = fastf_tps_setup(A, S, ssorted, G, sw, lane, kav != 0);
                    FASTF_PROF(if (lane == 0 && kav) { atomicAdd(&g_fastf_tps_prof[24], 1ull); atomicAdd(&g_fastf_tps_prof[25], (unsigned long long)later); })
                    if (later) fastf_tps_copy(A, S, krd, kav < 32u ? kav : 32u, lane);   // drain, then set up again
                }
                FASTF_PROF(if (w == 1) p_ccopy += (u64)(clock64() - p_t1); else p_csetup += (u64)(clock64() - p_t1);)
            }
        }
#if FASTF_TPS_PROF
        if (lane == 0) {
            atomicAdd(&g_fastf_tps_prof[3], p_pass); atomicAdd(&g_fastf_tps_prof[4], p_empty); atomicAdd(&g_fastf_tps_prof[5], p_ccopy);
            atomicAdd(&g_fastf_tps_prof[6], p_csetup); atomicAdd(&g_fastf_tps_prof[7], p_cempty); atomicAdd(&g_fastf_tps_prof[8], p_batches);
            atomicAdd(&g_fastf_tps_prof[9], p_tokens); atomicAdd(&g_fastf_tps_prof[10], (u64)(clock64() - p_t00));
        }
#endif
    }
}
