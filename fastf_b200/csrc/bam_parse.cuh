// K2 -- BAM record-boundary scan + warp-cooperative aux-tag parse.
//
// Replaces, for every record, htslib's sam_read1 framing and the reference's per-read tag logic:
//   bam_aux_get/bam_aux2Z("CB") + hash_table_lookup(ht_cell)      reference src/bam2db_ds.c:366-382
//   bam_aux_get/bam_aux2i("xf") in {25,17}                         reference src/bam2db_ds.c:394-400
//   bam_aux_get/bam_aux2Z("GX") + hash_table_lookup(ht_feature)   reference src/bam2db_ds.c:403-411
//   bam_aux_get/bam_aux2Z("UB") + encode_DNA                       reference src/bam2db_ds.c:412-419, 5-51
// Aux layout and htslib semantics (first matching tag wins; Z/H only for strings; c C s S i I for ints;
// a malformed field hides every tag at or after it) are from the SAM/BAM specification, section 4.2.4.
//
// Mapping: one warp per BGZF block.  htslib writers never split a record across BGZF blocks, so a
// block starts on a record boundary; the warp walks the block_size chain (the walk must end exactly
// at ISIZE, otherwise FASTF_ST_REC_STRADDLE is raised and the host falls back).  All lanes keep the
// same cursor; string scans (NUL search), hashing, table compares and the 2-bit UMI packing are done
// one byte per lane with ballots / redux.  The kernel emits, per block, the record count, the number
// of "CB-valid" records (the ones that consume an MT19937 draw) and one packed u64 candidate per
// CB-valid record, in file order, into a per-block staging slice.  A later prefix sum over the
// per-block counts yields the global read ordinal (= MT draw index) of every candidate.
#pragma once
#include "common.cuh"
#include "strtable.h"

struct FastfKeyLayout {
    u32 umi_max_bytes;   // 1..4 -> UMIs up to 4*umi_max_bytes bases
    u32 bits_umi;        // 1 (non-NULL flag) + 8*umi_max_bytes + 3 (blob length)
    u32 bits_gene;
    u32 bits_cell;       // bits_cell + bits_gene + bits_umi <= 63
};

#ifndef FASTF_EMU
__device__ __forceinline__ void fastf_prefetch_l1(const void *p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
#else
inline void fastf_prefetch_l1(const void *) {}
#endif

// Byte accessors over the inflated stream: the shared-memory window of the current warp (normal case) or
// global memory (records larger than the window).  off is an offset into the chunk's inflated buffer.
struct FastfWinAcc {
    const u8 *W;
    u64 wbase;   // multiple of 16
    __device__ __forceinline__ u32 byte(u64 off) const { return W[off - wbase]; }
    // the aligned 32-bit word that holds byte `off` (off rounded down to a multiple of 4)
    __device__ __forceinline__ u32 word(u64 off) const { return *reinterpret_cast<const u32 *>(W + ((off - wbase) & ~3ull)); }
};
struct FastfGlobAcc {
    const u8 *infl;   // 16-byte aligned base
    __device__ __forceinline__ u32 byte(u64 off) const { return infl[off]; }
    __device__ __forceinline__ u32 word(u64 off) const { return *reinterpret_cast<const u32 *>(infl + (off & ~3ull)); }
};
// position of the first NUL byte in [s, rend), or rend if there is none: four bytes per load
template <class Acc> __device__ __forceinline__ u64 fastf_find_nul(const Acc &A, u64 s, u64 rend)
{
    while (s < rend) {
        const u64 a = s & ~3ull;
        u32 w = A.word(s);
        w |= (1u << (8u * (u32)(s & 3ull))) - 1u;               // bytes in front of s do not count
        const u32 z = (w - 0x01010101u) & ~w & 0x80808080u;     // 0x80 in every byte that is zero
        if (z) {
            const u64 p = a + (((u32)__ffs((int)z) - 1u) >> 3);
            return p < rend ? p : rend;
        }
        s = a + 4;
    }
    return rend;
}
// the four bytes at off .. off+3 (any alignment), all of which must be readable: two aligned word loads instead of four byte loads
template <class Acc> __device__ __forceinline__ u32 fastf_acc_4bytes(const Acc &A, u64 off)
{
    const u32 sh = 8u * (u32)(off & 3ull);
    const u32 lo = A.word(off);
    if (sh == 0) return lo;
    return (lo >> sh) | (A.word(off + 3) << (32u - sh));
}
// little-endian 16 / 32-bit values at any alignment out of aligned word loads (the words that hold the bytes asked for, nothing beyond)
template <class Acc> __device__ __forceinline__ u32 fastf_acc_u16(const Acc &A, u64 off)
{
    const u32 sh = 8u * (u32)(off & 3ull);
    const u32 lo = A.word(off) >> sh;
    return (sh == 24u ? (lo | (A.word(off + 1) << 8)) : lo) & 0xffffu;
}
template <class Acc> __device__ __forceinline__ u32 fastf_acc_u32(const Acc &A, u64 off) { return fastf_acc_4bytes(A, off); }

// warp-cooperative lookup of the len bytes at offset s in a string table; every lane gets the value (0 = absent)
template <class Acc>
__device__ __forceinline__ u32 fastf_table_lookup(const FastfStrTableView &T, u32 my_pw1, u32 my_pw2, const Acc &A, u64 s, u32 len, u32 lane)
{
    u32 h1 = 0, h2 = 0;
    u32 c = 0;
    do {
        u32 i = c + lane;
        u32 byte = (i < len) ? A.byte(s + i) + 1u : 0u;
        u32 s1 = __reduce_add_sync(FASTF_FULL_MASK, byte * my_pw1);
        u32 s2 = __reduce_add_sync(FASTF_FULL_MASK, byte * my_pw2);
        h1 = h1 * FASTF_H1_Q + s1;
        h2 = h2 * FASTF_H2_Q + s2;
        c += 32;
    } while (c < len);
    u32 slot = fastf_hash_finalize(h1) & T.mask;
    for (;;) {
        FastfStrSlot e = T.slots[slot];
        if (e.value == 0) return 0;
        if (e.tag == h2 && e.len == len) {
            bool same = true;
            for (u32 c2 = 0; c2 < len; c2 += 32) {
                u32 i = c2 + lane;
                bool ok = (i >= len) || (A.byte(s + i) == T.pool[e.off + i]);
                same = same && __all_sync(FASTF_FULL_MASK, ok);
            }
            if (same) return e.value;
        }
        slot = (slot + 1) & T.mask;
    }
}

struct FastfAuxHit { u64 off; u32 len; u32 type; };   // off = offset of the value inside the inflated buffer

#define FASTF_PARSE_WARPS 4
#define FASTF_PARSE_WIN 2048   // bytes of the block staged in shared memory per warp

// BAM header walk (what sam_hdr_read does at reference src/bam2db_ds.c:340): "BAM\1", l_text, text, n_ref,
// (l_name, name, l_ref) x n_ref.  One thread; writes the inflated offset of the first alignment record.
__global__ void fastf_bam_header_kernel(const u8 *__restrict__ infl, u64 n, u64 *__restrict__ first_record_off, u32 *__restrict__ status)
{
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    *first_record_off = n;
    if (n < 12 || infl[0] != 'B' || infl[1] != 'A' || infl[2] != 'M' || infl[3] != 1) { *status |= FASTF_ST_BAD_HEADER; return; }
    u64 p = 8ull + (u64)fastf_ld_u32(infl + 4);
    if (p + 4 > n) { *status |= FASTF_ST_BAD_HEADER; return; }
    const u32 n_ref = fastf_ld_u32(infl + p);
    p += 4;
    for (u32 i = 0; i < n_ref; i++) {
        if (p + 4 > n) { *status |= FASTF_ST_BAD_HEADER; return; }
        p += 8ull + (u64)fastf_ld_u32(infl + p);
    }
    if (p > n) { *status |= FASTF_ST_BAD_HEADER; return; }
    *first_record_off = p;
}

// One alignment record [rec, rend) (after its block_size word): the reference's per-read decision up to the draw.
// Returns 0 = not CB-valid (no candidate), 1 = candidate with *key set.  A candidate that would not be inserted is FASTF_INVALID_KEY,
// or with KEEP_CELL (the cell-rate grid, whose union table is remapped per cell rate later) its cell alone: cidx << (bits_gene +
// bits_umi), gene field 0, which no insertable key has (feature indices start at 1).
template <bool KEEP_CELL, class Acc>
__device__ __forceinline__ u32 fastf_parse_record(const Acc &A, u64 rec, u64 rend, u32 bs, const FastfStrTableView &cells, const FastfStrTableView &genes, const FastfKeyLayout &L,
                                                  u32 c_pw1, u32 c_pw2, u32 g_pw1, u32 g_pw2, u32 lane, u32 *status, u64 *key_out)
{
    const u32 l_read_name = A.byte(rec + 8);
    const u32 n_cigar = fastf_acc_u16(A, rec + 12);
    const i32 l_seq = (i32)fastf_acc_u32(A, rec + 16);
    const i64 aoff = 32 + (i64)l_read_name + 4 * (i64)n_cigar + (((i64)l_seq + 1) >> 1) + (i64)l_seq;
    if (l_seq < 0 || aoff > (i64)bs) { *status |= FASTF_ST_REC_CORRUPT; return 2; }

    // ---- aux walk: find the first CB, xf, GX, UB ----
    FastfAuxHit cb = {0, 0, 0}, xf = {0, 0, 0}, gx = {0, 0, 0}, ub = {0, 0, 0};
    u32 found = 0;
    u64 q = rec + (u64)aoff;
    while (rend - q >= 3 && found != 15u) {
        u32 t0, t1, ty;
        if (rend - q >= 4) { const u32 hd = fastf_acc_4bytes(A, q); t0 = hd & 255u; t1 = (hd >> 8) & 255u; ty = (hd >> 16) & 255u; }
        else { t0 = A.byte(q); t1 = A.byte(q + 1); ty = A.byte(q + 2); }
        const u64 v = q + 3;
        u64 next;
        u32 vlen = 0;
        if (ty == 'Z' || ty == 'H') {
            bool term = false;
            u64 s = v;
            while (s < rend) {
                u64 i = s + lane;
                bool z = (i < rend) && (A.byte(i) == 0);
                u32 m = __ballot_sync(FASTF_FULL_MASK, z);
                if (m) { s += (u32)__ffs((int)m) - 1u; term = true; break; }
                s += 32;
            }
            if (!term) break;   // htslib: a malformed field hides this and every later tag; not a failure
            vlen = (u32)(s - v);
            next = s + 1;
        } else {
            u64 sz;
            switch (ty) {
            case 'A': case 'c': case 'C': sz = 1; break;
            case 's': case 'S': sz = 2; break;
            case 'i': case 'I': case 'f': sz = 4; break;
            case 'd': sz = 8; break;
            case 'B': {
                if (rend - v < 5) { sz = ~0ull; break; }
                u32 sub = A.byte(v);
                u64 cnt = fastf_acc_u32(A, v + 1);
                u64 es = (sub == 'c' || sub == 'C') ? 1 : (sub == 's' || sub == 'S') ? 2 : (sub == 'i' || sub == 'I' || sub == 'f') ? 4 : 0;
                sz = es ? 5 + es * cnt : ~0ull;
                break;
            }
            default: sz = ~0ull;
            }
            if (sz == ~0ull || sz > rend - v) break;
            next = v + sz;
        }
        if (t0 == 'C' && t1 == 'B' && !(found & 1u)) { cb.off = v; cb.len = vlen; cb.type = ty; found |= 1u; }
        else if (t0 == 'x' && t1 == 'f' && !(found & 2u)) { xf.off = v; xf.type = ty; found |= 2u; }
        else if (t0 == 'G' && t1 == 'X' && !(found & 4u)) { gx.off = v; gx.len = vlen; gx.type = ty; found |= 4u; }
        else if (t0 == 'U' && t1 == 'B' && !(found & 8u)) { ub.off = v; ub.len = vlen; ub.type = ty; found |= 8u; }
        q = next;
    }

    // ---- CB gate: present, string-typed, in the sampled-cell table ----
    if (!(found & 1u) || !(cb.type == 'Z' || cb.type == 'H')) return 0;
    const u32 cidx = fastf_table_lookup(cells, c_pw1, c_pw2, A, cb.off, cb.len, lane);
    if (cidx == 0) return 0;

    // ---- this record consumes a draw; decide whether it would be inserted if kept ----
    u64 key = KEEP_CELL ? (u64)cidx << (L.bits_gene + L.bits_umi) : FASTF_INVALID_KEY;
    i64 xfv = 0;
    if (found & 2u) {
        const u64 x = xf.off;
        switch (xf.type) {
        case 'c': xfv = (i64)(int8_t)A.byte(x); break;
        case 'C': xfv = A.byte(x); break;
        case 's': xfv = (i64)(int16_t)fastf_acc_u16(A, x); break;
        case 'S': xfv = fastf_acc_u16(A, x); break;
        case 'i': xfv = (i64)(i32)fastf_acc_u32(A, x); break;
        case 'I': xfv = fastf_acc_u32(A, x); break;
        default: xfv = 0;
        }
    }
    const int xfi = (int)xfv;   // the reference stores bam_aux2i() in an int
    if ((xfi == 25 || xfi == 17) && (found & 4u) && (gx.type == 'Z' || gx.type == 'H') && (found & 8u) && (ub.type == 'Z' || ub.type == 'H')) {
        const u32 gidx = fastf_table_lookup(genes, g_pw1, g_pw2, A, gx.off, gx.len, lane);
        if (gidx != 0) {
            if (ub.len > 4u * L.umi_max_bytes) {
                *status |= FASTF_ST_UMI_TOO_LONG;
            } else {
                u32 code = 0, badbase = 0;
                if (lane < ub.len) {
                    u32 ch = A.byte(ub.off + lane);
                    code = ch == 'A' ? 0u : ch == 'C' ? 1u : ch == 'G' ? 2u : ch == 'T' ? 3u : 4u;
                    badbase = code > 3u;
                }
                u32 hi = __reduce_or_sync(FASTF_FULL_MASK, (lane < 16u && !badbase) ? (code << (30u - 2u * lane)) : 0u);
                u32 anybad = __any_sync(FASTF_FULL_MASK, badbase);
                u64 ucode = 0;   // SQL NULL
                if (!anybad) {
                    u64 content = (u64)(hi >> (32u - 8u * L.umi_max_bytes));
                    u64 nbytes = (ub.len + 3u) >> 2;
                    ucode = (1ull << (L.bits_umi - 1u)) | (content << 3) | nbytes;
                }
                key = ((u64)cidx << (L.bits_gene + L.bits_umi)) | ((u64)gidx << L.bits_umi) | ucode;
            }
        }
    }
    *key_out = key;
    return 1;
}

// ---- thread-per-record variant (no warp collectives): lane i of the warp walks record i of the staged batch ----
// Everything a lane touches lies in its warp's shared-memory window, so positions are 32-bit offsets from the start of the window:
// the 64-bit stream offsets of the generic accessors doubled the address arithmetic of what is an instruction-bound kernel.
struct FastfWin32 {
    const u8 *W;   // 16-byte aligned; readable FASTF_PARSE_PAD bytes beyond the staged bytes
    __device__ __forceinline__ u32 byte(u32 o) const { return W[o]; }
    __device__ __forceinline__ u32 word(u32 o) const { return *reinterpret_cast<const u32 *>(W + (o & ~3u)); }
    // the four bytes at o .. o+3, any alignment: two aligned words and a funnel shift (an aligned o reads the same word twice)
    __device__ __forceinline__ u32 bytes4(u32 o) const
    {
        const u32 lo = word(o), hi = word(o + 3u), sh = 8u * (o & 3u);
#ifdef FASTF_EMU
        return sh ? (lo >> sh) | (hi << (32u - sh)) : lo;
#else
        return __funnelshift_r(lo, hi, sh);
#endif
    }
    __device__ __forceinline__ u32 u16at(u32 o) const { return bytes4(o) & 0xffffu; }
};
#define FASTF_PARSE_PAD 16u
// position of the first NUL byte in [s, rend), or rend if there is none: four bytes per load
__device__ __forceinline__ u32 fastf_find_nul32(const FastfWin32 &A, u32 s, u32 rend)
{
    u32 a = s & ~3u;
    u32 w = A.word(a) | ((1u << (8u * (s & 3u))) - 1u);   // bytes in front of s do not count
    for (;;) {
        const u32 z = (w - 0x01010101u) & ~w & 0x80808080u;   // 0x80 in every byte that is zero
        if (z) {
            const u32 p = a + (((u32)__ffs((int)z) - 1u) >> 3);
            return p < rend ? p : rend;
        }
        a += 4u;
        if (a >= rend) return rend;
        w = A.word(a);
    }
}
__device__ __forceinline__ u32 fastf_table_lookup_lane(const FastfStrTableView &T, const FastfWin32 &A, u32 s, u32 len)
{
    u32 h1 = 0, h2 = 0;
    u32 c = 0;
    do {
        u32 s1 = 0, s2 = 0;
        const u32 m = len - c < 32u ? len - c : 32u;
        for (u32 j = 0; j < m; j++) {
            const u32 byte = A.byte(s + c + j) + 1u;
            s1 += byte * T.pw1[j];
            s2 += byte * T.pw2[j];
        }
        h1 = h1 * FASTF_H1_Q + s1;
        h2 = h2 * FASTF_H2_Q + s2;
        c += 32;
    } while (c < len);
    u32 slot = fastf_hash_finalize(h1) & T.mask;
    for (;;) {
        const uint4 raw = *reinterpret_cast<const uint4 *>(&T.slots[slot]);   // {tag, off, len, value}
        if (raw.w == 0) return 0;
        if (raw.x == h2 && raw.z == len) {
            // pool strings start on 4-byte boundaries (FastfStrTableHost::insert): compare word-wise
            const u32 *pw = reinterpret_cast<const u32 *>(T.pool + raw.y);
            bool same = true;
            u32 i = 0;
            for (; i + 4 <= len && same; i += 4) same = pw[i >> 2] == A.bytes4(s + i);
            if (same && i < len) {
                const u32 keep = (1u << (8u * (len - i))) - 1u;   // 1..3 trailing bytes
                same = ((pw[i >> 2] ^ A.bytes4(s + i)) & keep) == 0;
            }
            if (same) return raw.w;
        }
        slot = (slot + 1) & T.mask;
    }
}

// scalar twin of fastf_parse_record (same decisions, one thread); rec / rend are offsets into the window, bs = rend - rec
template <bool KEEP_CELL>
__device__ __forceinline__ u32 fastf_parse_record_lane(const FastfWin32 &A, u32 rec, u32 rend, u32 bs, const FastfStrTableView &cells, const FastfStrTableView &genes, const FastfKeyLayout &L,
                                                       u32 *status, u64 *key_out)
{
    const u32 l_read_name = A.byte(rec + 8u);
    const u32 n_cigar = A.u16at(rec + 12u);
    const i32 l_seq = (i32)A.bytes4(rec + 16u);
    const i64 aoff = 32 + (i64)l_read_name + 4 * (i64)n_cigar + (((i64)l_seq + 1) >> 1) + (i64)l_seq;
    if (l_seq < 0 || aoff > (i64)bs) { *status |= FASTF_ST_REC_CORRUPT; return 2; }
    u32 cb_off = 0, cb_len = 0, cb_type = 0, xf_off = 0, xf_type = 0, gx_off = 0, gx_len = 0, gx_type = 0, ub_off = 0, ub_len = 0, ub_type = 0;
    u32 found = 0;
    u32 q = rec + (u32)aoff;
    while (rend - q >= 3u && found != 15u) {
        const u32 hd = A.bytes4(q);   // tag, tag, type (+ one byte that may lie behind the record: read, not used)
        const u32 tag = hd & 0xffffu, ty = (hd >> 16) & 255u;
        const u32 v = q + 3u;
        u32 next, vlen = 0;
        if (ty == 'Z' || ty == 'H') {
            const u32 s = fastf_find_nul32(A, v, rend);
            if (s >= rend) break;   // unterminated: this and every later tag is invisible (htslib)
            vlen = s - v;
            next = s + 1u;
        } else {
            u64 sz;
            switch (ty) {
            case 'A': case 'c': case 'C': sz = 1; break;
            case 's': case 'S': sz = 2; break;
            case 'i': case 'I': case 'f': sz = 4; break;
            case 'd': sz = 8; break;
            case 'B': {
                if (rend - v < 5u) { sz = ~0ull; break; }
                const u32 sub = A.byte(v);
                const u64 cnt = A.bytes4(v + 1u);
                const u64 es = (sub == 'c' || sub == 'C') ? 1 : (sub == 's' || sub == 'S') ? 2 : (sub == 'i' || sub == 'I' || sub == 'f') ? 4 : 0;
                sz = es ? 5 + es * cnt : ~0ull;
                break;
            }
            default: sz = ~0ull;
            }
            if (sz == ~0ull || sz > (u64)(rend - v)) break;
            next = v + (u32)sz;
        }
        if (tag == ('C' | ('B' << 8)) && !(found & 1u)) { cb_off = v; cb_len = vlen; cb_type = ty; found |= 1u; }
        else if (tag == ('x' | ('f' << 8)) && !(found & 2u)) { xf_off = v; xf_type = ty; found |= 2u; }
        else if (tag == ('G' | ('X' << 8)) && !(found & 4u)) { gx_off = v; gx_len = vlen; gx_type = ty; found |= 4u; }
        else if (tag == ('U' | ('B' << 8)) && !(found & 8u)) { ub_off = v; ub_len = vlen; ub_type = ty; found |= 8u; }
        q = next;
    }
    if (!(found & 1u) || !(cb_type == 'Z' || cb_type == 'H')) return 0;
    const u32 cidx = fastf_table_lookup_lane(cells, A, cb_off, cb_len);
    if (cidx == 0) return 0;
    u64 key = KEEP_CELL ? (u64)cidx << (L.bits_gene + L.bits_umi) : FASTF_INVALID_KEY;
    i64 xfv = 0;
    if (found & 2u) {
        const u32 x = xf_off;
        switch (xf_type) {
        case 'c': xfv = (i64)(int8_t)A.byte(x); break;
        case 'C': xfv = A.byte(x); break;
        case 's': xfv = (i64)(int16_t)A.u16at(x); break;
        case 'S': xfv = A.u16at(x); break;
        case 'i': xfv = (i64)(i32)A.bytes4(x); break;
        case 'I': xfv = A.bytes4(x); break;
        default: xfv = 0;
        }
    }
    const int xfi = (int)xfv;   // the reference stores bam_aux2i() in an int
    if ((xfi == 25 || xfi == 17) && (found & 4u) && (gx_type == 'Z' || gx_type == 'H') && (found & 8u) && (ub_type == 'Z' || ub_type == 'H')) {
        const u32 gidx = fastf_table_lookup_lane(genes, A, gx_off, gx_len);
        if (gidx != 0) {
            if (ub_len > 4u * L.umi_max_bytes) {
                *status |= FASTF_ST_UMI_TOO_LONG;
            } else {
                // encode_DNA: A C G T -> 0 1 2 3 = bits 1 and 2 of the ASCII code, xor-ed; any other byte makes the UMI NULL
                u32 hi = 0, anybad = 0;
                for (u32 i = 0; i < ub_len; i++) {
                    const u32 ch = A.byte(ub_off + i);
                    const u32 code = ((ch >> 1) ^ (ch >> 2)) & 3u;
                    anybad |= ch ^ ((0x54474341u >> (8u * code)) & 255u);
                    hi |= code << (30u - 2u * i);
                }
                u64 ucode = 0;   // SQL NULL
                if (!anybad) {
                    u64 content = (u64)(hi >> (32u - 8u * L.umi_max_bytes));
                    u64 nbytes = (ub_len + 3u) >> 2;
                    ucode = (1ull << (L.bits_umi - 1u)) | (content << 3) | nbytes;
                }
                key = ((u64)cidx << (L.bits_gene + L.bits_umi)) | ((u64)gidx << L.bits_umi) | ucode;
            }
        }
    }
    *key_out = key;
    return 1;
}

#undef FASTF_PARSE_WIN
#define FASTF_PARSE_WIN 12224   // bytes of the block staged per warp and batch (4 warps x 12224 B stay under the 48 KB static limit)

// One warp per BGZF block.  Per batch: (1) the warp copies the next FASTF_PARSE_WIN bytes of the block into shared
// memory with coalesced 16-byte loads, (2) walks the block_size chain in the window (<= 32 records, lane k keeps
// record k), (3) every lane parses ITS OWN record out of shared memory (aux walk, table lookups, UMI packing --
// 32 records in flight per warp instead of 32 lanes repeating one record's scalar work), (4) the CB-valid records'
// keys are compacted in record order with a ballot.  Records larger than the window take the warp-cooperative
// global-memory path.  infl_total = readable bytes of the inflated buffer (>= end of the last block, multiple of 16).
// KEEP_CELL: see fastf_parse_record (false for every job but the cell-rate grid's).
template <bool KEEP_CELL>
__global__ void __launch_bounds__(FASTF_PARSE_WARPS * 32)
fastf_bam_parse_kernel(const u8 *__restrict__ infl, u64 infl_total, const u64 *__restrict__ blk_off, const u32 *__restrict__ blk_isize, u32 nblocks, const u64 *__restrict__ first_record_off_ptr,
                       FastfStrTableView cells, FastfStrTableView genes, FastfKeyLayout L,
                       const u64 *__restrict__ stage_off, u64 *__restrict__ stage, u32 *__restrict__ blk_nrec, u32 *__restrict__ blk_ncbv, u32 *__restrict__ blk_status)
{
    __shared__ __align__(16) u8 s_win[FASTF_PARSE_WARPS][FASTF_PARSE_WIN + FASTF_PARSE_PAD];
    __shared__ __align__(8) u64 s_mbar[FASTF_PARSE_WARPS];   // one TMA completion barrier per warp (its window is private)
    const u32 lane = threadIdx.x & 31u;
    const u32 b = blockIdx.x * FASTF_PARSE_WARPS + (threadIdx.x >> 5);
    if (b >= nblocks) return;
    u8 *W = s_win[threadIdx.x >> 5];
    u64 *mbar = &s_mbar[threadIdx.x >> 5];
    u32 mbar_parity = 0;
    if (lane == 0) fastf_mbar_init(mbar, 1);
    __syncwarp();
    const u64 bstart = blk_off[b], bend = bstart + blk_isize[b];
    const u64 first_record_off = *first_record_off_ptr;   // end of the BAM header (chunk 0) or 0
    u64 p = bstart > first_record_off ? bstart : first_record_off;
    u64 *out = stage + stage_off[b];
    const u64 cap = stage_off[b + 1] - stage_off[b];   // stage_off has nblocks + 1 entries; only a wrong record-start guess (FASTF_BAM_STRADDLE) can exceed it
    u32 nrec = 0, ncbv = 0, status = 0;

    while (p < bend) {
        if (bend - p < 4) { status |= FASTF_ST_REC_STRADDLE; break; }
        // (1) stage the window
        const u64 wbase = p & ~15ull;
        u64 wend = wbase + FASTF_PARSE_WIN < infl_total ? wbase + FASTF_PARSE_WIN : infl_total;
        {
            const u64 need = ((bend + 15ull) & ~15ull) < wend ? ((bend + 15ull) & ~15ull) : wend;   // nothing beyond the block is needed
            // the window arrives as ONE bulk copy of the TMA engine (a loop of 16-byte loads kept the warp waiting on DRAM round trips:
            // 28 % of the kernel's stall samples in round 1)
            __syncwarp();
            if (lane == 0) fastf_tma_load_1d(W, infl + wbase, (u32)(need - wbase), mbar);
            fastf_mbar_wait(mbar, mbar_parity);
            mbar_parity ^= 1u;
            __syncwarp();
            wend = need;
        }
        const FastfWin32 WA = {W};
        // (2) chain walk: up to 32 records that lie completely inside the window (offsets from the start of the window)
        u32 myrec = 0, mybs = 0, nb = 0, stop = 0;
        const u32 wlen = (u32)(wend - wbase), brel = (u32)(bend - wbase);   // the block ends at most 64 KiB + 15 behind wbase
        u32 qo = (u32)(p - wbase);
        while (nb < 32u && qo < brel) {
            if (brel - qo < 4u) { stop = FASTF_ST_REC_STRADDLE; break; }
            if (qo + 4u > wlen) break;
            const u32 bs = WA.bytes4(qo);
            if ((i32)bs < 32) { stop = FASTF_ST_REC_CORRUPT; break; }
            if ((u64)qo + 4u + (u64)bs > (u64)brel) { stop = FASTF_ST_REC_STRADDLE; break; }
            if (qo + 4u + bs > wlen) break;   // no overflow: bs <= brel < 2^17 here
            if (lane == nb) { myrec = qo + 4u; mybs = bs; }
            nb++;
            qo += 4u + bs;
        }
        const u64 q = wbase + qo;
        if (nb == 0 && !stop) {
            // the record at p is larger than the window: warp-cooperative walk in global memory
            const u32 bs = fastf_ld_u32(infl + p);
            if ((i32)bs < 32) { status |= FASTF_ST_REC_CORRUPT; break; }
            if (p + 4 + (u64)bs > bend) { status |= FASTF_ST_REC_STRADDLE; break; }
            const FastfGlobAcc GA = {infl};
            u64 key = 0;
            const u32 r = fastf_parse_record<KEEP_CELL>(GA, p + 4, p + 4 + bs, bs, cells, genes, L, cells.pw1[lane], cells.pw2[lane], genes.pw1[lane], genes.pw2[lane], lane, &status, &key);
            if (r == 2) break;
            p += 4 + (u64)bs;
            nrec++;
            if (r == 1) {
                if (ncbv >= cap) { status |= FASTF_ST_REC_CORRUPT; break; }
                if (lane == 0) out[ncbv] = key;
                ncbv++;
            }
            continue;
        }
        // (3) one record per lane
        u64 key = 0;
        u32 r = 0, st = 0;
        if (lane < nb) r = fastf_parse_record_lane<KEEP_CELL>(WA, myrec, myrec + mybs, mybs, cells, genes, L, &st, &key);
        // (4) ordered compaction; a corrupt record ends the block at that record
        const u32 badm = __ballot_sync(FASTF_FULL_MASK, r == 2);
        u32 good = nb;
        if (badm) good = (u32)__ffs((int)badm) - 1u;
        const u32 cm = __ballot_sync(FASTF_FULL_MASK, r == 1 && lane < good);
        if (ncbv + (u32)__popc(cm) > cap) { status |= FASTF_ST_REC_CORRUPT; break; }
        if (r == 1 && lane < good) out[ncbv + (u32)__popc(cm & fastf_lanemask_lt())] = key;
        ncbv += (u32)__popc(cm);
        nrec += good;
        status |= __reduce_or_sync(FASTF_FULL_MASK, lane <= good ? st : 0u);
        if (badm) break;
        p = q;
        if (stop) { status |= stop; break; }
    }
    if (lane == 0) { blk_nrec[b] = nrec; blk_ncbv[b] = ncbv; blk_status[b] = status; }
}

// Gather the per-block staging slices into the contiguous, file-ordered candidate array.
// dst_base[b] = global index of block b's first candidate (exclusive scan of blk_ncbv + running base).
__global__ void __launch_bounds__(256)
fastf_stage_gather_kernel(const u64 *__restrict__ stage, const u64 *__restrict__ stage_off, const u32 *__restrict__ blk_ncbv, const u64 *__restrict__ dst_base, u32 nblocks, u64 *__restrict__ cand)
{
    const u32 warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31u;
    if (warp >= nblocks) return;
    const u64 *src = stage + stage_off[warp];
    u64 *dst = cand + dst_base[warp];
    const u32 n = blk_ncbv[warp];
    for (u32 i = lane; i < n; i += 32) dst[i] = src[i];
}
