// Part of the libfastf_gpu translation unit (capi.cu includes it, in this order; it is not a header of its own):
// freq: the FASTQ streamed through HBM in chunks, keys accumulated, one sort + run-length at the end.
#pragma once

// ---------------------------------------------------------------------------------------------------
// freq
// ---------------------------------------------------------------------------------------------------
// The text (inflated FASTQ) streams through HBM chunk by chunk; what stays resident is one u64 key per read.  A chunk's text sits
// at buf + FASTF_FREQ_CARRY with the last bytes of the text before it copied in front, so that a sequence line that crosses the
// chunk boundary is seen whole by exactly one chunk (fastf_freq_keys_kernel).
#define FASTF_FREQ_CARRY 64u   // >= 2 * FASTF_FREQ_EXC_STRIDE, multiple of 16
struct FreqStream {
    DevBuf tiles, tot, keys, exc_cnt, exc_ord, exc_bytes;
    PinBuf host;
    Timer t_keys;
    u64 nl_total = 0;            // newlines of the text so far
    u64 bytes_total = 0;
    u64 keys_used = 0;           // records with a key slot so far
    u32 exc_cap = 0, n_exc = 0;
    u8 tail[FASTF_FREQ_CARRY];   // host copy of the last bytes of the text so far
    u32 tail_len = 0;
    u32 key_len = 0;
};
static int freq_stream_init(fastf_ctx *ctx, FreqStream &Q, u32 key_len, cudaStream_t s)
{
    Q.key_len = key_len;
    if (Q.t_keys.init()) return ctx_fail(ctx, "freq: event creation failed");
    TRY(pin_reserve(ctx, Q.host, 256));
    TRY(dev_reserve(ctx, Q.tot, sizeof(u32)));
    TRY(dev_reserve(ctx, Q.exc_cnt, sizeof(u32)));
    CK(cudaMemsetAsync(Q.exc_cnt.p, 0, sizeof(u32), s));
    return 0;
}
// one chunk: buf holds chunk_bytes of text at buf + FASTF_FREQ_CARRY (the bytes in front are free)
static int freq_stream_chunk(fastf_ctx *ctx, FreqStream &Q, u8 *buf, u64 chunk_bytes, bool last, fastf_freq_result *res, cudaStream_t s)
{
    const u32 carry = Q.tail_len;
    if (carry) CK(cudaMemcpyAsync(buf + FASTF_FREQ_CARRY - carry, Q.tail, carry, cudaMemcpyHostToDevice, s));
    const u64 lead = FASTF_FREQ_CARRY - carry;           // first byte of the text inside buf
    const u8 *text = buf + (lead & ~15ull);              // 16-byte aligned for the vector loads
    const u64 skip = lead & 15ull;
    const u64 n = skip + carry + chunk_bytes;
    const u64 ntiles64 = (n + FASTF_NL_TILE - 1) / FASTF_NL_TILE;
    if (ntiles64 >= 0xffffffffull) return ctx_fail(ctx, "freq: chunk too large");
    const u32 ntiles = (u32)std::max<u64>(ntiles64, 1);
    TRY(dev_reserve(ctx, Q.tiles, (size_t)ntiles * sizeof(u32)));
    Q.t_keys.collect(&res->ms_keys);
    Q.t_keys.start(s);
    FASTF_LAUNCH(fastf_nl_count_kernel, ntiles, FASTF_NL_THREADS, 0, s, text, n, Q.tiles.as<u32>(), skip);
    CKL("nl_count");
    TRY(launch_scan_rows(ctx, Q.tiles.as<u32>(), ntiles, 1, Q.tot.as<u32>(), s));
    CK(cudaMemcpyAsync(Q.host.p, Q.tot.p, sizeof(u32), cudaMemcpyDeviceToHost, s));
    const u32 new_tail = (u32)std::min<u64>(FASTF_FREQ_CARRY, carry + chunk_bytes);
    if (new_tail) CK(cudaMemcpyAsync(Q.host.as<u8>() + 64, text + n - new_tail, new_tail, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    const u64 nl_here = Q.host.as<u32>()[0];             // newlines of carry + chunk (a chunk holds < 2^32 bytes)
    u64 nl_carry = 0;
    for (u32 i = 0; i < carry; i++) nl_carry += Q.tail[i] == '\n';
    const u64 nl_base = Q.nl_total - nl_carry;           // global index of the first newline of this text
    Q.nl_total = nl_base + nl_here;
    Q.bytes_total += chunk_bytes;
    // key slots: record r exists as soon as newline 4r does
    const u64 n_keys = Q.nl_total ? (Q.nl_total - 1) / 4 + 1 : 0;
    if (n_keys >= 0xffffffffull) return ctx_fail(ctx, "freq: more than 2^32-1 reads in one pass");
    TRY(dev_reserve(ctx, Q.keys, std::max<u64>(n_keys, 1) * sizeof(u64), Q.keys_used * sizeof(u64), s));
    if (Q.exc_cap == 0) Q.exc_cap = 1u << 16;
    const u32 exc_before = Q.n_exc;
    for (int attempt = 0; attempt < 2; attempt++) {
        TRY(dev_reserve(ctx, Q.exc_ord, (size_t)Q.exc_cap * sizeof(u32), (size_t)exc_before * sizeof(u32), s));
        TRY(dev_reserve(ctx, Q.exc_bytes, (size_t)Q.exc_cap * FASTF_FREQ_EXC_STRIDE, (size_t)exc_before * FASTF_FREQ_EXC_STRIDE, s));
        CK(cudaMemcpyAsync(Q.exc_cnt.p, &exc_before, sizeof(u32), cudaMemcpyHostToDevice, s));
        FASTF_LAUNCH(fastf_freq_keys_kernel, ntiles, FASTF_NL_THREADS, 0, s, text, n, (const u32 *)Q.tiles.as<u32>(), Q.key_len, Q.keys.as<u64>(), n_keys, Q.exc_cnt.as<u32>(), Q.exc_cap,
                     Q.exc_ord.as<u32>(), Q.exc_bytes.as<u8>(), skip, nl_base, skip + carry, (u32)last);
        CKL("freq_keys");
        CK(cudaMemcpyAsync(Q.host.p, Q.exc_cnt.p, sizeof(u32), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        Q.n_exc = Q.host.as<u32>()[0];
        if (Q.n_exc <= Q.exc_cap) break;
        Q.exc_cap = std::max(Q.n_exc, Q.exc_cap * 2);   // rerun this chunk with room for every exceptional read
    }
    Q.t_keys.stop(s);
    Q.keys_used = n_keys;
    memcpy(Q.tail, Q.host.as<u8>() + 64, new_tail);
    Q.tail_len = new_tail;
    return 0;
}

// after the last chunk: compact the good keys with their read ordinals, sort, run-length encode, copy back
static int freq_stream_finish(fastf_ctx *ctx, FreqStream &Q, fastf_freq_result *res, cudaStream_t s)
{
    DevBuf ckeys, cidx, kalt, valt, orand, tiles, tot;
    PinBuf host;
    SortScratch S;
    RleScratch R;
    Timer t_sort, t_rle;
    DrainOnExit drain{ctx};
    if (t_sort.init() || t_rle.init()) return ctx_fail(ctx, "freq: event creation failed");
    TRY(pin_reserve(ctx, host, 64));
    TRY(dev_reserve(ctx, orand, 2 * sizeof(u64)));
    TRY(dev_reserve(ctx, tot, sizeof(u32)));
    Q.t_keys.collect(&res->ms_keys);
    const u64 n = Q.bytes_total, n_newlines = Q.nl_total;
    const u8 last = Q.tail_len ? Q.tail[Q.tail_len - 1] : (u8)'\n';
    const u64 n_lines = n_newlines + ((n && last != '\n') ? 1 : 0);
    // get_fastq reads four lines per record; a record exists as soon as its id line does (reference src/filter.c:22-34)
    res->n_lines = n_lines;
    res->last_byte_is_newline = (u8)(n == 0 || last == '\n');
    res->n_reads = (n_lines + 3) / 4;
    // records whose sequence line starts after newline 4r: r = 0 .. n_keys_dev-1 where newline 4r exists; a trailing record whose
    // id line is not newline-terminated has an empty key (NUL immediately): the host handles it
    const u64 n_keys_dev = Q.keys_used;
    const u32 n_exc = Q.n_exc;
    const u64 n_good = n_keys_dev - n_exc;
    u64 ngroups = 0;
    if (n_good) {
        const u32 ctiles = (u32)((n_keys_dev + FASTF_CP_TILE - 1) / FASTF_CP_TILE);
        TRY(dev_reserve(ctx, tiles, (size_t)ctiles * sizeof(u32)));
        TRY(dev_reserve(ctx, ckeys, n_good * sizeof(u64)));
        TRY(dev_reserve(ctx, cidx, n_good * sizeof(u32)));
        TRY(dev_reserve(ctx, kalt, n_good * sizeof(u64)));
        TRY(dev_reserve(ctx, valt, n_good * sizeof(u32)));
        t_sort.start(s);
        FASTF_LAUNCH(fastf_compact_count_kernel, ctiles, FASTF_CP_THREADS, 0, s, (const u64 *)Q.keys.as<u64>(), n_keys_dev, tiles.as<u32>());
        CKL("compact_count");
        TRY(launch_scan_rows(ctx, tiles.as<u32>(), ctiles, 1, tot.as<u32>(), s));
        FASTF_LAUNCH(fastf_compact_scatter_kernel, ctiles, FASTF_CP_THREADS, 0, s, (const u64 *)Q.keys.as<u64>(), n_keys_dev, (const u32 *)tiles.as<u32>(), ckeys.as<u64>(), cidx.as<u32>());
        CKL("compact_scatter");
        Q.keys.release();   // the compacted copy is what is sorted
        u64 varying = 0;
        TRY(varying_bits(ctx, orand, host, ckeys.as<u64>(), n_good, &varying, s));
        u32 shifts[8];
        const int npass = plan_windows(varying, shifts);
        bool in_alt = false;
        TRY(sort_keys(ctx, S, ckeys.as<u64>(), kalt.as<u64>(), cidx.as<u32>(), valt.as<u32>(), n_good, shifts, npass, &in_alt, s));
        t_sort.stop(s);
        t_rle.start(s);
        u64 nd = 0;
        TRY(rle_groups(ctx, R, in_alt ? kalt.as<u64>() : ckeys.as<u64>(), in_alt ? valt.as<u32>() : cidx.as<u32>(), n_good, 0, 64, 0, &ngroups, &nd, s));
        t_rle.stop(s);
    }
    // ---- results to host ----
    res->n_keys = ngroups;
    res->key = (u64 *)malloc(std::max<u64>(ngroups, 1) * sizeof(u64));
    res->count = (u32 *)malloc(std::max<u64>(ngroups, 1) * sizeof(u32));
    res->first = (u32 *)malloc(std::max<u64>(ngroups, 1) * sizeof(u32));
    res->n_exceptions = n_exc;
    res->exc_stride = FASTF_FREQ_EXC_STRIDE;
    res->exc_ordinal = (u32 *)malloc(std::max<u64>(n_exc, 1) * sizeof(u32));
    res->exc_bytes = (u8 *)malloc(std::max<u64>(n_exc, 1) * FASTF_FREQ_EXC_STRIDE);
    if (!res->key || !res->count || !res->first || !res->exc_ordinal || !res->exc_bytes) return ctx_fail(ctx, "freq: out of host memory");
    if (ngroups) {
        // with group_shift 0 every distinct key is a group and counts all its copies: count = next first - first
        TRY(d2h_pageable(ctx, res->key, R.grp_key.p, ngroups * sizeof(u64), s));
        TRY(d2h_pageable(ctx, res->first, R.grp_val.p, ngroups * sizeof(u32), s));
        TRY(d2h_pageable(ctx, res->count, R.grp_first.p, ngroups * sizeof(u32), s));
    }
    if (n_exc) {
        CK(cudaMemcpyAsync(res->exc_ordinal, Q.exc_ord.p, (size_t)n_exc * sizeof(u32), cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(res->exc_bytes, Q.exc_bytes.p, (size_t)n_exc * FASTF_FREQ_EXC_STRIDE, cudaMemcpyDeviceToHost, s));
    }
    CK(cudaStreamSynchronize(s));
    // grp_first[g] = index of the group's first element in the sorted array -> multiplicity by differencing
    for (u64 g = 0; g < ngroups; g++) {
        u64 nxt = (g + 1 < ngroups) ? res->count[g + 1] : n_good;
        res->count[g] = (u32)(nxt - res->count[g]);
    }
    t_sort.collect(&res->ms_sort);
    t_rle.collect(&res->ms_rle);
    return 0;
}

static bool looks_like_gzip(const u8 *p, size_t n) { return n >= 2 && p[0] == 0x1f && p[1] == 0x8b; }

// blocks per streamed chunk of the tag / freq jobs: two rounds of the persistent inflate kernel (tests shrink it to force many chunks)
static size_t stream_chunk_blocks(const fastf_ctx *ctx)
{
    if (ctx->taghist_chunk_blocks) return (size_t)ctx->taghist_chunk_blocks;
    if (const char *e = getenv("FASTF_STREAM_CHUNK_BLOCKS")) { const long v = atol(e); if (v > 0) return (size_t)v; }   // tests: many chunks on small inputs
    return 2ull * (size_t)ctx->n_sm * FASTF_TPS_STREAMS;
}

// freq over one input: chunks of whole BGZF blocks (or pieces of plain text) -> newline scan -> keys; then sort + run-length
static int freq_run(fastf_ctx *ctx, const void *host_bytes, size_t n, const u8 *dev_bytes, const std::vector<FastfBgzfBlock> *pre, uint32_t key_len, uint32_t lanes, fastf_freq_result *res)
{
    if (key_len == 0 || key_len > FASTF_FREQ_MAX_KEY) return ctx_fail(ctx, "freq: len_cellbarcode + len_umi must be 1..%d (got %u)", FASTF_FREQ_MAX_KEY, key_len);
    cudaStream_t s = ctx->compute;
    Event e0, e1;
    CK(e0.create());
    CK(e1.create());
    InflatedFile F;
    FreqStream Q;
    DevBuf plain;
    DrainOnExit drain{ctx};
    std::vector<FastfBgzfBlock> all, part;
    TRY(freq_stream_init(ctx, Q, key_len, s));
    cudaEventRecord(e0, s);
    if (dev_bytes || looks_like_gzip((const u8 *)host_bytes, n)) {
        const std::vector<FastfBgzfBlock> *blocks = pre;
        if (!dev_bytes) {
            // plain (non-BGZF) gzip cannot be inflated block-parallel: refuse loudly rather than fall back to the CPU
            const u8 *h = (const u8 *)host_bytes;
            if (n < 18 || !(h[3] & 4)) return ctx_fail(ctx, "freq: input is single-member gzip, not BGZF; recompress with bgzip (no CPU fallback; the reference reads it through zlib's gzopen)");
            size_t used = 0;
            const int irc = fastf_bgzf_index(h, n, 0, all, &used);
            if (irc != FASTF_BGZF_OK) return ctx_fail(ctx, "inflate: not a whole BGZF stream (index error %d at byte %zu of %zu)", irc, used, n);
            blocks = &all;
        }
        // chunks of whole BGZF blocks: inflate -> newline scan -> keys; only the keys stay resident
        const size_t nb = blocks->size(), per = stream_chunk_blocks(ctx);
        res->n_blocks = nb;
        for (size_t b0 = 0; b0 < nb || b0 == 0; b0 += per) {
            const size_t b1 = std::min(nb, b0 + per);
            part.assign(blocks->begin() + (ptrdiff_t)b0, blocks->begin() + (ptrdiff_t)b1);
            float ms_infl = 0;
            TRY(inflate_whole(ctx, F, host_bytes, n, dev_bytes, &part, lanes, &ms_infl, s, FASTF_FREQ_CARRY));
            res->ms_inflate += ms_infl;
            res->status |= F.status;
            TRY(freq_stream_chunk(ctx, Q, F.infl.as<u8>(), F.infl_bytes, b1 >= nb, res, s));
            if (nb == 0) break;
        }
    } else {
        // plain text: pieces of the host buffer
        size_t PIECE = (size_t)256 << 20;
        if (const char *e = getenv("FASTF_STREAM_CHUNK_BLOCKS")) { const long v = atol(e); if (v > 0) PIECE = (size_t)v * 1000; }   // tests: pieces of a few KB
        TRY(dev_reserve(ctx, plain, std::min<size_t>(n, PIECE) + FASTF_FREQ_CARRY + 64));
        for (size_t o = 0; o < n || o == 0; o += PIECE) {
            const size_t m = std::min(PIECE, n - o);
            if (m) CK(cudaMemcpyAsync(plain.as<u8>() + FASTF_FREQ_CARRY, (const u8 *)host_bytes + o, m, cudaMemcpyHostToDevice, s));
            TRY(freq_stream_chunk(ctx, Q, plain.as<u8>(), m, o + m >= n, res, s));
            if (n == 0) break;
        }
    }
    res->compressed_bytes = n;
    res->inflated_bytes = Q.bytes_total;
    TRY(freq_stream_finish(ctx, Q, res, s));
    cudaEventRecord(e1, s);
    cudaEventSynchronize(e1);
    cudaEventElapsedTime(&res->ms_device_total, e0, e1);
    return 0;
}

// a failed call leaves no result arrays behind
static int freq_common(fastf_ctx *ctx, const void *host_bytes, size_t n, const u8 *dev_bytes, const std::vector<FastfBgzfBlock> *pre, uint32_t key_len, uint32_t lanes, fastf_freq_result *res)
{
    CK(cudaSetDevice(ctx->device));
    memset(res, 0, sizeof *res);
    const u32 l0 = ctx->launches;
    const int rc = freq_run(ctx, host_bytes, n, dev_bytes, pre, key_len, lanes, res);
    res->n_launches = ctx->launches - l0;
    if (rc) fastf_freq_result_free(res);
    return rc;
}

extern "C" int fastf_freq_gpu(fastf_ctx *ctx, const void *host_bytes, size_t n, uint32_t key_len, uint32_t inflate_lanes, fastf_freq_result *res)
{
    return freq_common(ctx, host_bytes, n, nullptr, nullptr, key_len, inflate_lanes, res);
}
extern "C" int fastf_freq_gpu_device(fastf_ctx *ctx, const void *dev_bytes, size_t nbytes, const uint64_t *in_off, const uint32_t *in_len, const uint32_t *isize, uint64_t nblocks, uint32_t key_len,
                                     uint32_t inflate_lanes, fastf_freq_result *res)
{
    if (((uintptr_t)dev_bytes & 3u) != 0) return ctx_fail(ctx, "freq_gpu_device: dev_bytes must be 4-byte aligned");
    std::vector<FastfBgzfBlock> blocks(nblocks);
    for (u64 i = 0; i < nblocks; i++) {
        if (in_off[i] + in_len[i] + 8 > nbytes || isize[i] > 65536) return ctx_fail(ctx, "freq_gpu_device: block %llu outside the buffer", (unsigned long long)i);
        blocks[i].in_off = in_off[i]; blocks[i].in_len = in_len[i]; blocks[i].isize = isize[i]; blocks[i].crc32 = 0;
    }
    return freq_common(ctx, nullptr, nbytes, (const u8 *)dev_bytes, &blocks, key_len, inflate_lanes, res);
}
