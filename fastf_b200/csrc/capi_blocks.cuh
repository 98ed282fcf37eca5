// Part of the libfastf_gpu translation unit (capi.cu includes it, in this order; it is not a header of its own):
// device-level building blocks of multi-GPU hosts and the host-buffer wrappers around single kernels (tests, smoke).
#pragma once

// ---------------------------------------------------------------------------------------------------
// device-level building blocks
// ---------------------------------------------------------------------------------------------------
extern "C" int fastf_sort_u64_device(fastf_ctx *ctx, uint64_t *dev_keys, uint32_t *dev_vals, uint64_t n, uint32_t key_bits)
{
    CK(cudaSetDevice(ctx->device));
    if (n == 0) return 0;
    SortScratch S;
    DevBuf alt, valt;
    int rc = dev_reserve(ctx, alt, n * sizeof(u64));
    if (!rc && dev_vals) rc = dev_reserve(ctx, valt, n * sizeof(u32));
    u32 shifts[8];
    int npass = 0;
    for (u32 b = 0; b < key_bits && npass < 8; b += 8) shifts[npass++] = b;
    bool in_alt = false;
    if (!rc) rc = sort_keys(ctx, S, dev_keys, alt.as<u64>(), dev_vals, valt.as<u32>(), n, shifts, npass, &in_alt, ctx->compute);
    if (!rc && in_alt) {
        rc = cudaMemcpyAsync(dev_keys, alt.p, n * sizeof(u64), cudaMemcpyDeviceToDevice, ctx->compute) != cudaSuccess;
        if (!rc && dev_vals) rc = cudaMemcpyAsync(dev_vals, valt.p, n * sizeof(u32), cudaMemcpyDeviceToDevice, ctx->compute) != cudaSuccess;
    }
    if (cudaStreamSynchronize(ctx->compute) != cudaSuccess && !rc) rc = ctx_fail(ctx, "sort_u64_device: stream error");
    sort_scratch_release(ctx, S);
    dev_release(ctx, alt);
    dev_release(ctx, valt);
    return rc;
}

// same, results left on the device in caller-provided arrays of capacity >= n (multi-GPU driver: the pieces travel over NCCL)
extern "C" int fastf_dedup_count_device_out(fastf_ctx *ctx, const uint64_t *dev_sorted_keys, uint64_t n, uint32_t bits_gene, uint32_t bits_umi, uint64_t *nnz, uint32_t *dev_gene, uint32_t *dev_cell,
                                            uint32_t *dev_count)
{
    CK(cudaSetDevice(ctx->device));
    RleScratch R;
    u64 ng = 0;
    int rc = rle_groups(ctx, R, dev_sorted_keys, nullptr, n, bits_umi, bits_umi - 1, bits_gene, &ng, nullptr, ctx->compute);
    if (!rc && ng) {
        rc = cudaMemcpyAsync(dev_gene, R.out_gene.p, ng * sizeof(u32), cudaMemcpyDeviceToDevice, ctx->compute) != cudaSuccess ||
             cudaMemcpyAsync(dev_cell, R.out_cell.p, ng * sizeof(u32), cudaMemcpyDeviceToDevice, ctx->compute) != cudaSuccess ||
             cudaMemcpyAsync(dev_count, R.count.p, ng * sizeof(u32), cudaMemcpyDeviceToDevice, ctx->compute) != cudaSuccess;
        if (rc) ctx_fail(ctx, "dedup_count_device_out: copy failed");
    }
    if (cudaStreamSynchronize(ctx->compute) != cudaSuccess && !rc) rc = ctx_fail(ctx, "dedup_count_device_out: stream error");
    *nnz = ng;
    rle_scratch_release(ctx, R);
    return rc;
}

extern "C" int fastf_dedup_count_device(fastf_ctx *ctx, const uint64_t *dev_sorted_keys, uint64_t n, uint32_t bits_gene, uint32_t bits_umi, uint64_t *nnz, uint32_t **m_gene, uint32_t **m_cell,
                                        uint32_t **m_count)
{
    CK(cudaSetDevice(ctx->device));
    RleScratch R;
    u64 ng = 0;
    int rc = rle_groups(ctx, R, dev_sorted_keys, nullptr, n, bits_umi, bits_umi - 1, bits_gene, &ng, nullptr, ctx->compute);
    if (!rc) rc = coo_to_host(ctx, R, ng, m_gene, m_cell, m_count, ctx->compute);
    *nnz = ng;
    rle_scratch_release(ctx, R);
    return rc;
}

// Destination of a cell for the multi-GPU exchange: all keys of one (cell, gene) group must meet on one rank.  The "hash" is
// order preserving -- an equal-width range partition of the 1-based cell index, which is itself the position of the barcode in a
// file-ordered random sample, so depth is spread evenly -- and therefore the ranks' (cell, gene)-sorted COO pieces concatenate
// in rank order without a merge.
static inline __host__ __device__ u32 fastf_cell_dest(u32 cell, u32 n_cells, u32 nparts) { return (u32)(((u64)(cell - 1u) * nparts) / (n_cells ? n_cells : 1u)); }

__global__ void __launch_bounds__(256) fastf_tag_dest_kernel(u64 *__restrict__ keys, u64 n, u32 cell_shift, u32 key_bits, u32 n_cells, u32 nparts)
{
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    u64 k = keys[i];
    u32 d = fastf_cell_dest((u32)(k >> cell_shift), n_cells, nparts);
    keys[i] = k | ((u64)(d < nparts ? d : nparts - 1u) << key_bits);
}
// heads of runs of equal keys -> compacted, with the destination tag stripped; part boundaries by binary search
__global__ void __launch_bounds__(256) fastf_part_bounds_kernel(const u64 *__restrict__ keys, u64 n, u32 key_bits, u32 nparts, u64 *__restrict__ bounds)
{
    u32 p = threadIdx.x;
    if (p > nparts) return;
    u64 lo = 0, hi = n;
    while (lo < hi) { u64 mid = (lo + hi) >> 1; if ((keys[mid] >> key_bits) < (u64)p) lo = mid + 1; else hi = mid; }
    bounds[p] = lo;
}
__global__ void __launch_bounds__(256) fastf_strip_tag_kernel(u64 *__restrict__ keys, u64 n, u32 key_bits)
{
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) keys[i] &= (1ull << key_bits) - 1ull;
}

// Tag every key with its destination, sort (with rates: the rate index first, as the least significant digit), keep the first key of
// every run: the unique keys grouped by destination, each with its smallest rate index when rates are given.
static int unique_partition(fastf_ctx *ctx, const char *who, u64 *dev_keys, u32 *dev_rates, u64 n, u32 key_bits, u32 bits_gene, u32 bits_umi, u32 n_cells, u32 nparts, u64 *dev_out_keys,
                            u32 *dev_out_rates, u64 *part_counts)
{
    CK(cudaSetDevice(ctx->device));
    for (u32 p = 0; p < nparts; p++) part_counts[p] = 0;
    if (n == 0) return 0;
    if (nparts == 0 || nparts > 256 || key_bits + (nparts > 1 ? bits_for(nparts - 1) : 0) > 64)
        return ctx_fail(ctx, "%s: %u key bits leave no room for the destination tag of %u parts", who, key_bits, nparts);
    cudaStream_t s = ctx->compute;
    SortScratch S;
    RleScratch R;
    DevBuf alt, valt, orand, bounds;
    PinBuf host;
    int rc = 0;
    auto body = [&]() -> int {
        TRY(dev_reserve(ctx, alt, n * sizeof(u64)));
        if (dev_rates) TRY(dev_reserve(ctx, valt, n * sizeof(u32)));
        TRY(dev_reserve(ctx, orand, 2 * sizeof(u64)));
        TRY(dev_reserve(ctx, bounds, 257 * sizeof(u64)));
        TRY(pin_reserve(ctx, host, 257 * sizeof(u64)));
        FASTF_LAUNCH(fastf_tag_dest_kernel, (u32)((n + 255) / 256), 256, 0, s, dev_keys, n, bits_gene + bits_umi, key_bits, n_cells, nparts);
        CKL("tag_dest");
        u64 varying = 0;
        TRY(varying_bits(ctx, orand, host, dev_keys, n, &varying, s));
        u32 shifts[9];
        int npass = 0;
        if (dev_rates) shifts[npass++] = FASTF_SORT_VAL_DIGIT;
        npass += plan_windows(varying, shifts + npass);
        bool in_alt = false;
        TRY(sort_keys(ctx, S, dev_keys, alt.as<u64>(), dev_rates, dev_rates ? valt.as<u32>() : nullptr, n, shifts, npass, &in_alt, s));
        const u64 *sorted = in_alt ? alt.as<u64>() : dev_keys;
        const u32 *sorted_rates = dev_rates ? (in_alt ? valt.as<u32>() : dev_rates) : nullptr;
        // unique: every key is its own group (group_shift 0); grp_key = the distinct keys in sorted order, grp_val their first rate
        u64 nuniq = 0;
        TRY(rle_groups(ctx, R, sorted, sorted_rates, n, 0, 64, 0, &nuniq, nullptr, s));
        FASTF_LAUNCH(fastf_part_bounds_kernel, 1, 256, 0, s, (const u64 *)R.grp_key.as<u64>(), nuniq, key_bits, nparts, bounds.as<u64>());
        CKL("part_bounds");
        CK(cudaMemcpyAsync(dev_out_keys, R.grp_key.p, nuniq * sizeof(u64), cudaMemcpyDeviceToDevice, s));
        if (dev_rates) CK(cudaMemcpyAsync(dev_out_rates, R.grp_val.p, nuniq * sizeof(u32), cudaMemcpyDeviceToDevice, s));
        FASTF_LAUNCH(fastf_strip_tag_kernel, (u32)((nuniq + 255) / 256), 256, 0, s, dev_out_keys, nuniq, key_bits);
        CKL("strip_tag");
        CK(cudaMemcpyAsync(host.p, bounds.p, (nparts + 1) * sizeof(u64), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        for (u32 p = 0; p < nparts; p++) part_counts[p] = host.as<u64>()[p + 1] - host.as<u64>()[p];
        return 0;
    };
    rc = body();
    cudaStreamSynchronize(s);
    sort_scratch_release(ctx, S);
    rle_scratch_release(ctx, R);
    dev_release(ctx, alt); dev_release(ctx, valt); dev_release(ctx, orand); dev_release(ctx, bounds);
    pin_release(ctx, host);
    return rc;
}

extern "C" int fastf_unique_partition_device(fastf_ctx *ctx, uint64_t *dev_keys, uint64_t n, uint32_t key_bits, uint32_t bits_gene, uint32_t bits_umi, uint32_t n_cells, uint32_t nparts,
                                             uint64_t *dev_out_keys, uint64_t *part_counts)
{
    return unique_partition(ctx, "unique_partition", dev_keys, nullptr, n, key_bits, bits_gene, bits_umi, n_cells, nparts, dev_out_keys, nullptr, part_counts);
}

extern "C" int fastf_unique_partition_rates_device(fastf_ctx *ctx, uint64_t *dev_keys, uint32_t *dev_rates, uint64_t n, uint32_t key_bits, uint32_t bits_gene, uint32_t bits_umi, uint32_t n_cells,
                                                   uint32_t nparts, uint64_t *dev_out_keys, uint32_t *dev_out_rates, uint64_t *part_counts)
{
    if (n && (!dev_rates || !dev_out_rates)) return ctx_fail(ctx, "unique_partition_rates: null rate arrays");
    return unique_partition(ctx, "unique_partition_rates", dev_keys, dev_rates, n, key_bits, bits_gene, bits_umi, n_cells, nparts, dev_out_keys, dev_out_rates, part_counts);
}

// ---------------------------------------------------------------------------------------------------
// host-buffer wrappers around single kernels (tests, smoke)
// ---------------------------------------------------------------------------------------------------
struct InflatedFile {
    DevBuf comp, infl;
    DeScratch de;
    BlockIndexDev idx;
    u64 n_blocks = 0, infl_bytes = 0;
    u32 status = 0;
};
static void inflated_release(fastf_ctx *ctx, InflatedFile &F) { dev_release(ctx, F.comp); dev_release(ctx, F.infl); dev_release(ctx, F.de.counter); dev_release(ctx, F.de.sorted); index_release(ctx, F.idx); }

// Inflate a whole BGZF image (host bytes, or device bytes + host index) into F.infl in one launch.
// out_prefix: bytes kept free (and preserved across calls) in front of the inflated blocks -- streamed text carries the tail of the previous chunk there.
static int inflate_whole(fastf_ctx *ctx, InflatedFile &F, const void *host_bytes, size_t n, const u8 *dev_bytes, const std::vector<FastfBgzfBlock> *pre, u32 lanes, float *ms, cudaStream_t s, u64 out_prefix = 0)
{
    std::vector<FastfBgzfBlock> local;
    const std::vector<FastfBgzfBlock> *blocks = pre;
    if (!pre) {
        size_t used = 0;
        int rc = fastf_bgzf_index((const u8 *)host_bytes, n, 0, local, &used);
        if (rc != FASTF_BGZF_OK) return ctx_fail(ctx, "inflate: not a whole BGZF stream (index error %d at byte %zu of %zu)", rc, used, n);
        blocks = &local;
    }
    const size_t nb = blocks->size();
    if (nb >= 0xffffffffull) return ctx_fail(ctx, "inflate: too many blocks");
    TRY(index_reserve(ctx, F.idx, (u32)std::max<size_t>(nb, 1)));
    // host bytes: only the span of these blocks travels (a pre-indexed subset = one chunk of a larger file), offsets are rebased
    const u64 lo = (!dev_bytes && nb) ? ((*blocks)[0].in_off & ~3ull) : 0;
    const u64 hi = (!dev_bytes && nb) ? std::min<u64>((*blocks)[nb - 1].in_off + (*blocks)[nb - 1].in_len + 8, n) : (dev_bytes ? 0 : n);
    u64 total = 0;
    for (size_t i = 0; i < nb; i++) {
        F.idx.h_in_off[i] = (*blocks)[i].in_off - lo; F.idx.h_in_len[i] = (*blocks)[i].in_len; F.idx.h_isize[i] = (*blocks)[i].isize;
        F.idx.h_out_off[i] = out_prefix + total; F.idx.h_stage_off[i] = 0;
        total += (*blocks)[i].isize;
    }
    const u8 *comp = dev_bytes;
    u64 comp_total = n & ~(u64)3;
    const u64 span = hi > lo ? hi - lo : 0;
    if (!dev_bytes) {
        const u64 padded = (span + 3) & ~3ull;
        TRY(dev_reserve(ctx, F.comp, padded + 16));
        comp = F.comp.as<u8>();
        comp_total = padded;
    }
    TRY(dev_reserve(ctx, F.infl, out_prefix + total + 64, out_prefix, s));
    TRY(index_upload(ctx, F.idx, s));
    {
        const u32 l = lanes & 0xffu;
        lanes = ((l == 8 || l == 16 || l == 32 || (l >= 1 && l <= 4)) ? l : FASTF_INFLATE_DEFAULT) | (lanes & (FASTF_INFLATE_HW_ENGINE | FASTF_INFLATE_NO_CRC | FASTF_BAM_STRADDLE));
    }
    // One launch over all blocks.  (Measured on freq, 117 k blocks: sending the host bytes in groups of two kernel rounds on the copy
    // stream while the previous group inflates is SLOWER end to end, 491 vs 514 M reads/s, and four launches instead of one cost the
    // device-resident path 7 %: every launch pays for building 128 tables per SM before its decoders start, and for its tail.
    // FASTF_INFLATE_GROUP=<blocks> re-enables the grouping for experiments.)  The inflate clock is the sum of the launches.
    size_t group = std::max<size_t>(nb, 1);
    if (const char *e = getenv("FASTF_INFLATE_GROUP")) { const long v = atol(e); group = v > 0 ? (size_t)v : std::max<size_t>(nb, 1); }   // A/B knob: 0 = one launch
    std::vector<cudaEvent_t> ev;
    cudaEvent_t ev_copy = nullptr;
    if (!dev_bytes) CK(cudaEventCreateWithFlags(&ev_copy, cudaEventDisableTiming));
    int rc_l = 0;
    for (size_t g0 = 0; g0 < nb && !rc_l; g0 += group) {
        const size_t g1 = std::min(nb, g0 + group);
        if (!dev_bytes) {
            // bytes of this group: from its first payload (the very first group: from lo) to the end of its last block's trailer
            const u64 b0 = g0 == 0 ? 0 : (F.idx.h_in_off[g0] & ~3ull);
            const u64 b1 = std::min<u64>(F.idx.h_in_off[g1 - 1] + F.idx.h_in_len[g1 - 1] + 8, span);
            if (b1 > b0) CK(cudaMemcpyAsync(F.comp.as<u8>() + b0, (const u8 *)host_bytes + lo + b0, b1 - b0, cudaMemcpyHostToDevice, ctx->copy));
            CK(cudaEventRecord(ev_copy, ctx->copy));
            CK(cudaStreamWaitEvent(s, ev_copy, 0));
        }
        if (ms) { cudaEvent_t a = nullptr, b = nullptr; CK(cudaEventCreate(&a)); CK(cudaEventCreate(&b)); ev.push_back(a); ev.push_back(b); CK(cudaEventRecord(a, s)); }
        rc_l = launch_inflate(ctx, lanes, comp, comp_total, F.idx.in_off + g0, F.idx.in_len + g0, F.idx.out_off + g0, F.idx.isize + g0, (u32)(g1 - g0), F.infl.as<u8>(), F.idx.st_infl + g0, s, &F.de,
                              F.idx.h_in_off + g0, F.idx.h_in_len + g0, F.idx.h_out_off + g0, F.idx.h_isize + g0);
        if (ms) CK(cudaEventRecord(ev.back(), s));
        if (!rc_l) rc_l = launch_crc(ctx, lanes, comp, dev_bytes ? (u64)n : comp_total, F.idx.in_off + g0, F.idx.in_len + g0, F.infl.as<u8>(), F.idx.out_off + g0, F.idx.isize + g0, (u32)(g1 - g0),
                                     F.idx.st_infl + g0, s);
    }
    if (rc_l) { for (auto e : ev) cudaEventDestroy(e); if (ev_copy) cudaEventDestroy(ev_copy); return rc_l; }
    // OR of the per-block status words
    std::vector<u32> st(nb);
    if (nb) CK(cudaMemcpyAsync(st.data(), F.idx.st_infl, nb * sizeof(u32), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (!dev_bytes) CK(cudaStreamSynchronize(ctx->copy));
    if (ms) {
        *ms = 0;
        for (size_t i = 0; i + 1 < ev.size(); i += 2) { float t = 0; cudaEventElapsedTime(&t, ev[i], ev[i + 1]); *ms += t; }
    }
    for (auto e : ev) cudaEventDestroy(e);
    if (ev_copy) cudaEventDestroy(ev_copy);
    F.status = 0;
    for (size_t i = 0; i < nb; i++) F.status |= st[i];
    F.n_blocks = nb;
    F.infl_bytes = total;
    if (F.status) {
        char buf[256];
        return ctx_fail(ctx, "inflate: malformed deflate data: %s", status_string(F.status, buf, sizeof buf));
    }
    return 0;
}

extern "C" int fastf_inflate_host(fastf_ctx *ctx, const void *bgzf_bytes, size_t n, int lanes, void **out, size_t *out_n, float *ms)
{
    CK(cudaSetDevice(ctx->device));
    *out = nullptr;
    *out_n = 0;
    InflatedFile F;
    int rc = inflate_whole(ctx, F, bgzf_bytes, n, nullptr, nullptr, (u32)lanes, ms, ctx->compute);
    if (!rc) {
        *out = malloc(F.infl_bytes ? F.infl_bytes : 1);
        if (!*out) rc = ctx_fail(ctx, "inflate_host: out of host memory");
        if (!rc && F.infl_bytes) rc = fastf_memcpy_d2h(ctx, *out, F.infl.p, F.infl_bytes);
        *out_n = F.infl_bytes;
    }
    inflated_release(ctx, F);
    return rc;
}

static int mt_host_common(fastf_ctx *ctx, uint32_t seed, uint64_t n, uint64_t threshold, uint32_t *out_words, uint32_t *out_bits)
{
    CK(cudaSetDevice(ctx->device));
    if (n == 0) return 0;
    const u64 pairs = (n + 1247) / 1248;
    DevBuf state, out;
    int rc = dev_reserve(ctx, state, 624 * sizeof(u32));
    const size_t out_bytes = out_words ? (size_t)pairs * 1248 * sizeof(u32) : (size_t)pairs * 39 * sizeof(u32);
    if (!rc) rc = dev_reserve(ctx, out, out_bytes);
    if (!rc) {
        FASTF_LAUNCH(fastf_mt19937_kernel, 1, FASTF_MT_THREADS, 0, ctx->compute, seed, state.as<u32>(), 1u, (u64)0, pairs, threshold, out_words ? out.as<u32>() : (u32 *)nullptr,
                     out_words ? (u32 *)nullptr : out.as<u32>());
        ctx->launches++;
        if (cudaGetLastError() != cudaSuccess) rc = ctx_fail(ctx, "mt19937 launch failed");
    }
    if (!rc) rc = out_words ? fastf_memcpy_d2h(ctx, out_words, out.p, (size_t)n * sizeof(u32)) : fastf_memcpy_d2h(ctx, out_bits, out.p, (size_t)((n + 31) / 32) * sizeof(u32));
    dev_release(ctx, state);
    dev_release(ctx, out);
    return rc;
}
extern "C" int fastf_mt19937_host_from(fastf_ctx *ctx, uint32_t seed, uint64_t first, uint64_t n, uint32_t *out_words)
{
    CK(cudaSetDevice(ctx->device));
    if (n == 0) return 0;
    const u64 pairs = (n + 1247) / 1248;
    DevBuf state, out;
    int rc = dev_reserve(ctx, state, 624 * sizeof(u32));
    if (!rc) rc = dev_reserve(ctx, out, (size_t)pairs * 1248 * sizeof(u32));
    if (!rc) rc = mt_state_at(ctx, seed, first, state.as<u32>(), ctx->compute);
    if (rc == 1 && !ctx->err[0]) ctx_fail(ctx, "mt19937_host_from: jump tables unavailable");
    if (!rc) {
        FASTF_LAUNCH(fastf_mt19937_kernel, 1, FASTF_MT_THREADS, 0, ctx->compute, seed, state.as<u32>(), 0u, (u64)0, pairs, (u64)0, out.as<u32>(), (u32 *)nullptr);
        ctx->launches++;
        if (cudaGetLastError() != cudaSuccess) rc = ctx_fail(ctx, "mt19937 launch failed");
    }
    if (!rc) rc = fastf_memcpy_d2h(ctx, out_words, out.p, (size_t)n * sizeof(u32));
    dev_release(ctx, state);
    dev_release(ctx, out);
    return rc;
}
extern "C" int fastf_mt19937_host(fastf_ctx *ctx, uint32_t seed, uint64_t n, uint32_t *out_words) { return mt_host_common(ctx, seed, n, 0, out_words, nullptr); }
extern "C" int fastf_mt19937_keepbits_host(fastf_ctx *ctx, uint32_t seed, uint64_t n, uint64_t threshold, uint32_t *out_bits) { return mt_host_common(ctx, seed, n, threshold, nullptr, out_bits); }

extern "C" int fastf_sort_u64_host(fastf_ctx *ctx, uint64_t *keys, uint32_t *vals, uint64_t n, uint32_t key_bits)
{
    CK(cudaSetDevice(ctx->device));
    if (n == 0) return 0;
    DevBuf dk, dv;
    int rc = dev_reserve(ctx, dk, n * sizeof(u64));
    if (!rc && vals) rc = dev_reserve(ctx, dv, n * sizeof(u32));
    if (!rc) rc = fastf_memcpy_h2d(ctx, dk.p, keys, n * sizeof(u64));
    if (!rc && vals) rc = fastf_memcpy_h2d(ctx, dv.p, vals, n * sizeof(u32));
    if (!rc) rc = fastf_sort_u64_device(ctx, dk.as<u64>(), vals ? dv.as<u32>() : nullptr, n, key_bits);
    if (!rc) rc = fastf_memcpy_d2h(ctx, keys, dk.p, n * sizeof(u64));
    if (!rc && vals) rc = fastf_memcpy_d2h(ctx, vals, dv.p, n * sizeof(u32));
    dev_release(ctx, dk);
    dev_release(ctx, dv);
    return rc;
}

// Distinct keys of a host array with their multiplicities: stable radix sort + run-length heads on the device (K4), the copies of
// a key = distance between consecutive heads.  What `-u/--umicopies` needs (reference src/bam2db_ds.c:527-530: COUNT(*) GROUP BY
// cell, feature, umi): out_keys ascending, out_counts[i] copies of out_keys[i]; both malloc'ed here, free() them.
extern "C" int fastf_unique_counts_host(fastf_ctx *ctx, const uint64_t *keys, uint64_t n, uint32_t key_bits, uint64_t **out_keys, uint32_t **out_counts, uint64_t *n_unique)
{
    CK(cudaSetDevice(ctx->device));
    *out_keys = nullptr; *out_counts = nullptr; *n_unique = 0;
    if (n == 0) return 0;
    DevBuf dk;
    RleScratch R;
    u64 ngroups = 0;
    int rc = dev_reserve(ctx, dk, n * sizeof(u64));
    if (!rc) rc = fastf_memcpy_h2d(ctx, dk.p, keys, n * sizeof(u64));
    if (!rc) rc = fastf_sort_u64_device(ctx, dk.as<u64>(), nullptr, n, key_bits);
    if (!rc) rc = rle_groups(ctx, R, dk.as<u64>(), nullptr, n, 0, 64, 0, &ngroups, nullptr, ctx->compute);
    u32 *first = nullptr;
    if (!rc) {
        *out_keys = (uint64_t *)malloc(std::max<u64>(ngroups, 1) * sizeof(uint64_t));
        *out_counts = (uint32_t *)malloc(std::max<u64>(ngroups, 1) * sizeof(uint32_t));
        first = (u32 *)malloc(std::max<u64>(ngroups, 1) * sizeof(u32));
        if (!*out_keys || !*out_counts || !first) rc = ctx_fail(ctx, "unique_counts: out of host memory for %llu groups", (unsigned long long)ngroups);
    }
    if (!rc && ngroups) rc = d2h_pageable(ctx, *out_keys, R.grp_key.p, ngroups * sizeof(u64), ctx->compute);
    if (!rc && ngroups) rc = d2h_pageable(ctx, first, R.grp_first.p, ngroups * sizeof(u32), ctx->compute);
    if (!rc) {
        for (u64 g = 0; g < ngroups; g++) (*out_counts)[g] = (u32)((g + 1 < ngroups ? (u64)first[g + 1] : n) - first[g]);
        *n_unique = ngroups;
    } else {
        free(*out_keys); free(*out_counts); *out_keys = nullptr; *out_counts = nullptr;
    }
    free(first);
    dev_release(ctx, dk);
    rle_scratch_release(ctx, R);
    return rc;
}

