// Part of the libfastf_gpu translation unit (capi.cu includes it, in this order; it is not a header of its own):
// launch helpers (inflate engines, CRC-32), string tables on the device, per-chunk block index.
#pragma once

// ---------------------------------------------------------------------------------------------------
// launch helpers
// ---------------------------------------------------------------------------------------------------
#define FASTF_INFLATE_HW_ENGINE 0x100u   // flag in the `inflate_lanes` argument (include/fastf_gpu.h)

// after a hardware-engine batch: actual byte counts -> status words
__global__ void __launch_bounds__(256) fastf_de_check_kernel(u32 *__restrict__ act_status, const u32 *__restrict__ isize, u32 n)
{
    u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) act_status[i] = (isize[i] != 0 && act_status[i] != isize[i]) ? (u32)FASTF_ST_SIZE_MISMATCH : 0u;
}

struct DeScratch {   // per-launch state of the inflate engines
#ifndef FASTF_EMU
    std::vector<CUmemDecompressParams> params;   // parameter array of a hardware-engine batch; must stay alive until the batch has run
#endif
    DevBuf counter;                               // work counter of the persistent thread-per-stream kernel
    DevBuf sorted;                                // its per-stream sorted-symbol lists (global scratch)
};
#define FASTF_INFLATE_TPS 1u   // inflate_lanes 1..4 select a shape of the thread-per-stream kernel; 8/16/32 the lock-step kernel
#define FASTF_INFLATE_DEFAULT 2u   // 0 = default: the thread-per-stream kernel

// CRC-32 of every inflated block against its BGZF trailer (htslib does this in bgzf_read_block); sets FASTF_ST_BAD_CRC in status[]
static int launch_crc(fastf_ctx *ctx, u32 lanes, const u8 *comp, u64 comp_total, const u64 *in_off, const u32 *in_len, const u8 *infl, const u64 *out_off, const u32 *isize, u32 nblocks,
                      u32 *status, cudaStream_t s)
{
    if (nblocks == 0 || (lanes & FASTF_INFLATE_NO_CRC)) return 0;
    u32 grid = (nblocks + FASTF_CRC_WARPS - 1) / FASTF_CRC_WARPS;
    if (grid > (u32)ctx->n_sm) grid = (u32)ctx->n_sm;   // one CTA per SM (the tables are built once per CTA); the rest is a grid-stride loop
#ifndef FASTF_EMU
    if (!ctx->crc_attr_set) { CK(cudaFuncSetAttribute(fastf_bgzf_crc32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FastfCrcTables))); ctx->crc_attr_set = true; }
#endif
    FASTF_LAUNCH(fastf_bgzf_crc32_kernel, grid, FASTF_CRC_WARPS * 32, sizeof(FastfCrcTables), s, comp, comp_total, in_off, in_len, infl, out_off, isize, nblocks, status);
    CKL("bgzf_crc32");
    return 0;
}

// h_* = host copies of the block index (needed to build the engine's parameter array)
static int launch_inflate(fastf_ctx *ctx, u32 lanes, const u8 *comp, u64 comp_total, const u64 *in_off, const u32 *in_len, const u64 *out_off, const u32 *isize, u32 nblocks, u8 *out,
                          u32 *status, cudaStream_t s, DeScratch *de, const u64 *h_in_off, const u32 *h_in_len, const u64 *h_out_off, const u32 *h_isize)
{
    if (nblocks == 0) return 0;
    if (lanes & FASTF_INFLATE_HW_ENGINE) {
#ifdef FASTF_EMU
        return ctx_fail(ctx, "inflate: the hardware decompression engine does not exist in the emulator build");
#else
        // Blackwell decompression engine: one DEFLATE operation per BGZF block, submitted as one batch in stream order.
        // dstActBytes lands in the status array and is turned into status bits by a small kernel afterwards.
        de->params.clear();
        de->params.reserve(nblocks);
        for (u32 i = 0; i < nblocks; i++) {
            if (h_isize[i] == 0) continue;   // empty (EOF) blocks produce nothing
            CUmemDecompressParams p;
            memset(&p, 0, sizeof p);
            p.srcNumBytes = h_in_len[i];
            p.dstNumBytes = h_isize[i];
            p.dstActBytes = (cuuint32_t *)(status + i);
            p.src = comp + h_in_off[i];
            p.dst = out + h_out_off[i];
            p.algo = CU_MEM_DECOMPRESS_ALGORITHM_DEFLATE;
            de->params.push_back(p);
        }
        CK(cudaMemsetAsync(status, 0, (size_t)nblocks * sizeof(u32), s));
        if (!de->params.empty()) {
            // the driver entry point is resolved through the runtime: no link-time dependency on libcuda (absent on build hosts)
            typedef CUresult (*decompress_fn)(CUmemDecompressParams *, size_t, unsigned int, size_t *, CUstream);
            static decompress_fn fn = nullptr;
            if (!fn) {
                void *sym = nullptr;
                cudaDriverEntryPointQueryResult q;
                if (cudaGetDriverEntryPoint("cuMemBatchDecompressAsync", &sym, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess || !sym)
                    return ctx_fail(ctx, "inflate: this driver does not export cuMemBatchDecompressAsync (hardware decompression engine unavailable)");
                fn = (decompress_fn)sym;
            }
            size_t erri = 0;
            CUresult r = fn(de->params.data(), de->params.size(), 0, &erri, (CUstream)s);
            if (r != CUDA_SUCCESS)
                return ctx_fail(ctx, "inflate: cuMemBatchDecompressAsync failed (CUresult %d) at operation %zu; is the hardware decompression engine available on this GPU?", (int)r, erri);
        }
        FASTF_LAUNCH(fastf_de_check_kernel, (nblocks + 255) / 256, 256, 0, s, status, isize, nblocks);
        CKL("de_check");
        return 0;
#endif
    }
    lanes &= 0xffu;   // the kernel shape; the flag bits (no-CRC, straddle) were for the callers
    if (lanes >= 1 && lanes <= 4) {
        // thread-per-stream kernel: persistent CTAs (one per SM), FASTF_TPS_STREAMS streams each; blocks are handed out by a global counter.
        // one shape is built: <FASTF_TPS_LANES decoding lanes per decoder warp, FASTF_TPS_SVC_WARPS service warps> (bgzf_inflate_tps.cuh); lanes 1..4 all select it
        const size_t smem = sizeof(FastfTpsStream) * FASTF_TPS_STREAMS + sizeof(FastfTpsShared);
        TRY(dev_reserve(ctx, de->counter, 64));
        CK(cudaMemsetAsync(de->counter.p, 0, sizeof(u32), s));
        FastfTpsArgs A;
        A.comp = comp; A.comp_total = comp_total; A.in_off = in_off; A.in_len = in_len; A.out_off = out_off; A.isize = isize; A.nblocks = nblocks; A.out = out; A.status = status;
        A.next_block = de->counter.as<u32>();
        u32 grid = (nblocks + FASTF_TPS_STREAMS - 1) / FASTF_TPS_STREAMS;
        if (grid > (u32)ctx->n_sm) grid = (u32)ctx->n_sm;
        TRY(dev_reserve(ctx, de->sorted, (size_t)grid * FASTF_TPS_STREAMS * FASTF_TPS_SORTED_U16 * sizeof(u16)));
        A.sorted = de->sorted.as<u16>();
#ifndef FASTF_EMU
        if (!ctx->tps_attr_set) {
            CK(cudaFuncSetAttribute(fastf_bgzf_inflate_tps_kernel<FASTF_TPS_LANES, FASTF_TPS_SVC_WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            ctx->tps_attr_set = true;
        }
#endif
        FASTF_LAUNCH((fastf_bgzf_inflate_tps_kernel<FASTF_TPS_LANES, FASTF_TPS_SVC_WARPS>), grid, FASTF_TPS_THREADS, smem, s, A);
        CKL("bgzf_inflate_tps");
        return 0;
    }
    if (lanes == 8) {
        FASTF_LAUNCH(fastf_bgzf_inflate_kernel<8>, (nblocks + 3) / 4, 32, 0, s, comp, comp_total, in_off, in_len, out_off, isize, nblocks, out, status);
    } else if (lanes == 16) {
        FASTF_LAUNCH(fastf_bgzf_inflate_kernel<16>, (nblocks + 1) / 2, 32, 0, s, comp, comp_total, in_off, in_len, out_off, isize, nblocks, out, status);
    } else {
        FASTF_LAUNCH(fastf_bgzf_inflate_kernel<32>, nblocks, 32, 0, s, comp, comp_total, in_off, in_len, out_off, isize, nblocks, out, status);
    }
    CKL("bgzf_inflate");
    return 0;
}

// exclusive scan of every row of a [nrows][n] u32 matrix in place; totals[nrows]
static int launch_scan_rows(fastf_ctx *ctx, u32 *data, u64 n, u32 nrows, u32 *totals, cudaStream_t s)
{
    FASTF_LAUNCH(fastf_scan_rows_kernel, nrows, FASTF_SCAN_THREADS, 0, s, data, n, totals);
    CKL("scan_rows");
    return 0;
}

// ---- LSD radix sort over a chosen set of 8-bit digit windows --------------------------------------
struct SortScratch {
    DevBuf hist, totals, dbase;
};
// Windows: greedy cover of the bit positions set in `varying` (bits that differ between keys).
static int plan_windows(u64 varying, u32 *shifts)
{
    int n = 0;
    u32 b = 0;
    while (b < 64) {
        if ((varying >> b) & 1ull) { shifts[n++] = b; b += 8; } else b++;
    }
    return n;
}
// Sorts n keys (and optional u32 payload).  keys/alt (and vals/vals_alt) are ping-pong buffers of n elements;
// *sorted_in_alt tells where the result ended up.  A pass whose shift is FASTF_SORT_VAL_DIGIT sorts by the payload's low byte.
static int sort_keys(fastf_ctx *ctx, SortScratch &S, u64 *keys, u64 *alt, u32 *vals, u32 *vals_alt, u64 n, const u32 *shifts, int npass, bool *sorted_in_alt, cudaStream_t s)
{
    *sorted_in_alt = false;
    if (n == 0 || npass == 0) return 0;
    if (n >= 0xffffffffull) return ctx_fail(ctx, "sort: %llu keys exceed the 2^32-1 limit of one device sort", (unsigned long long)n);
    const u32 ntiles = (u32)((n + FASTF_RS_TILE - 1) / FASTF_RS_TILE);
    TRY(dev_reserve(ctx, S.hist, (size_t)256 * ntiles * sizeof(u32)));
    TRY(dev_reserve(ctx, S.totals, 256 * sizeof(u32)));
    TRY(dev_reserve(ctx, S.dbase, 256 * sizeof(u32)));
    u64 *src = keys, *dst = alt;
    u32 *vsrc = vals, *vdst = vals_alt;
    for (int p = 0; p < npass; p++) {
        if (shifts[p] == FASTF_SORT_VAL_DIGIT && !vals) return ctx_fail(ctx, "sort: a payload-digit pass needs a payload");
        FASTF_LAUNCH(fastf_radix_hist_kernel, ntiles, FASTF_RS_THREADS, 0, s, (const u64 *)src, (const u32 *)vsrc, n, shifts[p], S.hist.as<u32>(), ntiles);
        CKL("radix_hist");
        TRY(launch_scan_rows(ctx, S.hist.as<u32>(), ntiles, 256, S.totals.as<u32>(), s));
        FASTF_LAUNCH(fastf_radix_digit_base_kernel, 1, 256, 0, s, (const u32 *)S.totals.as<u32>(), S.dbase.as<u32>());
        CKL("radix_digit_base");
        if (vals) {
            FASTF_LAUNCH(fastf_radix_scatter_kernel<true>, ntiles, FASTF_RS_THREADS, 0, s, (const u64 *)src, (const u32 *)vsrc, dst, vdst, n, shifts[p], (const u32 *)S.hist.as<u32>(),
                         (const u32 *)S.dbase.as<u32>(), ntiles);
        } else {
            FASTF_LAUNCH(fastf_radix_scatter_kernel<false>, ntiles, FASTF_RS_THREADS, 0, s, (const u64 *)src, (const u32 *)nullptr, dst, (u32 *)nullptr, n, shifts[p],
                         (const u32 *)S.hist.as<u32>(), (const u32 *)S.dbase.as<u32>(), ntiles);
        }
        CKL("radix_scatter");
        std::swap(src, dst);
        std::swap(vsrc, vdst);
    }
    *sorted_in_alt = (src == alt);
    return 0;
}
static void sort_scratch_release(fastf_ctx *ctx, SortScratch &S) { dev_release(ctx, S.hist); dev_release(ctx, S.totals); dev_release(ctx, S.dbase); }

// OR / AND of all keys -> which bit positions vary (device reduction, 16 bytes back)
__global__ void __launch_bounds__(256) fastf_key_bits_kernel(const u64 *__restrict__ keys, u64 n, u64 *__restrict__ or_and)
{
    u64 o = 0, a = ~0ull;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) { u64 k = keys[i]; o |= k; a &= k; }
    for (int d = 16; d; d >>= 1) { o |= __shfl_xor_sync(FASTF_FULL_MASK, o, d); a &= __shfl_xor_sync(FASTF_FULL_MASK, a, d); }
    if ((threadIdx.x & 31u) == 0) { atomicOr((unsigned long long *)&or_and[0], (unsigned long long)o); atomicAnd((unsigned long long *)&or_and[1], (unsigned long long)a); }
}

// ---- run-length / segmented count over sorted keys ------------------------------------------------
struct RleScratch {
    DevBuf tile_counts, tile_totals, grp_key, grp_first, grp_dstart, grp_val, count, out_gene, out_cell;
    PinBuf totals_host;
};
static void rle_scratch_release(fastf_ctx *ctx, RleScratch &R)
{
    dev_release(ctx, R.tile_counts); dev_release(ctx, R.tile_totals); dev_release(ctx, R.grp_key); dev_release(ctx, R.grp_first); dev_release(ctx, R.grp_dstart); dev_release(ctx, R.grp_val);
    dev_release(ctx, R.count); dev_release(ctx, R.out_gene); dev_release(ctx, R.out_cell);
    pin_release(ctx, R.totals_host);
}
// After this: R.grp_key/grp_first/grp_dstart(/grp_val)/count hold ngroups entries on device; with split_bits_gene > 0
// R.out_gene / R.out_cell hold the split group key.  pred: the depth sweep's rate predicate (radix_dedup.cuh), off by default.
static int rle_groups(fastf_ctx *ctx, RleScratch &R, const u64 *sorted, const u32 *vals, u64 n, u32 group_shift, u32 nn_bit, u32 split_bits_gene, u64 *ngroups_out, u64 *ndistinct_out,
                      cudaStream_t s, FastfRatePred pred = FastfRatePred{nullptr, nullptr, 0u})
{
    *ngroups_out = 0;
    if (ndistinct_out) *ndistinct_out = 0;
    if (n == 0) return 0;
    if (n >= 0xffffffffull) return ctx_fail(ctx, "rle: %llu keys exceed the 2^32-1 limit", (unsigned long long)n);
    const u32 ntiles = (u32)((n + FASTF_RLE_TILE - 1) / FASTF_RLE_TILE);
    TRY(dev_reserve(ctx, R.tile_counts, (size_t)2 * ntiles * sizeof(u32)));
    TRY(dev_reserve(ctx, R.tile_totals, 2 * sizeof(u32)));
    TRY(pin_reserve(ctx, R.totals_host, 2 * sizeof(u32)));
    FASTF_LAUNCH(fastf_rle_count_kernel, ntiles, FASTF_RLE_THREADS, 0, s, sorted, n, group_shift, nn_bit, pred, R.tile_counts.as<u32>(), ntiles);
    CKL("rle_count");
    TRY(launch_scan_rows(ctx, R.tile_counts.as<u32>(), ntiles, 2, R.tile_totals.as<u32>(), s));
    CK(cudaMemcpyAsync(R.totals_host.p, R.tile_totals.p, 2 * sizeof(u32), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    const u32 ngroups = R.totals_host.as<u32>()[0], ndistinct = R.totals_host.as<u32>()[1];
    TRY(dev_reserve(ctx, R.grp_key, (size_t)ngroups * sizeof(u64)));
    TRY(dev_reserve(ctx, R.grp_first, (size_t)ngroups * sizeof(u32)));
    TRY(dev_reserve(ctx, R.grp_dstart, (size_t)ngroups * sizeof(u32)));
    TRY(dev_reserve(ctx, R.count, (size_t)ngroups * sizeof(u32)));
    if (vals) TRY(dev_reserve(ctx, R.grp_val, (size_t)ngroups * sizeof(u32)));
    if (split_bits_gene) { TRY(dev_reserve(ctx, R.out_gene, (size_t)ngroups * sizeof(u32))); TRY(dev_reserve(ctx, R.out_cell, (size_t)ngroups * sizeof(u32))); }
    FASTF_LAUNCH(fastf_rle_emit_kernel, ntiles, FASTF_RLE_THREADS, 0, s, sorted, vals, n, group_shift, nn_bit, pred, (const u32 *)R.tile_counts.as<u32>(), ntiles, R.grp_key.as<u64>(),
                 R.grp_first.as<u32>(), R.grp_dstart.as<u32>(), vals ? R.grp_val.as<u32>() : (u32 *)nullptr);
    CKL("rle_emit");
    if (ngroups) {
        FASTF_LAUNCH(fastf_rle_finish_kernel, (ngroups + 255) / 256, 256, 0, s, (const u32 *)R.grp_dstart.as<u32>(), ngroups, ndistinct, R.count.as<u32>(), (const u64 *)R.grp_key.as<u64>(),
                     split_bits_gene, split_bits_gene ? R.out_gene.as<u32>() : (u32 *)nullptr, split_bits_gene ? R.out_cell.as<u32>() : (u32 *)nullptr);
        CKL("rle_finish");
    }
    *ngroups_out = ngroups;
    if (ndistinct_out) *ndistinct_out = ndistinct;
    return 0;
}

// ---------------------------------------------------------------------------------------------------
// string tables -> device
// ---------------------------------------------------------------------------------------------------
struct DevTable {
    DevBuf slots, pool;
    FastfStrTableView view;
    u32 count = 0;
};
static int table_upload(fastf_ctx *ctx, DevTable &T, const char *keys, const u32 *off, u32 n)
{
    FastfStrTableHost H;
    H.init(n);
    for (u32 i = 0; i < n; i++) {
        // first insertion wins; the reference's hash_table_insert refuses duplicates (src/hashtable.c:70-95)
        H.insert(keys + off[i], off[i + 1] - off[i], i + 1);
    }
    H.finish();
    TRY(dev_reserve(ctx, T.slots, H.slots.size() * sizeof(FastfStrSlot)));
    TRY(dev_reserve(ctx, T.pool, H.pool.size()));
    CK(cudaMemcpy(T.slots.p, H.slots.data(), H.slots.size() * sizeof(FastfStrSlot), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(T.pool.p, H.pool.data(), H.pool.size(), cudaMemcpyHostToDevice));
    T.view.slots = T.slots.as<FastfStrSlot>();
    T.view.pool = T.pool.as<uint8_t>();
    T.view.mask = H.mask;
    memcpy(T.view.pw1, H.pw1, sizeof H.pw1);
    memcpy(T.view.pw2, H.pw2, sizeof H.pw2);
    T.count = n;
    return 0;
}
static u32 bits_for(u32 max_value)
{
    u32 b = 1;
    while (b < 32 && (max_value >> b)) b++;
    return b;
}

// ---------------------------------------------------------------------------------------------------
// chunked BGZF -> inflated bytes machinery shared by bam2db and freq
// ---------------------------------------------------------------------------------------------------
struct BlockIndexDev {   // per-chunk block index on device (one allocation, 8-byte fields first)
    DevBuf buf;
    PinBuf host;
    u32 cap_blocks = 0;
    u64 *in_off, *out_off, *stage_off, *dst_base;
    u32 *in_len, *isize, *nrec, *ncbv, *st_infl, *st_parse;
    u64 *h_in_off, *h_out_off, *h_stage_off;
    u32 *h_in_len, *h_isize;
};
static size_t index_bytes_dev(u32 nb) { return (size_t)nb * (4 * sizeof(u64) + 6 * sizeof(u32)); }
static size_t index_bytes_up(u32 nb) { return (size_t)nb * (3 * sizeof(u64) + 2 * sizeof(u32)); }
static int index_reserve(fastf_ctx *ctx, BlockIndexDev &I, u32 nb)
{
    if (nb <= I.cap_blocks) return 0;
    u32 cap = std::max(nb, I.cap_blocks * 2);
    cap = (cap + 63u) & ~63u;
    TRY(dev_reserve(ctx, I.buf, index_bytes_dev(cap)));
    TRY(pin_reserve(ctx, I.host, index_bytes_up(cap)));
    I.cap_blocks = cap;
    // upload region first (in_off, out_off, stage_off, in_len, isize), device-only region after
    u8 *d = I.buf.as<u8>();
    I.in_off = (u64 *)d; d += (size_t)cap * 8;
    I.out_off = (u64 *)d; d += (size_t)cap * 8;
    I.stage_off = (u64 *)d; d += (size_t)cap * 8;
    I.in_len = (u32 *)d; d += (size_t)cap * 4;
    I.isize = (u32 *)d; d += (size_t)cap * 4;
    I.dst_base = (u64 *)d; d += (size_t)cap * 8;
    I.nrec = (u32 *)d; d += (size_t)cap * 4;
    I.ncbv = (u32 *)d; d += (size_t)cap * 4;
    I.st_infl = (u32 *)d; d += (size_t)cap * 4;
    I.st_parse = (u32 *)d;
    u8 *h = I.host.as<u8>();
    I.h_in_off = (u64 *)h; h += (size_t)cap * 8;
    I.h_out_off = (u64 *)h; h += (size_t)cap * 8;
    I.h_stage_off = (u64 *)h; h += (size_t)cap * 8;
    I.h_in_len = (u32 *)h; h += (size_t)cap * 4;
    I.h_isize = (u32 *)h;
    return 0;
}
// The block index of a chunk (a few MB) is PULLED by a kernel out of the pinned host arrays instead of being pushed through the
// copy engine: there it queues behind the bulk H2D copies of the next chunks' compressed bytes (FIFO per direction) and the inflate
// that waits for it starts up to three copies late (measured: the first inflate of a host-fed job 90 ms after its bytes arrived).
__global__ void __launch_bounds__(256) fastf_pull_words_kernel(u32 *__restrict__ dst, const u32 *__restrict__ src_host, u64 n_words)
{
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n_words; i += (u64)gridDim.x * blockDim.x) dst[i] = src_host[i];
}
static int index_upload(fastf_ctx *ctx, BlockIndexDev &I, cudaStream_t s)
{
    const size_t bytes = index_bytes_up(I.cap_blocks);
#ifdef FASTF_EMU
    CK(cudaMemcpyAsync(I.buf.p, I.host.p, bytes, cudaMemcpyHostToDevice, s));
#else
    void *src = nullptr;
    CK(cudaHostGetDevicePointer(&src, I.host.p, 0));
    FASTF_LAUNCH(fastf_pull_words_kernel, 2 * ctx->n_sm, 256, 0, s, I.buf.as<u32>(), (const u32 *)src, (u64)(bytes / 4));
    CKL("pull_index");
#endif
    return 0;
}
static void index_release(fastf_ctx *ctx, BlockIndexDev &I) { dev_release(ctx, I.buf); pin_release(ctx, I.host); I.cap_blocks = 0; }
