// K4 -- (cell, gene, UMI) deduplication and per-(gene, cell) UMI counting on device.
//
// Replaces the reference's sqlite aggregation: the INSERT loop (reference src/bam2db_ds.c:351-435)
// followed by  CREATE TABLE mtx AS SELECT feature_index, cell_index, COUNT(DISTINCT encoded_umi)
// ... GROUP BY cell_index, feature_index  (reference src/bam2db_ds.c:480-483).
//
//   packed u64 keys  --LSD radix sort (8-bit digits)-->  sorted keys
//   --run-length heads-->  distinct (cell, gene, umi)  --segmented count-->  COO rows sorted by (cell, gene)
//
// The sort is a stable least-significant-digit radix sort written for this key shape: per pass a
// tile histogram kernel, a per-digit row scan (scan_mt_sample.cuh) and a scatter kernel that ranks
// keys inside a tile with warp match-any, reorders them through shared memory and writes each digit
// run contiguously.  The same kernels sort (key, u32 value) pairs for `freq`, and (key, rate index)
// pairs for the depth sweep, whose first pass sorts by the value.
#pragma once
#include "common.cuh"

#define FASTF_RS_THREADS 256
#define FASTF_RS_ITEMS 8
#define FASTF_RS_TILE (FASTF_RS_THREADS * FASTF_RS_ITEMS)   // 2048 keys per tile
#define FASTF_RS_WARPS (FASTF_RS_THREADS / 32)

// shift == FASTF_SORT_VAL_DIGIT: the pass sorts by the low 8 bits of the u32 payload instead of a window of the key (the depth
// sweep's rate index, sorted as the least significant digit so that equal keys end up in ascending payload order)
#define FASTF_SORT_VAL_DIGIT 64u
template <bool HAS_VAL>
__device__ __forceinline__ u32 fastf_radix_digit(u64 key, u32 val, u32 shift) { return (HAS_VAL && shift == FASTF_SORT_VAL_DIGIT) ? (val & 255u) : ((u32)(key >> shift) & 255u); }

// hist layout: [256 digits][ntiles]  (row = digit, so that one CTA scans one digit row)
__global__ void __launch_bounds__(FASTF_RS_THREADS) fastf_radix_hist_kernel(const u64 *__restrict__ keys, const u32 *__restrict__ vals, u64 n, u32 shift, u32 *__restrict__ hist, u32 ntiles)
{
    __shared__ u32 s_cnt[256];
    s_cnt[threadIdx.x] = 0;
    __syncthreads();
    const u64 base = (u64)blockIdx.x * FASTF_RS_TILE;
#pragma unroll
    for (int k = 0; k < FASTF_RS_ITEMS; k++) {
        u64 i = base + (u64)k * FASTF_RS_THREADS + threadIdx.x;
        if (i < n) atomicAdd(&s_cnt[shift == FASTF_SORT_VAL_DIGIT ? (vals[i] & 255u) : ((u32)(keys[i] >> shift) & 255u)], 1u);
    }
    __syncthreads();
    hist[(u64)threadIdx.x * ntiles + blockIdx.x] = s_cnt[threadIdx.x];
}

// tile_off = hist after the per-digit row scan (exclusive within the digit); digit_base = exclusive scan of the digit totals.
template <bool HAS_VAL>
__global__ void __launch_bounds__(FASTF_RS_THREADS)
fastf_radix_scatter_kernel(const u64 *__restrict__ keys_in, const u32 *__restrict__ vals_in, u64 *__restrict__ keys_out, u32 *__restrict__ vals_out, u64 n, u32 shift,
                           const u32 *__restrict__ tile_off, const u32 *__restrict__ digit_base, u32 ntiles)
{
    __shared__ u64 s_keys[FASTF_RS_TILE];
    __shared__ u32 s_vals[HAS_VAL ? FASTF_RS_TILE : 1];
    __shared__ u32 s_cnt[FASTF_RS_WARPS][256];
    __shared__ u32 s_dbase[256];   // first sorted position of digit d inside the tile
    __shared__ u32 s_gbase[256];   // global output index of that position
    const u32 tid = threadIdx.x, lane = tid & 31u, w = tid >> 5;
    const u64 base = (u64)blockIdx.x * FASTF_RS_TILE;
    const u32 nvalid = (u32)((n - base) < (u64)FASTF_RS_TILE ? (n - base) : (u64)FASTF_RS_TILE);
    for (u32 i = tid; i < FASTF_RS_WARPS * 256; i += FASTF_RS_THREADS) (&s_cnt[0][0])[i] = 0;
    __syncthreads();

    // warp w owns tile elements [w*256, w*256+256) in 8 rounds of 32 consecutive keys: ranks stay stable
    u64 key[FASTF_RS_ITEMS];
    u32 val[FASTF_RS_ITEMS];
    u32 rank[FASTF_RS_ITEMS];
#pragma unroll
    for (int r = 0; r < FASTF_RS_ITEMS; r++) {
        const u32 idx = w * (32 * FASTF_RS_ITEMS) + r * 32 + lane;
        const bool ok = idx < nvalid;
        key[r] = ok ? keys_in[base + idx] : ~0ull;   // padding sorts last inside digit 255 and is never written
        if (HAS_VAL) val[r] = ok ? vals_in[base + idx] : 0u;
        const u32 d = ok ? fastf_radix_digit<HAS_VAL>(key[r], HAS_VAL ? val[r] : 0u, shift) : 255u;
        const u32 peers = __match_any_sync(FASTF_FULL_MASK, d);
        const u32 before = s_cnt[w][d];
        __syncwarp();
        if (lane == (u32)__ffs((int)peers) - 1u) s_cnt[w][d] = before + (u32)__popc(peers);
        __syncwarp();
        rank[r] = before + (u32)__popc(peers & fastf_lanemask_lt());
    }
    __syncthreads();
    // thread d: per-warp exclusive offsets of digit d, then exclusive scan over digits
    u32 total = 0;
#pragma unroll
    for (int ww = 0; ww < FASTF_RS_WARPS; ww++) { u32 c = s_cnt[ww][tid]; s_cnt[ww][tid] = total; total += c; }
    u32 dummy;
    const u32 dstart = fastf_block_exscan<FASTF_RS_THREADS>(total, &dummy);
    s_dbase[tid] = dstart;
    s_gbase[tid] = digit_base[tid] + tile_off[(u64)tid * ntiles + blockIdx.x];
    __syncthreads();
#pragma unroll
    for (int r = 0; r < FASTF_RS_ITEMS; r++) {
        const u32 idx = w * (32 * FASTF_RS_ITEMS) + r * 32 + lane;
        const u32 d = idx < nvalid ? fastf_radix_digit<HAS_VAL>(key[r], HAS_VAL ? val[r] : 0u, shift) : 255u;
        const u32 pos = s_dbase[d] + s_cnt[w][d] + rank[r];
        s_keys[pos] = key[r];
        if (HAS_VAL) s_vals[pos] = val[r];
    }
    __syncthreads();
    for (u32 p = tid; p < nvalid; p += FASTF_RS_THREADS) {
        const u64 k = s_keys[p];
        const u32 d = fastf_radix_digit<HAS_VAL>(k, HAS_VAL ? s_vals[p] : 0u, shift);
        const u64 g = (u64)s_gbase[d] + (p - s_dbase[d]);
        keys_out[g] = k;
        if (HAS_VAL) vals_out[g] = s_vals[p];
    }
}

// exclusive scan of the 256 digit totals (one CTA of 256 threads)
__global__ void __launch_bounds__(256) fastf_radix_digit_base_kernel(const u32 *__restrict__ totals, u32 *__restrict__ digit_base)
{
    u32 dummy;
    digit_base[threadIdx.x] = fastf_block_exscan<256>(totals[threadIdx.x], &dummy);
}

// ------------------------------------------------------------------------------------------------
// Run-length / segmented count over SORTED keys (two-phase: tile counts -> row scan -> emit).
//   group  = key >> group_shift                      ((cell, gene) for bam2db; the whole key for freq)
//   a key "counts" when it differs from its predecessor and its non-NULL bit (bit nn_bit) is set
//   (COUNT(DISTINCT x) ignores NULL, reference src/bam2db_ds.c:481); nn_bit >= 64 means "always set".
// Emits per group: its group value, the index of its first element, and the number of counting keys
// that precede it (exclusive); counts are differences of consecutive entries.
// ------------------------------------------------------------------------------------------------
#define FASTF_RLE_THREADS 256
#define FASTF_RLE_ITEMS 8
#define FASTF_RLE_TILE (FASTF_RLE_THREADS * FASTF_RLE_ITEMS)

// Rate predicate of the depth sweep (rate == nullptr: off).  The keys are then DISTINCT, rate[i] is the smallest rate index that
// keeps key i and grate[i] the smallest rate index that keeps any key of the group starting at i (no group starts at i: ~0u).  At
// rate `max` a key counts when rate[i] <= max and a group exists when grate[i] <= max.  A group that does not exist at `max` holds
// no counting key, so the counts (differences of the emitted groups' prefixes) stay exact.
struct FastfRatePred {
    const u32 *rate, *grate;
    u32 max;
};

__device__ __forceinline__ void fastf_rle_flags(const u64 *__restrict__ keys, u64 i, u32 group_shift, u32 nn_bit, const FastfRatePred &P, bool *head, bool *distinct)
{
    const u64 k = keys[i];
    if (P.rate) {
        *head = P.grate[i] <= P.max;
        *distinct = (nn_bit >= 64 || ((k >> nn_bit) & 1ull)) && P.rate[i] <= P.max;
        return;
    }
    const bool first = (i == 0);
    const u64 prev = first ? 0 : keys[i - 1];
    *head = first || ((k >> group_shift) != (prev >> group_shift));
    const bool nn = nn_bit >= 64 ? true : ((k >> nn_bit) & 1ull);
    *distinct = nn && (first || k != prev);
}

// tile_counts layout: [2][ntiles]: row 0 = group heads, row 1 = counting keys
__global__ void __launch_bounds__(FASTF_RLE_THREADS)
fastf_rle_count_kernel(const u64 *__restrict__ keys, u64 n, u32 group_shift, u32 nn_bit, FastfRatePred pred, u32 *__restrict__ tile_counts, u32 ntiles)
{
    __shared__ u32 s_h, s_d;
    if (threadIdx.x == 0) { s_h = 0; s_d = 0; }
    __syncthreads();
    const u64 base = (u64)blockIdx.x * FASTF_RLE_TILE;
    u32 h = 0, d = 0;
#pragma unroll
    for (int k = 0; k < FASTF_RLE_ITEMS; k++) {
        u64 i = base + (u64)k * FASTF_RLE_THREADS + threadIdx.x;
        if (i < n) { bool hh, dd; fastf_rle_flags(keys, i, group_shift, nn_bit, pred, &hh, &dd); h += hh; d += dd; }
    }
    h = __reduce_add_sync(FASTF_FULL_MASK, h);
    d = __reduce_add_sync(FASTF_FULL_MASK, d);
    if ((threadIdx.x & 31u) == 0) { atomicAdd(&s_h, h); atomicAdd(&s_d, d); }
    __syncthreads();
    if (threadIdx.x == 0) { tile_counts[blockIdx.x] = s_h; tile_counts[ntiles + blockIdx.x] = s_d; }
}

// vals (optional) = payload of the sorted keys; grp_val gets the payload of each group's first element
// (for freq: the read ordinal of the key's first occurrence, because the sort is stable).
__global__ void __launch_bounds__(FASTF_RLE_THREADS)
fastf_rle_emit_kernel(const u64 *__restrict__ keys, const u32 *__restrict__ vals, u64 n, u32 group_shift, u32 nn_bit, FastfRatePred pred, const u32 *__restrict__ tile_off, u32 ntiles,
                      u64 *__restrict__ grp_key, u32 *__restrict__ grp_first, u32 *__restrict__ grp_dstart, u32 *__restrict__ grp_val)
{
    const u64 base = (u64)blockIdx.x * FASTF_RLE_TILE + (u64)threadIdx.x * FASTF_RLE_ITEMS;
    u32 hflags = 0, dflags = 0, hc = 0, dc = 0;
#pragma unroll
    for (int k = 0; k < FASTF_RLE_ITEMS; k++) {
        u64 i = base + k;
        if (i < n) { bool hh, dd; fastf_rle_flags(keys, i, group_shift, nn_bit, pred, &hh, &dd); hflags |= (u32)hh << k; dflags |= (u32)dd << k; hc += hh; dc += dd; }
    }
    u32 tot;
    u32 hex = fastf_block_exscan<FASTF_RLE_THREADS>(hc, &tot) + tile_off[blockIdx.x];
    u32 dex = fastf_block_exscan<FASTF_RLE_THREADS>(dc, &tot) + tile_off[ntiles + blockIdx.x];
#pragma unroll
    for (int k = 0; k < FASTF_RLE_ITEMS; k++) {
        if (hflags & (1u << k)) {
            u64 i = base + k;
            grp_key[hex] = keys[i] >> group_shift;
            grp_first[hex] = (u32)i;
            grp_dstart[hex] = dex;
            if (vals) grp_val[hex] = vals[i];
            hex++;
        }
        if (dflags & (1u << k)) dex++;
    }
}

// count[g] = next[g+1] - next[g] with next[ngroups] = end_total; optional split of the group key
// into (cell = key >> bits_gene, gene = key & mask) for the COO output.
__global__ void __launch_bounds__(256)
fastf_rle_finish_kernel(const u32 *__restrict__ start, u32 ngroups, u32 end_total, u32 *__restrict__ count,
                        const u64 *__restrict__ grp_key, u32 bits_gene, u32 *__restrict__ out_gene, u32 *__restrict__ out_cell)
{
    u32 g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= ngroups) return;
    u32 nxt = (g + 1 < ngroups) ? start[g + 1] : end_total;
    count[g] = nxt - start[g];
    if (out_gene) {
        u64 k = grp_key[g];
        out_gene[g] = (u32)(k & ((1ull << bits_gene) - 1ull));
        out_cell[g] = (u32)(k >> bits_gene);
    }
}

// Depth sweep: grate[] of FastfRatePred over DISTINCT sorted keys.  The first key of every group gets the minimum of rate[] over
// its group, every other key ~0u.  A warp takes the groups that start in its 32 keys one after another and reads each with all 32
// lanes, so a long group (thousands of UMIs of one gene in one cell) costs len/32 coalesced steps, not len dependent ones.
__global__ void __launch_bounds__(256)
fastf_group_rate_kernel(const u64 *__restrict__ keys, const u32 *__restrict__ rate, u64 n, u32 group_shift, u32 *__restrict__ grate)
{
    const u32 lane = threadIdx.x & 31u;
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u64 warp0 = j - lane;
    const bool start = j < n && (j == 0 || (keys[j - 1] >> group_shift) != (keys[j] >> group_shift));
    if (j < n && !start) grate[j] = ~0u;
    u32 pending = __ballot_sync(FASTF_FULL_MASK, start);
    while (pending) {
        const u32 src = (u32)__ffs((int)pending) - 1u;
        pending &= pending - 1u;
        const u64 s0 = warp0 + src;
        const u64 g = keys[s0] >> group_shift;
        u32 m = ~0u;
        for (u64 k0 = s0;; k0 += 32) {
            const u64 k = k0 + lane;
            const bool in = k < n && (keys[k] >> group_shift) == g;
            if (in && rate[k] < m) m = rate[k];
            if (__ballot_sync(FASTF_FULL_MASK, in) != FASTF_FULL_MASK) break;   // a group is contiguous: its end is in this step
        }
        m = __reduce_min_sync(FASTF_FULL_MASK, m);
        if (lane == src) grate[s0] = m;
    }
}
