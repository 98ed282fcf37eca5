// Prefix sums, the MT19937 keep-bit stream (K3), the depth-sampling compaction (K3b) and its several-rate form (the depth sweep).
#pragma once
#include "common.cuh"

// ------------------------------------------------------------------------------------------------
// Row scan: CTA r turns row r of a [nrows][n] u32 matrix into its exclusive prefix sum in place and
// stores the row total.  Used for: per-tile counts of every two-phase compaction, the per-digit tile
// histograms of the radix sort (256 rows), the per-chunk BGZF block counts.
// ------------------------------------------------------------------------------------------------
#define FASTF_SCAN_THREADS 1024
__global__ void __launch_bounds__(FASTF_SCAN_THREADS) fastf_scan_rows_kernel(u32 *__restrict__ data, u64 n, u32 *__restrict__ totals)
{
    u32 *row = data + (u64)blockIdx.x * n;
    u32 carry = 0;
    for (u64 base = 0; base < n; base += FASTF_SCAN_THREADS) {
        u64 i = base + threadIdx.x;
        u32 v = i < n ? row[i] : 0u;
        u32 tot;
        u32 ex = fastf_block_exscan<FASTF_SCAN_THREADS>(v, &tot);
        if (i < n) row[i] = carry + ex;
        carry += tot;
    }
    if (threadIdx.x == 0) totals[blockIdx.x] = carry;
}

// Per-chunk bookkeeping after the parse kernel: exclusive scan of the per-block CB-valid counts on top
// of the running candidate count -> dst_base[b]; accumulates the running record / candidate totals and
// ORs all block status words.  counters = {n_records, n_candidates, status_or}.  One CTA.
__global__ void __launch_bounds__(FASTF_SCAN_THREADS)
fastf_chunk_counts_kernel(const u32 *__restrict__ blk_nrec, const u32 *__restrict__ blk_ncbv, const u32 *__restrict__ blk_status_infl, const u32 *__restrict__ blk_status_parse,
                          u32 nblocks, u64 *__restrict__ dst_base, u64 *__restrict__ counters)
{
    __shared__ u64 s_rec;
    __shared__ u32 s_status;
    if (threadIdx.x == 0) { s_rec = 0; s_status = 0; }
    __syncthreads();
    u64 carry = counters[1];
    u64 rec = 0;
    u32 st = 0;
    for (u32 base = 0; base < nblocks; base += FASTF_SCAN_THREADS) {
        u32 i = base + threadIdx.x;
        u32 v = i < nblocks ? blk_ncbv[i] : 0u;
        if (i < nblocks) { rec += blk_nrec[i]; st |= blk_status_infl[i] | blk_status_parse[i]; }
        u32 tot;
        u32 ex = fastf_block_exscan<FASTF_SCAN_THREADS>(v, &tot);
        if (i < nblocks) dst_base[i] = carry + ex;
        carry += tot;
    }
    atomicAdd((unsigned long long *)&s_rec, (unsigned long long)rec);
    atomicOr(&s_status, st);
    __syncthreads();
    if (threadIdx.x == 0) {
        counters[0] += s_rec;
        counters[1] = carry;
        counters[2] |= (u64)s_status;
    }
}

// ------------------------------------------------------------------------------------------------
// K3: MT19937 (Matsumoto-Nishimura mt19937ar; reference src/mt19937ar.c:60-73 seeding, :111-129
// twist, :133-137 tempering) generated on device in twist batches.  One CTA owns the 624-word state
// in shared memory (double buffered); a twist is three dependent phases of <= 227 independent lanes
// (x[i] needs x[i+397] for i < 227 and the freshly written x[i-227] afterwards).  The kernel writes
// either the tempered words (tests) or, for the sampler, one KEEP BIT per draw:
//     keep(u)  <=>  u * (1.0/4294967295.0) < (double)rate_depth  <=>  u < T     (host computes T)
// bit s of the output is the decision for stream index s (counted from init_genrand(seed)).
// ------------------------------------------------------------------------------------------------
#define FASTF_MT_THREADS 256
__device__ __forceinline__ u32 fastf_mt_tw(u32 a, u32 b) { u32 y = (a & 0x80000000u) | (b & 0x7fffffffu); return (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u); }
__device__ __forceinline__ u32 fastf_mt_temper(u32 y)
{
    y ^= y >> 11;
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= y >> 18;
    return y;
}
// Produces twist pairs [pair0, pair0 + n_pairs): stream indices [pair0*1248, (pair0+n_pairs)*1248).
// state (624 words in global memory) carries the generator between launches so the stream can be
// extended chunk by chunk while the inflate kernel runs on another stream; it is always stored back.  Exactly one of out_words / out_bits is non-null.
// do_seed != 0: start from init_genrand(seed); otherwise continue from `state` (left by a previous launch or by the jump kernel).
// pair0 only positions the output (pair p writes words [p*1248, ..) or bit words [p*39, ..)).
__global__ void __launch_bounds__(FASTF_MT_THREADS) fastf_mt19937_kernel(u32 seed, u32 *__restrict__ state, u32 do_seed, u64 pair0, u64 n_pairs, u64 threshold,
                                                                        u32 *__restrict__ out_words, u32 *__restrict__ out_bits)
{
    __shared__ u32 st[2][624];
    __shared__ u32 tmp[1248];
    const u32 tid = threadIdx.x;
    // several CTAs = several independent segments of the stream: CTA b continues from state b (put there by the batched jump
    // kernel) and writes pairs [pair0 + b*n_pairs, pair0 + (b+1)*n_pairs)
    state += (size_t)blockIdx.x * 624;
    pair0 += (u64)blockIdx.x * n_pairs;
    if (do_seed) {
        if (tid == 0) {
            u32 x = seed;
            st[0][0] = x;
            for (u32 i = 1; i < 624; i++) { x = 1812433253u * (x ^ (x >> 30)) + i; st[0][i] = x; }
        }
    } else {
        for (u32 i = tid; i < 624; i += FASTF_MT_THREADS) st[0][i] = state[i];
    }
    __syncthreads();
    u32 a = 0;
    for (u64 pair = pair0; pair < pair0 + n_pairs; pair++) {
        for (u32 half = 0; half < 2; half++) {
            const u32 *cur = st[a];
            u32 *nxt = st[a ^ 1u];
            if (tid < 227) nxt[tid] = cur[tid + 397] ^ fastf_mt_tw(cur[tid], cur[tid + 1]);
            __syncthreads();
            if (tid < 227) nxt[227 + tid] = nxt[tid] ^ fastf_mt_tw(cur[227 + tid], cur[228 + tid]);
            __syncthreads();
            if (tid < 169) nxt[454 + tid] = nxt[227 + tid] ^ fastf_mt_tw(cur[454 + tid], cur[455 + tid]);
            else if (tid == 169) nxt[623] = nxt[396] ^ fastf_mt_tw(cur[623], nxt[0]);
            __syncthreads();
            for (u32 i = tid; i < 624; i += FASTF_MT_THREADS) tmp[half * 624 + i] = fastf_mt_temper(nxt[i]);
            a ^= 1u;
        }
        __syncthreads();
        if (out_words) {
            for (u32 i = tid; i < 1248; i += FASTF_MT_THREADS) out_words[pair * 1248 + i] = tmp[i];
        } else {
            // 1248 draws = 39 output words; warp w packs words w, w+8, ...
            const u32 lane = tid & 31u, w = tid >> 5;
            for (u32 word = w; word < 39; word += FASTF_MT_THREADS / 32) {
                bool keep = (u64)tmp[word * 32 + lane] < threshold;
                u32 m = __ballot_sync(FASTF_FULL_MASK, keep);
                if (lane == 0) out_bits[pair * 39 + word] = m;
            }
        }
        __syncthreads();
    }
    for (u32 i = tid; i < 624; i += FASTF_MT_THREADS) state[i] = st[a][i];
}

// Jump-ahead (mt_jump.h): state <- g(F) state for one polynomial g (FASTF_MT_POLY_WORDS 64-bit words, bit i = g_i):
//     new[j] = XOR over set bits i of x_{i+j},   x_0.. = the raw recurrence words generated from the current window.
// One CTA; scratch holds FASTF_MT_DEG + 624 words.
#define FASTF_MTJ_THREADS 1024
__global__ void __launch_bounds__(FASTF_MTJ_THREADS) fastf_mt_jump_kernel(u32 *__restrict__ state, const u64 *__restrict__ poly, u32 *__restrict__ scratch)
{
    const u32 tid = threadIdx.x;
    for (u32 i = tid; i < 624; i += FASTF_MTJ_THREADS) scratch[i] = state[i];
    __syncthreads();
    // x_k = x_{k-227} ^ tw(x_{k-624}, x_{k-623}): 227 independent words per step
    for (u32 base = 624; base < 19937u + 624u; base += 227u) {
        const u32 k = base + tid;
        if (tid < 227u && k < 19937u + 624u) scratch[k] = scratch[k - 227] ^ fastf_mt_tw(scratch[k - 624], scratch[k - 623]);
        __syncthreads();
    }
    if (tid < 624u) {
        u32 acc = 0;
        for (u32 w = 0; w < 312u; w++) {
            u64 bits = poly[w];
            const u32 b0 = w * 64u + tid;
            while (bits) {
                const u32 b = (u32)__ffsll((long long)bits) - 1u;
                bits &= bits - 1ull;
                acc ^= scratch[b0 + b];
            }
        }
        state[tid] = acc;
    }
}

// Batched jump: CTA b leaves in states[b] the window at stream index origin0 + b * stride (seed, then one polynomial per set bit).
// scratch: gridDim.x regions of FASTF_MTJ_SCRATCH words.
#define FASTF_MTJ_SCRATCH (19937 + 624 + 63)
__global__ void __launch_bounds__(FASTF_MTJ_THREADS) fastf_mt_jump_batch_kernel(u32 seed, const u64 *__restrict__ polys, u32 n_polys, u64 origin0, u64 stride, u32 *__restrict__ states,
                                                                               u32 *__restrict__ scratch_all)
{
    __shared__ u32 win[624];
    const u32 tid = threadIdx.x;
    u32 *scratch = scratch_all + (size_t)blockIdx.x * FASTF_MTJ_SCRATCH;
    const u64 origin = origin0 + (u64)blockIdx.x * stride;
    if (tid == 0) {
        u32 x = seed;
        win[0] = x;
        for (u32 i = 1; i < 624; i++) { x = 1812433253u * (x ^ (x >> 30)) + i; win[i] = x; }
    }
    __syncthreads();
    for (u32 kbit = 0; kbit < n_polys; kbit++) {
        if (!((origin >> kbit) & 1ull)) continue;   // uniform across the CTA
        const u64 *poly = polys + (size_t)kbit * 312u;
        for (u32 i = tid; i < 624; i += FASTF_MTJ_THREADS) scratch[i] = win[i];
        __syncthreads();
        for (u32 base = 624; base < 19937u + 624u; base += 227u) {
            const u32 k = base + tid;
            if (tid < 227u && k < 19937u + 624u) scratch[k] = scratch[k - 227] ^ fastf_mt_tw(scratch[k - 624], scratch[k - 623]);
            __syncthreads();
        }
        if (tid < 624u) {
            u32 acc = 0;
            for (u32 w = 0; w < 312u; w++) {
                u64 bits = poly[w];
                const u32 b0 = w * 64u + tid;
                while (bits) {
                    const u32 b = (u32)__ffsll((long long)bits) - 1u;
                    bits &= bits - 1ull;
                    acc ^= scratch[b0 + b];
                }
            }
            win[tid] = acc;
        }
        __syncthreads();
    }
    for (u32 i = tid; i < 624; i += FASTF_MTJ_THREADS) states[(size_t)blockIdx.x * 624 + i] = win[i];
}

// ------------------------------------------------------------------------------------------------
// K3b: depth sampling.  Candidate i (file order) is the (ordinal_base + i)-th CB-valid read, i.e. it
// consumes stream index d0 + ordinal_base + i (reference src/bam2db_ds.c:385-390; SampleInt's draws
// come first, src/utils.c:53-62).  kept && key != INVALID rows are compacted, stably, into `kept`.
// Two-phase: tile counts -> row scan -> scatter.
// ------------------------------------------------------------------------------------------------
#define FASTF_SAMPLE_THREADS 256
#define FASTF_SAMPLE_ITEMS 8
#define FASTF_SAMPLE_TILE (FASTF_SAMPLE_THREADS * FASTF_SAMPLE_ITEMS)

__device__ __forceinline__ bool fastf_keep_bit(const u32 *__restrict__ bits, u64 s) { return (bits[s >> 5] >> (s & 31u)) & 1u; }

// counters: [0] sampled (kept draws), [1] valid (kept && insertable)
__global__ void __launch_bounds__(FASTF_SAMPLE_THREADS)
fastf_sample_count_kernel(const u64 *__restrict__ cand, u64 n, const u32 *__restrict__ keepbits, u64 first_draw, u32 *__restrict__ tile_valid, u64 *__restrict__ counters)
{
    __shared__ u32 s_kept, s_valid;
    if (threadIdx.x == 0) { s_kept = 0; s_valid = 0; }
    __syncthreads();
    const u64 base = (u64)blockIdx.x * FASTF_SAMPLE_TILE;
    u32 kept = 0, valid = 0;
#pragma unroll
    for (int k = 0; k < FASTF_SAMPLE_ITEMS; k++) {
        u64 i = base + (u64)k * FASTF_SAMPLE_THREADS + threadIdx.x;
        if (i < n) {
            bool kp = fastf_keep_bit(keepbits, first_draw + i);
            kept += kp;
            valid += kp && (cand[i] != FASTF_INVALID_KEY);
        }
    }
    kept = __reduce_add_sync(FASTF_FULL_MASK, kept);
    valid = __reduce_add_sync(FASTF_FULL_MASK, valid);
    if ((threadIdx.x & 31u) == 0) { atomicAdd(&s_kept, kept); atomicAdd(&s_valid, valid); }
    __syncthreads();
    if (threadIdx.x == 0) {
        tile_valid[blockIdx.x] = s_valid;
        atomicAdd((unsigned long long *)&counters[0], (unsigned long long)s_kept);
        atomicAdd((unsigned long long *)&counters[1], (unsigned long long)s_valid);
    }
}

__global__ void __launch_bounds__(FASTF_SAMPLE_THREADS)
fastf_sample_scatter_kernel(const u64 *__restrict__ cand, u64 n, const u32 *__restrict__ keepbits, u64 first_draw, const u32 *__restrict__ tile_off, u64 *__restrict__ kept)
{
    // blocked arrangement (thread t owns ITEMS consecutive candidates) keeps file order under a single block scan
    const u64 base = (u64)blockIdx.x * FASTF_SAMPLE_TILE + (u64)threadIdx.x * FASTF_SAMPLE_ITEMS;
    u64 keys[FASTF_SAMPLE_ITEMS];
    u32 flags = 0, cnt = 0;
#pragma unroll
    for (int k = 0; k < FASTF_SAMPLE_ITEMS; k++) {
        u64 i = base + k;
        bool v = false;
        if (i < n) {
            keys[k] = cand[i];
            v = fastf_keep_bit(keepbits, first_draw + i) && keys[k] != FASTF_INVALID_KEY;
        }
        flags |= (u32)v << k;
        cnt += v;
    }
    u32 tot;
    u32 ex = fastf_block_exscan<FASTF_SAMPLE_THREADS>(cnt, &tot);
    u64 o = (u64)tile_off[blockIdx.x] + ex;
#pragma unroll
    for (int k = 0; k < FASTF_SAMPLE_ITEMS; k++)
        if (flags & (1u << k)) kept[o++] = keys[k];
}

// ------------------------------------------------------------------------------------------------
// Depth sweep: one pass samples at K rates.  The draws arrive as tempered words u (fastf_mt19937_kernel
// out_words); the K keep thresholds are sorted ascending, and the rate index of a draw is
//     b(u) = min{ i : u < T_i }  (K when there is none)  =  number of thresholds <= u,
// so a read is kept at rate i <=> b <= i: the reads kept at a lower rate are a subset of those kept
// at a higher one.  Counts go into per-rate histograms (their prefix sums are the per-rate counters);
// the valid candidates with b < K are compacted in file order as (key, b).
// ------------------------------------------------------------------------------------------------
struct FastfSweepRates {
    u64 t[FASTF_SWEEP_MAX_RATES];   // ascending thresholds, t[0..k)
    u32 k;
};

__device__ __forceinline__ u32 fastf_rate_index(const u64 *t, u32 k, u32 u)
{
    u32 b = 0;
    for (u32 j = 0; j < k; j++) b += (u64)u >= t[j];
    return b;
}

// hist: u64[2][FASTF_SWEEP_MAX_RATES]: row 0 = CB-valid reads with rate index b, row 1 = those whose key is insertable
__global__ void __launch_bounds__(FASTF_SAMPLE_THREADS)
fastf_sweep_count_kernel(const u64 *__restrict__ cand, u64 n, const u32 *__restrict__ words, u64 first_draw, FastfSweepRates R, u32 *__restrict__ tile_valid, u64 *__restrict__ hist)
{
    __shared__ u64 s_t[FASTF_SWEEP_MAX_RATES];
    __shared__ u32 s_h[2][FASTF_SWEEP_MAX_RATES];
    __shared__ u32 s_valid;
    const u32 K = R.k;
    if (threadIdx.x < FASTF_SWEEP_MAX_RATES) { s_t[threadIdx.x] = R.t[threadIdx.x]; s_h[0][threadIdx.x] = 0; s_h[1][threadIdx.x] = 0; }
    if (threadIdx.x == 0) s_valid = 0;
    __syncthreads();
    const u64 base = (u64)blockIdx.x * FASTF_SAMPLE_TILE;
    u32 valid = 0;
#pragma unroll
    for (int k = 0; k < FASTF_SAMPLE_ITEMS; k++) {
        u64 i = base + (u64)k * FASTF_SAMPLE_THREADS + threadIdx.x;
        if (i < n) {
            const u32 b = fastf_rate_index(s_t, K, words[first_draw + i]);
            if (b < K) {
                atomicAdd(&s_h[0][b], 1u);
                if (cand[i] != FASTF_INVALID_KEY) { atomicAdd(&s_h[1][b], 1u); valid++; }
            }
        }
    }
    valid = __reduce_add_sync(FASTF_FULL_MASK, valid);
    if ((threadIdx.x & 31u) == 0) atomicAdd(&s_valid, valid);
    __syncthreads();
    if (threadIdx.x == 0) tile_valid[blockIdx.x] = s_valid;
    if (threadIdx.x < K) {
        if (s_h[0][threadIdx.x]) atomicAdd((unsigned long long *)&hist[threadIdx.x], (unsigned long long)s_h[0][threadIdx.x]);
        if (s_h[1][threadIdx.x]) atomicAdd((unsigned long long *)&hist[FASTF_SWEEP_MAX_RATES + threadIdx.x], (unsigned long long)s_h[1][threadIdx.x]);
    }
}

__global__ void __launch_bounds__(FASTF_SAMPLE_THREADS)
fastf_sweep_scatter_kernel(const u64 *__restrict__ cand, u64 n, const u32 *__restrict__ words, u64 first_draw, FastfSweepRates R, const u32 *__restrict__ tile_off, u64 *__restrict__ kept,
                           u32 *__restrict__ kept_rate)
{
    __shared__ u64 s_t[FASTF_SWEEP_MAX_RATES];
    const u32 K = R.k;
    if (threadIdx.x < FASTF_SWEEP_MAX_RATES) s_t[threadIdx.x] = R.t[threadIdx.x];
    __syncthreads();
    // blocked arrangement as in fastf_sample_scatter_kernel: file order under a single block scan
    const u64 base = (u64)blockIdx.x * FASTF_SAMPLE_TILE + (u64)threadIdx.x * FASTF_SAMPLE_ITEMS;
    u64 keys[FASTF_SAMPLE_ITEMS];
    u32 rb[FASTF_SAMPLE_ITEMS];
    u32 flags = 0, cnt = 0;
#pragma unroll
    for (int k = 0; k < FASTF_SAMPLE_ITEMS; k++) {
        u64 i = base + k;
        bool v = false;
        rb[k] = K;
        if (i < n) {
            rb[k] = fastf_rate_index(s_t, K, words[first_draw + i]);
            if (rb[k] < K) { keys[k] = cand[i]; v = keys[k] != FASTF_INVALID_KEY; }
        }
        flags |= (u32)v << k;
        cnt += v;
    }
    u32 tot;
    u32 ex = fastf_block_exscan<FASTF_SAMPLE_THREADS>(cnt, &tot);
    u64 o = (u64)tile_off[blockIdx.x] + ex;
#pragma unroll
    for (int k = 0; k < FASTF_SAMPLE_ITEMS; k++)
        if (flags & (1u << k)) { kept[o] = keys[k]; kept_rate[o] = rb[k]; o++; }
}
