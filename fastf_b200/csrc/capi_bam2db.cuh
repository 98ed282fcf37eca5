// Part of the libfastf_gpu translation unit (capi.cu includes it, in this order; it is not a header of its own):
// the bam2db job: chunk pipeline (copy ring, inflate / CRC / parse / gather per chunk), MT19937 keep bits, sampling, sort, dedup / count, results;
// the depth sweep (several rates out of one job); the cell-rate grid (several cell tables and depth rates out of one job).
#pragma once

// ---------------------------------------------------------------------------------------------------
// bam2db job
// ---------------------------------------------------------------------------------------------------
#define FASTF_DEFAULT_CHUNK (512ull << 20)
#define FASTF_MAX_BLOCKS_PER_CHUNK (1u << 22)

struct ChunkSlot {
    BlockIndexDev idx;
    DevBuf stage;         // per-block candidate staging
    DevBuf virt;          // FASTF_BAM_STRADDLE: record-start guesses and virtual blocks
    DevBuf infl;          // inflated bytes of the chunk (double buffered: chunk i+1 inflates while chunk i is parsed)
    DeScratch de;
    Event ev_infl, ev_gather;
    PinBuf snap;          // counters snapshot {n_records, n_candidates, status_or, chunk_candidates}
    Event ev_copy, ev_done;
    u32 nblocks = 0;
    bool pending = false; // parse launched, gather not yet
};

struct fastf_bam2db_job {
    fastf_ctx *ctx;
    fastf_bam2db_params prm;
    FastfKeyLayout L;
    DevTable cells, genes;
    u32 lanes;
    u64 chunk_bytes;
    ChunkSlot slot[2];
    u32 next_slot = 0;
    // compressed bytes of host-fed chunks: a ring of three, so that the copy of chunk i is issued before the host waits for
    // anything and overlaps the inflate of chunks i-2 and i-1
    struct CompRing { DevBuf buf; Event ev_copy, ev_free; bool used = false; } comp_ring[3];
    u32 comp_seq = 0;
    u64 ring_estimate = 0;
    // FASTF_FEED_TIMING=1: where a host-fed job spends its time (stderr at finish): H2D copies by CUDA events, host waits by wall clock
    bool feed_timing = false;
    std::vector<std::pair<Event, Event>> ft_copy_ev, ft_infl_ev;
    std::vector<Event> ft_parse_ev;
    std::vector<double> ft_host_submit;
    u64 ft_copy_bytes = 0;
    double ft_wait_s = 0, ft_index_s = 0, ft_feed_s = 0;
    // Blocks wait here until a chunk is full, ACROSS feed calls: the persistent inflate kernel keeps n_sm x FASTF_TPS_STREAMS blocks
    // in flight, so a launch over an exact multiple of that many blocks has no half-empty last round (measured: +11 % inflate
    // throughput over 2 GiB chunks cut at the feed boundaries).
    struct PendingChunk {
        std::vector<FastfBgzfBlock> blocks;
        u64 infl = 0;
        const u8 *comp_dev = nullptr;   // device feeds: the caller's buffer
        u64 comp_total = 0;
        CompRing *ring = nullptr;       // host feeds: where the compressed bytes are being staged
        u64 fill = 0;                   // bytes staged so far (multiple of 4)
    } pending;
    u64 chunk_blocks = FASTF_MAX_BLOCKS_PER_CHUNK;
    DevBuf counters;          // u64[4]: n_records, n_candidates, status_or, (unused)
    DevBuf hdr_off;           // u64: offset of the first alignment record inside the current chunk
    DevBuf cand;              // all candidates (CB-valid reads) in file order
    u64 cand_cap = 0;
    u64 n_records = 0, n_cand = 0;   // host copies after the last finalized chunk
    u32 status = 0;
    bool header_done = false;
    std::vector<u8> carry;    // partial BGZF block left over by fastf_bam2db_feed
    // MT19937 keep bits from the job's first draw on (the depth sweep: tempered words, one u32 per draw)
    DevBuf keepbits, mt_states, mt_scratch;
    Event ev_mt;
    // sampling / sort / count
    bool sampled_done = false;
    u32 sweep_rates = 0;          // sampled by the depth sweep at this many rates (0: at the job's one rate)
    DevBuf tile_valid, tile_tot, kept, orand;
    DevBuf sample_counters;       // u64[2][FASTF_SWEEP_MAX_RATES]: sampled / valid reads per rate index (one rate: [0] / [FASTF_SWEEP_MAX_RATES])
    DevBuf kept_rate, rate_alt;   // depth sweep: rate index of every kept row, and its sort ping-pong buffer
    RleScratch rateS;             // depth sweep: the per-rate count over the distinct keys (held in rleS)
    PinBuf small_host;
    u64 n_sampled = 0, n_valid = 0;
    // cell-rate grid (fastf_bam2db_begin_grid): `cand` holds the union table's candidates and stays; per cell rate, the remap table
    // and the candidate array of that rate's own table (also the sort's ping-pong buffer once it has been sampled)
    bool grid = false;
    DevBuf grid_remap, grid_cand;
    SortScratch sortS;
    RleScratch rleS;
    // stats
    u64 n_blocks = 0, comp_bytes = 0, infl_bytes = 0;
    u64 n_blocks_fed = 0, n_blocks_done = 0;   // blocks handed to run_blocks / blocks whose candidate counts have come back
    u32 launches0 = 0, n_chunks = 0;
    Timer t_infl[2], t_crc[2], t_parse[2], t_gather[2], t_mt, t_sample, t_sort, t_count;
    Event ev_first, ev_last;
    bool first_recorded = false;
    float ms_inflate = 0, ms_crc = 0, ms_parse = 0, ms_gather = 0, ms_mt = 0, ms_sample = 0, ms_sort = 0, ms_count = 0;
};

static u32 stage_cap_for(u32 isize) { return isize / 36u + 1u; }   // a record is >= 4 + 32 bytes

extern "C" void fastf_bam2db_job_free(fastf_bam2db_job *job)
{
    if (!job) return;
    fastf_ctx *ctx = job->ctx;
    cudaSetDevice(ctx->device);
    // the job's buffers go back to the pools when it is deleted: nothing queued may still touch them
    cudaStreamSynchronize(ctx->compute);
    cudaStreamSynchronize(ctx->copy);
    cudaStreamSynchronize(ctx->infl);
    cudaStreamSynchronize(ctx->mt);
    ctx->hint_cand = std::max(ctx->hint_cand, job->cand.cap);
    for (auto &R : job->comp_ring) ctx->hint_ring = std::max(ctx->hint_ring, R.buf.cap);
    delete job;
}

extern "C" int fastf_bam2db_begin(fastf_ctx *ctx, const fastf_bam2db_params *p, fastf_bam2db_job **out)
{
    *out = nullptr;
    CK(cudaSetDevice(ctx->device));
    if (!p || (p->n_cells && (!p->cell_keys || !p->cell_off)) || (p->n_genes && (!p->gene_keys || !p->gene_off))) return ctx_fail(ctx, "bam2db_begin: null table pointers");
    if (p->keep_threshold > 4294967296ull) return ctx_fail(ctx, "bam2db_begin: keep_threshold > 2^32");
    fastf_bam2db_job *job = new fastf_bam2db_job();
    { const char *e = getenv("FASTF_FEED_TIMING"); job->feed_timing = e && *e && *e != '0'; }
    job->ctx = ctx;
    job->prm = *p;
    job->launches0 = ctx->launches;
    {
        const u32 l = p->inflate_lanes & 0xffu;
        job->lanes = ((l == 8 || l == 16 || l == 32 || (l >= 1 && l <= 4)) ? l : FASTF_INFLATE_DEFAULT) | (p->inflate_lanes & (FASTF_INFLATE_HW_ENGINE | FASTF_INFLATE_NO_CRC | FASTF_BAM_STRADDLE));
    }
    job->chunk_bytes = p->chunk_inflated_bytes ? std::max<u64>(p->chunk_inflated_bytes, 1u << 20) : FASTF_DEFAULT_CHUNK;
    // the persistent thread-per-stream kernel keeps 64 streams per SM busy: give every launch several blocks per stream
    if (!p->chunk_inflated_bytes && (job->lanes & 0xffu) >= 1 && (job->lanes & 0xffu) <= 4) {
        u64 rounds = 2;   // full rounds of the persistent kernel per chunk (2 -> 66304 blocks, <= 4.3 GB on 148 SMs)
        if (const char *e = getenv("FASTF_CHUNK_ROUNDS")) { const long v = atol(e); if (v >= 1 && v <= 16) rounds = (u64)v; }
        job->chunk_blocks = rounds * (u64)ctx->n_sm * FASTF_TPS_STREAMS;
        job->chunk_bytes = job->chunk_blocks * 65536ull;
    }
    if (job->lanes & FASTF_BAM_STRADDLE) {
        // records may run across block boundaries: keep the whole file in one chunk so that none is cut by a chunk boundary
        if (p->headerless) { delete job; return ctx_fail(ctx, "bam2db_begin: FASTF_BAM_STRADDLE needs the whole file in one job (a later shard does not know where its first record starts)"); }
        job->chunk_blocks = FASTF_MAX_BLOCKS_PER_CHUNK;
        job->chunk_bytes = ~0ull >> 2;
    }
    FastfKeyLayout &L = job->L;
    L.umi_max_bytes = p->umi_max_bytes ? p->umi_max_bytes : 3;
    if (L.umi_max_bytes > 4) { delete job; return ctx_fail(ctx, "bam2db_begin: umi_max_bytes must be 1..4 (UMIs up to 16 bases)"); }
    L.bits_umi = 1 + 8 * L.umi_max_bytes + 3;
    L.bits_gene = bits_for(p->n_genes);
    L.bits_cell = bits_for(p->n_cells);
    if (L.bits_cell + L.bits_gene + L.bits_umi > 63) { delete job; return ctx_fail(ctx, "bam2db_begin: key layout needs %u bits (> 63)", L.bits_cell + L.bits_gene + L.bits_umi); }
    int rc = 0;
    rc = rc || table_upload(ctx, job->cells, p->cell_keys, p->cell_off, p->n_cells);
    rc = rc || table_upload(ctx, job->genes, p->gene_keys, p->gene_off, p->n_genes);
    rc = rc || dev_reserve(ctx, job->counters, 4 * sizeof(u64));
    rc = rc || dev_reserve(ctx, job->hdr_off, sizeof(u64));
    rc = rc || dev_reserve(ctx, job->sample_counters, 2 * FASTF_SWEEP_MAX_RATES * sizeof(u64));
    rc = rc || dev_reserve(ctx, job->orand, 2 * sizeof(u64));
    rc = rc || pin_reserve(ctx, job->small_host, 2 * FASTF_SWEEP_MAX_RATES * sizeof(u64));
    for (int i = 0; i < 2 && !rc; i++) {
        rc = rc || pin_reserve(ctx, job->slot[i].snap, 4 * sizeof(u64));
        rc = rc || job->slot[i].ev_copy.create(cudaEventDisableTiming) != cudaSuccess;
        rc = rc || job->slot[i].ev_done.create(cudaEventDisableTiming) != cudaSuccess;
        rc = rc || job->slot[i].ev_infl.create(cudaEventDisableTiming) != cudaSuccess;
        rc = rc || job->slot[i].ev_gather.create(cudaEventDisableTiming) != cudaSuccess;
        rc = rc || job->t_infl[i].init() || job->t_crc[i].init() || job->t_parse[i].init() || job->t_gather[i].init();
    }
    for (auto &R : job->comp_ring) {
        rc = rc || R.ev_copy.create(cudaEventDisableTiming) != cudaSuccess;
        rc = rc || R.ev_free.create(cudaEventDisableTiming) != cudaSuccess;
    }
    rc = rc || job->t_mt.init() || job->t_sample.init() || job->t_sort.init() || job->t_count.init();
    rc = rc || job->ev_mt.create(cudaEventDisableTiming) != cudaSuccess;
    rc = rc || job->ev_first.create() != cudaSuccess || job->ev_last.create() != cudaSuccess;
    if (!rc) rc = cudaMemsetAsync(job->counters.p, 0, 4 * sizeof(u64), ctx->compute) != cudaSuccess;
    job->header_done = p->headerless != 0;

    if (rc) { if (!ctx->err[0]) ctx_fail(ctx, "bam2db_begin: resource setup failed"); fastf_bam2db_job_free(job); return 1; }
    *out = job;
    return 0;
}

// The jump polynomials x^(2^k) mod phi (mt_jump.h) on the device, uploaded once per context, with their count in *n_polys.  They
// reach stream indices below 2^n_polys; `last_origin` is the largest index the caller jumps to.  The tables are a pure function of
// constants and the draw index of a job is d0 plus a count of reads, so a failure here is a bug, not a property of the input.
static int mt_jump_polys(fastf_ctx *ctx, const char *who, u64 last_origin, u32 *n_polys)
{
    const fastf_mtj::Tables &T = fastf_mtj::tables();
    if (!T.ok) return ctx_fail(ctx, "%s: the MT19937 jump tables could not be built (Berlekamp-Massey did not find the degree-19937 polynomial)", who);
    if ((last_origin >> T.pow2.size()) != 0)
        return ctx_fail(ctx, "%s: MT19937 stream index %llu is beyond the jump tables (< 2^%zu)", who, (unsigned long long)last_origin, T.pow2.size());
    if (!ctx->mtj_polys) {
        std::vector<uint64_t> flat(T.pow2.size() * FASTF_MT_POLY_WORDS);
        for (size_t k = 0; k < T.pow2.size(); k++) memcpy(flat.data() + k * FASTF_MT_POLY_WORDS, T.pow2[k].data(), FASTF_MT_POLY_WORDS * sizeof(uint64_t));
        CK(cudaMalloc(&ctx->mtj_polys, flat.size() * sizeof(uint64_t)));
        CK(cudaMemcpy(ctx->mtj_polys, flat.data(), flat.size() * sizeof(uint64_t), cudaMemcpyHostToDevice));
    }
    *n_polys = (u32)T.pow2.size();
    return 0;
}

// Keep bits (words: tempered words) for stream indices [first, first + n) into job->keepbits from bit (word) 0 on, generated by
// up to FASTF_MT_SEGMENTS CTAs at once: every CTA jumps to the start of its own segment of the reference's single stream, then
// runs the normal twist.  Runs on the mt stream.
#define FASTF_MT_SEGMENTS 32
static int mt_generate_parallel(fastf_bam2db_job *job, const char *who, u64 first, u64 n, bool words)
{
    fastf_ctx *ctx = job->ctx;
    cudaStream_t s = ctx->mt;
    const u64 pairs = (n + 1247) / 1248;
    const u32 K = (u32)std::min<u64>(FASTF_MT_SEGMENTS, std::max<u64>(1, pairs / 64));
    const u64 ppc = (pairs + K - 1) / K;
    u32 n_polys = 0;
    TRY(mt_jump_polys(ctx, who, first + (u64)K * ppc * 1248ull, &n_polys));
    TRY(dev_reserve(ctx, job->mt_states, (size_t)K * 624 * sizeof(u32)));
    TRY(dev_reserve(ctx, job->mt_scratch, (size_t)K * FASTF_MTJ_SCRATCH * sizeof(u32)));
    TRY(dev_reserve(ctx, job->keepbits, (size_t)K * ppc * (words ? 1248 : 39) * sizeof(u32)));
    job->t_mt.start(s);
    FASTF_LAUNCH(fastf_mt_jump_batch_kernel, K, FASTF_MTJ_THREADS, 0, s, job->prm.seed, (const u64 *)ctx->mtj_polys, n_polys, first, ppc * 1248ull, job->mt_states.as<u32>(),
                 job->mt_scratch.as<u32>());
    CKL("mt_jump_batch");
    FASTF_LAUNCH(fastf_mt19937_kernel, K, FASTF_MT_THREADS, 0, s, job->prm.seed, job->mt_states.as<u32>(), 0u, (u64)0, ppc, job->prm.keep_threshold,
                 words ? job->keepbits.as<u32>() : (u32 *)nullptr, words ? (u32 *)nullptr : job->keepbits.as<u32>());
    CKL("mt19937");
    job->t_mt.stop(s);
    return 0;
}

// Wait for the slot's counters, size the candidate array, gather the slot's staged candidates.
static int finalize_slot(fastf_bam2db_job *job, u32 si)
{
    fastf_ctx *ctx = job->ctx;
    ChunkSlot &S = job->slot[si];
    if (!S.pending) return 0;
    const double ft_w0 = job->feed_timing ? wall_seconds() : 0;
    CK(cudaEventSynchronize(S.ev_done));
    if (job->feed_timing) job->ft_wait_s += wall_seconds() - ft_w0;
    const u64 *snap = S.snap.as<u64>();
    const u64 n_records = snap[0], n_cand = snap[1];
    job->n_blocks_done += S.nblocks;
    job->status |= (u32)snap[2];
    if (job->status) {
        char buf[256];
        if (job->status == FASTF_ST_UMI_TOO_LONG)
            return ctx_fail(ctx, "bam2db: umi-too-long: a UB tag holds more than %u bases; begin the job with a larger umi_max_bytes", 4u * job->L.umi_max_bytes);
        return ctx_fail(ctx, "bam2db: malformed input in chunk ending at block %llu: %s", (unsigned long long)job->n_blocks, status_string(job->status, buf, sizeof buf));
    }
    if (n_cand > job->cand_cap) {
        u64 want = std::max<u64>(n_cand + n_cand / 2, 1u << 20);
        want = std::max<u64>(want, ctx->hint_cand / sizeof(u64));
        // the blocks already handed to the job will bring candidates at the rate seen so far
        if (job->n_blocks_done) want = std::max<u64>(want, (u64)((double)n_cand * (double)job->n_blocks_fed / (double)job->n_blocks_done * 1.03) + (1u << 16));
        TRY(dev_reserve(ctx, job->cand, want * sizeof(u64), job->n_cand * sizeof(u64), ctx->compute));
        job->cand_cap = job->cand.cap / sizeof(u64);
    }
    job->t_gather[si].collect(&job->ms_gather);
    job->t_gather[si].start(ctx->compute);
    if (S.nblocks) {
        FASTF_LAUNCH(fastf_stage_gather_kernel, (S.nblocks + 7) / 8, 256, 0, ctx->compute, (const u64 *)S.stage.as<u64>(), (const u64 *)S.idx.stage_off, (const u32 *)S.idx.ncbv,
                     (const u64 *)S.idx.dst_base, S.nblocks, job->cand.as<u64>());
        CKL("stage_gather");
    }
    job->t_gather[si].stop(ctx->compute);
    CK(cudaEventRecord(S.ev_gather, ctx->compute));   // the slot's index arrays are free for the next upload (inflate stream) after this
    CK(cudaEventRecord(job->ev_last, ctx->compute));
    job->n_records = n_records;
    job->n_cand = n_cand;
    S.pending = false;

    return 0;
}

// FASTF_BAM_STRADDLE: record-start guesses per BGZF block -> virtual blocks [v_k, v_next) for the per-block kernels (bam_straddle.cuh).
// scratch holds guess u64[nb] | virt_off u64[nb] | virt_size u32[nb]; status_word collects impossible layouts.
static int launch_virtual_blocks(fastf_ctx *ctx, DevBuf &scratch, const u8 *infl, u64 infl_bytes, const u64 *blk_off, const u32 *blk_isize, u32 nb, const u64 *hdr_off, u32 *status_word,
                                 const u64 **virt_off, const u32 **virt_size, cudaStream_t s)
{
    TRY(dev_reserve(ctx, scratch, (size_t)std::max<u32>(nb, 1) * 20 + 64));
    u64 *guess = scratch.as<u64>(), *voff = guess + nb;
    u32 *vsize = (u32 *)(voff + nb);
    if (nb) {
        FASTF_LAUNCH(fastf_bam_guess_kernel, (nb + 7) / 8, 256, 0, s, infl, infl_bytes, blk_off, blk_isize, nb, hdr_off, guess);
        CKL("bam_guess");
        FASTF_LAUNCH(fastf_bam_virtual_blocks_kernel, (nb + 255) / 256, 256, 0, s, (const u64 *)guess, nb, infl_bytes, voff, vsize, status_word);
        CKL("bam_virtual_blocks");
    }
    *virt_off = voff;
    *virt_size = vsize;
    return 0;
}

// One chunk: blocks with payload offsets relative to `comp_dev` (the caller's device buffer, or the ring entry the host bytes were
// staged into by stage_host_bytes: their H2D copies are already queued on the copy stream).
static int run_chunk(fastf_bam2db_job *job, const FastfBgzfBlock *blocks, u32 nb, const u8 *comp_dev, u64 comp_total, fastf_bam2db_job::CompRing *ring)
{
    fastf_ctx *ctx = job->ctx;
    const u32 si = job->next_slot;
    ChunkSlot &S = job->slot[si];
    if (ring) CK(cudaEventRecord(ring->ev_copy, ctx->copy));
    // the slot was used two chunks ago: its gather must have been issued (finalize) before we reuse its buffers
    TRY(finalize_slot(job, si));
    TRY(index_reserve(ctx, S.idx, nb + 1));
    const bool straddle = (job->lanes & FASTF_BAM_STRADDLE) != 0;
    u64 out_total = 0, stage_total = 0;
    for (u32 i = 0; i < nb; i++) {
        S.idx.h_in_off[i] = blocks[i].in_off;
        S.idx.h_in_len[i] = blocks[i].in_len;
        S.idx.h_isize[i] = blocks[i].isize;
        S.idx.h_out_off[i] = out_total;
        S.idx.h_stage_off[i] = stage_total;
        out_total += blocks[i].isize;
        // straddle mode: a virtual block holds the records that START between this block's guess and the next one's
        stage_total += straddle ? stage_cap_for(blocks[i].isize + (i + 1 < nb ? blocks[i + 1].isize : 0)) + 1u : stage_cap_for(blocks[i].isize);
    }
    S.idx.h_stage_off[nb] = stage_total;   // the kernels read the slice capacity as stage_off[b + 1] - stage_off[b]
    if (ring) CK(cudaStreamWaitEvent(ctx->infl, ring->ev_copy, 0));
    // S.infl / S.stage / S.idx were last used by chunk i-2, whose parse and gather have completed (finalize_slot above)
    TRY(dev_reserve(ctx, S.infl, out_total + 64));
    TRY(dev_reserve(ctx, S.stage, stage_total * sizeof(u64) + 64));
    if (!job->first_recorded) { CK(cudaEventRecord(job->ev_first, ctx->infl)); job->first_recorded = true; }
    // inflate runs on its own stream so that chunk i+1 inflates (SM kernel or hardware engine) while chunk i is parsed;
    // the gather of the slot's previous chunk (compute stream) still reads the index arrays we are about to overwrite
    CK(cudaStreamWaitEvent(ctx->infl, S.ev_gather, 0));
    TRY(index_upload(ctx, S.idx, ctx->infl));
    job->t_infl[si].collect(&job->ms_inflate);
    job->t_infl[si].start(ctx->infl);
    std::pair<Event, Event> fti;
    if (job->feed_timing && ring) { CK(fti.first.create()); CK(fti.second.create()); CK(cudaEventRecord(fti.first, ctx->infl)); job->ft_host_submit.push_back(wall_seconds()); }
    TRY(launch_inflate(ctx, job->lanes, comp_dev, comp_total, S.idx.in_off, S.idx.in_len, S.idx.out_off, S.idx.isize, nb, S.infl.as<u8>(), S.idx.st_infl, ctx->infl, &S.de, S.idx.h_in_off,
                       S.idx.h_in_len, S.idx.h_out_off, S.idx.h_isize));
    if (fti.first) { CK(cudaEventRecord(fti.second, ctx->infl)); job->ft_infl_ev.push_back(std::move(fti)); }
    job->t_infl[si].stop(ctx->infl);
    CK(cudaEventRecord(S.ev_infl, ctx->infl));
    CK(cudaStreamWaitEvent(ctx->compute, S.ev_infl, 0));
    job->t_crc[si].collect(&job->ms_crc);
    job->t_crc[si].start(ctx->compute);
    TRY(launch_crc(ctx, job->lanes, comp_dev, comp_total, S.idx.in_off, S.idx.in_len, S.infl.as<u8>(), S.idx.out_off, S.idx.isize, nb, S.idx.st_infl, ctx->compute));
    job->t_crc[si].stop(ctx->compute);
    if (ring) { CK(cudaEventRecord(ring->ev_free, ctx->compute)); ring->used = true; }   // compressed bytes no longer needed
    job->t_parse[si].collect(&job->ms_parse);
    job->t_parse[si].start(ctx->compute);
    if (!job->header_done) {
        FASTF_LAUNCH(fastf_bam_header_kernel, 1, 32, 0, ctx->compute, (const u8 *)S.infl.as<u8>(), out_total, job->hdr_off.as<u64>(), (u32 *)(job->counters.as<u64>() + 2));
        CKL("bam_header");
        job->header_done = true;
    } else {
        CK(cudaMemsetAsync(job->hdr_off.p, 0, sizeof(u64), ctx->compute));
    }
    const u64 *p_off = S.idx.out_off;
    const u32 *p_size = S.idx.isize;
    if (straddle) TRY(launch_virtual_blocks(ctx, S.virt, (const u8 *)S.infl.as<u8>(), out_total, S.idx.out_off, S.idx.isize, nb, job->hdr_off.as<u64>(), (u32 *)(job->counters.as<u64>() + 2), &p_off, &p_size,
                                            ctx->compute));
    if (nb) {
        const auto parse = job->grid ? fastf_bam_parse_kernel<true> : fastf_bam_parse_kernel<false>;
        FASTF_LAUNCH(parse, (nb + FASTF_PARSE_WARPS - 1) / FASTF_PARSE_WARPS, FASTF_PARSE_WARPS * 32, 0, ctx->compute, (const u8 *)S.infl.as<u8>(), (u64)((out_total + 15) & ~15ull),
                     p_off, p_size, nb, (const u64 *)job->hdr_off.as<u64>(), job->cells.view, job->genes.view, job->L, (const u64 *)S.idx.stage_off,
                     S.stage.as<u64>(), S.idx.nrec, S.idx.ncbv, S.idx.st_parse);
        CKL("bam_parse");
    }
    FASTF_LAUNCH(fastf_chunk_counts_kernel, 1, FASTF_SCAN_THREADS, 0, ctx->compute, (const u32 *)S.idx.nrec, (const u32 *)S.idx.ncbv, (const u32 *)S.idx.st_infl, (const u32 *)S.idx.st_parse, nb,
                 S.idx.dst_base, job->counters.as<u64>());
    CKL("chunk_counts");
    job->t_parse[si].stop(ctx->compute);
    CK(cudaMemcpyAsync(S.snap.p, job->counters.p, 4 * sizeof(u64), cudaMemcpyDeviceToHost, ctx->compute));
    CK(cudaEventRecord(S.ev_done, ctx->compute));
    if (job->feed_timing && ring) { Event e; CK(e.create()); CK(cudaEventRecord(e, ctx->compute)); job->ft_parse_ev.push_back(std::move(e)); }
    S.nblocks = nb;
    S.pending = true;
    job->n_blocks += nb;
    job->n_chunks++;
    job->infl_bytes += out_total;
    job->next_slot ^= 1u;
    // The previous chunk (slot si ^ 1) is gathered when its slot comes round again (top of the next run_chunk) or at the end of
    // the job: waiting for it here would keep the host from queueing more than one chunk ahead of the device.
    return 0;
}

static int submit_pending(fastf_bam2db_job *job)
{
    fastf_bam2db_job::PendingChunk &P = job->pending;
    if (P.blocks.empty()) return 0;
    const u8 *comp = P.ring ? P.ring->buf.as<u8>() : P.comp_dev;
    const u64 total = P.ring ? P.fill : P.comp_total;
    int rc = run_chunk(job, P.blocks.data(), (u32)P.blocks.size(), comp, total, P.ring);
    P.blocks.clear();
    P.infl = 0; P.comp_dev = nullptr; P.comp_total = 0; P.ring = nullptr; P.fill = 0;
    return rc;
}

// Queue the H2D copy of host bytes [lo, hi) behind what the pending chunk has staged so far; returns their offset in the ring entry.
static int stage_host_bytes(fastf_bam2db_job *job, const u8 *host_base, u64 lo, u64 hi, u64 *at)
{
    fastf_ctx *ctx = job->ctx;
    fastf_bam2db_job::PendingChunk &P = job->pending;
    if (!P.ring) {
        // The copy goes out before the host waits for anything.  The ring entry was last read by the chunk three back (inflate +
        // CRC), which the copy stream waits for on the device.
        P.ring = &job->comp_ring[job->comp_seq++ % 3u];
        P.fill = 0;
        if (P.ring->used) CK(cudaStreamWaitEvent(ctx->copy, P.ring->ev_free, 0));
    }
    const u64 bytes = hi - lo, padded = (bytes + 3) & ~3ull;
    // growing moves the buffer: the bytes staged so far travel along (dev_reserve drains the streams before it lets go of the old one),
    // so an entry starts at the size a whole chunk is expected to need
    u64 want = P.fill + padded + 16;
    if (want > P.ring->buf.cap) want = std::max<u64>(want, std::max<u64>(ctx->hint_ring, job->ring_estimate));
    TRY(dev_reserve(ctx, P.ring->buf, want, P.fill, ctx->copy));
    std::pair<Event, Event> ft;
    if (job->feed_timing) { CK(ft.first.create()); CK(ft.second.create()); CK(cudaEventRecord(ft.first, ctx->copy)); }
    CK(cudaMemcpyAsync(P.ring->buf.as<u8>() + P.fill, host_base + lo, bytes, cudaMemcpyHostToDevice, ctx->copy));
    if (job->feed_timing) { CK(cudaEventRecord(ft.second, ctx->copy)); job->ft_copy_ev.push_back(std::move(ft)); job->ft_copy_bytes += bytes; }
    *at = P.fill;
    P.fill += padded;
    return 0;
}

// Append indexed blocks (payload offsets relative to comp_dev, or to host_base for a host feed) to the pending chunk and launch
// every chunk that fills up.  What is left waits for the next feed or for drain_chunks.
static int run_blocks(fastf_bam2db_job *job, const std::vector<FastfBgzfBlock> &blocks, const u8 *comp_dev, u64 comp_total, const u8 *host_base)
{
    fastf_bam2db_job::PendingChunk &P = job->pending;
    const size_t n = blocks.size();
    size_t i = 0;
    job->n_blocks_fed += n;
    // compressed bytes a full chunk of this feed will stage (ring entries are sized once, see stage_host_bytes): never more than the feed holds
    if (host_base && n) {
        u64 isz = 0;
        for (size_t k = 0; k < n; k++) isz += blocks[k].isize;
        const double span = (double)(blocks[n - 1].in_off + blocks[n - 1].in_len + 8 - blocks[0].in_off);
        const double per_chunk = std::min<double>((double)job->chunk_blocks, (double)job->chunk_bytes / std::max<double>((double)isz / (double)n, 1.0));
        job->ring_estimate = (u64)std::min<double>(span, span / (double)n * 1.03 * per_chunk) + (1u << 20);
    }
    while (i < n) {
        // a chunk reads its compressed bytes from one buffer: blocks of another device buffer (or of the other kind of feed) start a new one
        if (!P.blocks.empty() && (host_base ? P.ring == nullptr : (P.ring != nullptr || P.comp_dev != comp_dev))) TRY(submit_pending(job));
        size_t j = i;
        u64 infl = P.infl;
        const u64 byte0 = blocks[i].in_off & ~3ull;
        while (j < n && P.blocks.size() + (j - i) < job->chunk_blocks && (P.blocks.empty() && j == i ? true : infl + blocks[j].isize <= job->chunk_bytes) &&
               (!host_base || j == i || P.fill + (blocks[j].in_off + blocks[j].in_len + 8 - byte0) <= job->chunk_bytes + (1u << 20))) {
            infl += blocks[j].isize;
            j++;
        }
        if (j == i) { TRY(submit_pending(job)); continue; }   // the pending chunk is full
        if (host_base) {
            // copy [first payload rounded down to 4, end of the last block's CRC32 / ISIZE trailer) and rebase the offsets
            const u64 hi = blocks[j - 1].in_off + blocks[j - 1].in_len + 8;
            u64 at = 0;
            TRY(stage_host_bytes(job, host_base, byte0, hi, &at));
            for (size_t k = i; k < j; k++) { FastfBgzfBlock b = blocks[k]; b.in_off = at + (b.in_off - byte0); P.blocks.push_back(b); }
        } else {
            P.comp_dev = comp_dev;
            P.comp_total = comp_total;
            P.blocks.insert(P.blocks.end(), blocks.begin() + i, blocks.begin() + j);
        }
        P.infl = infl;
        i = j;
        if (P.blocks.size() >= job->chunk_blocks || i < n) TRY(submit_pending(job));   // full, or the next block did not fit
    }
    return 0;
}

extern "C" int fastf_bam2db_feed(fastf_bam2db_job *job, const void *host_bytes, size_t n)
{
    fastf_ctx *ctx = job->ctx;
    CK(cudaSetDevice(ctx->device));
    if (job->sampled_done) return ctx_fail(ctx, "bam2db_feed: job already sampled");
    struct FeedClock { fastf_bam2db_job *j; double t0; ~FeedClock() { if (j->feed_timing) j->ft_feed_s += wall_seconds() - t0; } } feed_clock{job, job->feed_timing ? wall_seconds() : 0};
    const u8 *p = (const u8 *)host_bytes;
    job->comp_bytes += n;
    std::vector<FastfBgzfBlock> blocks;
    // 1. complete a partial block left over from the previous call
    while (!job->carry.empty() && n) {
        std::vector<u8> &c = job->carry;
        size_t want = 18;
        if (c.size() >= 18) {
            blocks.clear();
            size_t used = 0;
            int rc = fastf_bgzf_index(c.data(), c.size(), 0, blocks, &used);
            if (rc != FASTF_BGZF_OK && rc != FASTF_BGZF_NEED_MORE) return ctx_fail(ctx, "bam2db_feed: not a BGZF block (index error %d)", rc);
            if (!blocks.empty()) {
                // run the completed block(s) out of the carry buffer (pageable copy; rare path).  The copy must finish
                // before the carry buffer is edited, so drain the copy stream here.
                TRY(run_blocks(job, blocks, nullptr, 0, c.data()));
                CK(cudaStreamSynchronize(ctx->copy));
                c.erase(c.begin(), c.begin() + used);
                continue;
            }
            // header visible: total block size = BSIZE+1 (read it the same way the indexer does)
            u32 xlen = (u32)c[10] | ((u32)c[11] << 8);
            want = 12 + (size_t)xlen;
            if (c.size() >= want) {
                u32 bsize = 0;
                for (u32 x = 0; x + 4 <= xlen;) {
                    const u8 *sf = c.data() + 12 + x;
                    u32 slen = (u32)sf[2] | ((u32)sf[3] << 8);
                    if (sf[0] == 'B' && sf[1] == 'C' && slen == 2 && x + 6 <= xlen) bsize = ((u32)sf[4] | ((u32)sf[5] << 8)) + 1;
                    x += 4 + slen;
                }
                if (!bsize) return ctx_fail(ctx, "bam2db_feed: gzip member without a BGZF BC field");
                want = bsize;
            }
        }
        size_t take = std::min(n, want > c.size() ? want - c.size() : (size_t)1);
        c.insert(c.end(), p, p + take);
        p += take;
        n -= take;
    }
    if (!job->carry.empty()) {
        // n == 0: maybe the carry became a whole block exactly
        blocks.clear();
        size_t used = 0;
        int rc = fastf_bgzf_index(job->carry.data(), job->carry.size(), 0, blocks, &used);
        if (rc != FASTF_BGZF_OK && rc != FASTF_BGZF_NEED_MORE) return ctx_fail(ctx, "bam2db_feed: not a BGZF block (index error %d)", rc);
        if (!blocks.empty()) {
            TRY(run_blocks(job, blocks, nullptr, 0, job->carry.data()));
            CK(cudaStreamSynchronize(ctx->copy));
            job->carry.erase(job->carry.begin(), job->carry.begin() + used);
        }
        return 0;
    }
    if (!n) return 0;
    // 2. whole blocks straight out of the caller's buffer
    // (one chunk's worth of block headers at a time: the device starts on chunk i while the host walks the headers of chunk i+1)
    size_t used = 0;
    for (;;) {
        blocks.clear();
        size_t step = 0;
        int rc = fastf_bgzf_index(p + used, n - used, used, blocks, &step, job->chunk_bytes, (size_t)job->chunk_blocks);
        if (rc != FASTF_BGZF_OK && rc != FASTF_BGZF_NEED_MORE && rc != FASTF_BGZF_LIMIT) return ctx_fail(ctx, "bam2db_feed: not a BGZF stream at byte %zu (index error %d)", used + step, rc);
        used += step;
        if (!blocks.empty()) TRY(run_blocks(job, blocks, nullptr, 0, p));
        if (rc != FASTF_BGZF_LIMIT) break;
    }
    // 3. keep the tail.  The caller may reuse its buffer after we return: wait for the copies.
    if (used < n) job->carry.assign(p + used, p + n);
    CK(cudaStreamSynchronize(ctx->copy));
    return 0;
}

extern "C" int fastf_bam2db_feed_device(fastf_bam2db_job *job, const void *dev_bytes, size_t nbytes, const uint64_t *in_off, const uint32_t *in_len, const uint32_t *isize, uint64_t nblocks)
{
    fastf_ctx *ctx = job->ctx;
    CK(cudaSetDevice(ctx->device));
    if (job->sampled_done) return ctx_fail(ctx, "bam2db_feed_device: job already sampled");
    if (((uintptr_t)dev_bytes & 3u) != 0) return ctx_fail(ctx, "bam2db_feed_device: dev_bytes must be 4-byte aligned");
    std::vector<FastfBgzfBlock> blocks(nblocks);
    for (u64 i = 0; i < nblocks; i++) {
        if (in_off[i] + in_len[i] + 8 > nbytes || isize[i] > 65536) return ctx_fail(ctx, "bam2db_feed_device: block %llu outside the buffer", (unsigned long long)i);
        blocks[i].in_off = in_off[i]; blocks[i].in_len = in_len[i]; blocks[i].isize = isize[i]; blocks[i].crc32 = 0;
    }
    job->comp_bytes += nbytes;
    return run_blocks(job, blocks, (const u8 *)dev_bytes, nbytes & ~(u64)3, nullptr);
}

static int drain_chunks(fastf_bam2db_job *job)
{
    fastf_ctx *ctx = job->ctx;
    if (!job->carry.empty()) return ctx_fail(ctx, "bam2db: input ends inside a BGZF block (%zu trailing bytes)", job->carry.size());
    TRY(submit_pending(job));
    TRY(finalize_slot(job, job->next_slot));        // older one first (file order of the gathers does not matter, bases are absolute)
    TRY(finalize_slot(job, job->next_slot ^ 1u));
    return 0;
}

extern "C" int fastf_bam2db_counts(fastf_bam2db_job *job, uint64_t *n_records, uint64_t *n_cb_valid)
{
    fastf_ctx *ctx = job->ctx;
    CK(cudaSetDevice(ctx->device));
    TRY(drain_chunks(job));
    if (n_records) *n_records = job->n_records;
    if (n_cb_valid) *n_cb_valid = job->n_cand;
    return 0;
}

static int report_feed_timing(fastf_bam2db_job *job);

// The sampling pass over candidates cand[0, n) (file order) whose k-th meets draw first_draw + k: at the job's keep threshold (R null;
// draws as keep bits), or at the depth sweep's sorted thresholds R (draws as tempered words).  hist[p] / hist[FASTF_SWEEP_MAX_RATES + p]:
// reads / valid reads whose rate index is p (one rate: p = 0); the valid rows kept by the largest threshold land in job->kept, with the
// sweep's rate indices in job->kept_rate (file order).
static int sample_cands(fastf_bam2db_job *job, const char *who, u64 first_draw, const u64 *cand, u64 n, const FastfSweepRates *R, u64 *hist)
{
    fastf_ctx *ctx = job->ctx;
    if (n >= 0xffffffffull) return ctx_fail(ctx, "%s: %llu CB-valid reads exceed the 2^32-1 limit of one device; shard over more GPUs", who, (unsigned long long)n);
    const u32 K = R ? R->k : 1;
    const size_t hbytes = 2 * FASTF_SWEEP_MAX_RATES * sizeof(u64);
    memset(hist, 0, hbytes);
    u64 nk = 0;
    if (n) {
        // the number of draws is known now: generate exactly [first_draw, first_draw + n)
        TRY(mt_generate_parallel(job, who, first_draw, n, R != nullptr));
        CK(cudaEventRecord(job->ev_mt, ctx->mt));
        CK(cudaStreamWaitEvent(ctx->compute, job->ev_mt, 0));
        const u32 ntiles = (u32)((n + FASTF_SAMPLE_TILE - 1) / FASTF_SAMPLE_TILE);
        const u32 *draws = job->keepbits.as<u32>();
        TRY(dev_reserve(ctx, job->tile_valid, (size_t)ntiles * sizeof(u32)));
        TRY(dev_reserve(ctx, job->tile_tot, sizeof(u32)));
        CK(cudaMemsetAsync(job->sample_counters.p, 0, hbytes, ctx->compute));
        job->t_sample.start(ctx->compute);
        if (R) FASTF_LAUNCH(fastf_sweep_count_kernel, ntiles, FASTF_SAMPLE_THREADS, 0, ctx->compute, cand, n, draws, *R, job->tile_valid.as<u32>(), job->sample_counters.as<u64>());
        else FASTF_LAUNCH(fastf_sample_count_kernel, ntiles, FASTF_SAMPLE_THREADS, 0, ctx->compute, cand, n, draws, job->tile_valid.as<u32>(), job->sample_counters.as<u64>());
        CKL(R ? "sweep_count" : "sample_count");
        TRY(launch_scan_rows(ctx, job->tile_valid.as<u32>(), ntiles, 1, job->tile_tot.as<u32>(), ctx->compute));
        CK(cudaMemcpyAsync(job->small_host.p, job->sample_counters.p, hbytes, cudaMemcpyDeviceToHost, ctx->compute));
        CK(cudaStreamSynchronize(ctx->compute));
        memcpy(hist, job->small_host.p, hbytes);
        for (u32 p = 0; p < K; p++) nk += hist[FASTF_SWEEP_MAX_RATES + p];
        TRY(dev_reserve(ctx, job->kept, std::max<u64>(nk, 1) * sizeof(u64)));
        const u32 *tile_off = job->tile_valid.as<u32>();
        if (R) {
            TRY(dev_reserve(ctx, job->kept_rate, std::max<u64>(nk, 1) * sizeof(u32)));
            TRY(dev_reserve(ctx, job->rate_alt, std::max<u64>(nk, 1) * sizeof(u32)));
            FASTF_LAUNCH(fastf_sweep_scatter_kernel, ntiles, FASTF_SAMPLE_THREADS, 0, ctx->compute, cand, n, draws, *R, tile_off, job->kept.as<u64>(), job->kept_rate.as<u32>());
        } else {
            FASTF_LAUNCH(fastf_sample_scatter_kernel, ntiles, FASTF_SAMPLE_THREADS, 0, ctx->compute, cand, n, draws, tile_off, job->kept.as<u64>());
        }
        CKL(R ? "sweep_scatter" : "sample_scatter");
        job->t_sample.stop(ctx->compute);
        CK(cudaEventRecord(job->ev_last, ctx->compute));
    }
    job->n_sampled = 0;
    for (u32 p = 0; p < K; p++) job->n_sampled += hist[p];
    job->n_valid = nk;
    return 0;
}

// a job begun with fastf_bam2db_begin_grid is finished by fastf_bam2db_finish_grid only: its candidates carry the union table's cells
static int refuse_grid(fastf_bam2db_job *job, const char *who)
{
    if (job->grid) return ctx_fail(job->ctx, "%s: the job was begun with fastf_bam2db_begin_grid; finish it with fastf_bam2db_finish_grid", who);
    return 0;
}

// sample_cands over the job's own candidates, once, after the last feed; its CB-valid reads meet draws d0 + ordinal_base + k
static int sample_pass(fastf_bam2db_job *job, const char *who, u64 ordinal_base, const FastfSweepRates *R, u64 *hist)
{
    fastf_ctx *ctx = job->ctx;
    TRY(refuse_grid(job, who));
    if (job->sampled_done) return ctx_fail(ctx, "%s: the job was already sampled", who);
    TRY(drain_chunks(job));
    TRY(report_feed_timing(job));
    TRY(sample_cands(job, who, job->prm.d0 + ordinal_base, job->cand.as<u64>(), job->n_cand, R, hist));
    job->sampled_done = true;
    job->sweep_rates = R ? R->k : 0;
    return 0;
}

extern "C" int fastf_bam2db_sample(fastf_bam2db_job *job, uint64_t ordinal_base)
{
    fastf_ctx *ctx = job->ctx;
    CK(cudaSetDevice(ctx->device));
    u64 hist[2 * FASTF_SWEEP_MAX_RATES];
    return sample_pass(job, "bam2db_sample", ordinal_base, nullptr, hist);
}

extern "C" int fastf_bam2db_kept_device(fastf_bam2db_job *job, uint64_t **dev_keys, uint64_t *n)
{
    fastf_ctx *ctx = job->ctx;
    TRY(refuse_grid(job, "bam2db_kept_device"));
    if (!job->sampled_done) return ctx_fail(ctx, "bam2db_kept_device: call fastf_bam2db_sample first");
    if (job->sweep_rates) return ctx_fail(ctx, "bam2db_kept_device: the job was sampled by the depth sweep; use fastf_bam2db_kept_sweep_device");
    *dev_keys = job->kept.as<u64>();
    *n = job->n_valid;
    return 0;
}

extern "C" int fastf_bam2db_sample_counts(fastf_bam2db_job *job, uint64_t *sampled, uint64_t *valid)
{
    fastf_ctx *ctx = job->ctx;
    if (!job->sampled_done) return ctx_fail(ctx, "bam2db_sample_counts: call fastf_bam2db_sample first");
    if (sampled) *sampled = job->n_sampled;
    if (valid) *valid = job->n_valid;
    return 0;
}

extern "C" int fastf_bam2db_key_layout(fastf_bam2db_job *job, uint32_t *bits_cell, uint32_t *bits_gene, uint32_t *bits_umi)
{
    *bits_cell = job->L.bits_cell; *bits_gene = job->L.bits_gene; *bits_umi = job->L.bits_umi;
    return 0;
}

// sorted-unaware front half shared by finish and the device-level entry points: figure out which bits vary
static int varying_bits(fastf_ctx *ctx, DevBuf &orand, PinBuf &host, const u64 *keys, u64 n, u64 *varying, cudaStream_t s)
{
    u64 init[2] = {0ull, ~0ull};
    CK(cudaMemcpyAsync(orand.p, init, sizeof init, cudaMemcpyHostToDevice, s));
    u32 grid = (u32)std::min<u64>((n + 255) / 256, 148 * 8);
    FASTF_LAUNCH(fastf_key_bits_kernel, grid ? grid : 1, 256, 0, s, keys, n, orand.as<u64>());
    CKL("key_bits");
    CK(cudaMemcpyAsync(host.p, orand.p, 2 * sizeof(u64), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    *varying = host.as<u64>()[0] ^ host.as<u64>()[1];
    return 0;
}

static int coo_to_host(fastf_ctx *ctx, RleScratch &R, u64 nnz, u32 **m_gene, u32 **m_cell, u32 **m_count, cudaStream_t s)
{
    *m_gene = (u32 *)malloc(std::max<u64>(nnz, 1) * sizeof(u32));
    *m_cell = (u32 *)malloc(std::max<u64>(nnz, 1) * sizeof(u32));
    *m_count = (u32 *)malloc(std::max<u64>(nnz, 1) * sizeof(u32));
    if (!*m_gene || !*m_cell || !*m_count) return ctx_fail(ctx, "out of host memory for %llu COO rows", (unsigned long long)nnz);
    if (nnz) {
        TRY(d2h_pageable(ctx, *m_gene, R.out_gene.p, nnz * sizeof(u32), s));
        TRY(d2h_pageable(ctx, *m_cell, R.out_cell.p, nnz * sizeof(u32), s));
        TRY(d2h_pageable(ctx, *m_count, R.count.p, nnz * sizeof(u32), s));
        CK(cudaStreamSynchronize(s));
    }
    return 0;
}

// counters, sizes and the per-stage CUDA-event clocks of a job (no result arrays)
static int fill_stats(fastf_bam2db_job *job, fastf_bam2db_result *res)
{
    fastf_ctx *ctx = job->ctx;
    const FastfKeyLayout &L = job->L;
    res->total = job->n_records;
    res->cb_valid = job->n_cand;
    res->sampled = job->n_sampled;
    res->valid = job->n_valid;
    res->bits_cell = L.bits_cell; res->bits_gene = L.bits_gene; res->bits_umi = L.bits_umi; res->umi_max_bytes = L.umi_max_bytes;
    res->n_blocks = job->n_blocks; res->compressed_bytes = job->comp_bytes; res->inflated_bytes = job->infl_bytes;
    res->status = job->status;
    for (int i = 0; i < 2; i++) { job->t_infl[i].collect(&job->ms_inflate); job->t_crc[i].collect(&job->ms_crc); job->t_parse[i].collect(&job->ms_parse); job->t_gather[i].collect(&job->ms_gather); }
    job->t_mt.collect(&job->ms_mt); job->t_sample.collect(&job->ms_sample); job->t_sort.collect(&job->ms_sort); job->t_count.collect(&job->ms_count);
    res->ms_inflate = job->ms_inflate; res->ms_crc = job->ms_crc; res->ms_parse = job->ms_parse; res->ms_gather = job->ms_gather; res->ms_mt = job->ms_mt;
    res->ms_sample = job->ms_sample; res->ms_sort = job->ms_sort; res->ms_count = job->ms_count;
    if (job->first_recorded) {
        CK(cudaEventRecord(job->ev_last, ctx->compute));
        CK(cudaEventSynchronize(job->ev_last));
        CK(cudaEventElapsedTime(&res->ms_device_total, job->ev_first, job->ev_last));
    }
    res->n_launches = ctx->launches - job->launches0;
    res->n_chunks = job->n_chunks;
    return 0;
}

extern "C" int fastf_bam2db_stats(fastf_bam2db_job *job, fastf_bam2db_result *res)
{
    fastf_ctx *ctx = job->ctx;
    CK(cudaSetDevice(ctx->device));
    memset(res, 0, sizeof *res);
    CK(cudaStreamSynchronize(ctx->compute));
    CK(cudaStreamSynchronize(ctx->mt));
    return fill_stats(job, res);
}

// FASTF_FEED_TIMING=1: the host-fed job's copy / inflate / parse timeline on stderr (once, when the job is sampled)
static int report_feed_timing(fastf_bam2db_job *job)
{
    fastf_ctx *ctx = job->ctx;
    if (!job->feed_timing || job->ft_copy_ev.empty()) return 0;
    {
        CK(cudaStreamSynchronize(ctx->copy));
        double ms = 0, span = 0;
        for (auto &e : job->ft_copy_ev) { float t = 0; cudaEventElapsedTime(&t, e.first, e.second); ms += t; }
        { float t = 0; cudaEventElapsedTime(&t, job->ft_copy_ev.front().first, job->ft_copy_ev.back().second); span = t; }
        fprintf(stderr, "[fastf feed timing] H2D %zu copies, %.2f GB in %.1f ms of copy time = %.1f GB/s (first start to last end %.1f ms); host: %.1f ms inside feed calls, of which %.1f ms waiting for chunks to finish\n",
                job->ft_copy_ev.size(), job->ft_copy_bytes / 1e9, ms, job->ft_copy_bytes / 1e6 / std::max(ms, 1e-3), span, 1e3 * job->ft_feed_s, 1e3 * job->ft_wait_s);
        CK(cudaDeviceSynchronize());
        {
            // per chunk, ms since the first copy started: inflate start / end, parse end, and when the host submitted it
            cudaEvent_t o = job->ft_copy_ev.front().first;
            fprintf(stderr, "[fastf feed timing] chunk: host-submit | inflate start..end | parse end   (ms since the first H2D started; copies: start..end)\n");
            for (size_t k = 0; k < job->ft_infl_ev.size(); k++) {
                float a = 0, b = 0, c = 0;
                cudaEventElapsedTime(&a, o, job->ft_infl_ev[k].first); cudaEventElapsedTime(&b, o, job->ft_infl_ev[k].second);
                if (k < job->ft_parse_ev.size()) cudaEventElapsedTime(&c, o, job->ft_parse_ev[k]);
                fprintf(stderr, "[fastf feed timing]   %2zu: host %.1f | %.1f..%.1f | %.1f\n", k, 1e3 * (job->ft_host_submit[k] - job->ft_host_submit[0]), a, b, c);
            }
            for (size_t k = 0; k < job->ft_copy_ev.size(); k++) {
                float a = 0, b = 0;
                cudaEventElapsedTime(&a, o, job->ft_copy_ev[k].first); cudaEventElapsedTime(&b, o, job->ft_copy_ev[k].second);
                fprintf(stderr, "[fastf feed timing]   copy %2zu: %.1f..%.1f\n", k, a, b);
            }
        }
    }
    return 0;
}

extern "C" int fastf_bam2db_finish(fastf_bam2db_job *job, fastf_bam2db_result *res)
{
    fastf_ctx *ctx = job->ctx;
    CK(cudaSetDevice(ctx->device));
    memset(res, 0, sizeof *res);
    TRY(refuse_grid(job, "bam2db_finish"));
    if (job->sweep_rates) return ctx_fail(ctx, "bam2db_finish: the job was sampled by the depth sweep");
    if (!job->sampled_done) TRY(fastf_bam2db_sample(job, 0));
    const u64 n = job->n_valid;
    const FastfKeyLayout &L = job->L;
    if (job->prm.want_rows) {
        res->row_keys = (u64 *)malloc(std::max<u64>(n, 1) * sizeof(u64));
        if (!res->row_keys) return ctx_fail(ctx, "out of host memory for %llu rows", (unsigned long long)n);
        if (n) TRY(d2h_pageable(ctx, res->row_keys, job->kept.p, n * sizeof(u64), ctx->compute));
        res->n_rows = n;
    }
    u64 nnz = 0;
    if (n) {
        u64 varying = 0;
        job->t_sort.start(ctx->compute);
        TRY(varying_bits(ctx, job->orand, job->small_host, job->kept.as<u64>(), n, &varying, ctx->compute));
        u32 shifts[8];
        const int npass = plan_windows(varying, shifts);
        bool in_alt = false;
        // the candidate array is dead after sampling and at least as large as `kept`: reuse it as the ping-pong buffer
        TRY(sort_keys(ctx, job->sortS, job->kept.as<u64>(), job->cand.as<u64>(), nullptr, nullptr, n, shifts, npass, &in_alt, ctx->compute));
        job->t_sort.stop(ctx->compute);
        const u64 *sorted = in_alt ? job->cand.as<u64>() : job->kept.as<u64>();
        job->t_count.start(ctx->compute);
        TRY(rle_groups(ctx, job->rleS, sorted, nullptr, n, L.bits_umi, L.bits_umi - 1, L.bits_gene, &nnz, nullptr, ctx->compute));
        job->t_count.stop(ctx->compute);
        CK(cudaEventRecord(job->ev_last, ctx->compute));
    }
    TRY(coo_to_host(ctx, job->rleS, nnz, &res->m_gene, &res->m_cell, &res->m_count, ctx->compute));
    CK(cudaStreamSynchronize(ctx->compute));
    CK(cudaStreamSynchronize(ctx->mt));
    TRY(fill_stats(job, res));
    res->nnz = nnz;
    return 0;
}

// Depth sweep (include/fastf_gpu.h): draws as words -> per-rate histograms + (key, rate index) rows in file order -> ONE sort with the
// rate index as least significant digit -> distinct keys with their smallest rate index -> per rate, a predicated count over them.
// The front half (sample_pass) runs per job, the back half (sweep_count) wherever the rows of a key meet: in the same job for one
// GPU, on the receiving device of the exchange for several.

// thresholds in caller order -> R (ascending) and order[p] = caller index of sorted position p; ties keep caller order, so a row's
// rate index maps to the first of equal thresholds
static int sweep_rates(fastf_ctx *ctx, const char *who, uint32_t n_rates, const uint64_t *keep_thresholds, FastfSweepRates *R, u32 *order)
{
    if (n_rates < 1 || n_rates > FASTF_SWEEP_MAX_RATES || !keep_thresholds) return ctx_fail(ctx, "%s: 1..%u keep thresholds", who, (unsigned)FASTF_SWEEP_MAX_RATES);
    for (u32 i = 0; i < n_rates; i++)
        if (keep_thresholds[i] > 4294967296ull) return ctx_fail(ctx, "%s: keep_thresholds[%u] > 2^32", who, i);
    for (u32 i = 0; i < n_rates; i++) order[i] = i;
    std::stable_sort(order, order + n_rates, [&](u32 a, u32 b) { return keep_thresholds[a] < keep_thresholds[b]; });
    memset(R, 0, sizeof *R);
    R->k = n_rates;
    for (u32 p = 0; p < n_rates; p++) R->t[p] = keep_thresholds[order[p]];
    return 0;
}

// (key, rate index) rows in any order, repeated keys allowed; alt / rate_alt are ping-pong buffers of n elements.  One sort of
// (key, rate index), the rate index as the least significant digit: the first row of a run of equal keys carries the key's smallest
// rate index, and the run heads are the distinct keys (rleS.grp_key) with it (rleS.grp_val).  Then the smallest rate index of every
// (cell, gene) group, and per rate p (ascending threshold) one predicated count over the distinct keys, whose COO goes to the host
// arrays nnz[p] / m_*[p] (malloc'ed) before the next pass.  t_sort / t_count (nullable) time the sort and the count passes.
static int sweep_count(fastf_ctx *ctx, SortScratch &sortS, RleScratch &rleS, RleScratch &rateS, DevBuf &orand, PinBuf &host, u64 *keys, u64 *alt, u32 *rates, u32 *rate_alt, u64 n,
                       u32 key_bits, u32 bits_gene, u32 bits_umi, u32 K, Timer *t_sort, Timer *t_count, float *ms_count, u64 *nnz, u32 **m_gene, u32 **m_cell, u32 **m_count, cudaStream_t s)
{
    u64 nheads = 0;
    const u32 *grate = nullptr;   // FastfRatePred::grate of the distinct keys
    if (n) {
        u64 varying = 0;
        if (t_sort) t_sort->start(s);
        TRY(varying_bits(ctx, orand, host, keys, n, &varying, s));
        if (key_bits < 64) varying &= (1ull << key_bits) - 1ull;
        u32 shifts[9];
        shifts[0] = FASTF_SORT_VAL_DIGIT;
        const int npass = 1 + plan_windows(varying, shifts + 1);
        bool in_alt = false;
        TRY(sort_keys(ctx, sortS, keys, alt, rates, rate_alt, n, shifts, npass, &in_alt, s));
        const u64 *sorted = in_alt ? alt : keys;
        const u32 *sorted_rate = in_alt ? rate_alt : rates;
        u32 *gr = in_alt ? rates : rate_alt;   // the ping-pong buffer the sort left free
        TRY(rle_groups(ctx, rleS, sorted, sorted_rate, n, 0, 64, 0, &nheads, nullptr, s));
        FASTF_LAUNCH(fastf_group_rate_kernel, (u32)((nheads + 255) / 256), 256, 0, s, (const u64 *)rleS.grp_key.as<u64>(), (const u32 *)rleS.grp_val.as<u32>(), nheads, bits_umi, gr);
        grate = gr;
        CKL("group_rate");
        if (t_sort) t_sort->stop(s);
    }
    for (u32 p = 0; p < K; p++) {
        nnz[p] = 0;
        if (nheads) {
            if (t_count) t_count->start(s);
            TRY(rle_groups(ctx, rateS, rleS.grp_key.as<u64>(), nullptr, nheads, bits_umi, bits_umi - 1, bits_gene, &nnz[p], nullptr, s, FastfRatePred{rleS.grp_val.as<u32>(), grate, p}));
            if (t_count) { t_count->stop(s); t_count->collect(ms_count); }
        }
        TRY(coo_to_host(ctx, rateS, nnz[p], &m_gene[p], &m_cell[p], &m_count[p], s));
    }
    return 0;
}

// The depth sweep's results out of a job that sample_cands has just sampled at the thresholds `order` came from (hist: its histograms):
// the rows with their caller rate index, sweep_count with `alt` (a dead array of at least job->n_valid keys) as the keys' ping-pong
// buffer, per caller rate the counters and COO, and the job's stats (cb_valid = the job's candidates).
static int sweep_finish(fastf_bam2db_job *job, u32 K, const u32 *order, const u64 *hist, u64 *alt, fastf_bam2db_sweep_result *res)
{
    fastf_ctx *ctx = job->ctx;
    const FastfKeyLayout &L = job->L;
    const u64 nk = job->n_valid;   // valid rows kept by the largest threshold
    // the rows in file order, each with the caller index of its rate
    if (job->prm.want_rows) {
        res->row_keys = (u64 *)malloc(std::max<u64>(nk, 1) * sizeof(u64));
        res->row_rate = (u8 *)malloc(std::max<u64>(nk, 1));
        u32 *rb = (u32 *)malloc(std::max<u64>(nk, 1) * sizeof(u32));
        if (!res->row_keys || !res->row_rate || !rb) { free(rb); return ctx_fail(ctx, "out of host memory for %llu rows", (unsigned long long)nk); }
        int rc = 0;
        if (nk) rc = d2h_pageable(ctx, res->row_keys, job->kept.p, nk * sizeof(u64), ctx->compute) || d2h_pageable(ctx, rb, job->kept_rate.p, nk * sizeof(u32), ctx->compute);
        for (u64 r = 0; r < nk && !rc; r++) res->row_rate[r] = (u8)order[rb[r]];
        free(rb);
        if (rc) return rc;
        res->n_rows = nk;
    }
    fastf_bam2db_result *out = res->rate;
    u64 nnz[FASTF_SWEEP_MAX_RATES];
    u32 *mg[FASTF_SWEEP_MAX_RATES] = {}, *mc[FASTF_SWEEP_MAX_RATES] = {}, *mn[FASTF_SWEEP_MAX_RATES] = {};
    const int crc = sweep_count(ctx, job->sortS, job->rleS, job->rateS, job->orand, job->small_host, job->kept.as<u64>(), alt, job->kept_rate.as<u32>(), job->rate_alt.as<u32>(), nk,
                                L.bits_cell + L.bits_gene + L.bits_umi, L.bits_gene, L.bits_umi, K, &job->t_sort, &job->t_count, &job->ms_count, nnz, mg, mc, mn, ctx->compute);
    for (u32 p = 0; p < K; p++) { out[order[p]].m_gene = mg[p]; out[order[p]].m_cell = mc[p]; out[order[p]].m_count = mn[p]; }
    if (crc) return crc;
    u64 sampled = 0, valid = 0;
    for (u32 p = 0; p < K; p++) {
        fastf_bam2db_result &r = out[order[p]];
        sampled += hist[p];
        valid += hist[FASTF_SWEEP_MAX_RATES + p];
        r.sampled = sampled;
        r.valid = valid;
        r.nnz = nnz[p];
    }
    CK(cudaEventRecord(job->ev_last, ctx->compute));
    CK(cudaStreamSynchronize(ctx->compute));
    CK(cudaStreamSynchronize(ctx->mt));
    fastf_bam2db_result st;
    memset(&st, 0, sizeof st);
    TRY(fill_stats(job, &st));
    res->n_rates = K;
    for (u32 i = 0; i < K; i++) {
        fastf_bam2db_result &r = out[i];
        const fastf_bam2db_result keep = r;
        r = st;
        r.sampled = keep.sampled; r.valid = keep.valid; r.nnz = keep.nnz;
        r.m_gene = keep.m_gene; r.m_cell = keep.m_cell; r.m_count = keep.m_count;
    }
    return 0;
}

extern "C" int fastf_bam2db_finish_sweep(fastf_bam2db_job *job, uint32_t n_rates, const uint64_t *keep_thresholds, fastf_bam2db_sweep_result *res)
{
    const char *who = "bam2db_finish_sweep";
    fastf_ctx *ctx = job->ctx;
    CK(cudaSetDevice(ctx->device));
    memset(res, 0, sizeof *res);
    FastfSweepRates R;
    u32 order[FASTF_SWEEP_MAX_RATES];
    TRY(sweep_rates(ctx, who, n_rates, keep_thresholds, &R, order));
    TRY(refuse_grid(job, who));
    if (job->sampled_done) return ctx_fail(ctx, "bam2db_finish_sweep: the job was already sampled at one rate");
    u64 hist[2 * FASTF_SWEEP_MAX_RATES];
    TRY(sample_pass(job, who, 0, &R, hist));
    // the candidate array is dead after sampling and at least as large as `kept`: the keys' ping-pong buffer
    return sweep_finish(job, n_rates, order, hist, job->cand.as<u64>(), res);
}

// Cell-rate grid (include/fastf_gpu.h): the job parsed against the union of the cell tables, non-insertable reads keeping their cell
// (fastf_parse_record<true>).  Per cell rate: remap + compaction into the candidate array a job begun with that rate's table would
// have gathered (fastf_grid_count / scatter_kernel), then the depth sweep over it at the rate's d0.  job->cand is read by every rate.
extern "C" int fastf_bam2db_begin_grid(fastf_ctx *ctx, const fastf_bam2db_params *p, fastf_bam2db_job **out)
{
    TRY(fastf_bam2db_begin(ctx, p, out));
    (*out)->grid = true;
    return 0;
}

// the caller's remap tables: 1..FASTF_GRID_MAX_CELL_RATES of them, each a one-to-one map of the union cells it holds onto 1..n_cells
static int grid_check_cell_rates(fastf_bam2db_job *job, const char *who, uint32_t n_cell_rates, const fastf_bam2db_cell_rate *cell_rates)
{
    fastf_ctx *ctx = job->ctx;
    const u32 n_union = job->prm.n_cells;
    if (n_cell_rates < 1 || n_cell_rates > FASTF_GRID_MAX_CELL_RATES || !cell_rates) return ctx_fail(ctx, "%s: 1..%u cell rates", who, (unsigned)FASTF_GRID_MAX_CELL_RATES);
    for (u32 i = 0; i < n_cell_rates; i++) {
        const fastf_bam2db_cell_rate &c = cell_rates[i];
        if (n_union && !c.cell_index) return ctx_fail(ctx, "%s: cell_rates[%u].cell_index is NULL", who, i);
        if (c.n_cells > n_union) return ctx_fail(ctx, "%s: cell_rates[%u].n_cells = %u exceeds the union table's %u cells", who, i, c.n_cells, n_union);
        std::vector<u8> seen((size_t)c.n_cells + 1, 0);
        u32 held = 0;
        for (u32 u = 0; u < n_union; u++) {
            const u32 v = c.cell_index[u];
            if (!v) continue;
            if (v > c.n_cells) return ctx_fail(ctx, "%s: cell_rates[%u].cell_index[%u] = %u exceeds its n_cells = %u", who, i, u, v, c.n_cells);
            if (seen[v]) return ctx_fail(ctx, "%s: cell_rates[%u].cell_index holds %u twice", who, i, v);
            seen[v] = 1;
            held++;
        }
        if (held != c.n_cells) return ctx_fail(ctx, "%s: cell_rates[%u] maps %u union cells onto its n_cells = %u (every cell of its table must be in the union)", who, i, held, c.n_cells);
    }
    return 0;
}

extern "C" int fastf_bam2db_finish_grid(fastf_bam2db_job *job, uint32_t n_cell_rates, const fastf_bam2db_cell_rate *cell_rates, uint32_t n_rates, const uint64_t *keep_thresholds,
                                        fastf_bam2db_sweep_result *res)
{
    const char *who = "bam2db_finish_grid";
    fastf_ctx *ctx = job->ctx;
    CK(cudaSetDevice(ctx->device));
    // zeroed before anything is checked: the caller frees every res[i], also after a refusal
    for (u32 i = 0; res && i < std::min<u32>(n_cell_rates, FASTF_GRID_MAX_CELL_RATES); i++) memset(&res[i], 0, sizeof res[i]);
    if (!job->grid) return ctx_fail(ctx, "%s: the job was not begun with fastf_bam2db_begin_grid", who);
    if (!res) return ctx_fail(ctx, "%s: res is NULL", who);
    TRY(grid_check_cell_rates(job, who, n_cell_rates, cell_rates));
    FastfSweepRates R;
    u32 order[FASTF_SWEEP_MAX_RATES];
    TRY(sweep_rates(ctx, who, n_rates, keep_thresholds, &R, order));
    if (job->sampled_done) return ctx_fail(ctx, "%s: the job was already finished", who);
    TRY(drain_chunks(job));
    TRY(report_feed_timing(job));
    job->sampled_done = true;
    const FastfKeyLayout &L = job->L;
    const u32 n_union = job->prm.n_cells, cell_shift = L.bits_gene + L.bits_umi;
    const u64 n = job->n_cand;
    if (n >= 0xffffffffull) return ctx_fail(ctx, "%s: %llu CB-valid reads exceed the 2^32-1 limit of one device", who, (unsigned long long)n);
    const u32 ntiles = (u32)((n + FASTF_SAMPLE_TILE - 1) / FASTF_SAMPLE_TILE);
    if (n) {
        TRY(dev_reserve(ctx, job->grid_cand, n * sizeof(u64)));
        TRY(dev_reserve(ctx, job->grid_remap, (size_t)n_union * sizeof(u32)));
    }
    for (u32 i = 0; i < n_cell_rates; i++) {
        const fastf_bam2db_cell_rate &c = cell_rates[i];
        // this rate's own clocks (the previous rate's fill_stats collected every timer)
        job->ms_mt = job->ms_sample = job->ms_sort = job->ms_count = 0;
        u64 ni = 0;
        if (n) {
            // sample_cands of the previous rate may have left smaller tile arrays
            TRY(dev_reserve(ctx, job->tile_valid, (size_t)ntiles * sizeof(u32)));
            TRY(dev_reserve(ctx, job->tile_tot, sizeof(u32)));
            CK(cudaMemcpyAsync(job->grid_remap.p, c.cell_index, (size_t)n_union * sizeof(u32), cudaMemcpyHostToDevice, ctx->compute));
            job->t_sample.start(ctx->compute);
            FASTF_LAUNCH(fastf_grid_count_kernel, ntiles, FASTF_SAMPLE_THREADS, 0, ctx->compute, (const u64 *)job->cand.as<u64>(), n, (const u32 *)job->grid_remap.as<u32>(), n_union, cell_shift,
                         job->tile_valid.as<u32>());
            CKL("grid_count");
            TRY(launch_scan_rows(ctx, job->tile_valid.as<u32>(), ntiles, 1, job->tile_tot.as<u32>(), ctx->compute));
            FASTF_LAUNCH(fastf_grid_scatter_kernel, ntiles, FASTF_SAMPLE_THREADS, 0, ctx->compute, (const u64 *)job->cand.as<u64>(), n, (const u32 *)job->grid_remap.as<u32>(), n_union, cell_shift,
                         L.bits_umi, (const u32 *)job->tile_valid.as<u32>(), job->grid_cand.as<u64>());
            CKL("grid_scatter");
            job->t_sample.stop(ctx->compute);
            CK(cudaMemcpyAsync(job->small_host.p, job->tile_tot.p, sizeof(u32), cudaMemcpyDeviceToHost, ctx->compute));
            CK(cudaStreamSynchronize(ctx->compute));
            ni = job->small_host.as<u32>()[0];
            job->t_sample.collect(&job->ms_sample);
        }
        u64 hist[2 * FASTF_SWEEP_MAX_RATES];
        TRY(sample_cands(job, who, c.d0, job->grid_cand.as<u64>(), ni, &R, hist));
        // the compacted array is dead after sampling and holds at least `kept`: the keys' ping-pong buffer
        TRY(sweep_finish(job, n_rates, order, hist, job->grid_cand.as<u64>(), &res[i]));
        for (u32 j = 0; j < n_rates; j++) { res[i].rate[j].cb_valid = ni; res[i].rate[j].bits_cell = bits_for(c.n_cells); }
    }
    return 0;
}

extern "C" int fastf_bam2db_sample_sweep(fastf_bam2db_job *job, uint64_t ordinal_base, uint32_t n_rates, const uint64_t *sorted_thresholds, uint64_t *sampled, uint64_t *valid)
{
    const char *who = "bam2db_sample_sweep";
    fastf_ctx *ctx = job->ctx;
    CK(cudaSetDevice(ctx->device));
    FastfSweepRates R;
    u32 order[FASTF_SWEEP_MAX_RATES];
    TRY(sweep_rates(ctx, who, n_rates, sorted_thresholds, &R, order));
    for (u32 i = 1; i < n_rates; i++)
        if (sorted_thresholds[i] < sorted_thresholds[i - 1]) return ctx_fail(ctx, "%s: thresholds must be non-decreasing (sorted_thresholds[%u] < sorted_thresholds[%u])", who, i, i - 1);
    u64 hist[2 * FASTF_SWEEP_MAX_RATES];
    TRY(sample_pass(job, who, ordinal_base, &R, hist));
    u64 s = 0, v = 0;
    for (u32 p = 0; p < n_rates; p++) {
        s += hist[p];
        v += hist[FASTF_SWEEP_MAX_RATES + p];
        if (sampled) sampled[p] = s;
        if (valid) valid[p] = v;
    }
    return 0;
}

extern "C" int fastf_bam2db_kept_sweep_device(fastf_bam2db_job *job, uint64_t **dev_keys, uint32_t **dev_rates, uint64_t *n)
{
    fastf_ctx *ctx = job->ctx;
    if (!job->sweep_rates) return ctx_fail(ctx, "bam2db_kept_sweep_device: call fastf_bam2db_sample_sweep first");
    *dev_keys = job->kept.as<u64>();
    *dev_rates = job->kept_rate.as<u32>();
    *n = job->n_valid;
    return 0;
}

extern "C" int fastf_sweep_count_device(fastf_ctx *ctx, uint64_t *dev_keys, uint32_t *dev_rates, uint64_t n, uint32_t key_bits, uint32_t bits_gene, uint32_t bits_umi, uint32_t n_rates,
                                        uint64_t *nnz, uint32_t **m_gene, uint32_t **m_cell, uint32_t **m_count)
{
    CK(cudaSetDevice(ctx->device));
    if (n_rates < 1 || n_rates > FASTF_SWEEP_MAX_RATES) return ctx_fail(ctx, "sweep_count_device: 1..%u rates", (unsigned)FASTF_SWEEP_MAX_RATES);
    if (key_bits > 64 || bits_umi < 2 || bits_gene + bits_umi > key_bits) return ctx_fail(ctx, "sweep_count_device: key layout %u / %u / %u bits", key_bits, bits_gene, bits_umi);
    for (u32 p = 0; p < n_rates; p++) { nnz[p] = 0; m_gene[p] = m_cell[p] = m_count[p] = nullptr; }
    cudaStream_t s = ctx->compute;
    SortScratch S;
    RleScratch R, RR;
    DevBuf alt, ralt, orand;
    PinBuf host;
    DrainOnExit drain{ctx};
    int rc = dev_reserve(ctx, alt, std::max<u64>(n, 1) * sizeof(u64));
    if (!rc) rc = dev_reserve(ctx, ralt, std::max<u64>(n, 1) * sizeof(u32));
    if (!rc) rc = dev_reserve(ctx, orand, 2 * sizeof(u64));
    if (!rc) rc = pin_reserve(ctx, host, 2 * sizeof(u64));
    if (!rc) rc = sweep_count(ctx, S, R, RR, orand, host, dev_keys, alt.as<u64>(), dev_rates, ralt.as<u32>(), n, key_bits, bits_gene, bits_umi, n_rates, nullptr, nullptr, nullptr, nnz, m_gene, m_cell,
                              m_count, s);
    if (!rc && cudaStreamSynchronize(s) != cudaSuccess) rc = ctx_fail(ctx, "sweep_count_device: stream error");
    if (rc)
        for (u32 p = 0; p < n_rates; p++) { free(m_gene[p]); free(m_cell[p]); free(m_count[p]); m_gene[p] = m_cell[p] = m_count[p] = nullptr; nnz[p] = 0; }
    return rc;
}

extern "C" void fastf_bam2db_sweep_result_free(fastf_bam2db_sweep_result *res)
{
    if (!res) return;
    for (u32 i = 0; i < FASTF_SWEEP_MAX_RATES; i++) fastf_bam2db_result_free(&res->rate[i]);
    free(res->row_keys); free(res->row_rate);
    res->row_keys = nullptr;
    res->row_rate = nullptr;
    res->n_rows = 0;
}

extern "C" void fastf_bam2db_result_free(fastf_bam2db_result *res)
{
    if (!res) return;
    free(res->m_gene); free(res->m_cell); free(res->m_count); free(res->row_keys);
    res->m_gene = res->m_cell = res->m_count = nullptr;
    res->row_keys = nullptr;
}
