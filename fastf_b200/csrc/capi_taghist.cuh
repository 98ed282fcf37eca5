// Part of the libfastf_gpu translation unit (capi.cu includes it, in this order; it is not a header of its own):
// crb / extract: aux-tag histograms.
#pragma once

// ---------------------------------------------------------------------------------------------------
// crb / extract: histogram of one aux tag (or of the pair of two) over all records of a BAM image
// ---------------------------------------------------------------------------------------------------
extern "C" void fastf_taghist_result_free(fastf_taghist_result *res)
{
    if (!res) return;
    free(res->first); free(res->count); free(res->ivalue); free(res->a_off); free(res->a_len); free(res->b_len); free(res->strings);
    res->first = nullptr; res->count = nullptr; res->ivalue = nullptr; res->a_off = nullptr; res->a_len = nullptr; res->b_len = nullptr; res->strings = nullptr;
}

// One chunk's groups, merged on the host across chunks (a value's count adds up, its first occurrence is the smallest ordinal)
struct TagAgg { u64 count; u64 first; };

// One pass over the BAM image: chunks of whole blocks, each inflated and grouped on the device, the groups merged here
static int taghist_run(fastf_ctx *ctx, const void *host_bytes, size_t n, const char *tag_a, uint32_t mode, const char *tag_b, uint32_t inflate_lanes, fastf_taghist_result *res)
{
    cudaStream_t s = ctx->compute;
    InflatedFile F;
    DevBuf hdr_off, counters, stage_off, stage, keys, loc_a, loc_b, vals, kalt, valt, orand, coll, rep_a, rep_b, blob_off, blob, virt;
    const bool straddle = (inflate_lanes & FASTF_BAM_STRADDLE) != 0;   // records may cross BGZF block boundaries (bam_straddle.cuh): one chunk
    PinBuf host;
    SortScratch S;
    RleScratch R;
    Timer t_tags, t_sort, t_rle;
    Event e0, e1;
    DrainOnExit drain{ctx};
    std::vector<FastfBgzfBlock> all, part;
    std::vector<u64> h_stage_off, h_rep_a, h_rep_b, h_blob_off, h_key;
    std::vector<u32> h_start, h_first;
    std::vector<char> h_blob;
    // groups merged across chunks: strings keyed by "A \0 B" (values hold no NUL), integers by value
    std::unordered_map<std::string, TagAgg> smap;
    std::unordered_map<int32_t, TagAgg> imap;
    if (t_tags.init() || t_sort.init() || t_rle.init() || e0.create() != cudaSuccess || e1.create() != cudaSuccess) return ctx_fail(ctx, "taghist: event creation failed");
    {
        size_t used = 0;
        int rc = fastf_bgzf_index((const u8 *)host_bytes, n, 0, all, &used);
        if (rc != FASTF_BGZF_OK) return ctx_fail(ctx, "taghist: not a whole BGZF stream (index error %d at byte %zu of %zu)", rc, used, n);
    }
    CK(cudaEventRecord(e0, s));
    res->n_blocks = all.size(); res->compressed_bytes = n;
    TRY(pin_reserve(ctx, host, 64));
    TRY(dev_reserve(ctx, hdr_off, sizeof(u64)));
    TRY(dev_reserve(ctx, counters, 4 * sizeof(u64)));
    TRY(dev_reserve(ctx, orand, 2 * sizeof(u64)));
    TRY(dev_reserve(ctx, coll, sizeof(u32)));
    FastfTagQuery Q;
    Q.a0 = (u8)tag_a[0]; Q.a1 = (u8)tag_a[1];
    Q.b0 = tag_b ? (u8)tag_b[0] : 0u; Q.b1 = tag_b ? (u8)tag_b[1] : 0u;
    Q.mode = mode;
    // The file streams through HBM in chunks of whole blocks (two full rounds of the persistent inflate kernel each); every chunk
    // is grouped on the device, the per-chunk groups are merged here.
    size_t chunk_blocks = std::max<size_t>(1, ctx->taghist_chunk_blocks ? ctx->taghist_chunk_blocks : 2ull * (size_t)ctx->n_sm * FASTF_TPS_STREAMS);
    if (straddle) chunk_blocks = std::max<size_t>(all.size(), 1);
    else if (!ctx->taghist_chunk_blocks) {
        // a file whose inflated bytes, staging planes (worst case 2/3 of them) and key arrays fit HBM comfortably goes through in ONE
        // chunk: no host-side merge at all
        u64 infl_total = 0;
        for (auto &b : all) infl_total += b.isize;
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess && (double)infl_total * 2.6 + (double)n < 0.7 * (double)free_b && all.size() < 0xffffffffull) chunk_blocks = all.size();
    }
    u64 hit_base = 0;
    bool first_chunk = true, single = false;
    u64 single_groups = 0, single_hits = 0;
    res->hash_rounds = 1;
    smap.reserve(1u << 16);
    for (size_t c0 = 0; c0 < all.size() || first_chunk; c0 += chunk_blocks) {
        const size_t c1 = std::min(all.size(), c0 + chunk_blocks);
        part.assign(all.begin() + c0, all.begin() + c1);
        float ms_infl = 0;
        TRY(inflate_whole(ctx, F, host_bytes, n, nullptr, &part, inflate_lanes, &ms_infl, s));
        res->ms_inflate += ms_infl;
        res->inflated_bytes += F.infl_bytes;
        const u32 nb = (u32)F.n_blocks;
        // per-block staging slices (a record is >= 36 bytes)
        h_stage_off.resize((size_t)nb + 1);
        u64 plane = 0;
        for (u32 i = 0; i < nb; i++) {
            h_stage_off[i] = plane;
            plane += straddle ? stage_cap_for(F.idx.h_isize[i] + (i + 1 < nb ? F.idx.h_isize[i + 1] : 0)) + 1u : stage_cap_for(F.idx.h_isize[i]);
        }
        h_stage_off[nb] = plane;   // the kernel reads the slice capacity as stage_off[b + 1] - stage_off[b]
        TRY(dev_reserve(ctx, stage_off, h_stage_off.size() * sizeof(u64)));
        CK(cudaMemcpyAsync(stage_off.p, h_stage_off.data(), h_stage_off.size() * sizeof(u64), cudaMemcpyHostToDevice, s));
        TRY(dev_reserve(ctx, stage, std::max<u64>(plane, 1) * 3 * sizeof(u64)));
        u64 n_hits = 0, ngroups = 0, n_rec = 0;
        for (u32 round = 0;; round++) {
            if (round == 4) return ctx_fail(ctx, "taghist: 64-bit hash collisions in four rounds with different seeds");
            Q.seed = 0x9e3779b97f4a7c15ull * round;
            Q.key_mask = (round == 0 && ctx->taghist_round0_mask) ? ctx->taghist_round0_mask : ~0ull;
            if (round + 1 > res->hash_rounds) res->hash_rounds = round + 1;
            CK(cudaMemsetAsync(counters.p, 0, 4 * sizeof(u64), s));
            CK(cudaMemsetAsync(hdr_off.p, 0, sizeof(u64), s));
            t_tags.collect(&res->ms_tags);
            t_tags.start(s);
            if (first_chunk) {
                FASTF_LAUNCH(fastf_bam_header_kernel, 1, 32, 0, s, (const u8 *)F.infl.as<u8>(), F.infl_bytes, hdr_off.as<u64>(), (u32 *)(counters.as<u64>() + 2));
                CKL("bam_header");
            }
            const u64 *p_off = F.idx.out_off;
            const u32 *p_size = F.idx.isize;
            if (straddle) TRY(launch_virtual_blocks(ctx, virt, (const u8 *)F.infl.as<u8>(), F.infl_bytes, F.idx.out_off, F.idx.isize, nb, hdr_off.as<u64>(), (u32 *)(counters.as<u64>() + 2), &p_off, &p_size, s));
            if (nb) {
                FASTF_LAUNCH(fastf_bam_tags_kernel, (nb + FASTF_PARSE_WARPS - 1) / FASTF_PARSE_WARPS, FASTF_PARSE_WARPS * 32, 0, s, (const u8 *)F.infl.as<u8>(), (u64)((F.infl_bytes + 15) & ~15ull),
                             p_off, p_size, nb, (const u64 *)hdr_off.as<u64>(), Q, (const u64 *)stage_off.as<u64>(), stage.as<u64>(), plane, F.idx.nrec,
                             F.idx.ncbv, F.idx.st_parse);
                CKL("bam_tags");
            }
            FASTF_LAUNCH(fastf_chunk_counts_kernel, 1, FASTF_SCAN_THREADS, 0, s, (const u32 *)F.idx.nrec, (const u32 *)F.idx.ncbv, (const u32 *)F.idx.st_infl, (const u32 *)F.idx.st_parse, nb,
                         F.idx.dst_base, counters.as<u64>());
            CKL("chunk_counts");
            t_tags.stop(s);
            CK(cudaMemcpyAsync(host.p, counters.p, 4 * sizeof(u64), cudaMemcpyDeviceToHost, s));
            CK(cudaStreamSynchronize(s));
            n_rec = host.as<u64>()[0];
            n_hits = host.as<u64>()[1];
            res->status |= (u32)host.as<u64>()[2];
            if (res->status) {
                char buf[256];
                if (res->status & FASTF_ST_TAG_TYPE)
                    return ctx_fail(ctx, "taghist: tag-not-a-string: a record carries %c%c%s as a non-string value%s (the reference passes bam_aux2Z()'s NULL to strcmp/strcpy there)", tag_a[0],
                                    tag_a[1], tag_b ? " or its partner tag" : "", tag_b ? ", or lacks the partner tag" : "");
                return ctx_fail(ctx, "taghist: malformed input: %s", status_string(res->status, buf, sizeof buf));
            }
            if (hit_base + n_hits >= 0xffffffffull) return ctx_fail(ctx, "taghist: more than 2^32-1 tagged records");
            ngroups = 0;
            if (!n_hits) break;
            TRY(dev_reserve(ctx, keys, n_hits * sizeof(u64)));
            TRY(dev_reserve(ctx, loc_a, n_hits * sizeof(u64)));
            TRY(dev_reserve(ctx, loc_b, n_hits * sizeof(u64)));
            TRY(dev_reserve(ctx, kalt, n_hits * sizeof(u64)));
            TRY(dev_reserve(ctx, vals, n_hits * sizeof(u32)));
            TRY(dev_reserve(ctx, valt, n_hits * sizeof(u32)));
            t_sort.collect(&res->ms_sort);
            t_sort.start(s);
            u64 *planes[3] = {keys.as<u64>(), loc_a.as<u64>(), loc_b.as<u64>()};
            for (int k = 0; k < 3; k++) {
                FASTF_LAUNCH(fastf_stage_gather_kernel, (nb + 7) / 8, 256, 0, s, (const u64 *)(stage.as<u64>() + (u64)k * plane), (const u64 *)stage_off.as<u64>(), (const u32 *)F.idx.ncbv,
                             (const u64 *)F.idx.dst_base, nb, planes[k]);
                CKL("stage_gather");
            }
            FASTF_LAUNCH(fastf_iota_kernel, (u32)((n_hits + 255) / 256), 256, 0, s, vals.as<u32>(), n_hits);
            CKL("iota");
            u64 varying = 0;
            TRY(varying_bits(ctx, orand, host, keys.as<u64>(), n_hits, &varying, s));
            u32 shifts[8];
            const int npass = plan_windows(varying, shifts);
            bool in_alt = false;
            TRY(sort_keys(ctx, S, keys.as<u64>(), kalt.as<u64>(), vals.as<u32>(), valt.as<u32>(), n_hits, shifts, npass, &in_alt, s));
            t_sort.stop(s);
            const u64 *sorted = in_alt ? kalt.as<u64>() : keys.as<u64>();
            const u32 *perm = in_alt ? valt.as<u32>() : vals.as<u32>();
            t_rle.collect(&res->ms_rle);
            t_rle.start(s);
            u64 nd = 0;
            TRY(rle_groups(ctx, R, sorted, perm, n_hits, 0, 64, 0, &ngroups, &nd, s));
            u32 collided = 0;
            if (mode == FASTF_TAG_MODE_STRING) {
                CK(cudaMemsetAsync(coll.p, 0, sizeof(u32), s));
                FASTF_LAUNCH(fastf_taghist_verify_kernel, (u32)((n_hits + 255) / 256), 256, 0, s, (const u8 *)F.infl.as<u8>(), sorted, perm, (const u64 *)loc_a.as<u64>(),
                             (const u64 *)loc_b.as<u64>(), n_hits, coll.as<u32>());
                CKL("taghist_verify");
                CK(cudaMemcpyAsync(host.p, coll.p, sizeof(u32), cudaMemcpyDeviceToHost, s));
                CK(cudaStreamSynchronize(s));
                collided = host.as<u32>()[0];
            }
            t_rle.stop(s);
            if (!collided) break;   // every group holds one value: done.  Otherwise hash again with another seed.
        }
        // ---- this chunk's groups to the host, merged into the maps ----
        res->n_records += n_rec;
        res->n_hits += n_hits;
        if (ngroups) {
            h_start.resize(ngroups); h_first.resize(ngroups); h_key.resize(ngroups);
            CK(cudaMemcpyAsync(h_first.data(), R.grp_val.p, ngroups * sizeof(u32), cudaMemcpyDeviceToHost, s));
            CK(cudaMemcpyAsync(h_start.data(), R.grp_first.p, ngroups * sizeof(u32), cudaMemcpyDeviceToHost, s));
            CK(cudaMemcpyAsync(h_key.data(), R.grp_key.p, ngroups * sizeof(u64), cudaMemcpyDeviceToHost, s));
            if (mode == FASTF_TAG_MODE_STRING) {
                TRY(dev_reserve(ctx, rep_a, ngroups * sizeof(u64)));
                TRY(dev_reserve(ctx, rep_b, ngroups * sizeof(u64)));
                FASTF_LAUNCH(fastf_taghist_reps_kernel, (u32)((ngroups + 255) / 256), 256, 0, s, (const u32 *)R.grp_val.as<u32>(), (const u64 *)loc_a.as<u64>(), (const u64 *)loc_b.as<u64>(),
                             (u32)ngroups, rep_a.as<u64>(), rep_b.as<u64>());
                CKL("taghist_reps");
                h_rep_a.resize(ngroups); h_rep_b.resize(ngroups); h_blob_off.resize(ngroups);
                CK(cudaMemcpyAsync(h_rep_a.data(), rep_a.p, ngroups * sizeof(u64), cudaMemcpyDeviceToHost, s));
                CK(cudaMemcpyAsync(h_rep_b.data(), rep_b.p, ngroups * sizeof(u64), cudaMemcpyDeviceToHost, s));
            }
            CK(cudaStreamSynchronize(s));
            if (mode == FASTF_TAG_MODE_STRING) {
                u64 total = 0;
                for (u64 g = 0; g < ngroups; g++) { h_blob_off[g] = total; total += (h_rep_a[g] & 0xffffu) + (h_rep_b[g] & 0xffffu); }
                h_blob.resize(std::max<u64>(total, 1));
                TRY(dev_reserve(ctx, blob_off, ngroups * sizeof(u64)));
                TRY(dev_reserve(ctx, blob, std::max<u64>(total, 1)));
                CK(cudaMemcpyAsync(blob_off.p, h_blob_off.data(), ngroups * sizeof(u64), cudaMemcpyHostToDevice, s));
                FASTF_LAUNCH(fastf_taghist_strings_kernel, (u32)((ngroups * 32 + 255) / 256), 256, 0, s, (const u8 *)F.infl.as<u8>(), (const u64 *)rep_a.as<u64>(), (const u64 *)rep_b.as<u64>(),
                             (const u64 *)blob_off.as<u64>(), (u32)ngroups, blob.as<u8>());
                CKL("taghist_strings");
                if (total) CK(cudaMemcpyAsync(h_blob.data(), blob.p, total, cudaMemcpyDeviceToHost, s));
                CK(cudaStreamSynchronize(s));
            }
            if (c0 == 0 && c1 == all.size()) {
                // the whole file was one chunk: its groups are the result, no merge
                single = true;
                single_groups = ngroups;
                single_hits = n_hits;
                break;
            }
            std::string k;
            for (u64 g = 0; g < ngroups; g++) {
                const u64 cnt = (g + 1 < ngroups ? h_start[g + 1] : (u32)n_hits) - h_start[g], fst = hit_base + h_first[g];
                TagAgg *a;
                if (mode == FASTF_TAG_MODE_INT) a = &imap.emplace((int32_t)(u32)h_key[g], TagAgg{0, ~0ull}).first->second;
                else {
                    const u32 la = (u32)(h_rep_a[g] & 0xffffu), lb = (u32)(h_rep_b[g] & 0xffffu);
                    k.assign(h_blob.data() + h_blob_off[g], la);
                    k.push_back('\0');
                    k.append(h_blob.data() + h_blob_off[g] + la, lb);
                    a = &smap.emplace(k, TagAgg{0, ~0ull}).first->second;
                }
                a->count += cnt;
                if (fst < a->first) a->first = fst;
            }
        }
        hit_base += n_hits;
        first_chunk = false;
        if (all.empty()) break;
    }
    // ---- merged groups -> result arrays ----
    const u64 ngroups = single ? single_groups : (mode == FASTF_TAG_MODE_INT ? imap.size() : smap.size());
    res->n_groups = ngroups;
    const u64 ng1 = std::max<u64>(ngroups, 1);
    u64 sbytes = 0;
    for (auto &kv : smap) sbytes += kv.first.size() - 1;
    if (single && mode == FASTF_TAG_MODE_STRING) for (u64 g = 0; g < ngroups; g++) sbytes += (h_rep_a[g] & 0xffffu) + (h_rep_b[g] & 0xffffu);
    res->first = (u32 *)malloc(ng1 * sizeof(u32));
    res->count = (u32 *)malloc(ng1 * sizeof(u32));
    res->ivalue = (int32_t *)malloc(ng1 * sizeof(int32_t));
    res->a_off = (u64 *)malloc(ng1 * sizeof(u64));
    res->a_len = (u32 *)malloc(ng1 * sizeof(u32));
    res->b_len = (u32 *)malloc(ng1 * sizeof(u32));
    res->strings = (char *)malloc(std::max<u64>(sbytes, 1));
    res->strings_bytes = sbytes;
    if (!res->first || !res->count || !res->ivalue || !res->a_off || !res->a_len || !res->b_len || !res->strings) return ctx_fail(ctx, "taghist: out of host memory");
    u64 g = 0, at = 0;
    if (single) {
        for (; g < ngroups; g++) {
            res->count[g] = (u32)((g + 1 < ngroups ? h_start[g + 1] : (u32)single_hits) - h_start[g]);
            res->first[g] = h_first[g];
            res->ivalue[g] = (int32_t)(u32)h_key[g];
            res->a_off[g] = mode == FASTF_TAG_MODE_STRING ? h_blob_off[g] : 0;
            res->a_len[g] = mode == FASTF_TAG_MODE_STRING ? (u32)(h_rep_a[g] & 0xffffu) : 0;
            res->b_len[g] = mode == FASTF_TAG_MODE_STRING ? (u32)(h_rep_b[g] & 0xffffu) : 0;
        }
        if (mode == FASTF_TAG_MODE_STRING && sbytes) memcpy(res->strings, h_blob.data(), sbytes);
    }
    for (auto &kv : imap) { res->ivalue[g] = kv.first; res->first[g] = (u32)kv.second.first; res->count[g] = (u32)kv.second.count; res->a_off[g] = 0; res->a_len[g] = 0; res->b_len[g] = 0; g++; }
    for (auto &kv : smap) {
        const std::string &k = kv.first;
        const size_t la = k.find('\0'), lb = k.size() - la - 1;
        res->ivalue[g] = 0; res->first[g] = (u32)kv.second.first; res->count[g] = (u32)kv.second.count;
        res->a_off[g] = at; res->a_len[g] = (u32)la; res->b_len[g] = (u32)lb;
        memcpy(res->strings + at, k.data(), la);
        memcpy(res->strings + at + la, k.data() + la + 1, lb);
        at += la + lb;
        g++;
    }
    CK(cudaEventRecord(e1, s));
    CK(cudaEventSynchronize(e1));
    t_tags.collect(&res->ms_tags); t_sort.collect(&res->ms_sort); t_rle.collect(&res->ms_rle);
    cudaEventElapsedTime(&res->ms_device_total, e0, e1);
    return 0;
}

extern "C" int fastf_taghist_gpu(fastf_ctx *ctx, const void *host_bytes, size_t n, const char *tag_a, uint32_t mode, const char *tag_b, uint32_t inflate_lanes, fastf_taghist_result *res)
{
    CK(cudaSetDevice(ctx->device));
    memset(res, 0, sizeof *res);
    if (!tag_a || !tag_a[0] || !tag_a[1]) return ctx_fail(ctx, "taghist: a tag is two characters");
    if (tag_b && (!tag_b[0] || !tag_b[1])) return ctx_fail(ctx, "taghist: a tag is two characters");
    if (mode > FASTF_TAG_MODE_INT || (mode == FASTF_TAG_MODE_INT && tag_b)) return ctx_fail(ctx, "taghist: mode 0 = string (optionally a pair), 1 = integer");
    if (!looks_like_gzip((const u8 *)host_bytes, n)) return ctx_fail(ctx, "taghist: not a BGZF stream");
    res->mode = mode;
    const u32 l0 = ctx->launches;
    const int rc = taghist_run(ctx, host_bytes, n, tag_a, mode, tag_b, inflate_lanes, res);
    res->n_launches = ctx->launches - l0;
    if (rc) fastf_taghist_result_free(res);   // a failed call leaves no result arrays behind
    return rc;
}

/* test hooks: a smaller streaming chunk (so that tiny fixtures exercise the cross-chunk merge), and a mask ANDed onto the hash keys of
 * the FIRST round only, which forces collisions there: the byte-for-byte verification must catch them and the second round must win */
extern "C" void fastf_taghist_test_hooks(fastf_ctx *ctx, uint64_t chunk_blocks, uint64_t round0_key_mask)
{
    ctx->taghist_chunk_blocks = chunk_blocks;
    ctx->taghist_round0_mask = round0_key_mask;
}

extern "C" void fastf_freq_result_free(fastf_freq_result *res)
{
    if (!res) return;
    free(res->key); free(res->count); free(res->first); free(res->exc_ordinal); free(res->exc_bytes);
    res->key = nullptr; res->count = nullptr; res->first = nullptr; res->exc_ordinal = nullptr; res->exc_bytes = nullptr;
}
