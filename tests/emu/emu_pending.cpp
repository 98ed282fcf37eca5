// TEST INFRASTRUCTURE ONLY: the thread-per-stream inflate kernel, built with its role counters (-DFASTF_TPS_PROF=1), under the SIMT
// emulator on BGZF blocks of dynamic -> stored -> fixed -> dynamic deflate blocks.  A stream is set up for its next deflate block
// while the previous block's tokens are still in the ring; a stored block met then must wait until the ring is empty.  Every block
// is checked byte for byte against zlib, and the counters must show set-ups with tokens pending and stored blocks left for later.
// Usage: emu_pending
static inline long long clock64() { return 0; }   // the role counters time the service steps; the emulator has no clock
#include "../../fastf_b200/csrc/bgzf_inflate.cuh"
#include "../../fastf_b200/csrc/bgzf_inflate_tps.cuh"
#include "../../fastf_b200/csrc/bgzf_index.h"
#include <random>
#include <zlib.h>

#if !FASTF_TPS_PROF
#error "build with -DFASTF_TPS_PROF=1"
#endif

// text-like bytes: words from a small vocabulary (many matches, a skewed literal alphabet)
static std::vector<uint8_t> text(std::mt19937 &rng, size_t n)
{
    static const char *words[] = {"ACGT", "TTAGGG", "CB:Z:", "UB:Z:", "GX:Z:ENSG000", "read", "\t", "\n", "AAACCCAAGT", "GGGTTT", "xf:i:25"};
    std::vector<uint8_t> v;
    while (v.size() < n) {
        const char *w = words[rng() % (sizeof words / sizeof *words)];
        v.insert(v.end(), w, w + strlen(w));
        if (rng() % 5 == 0) v.push_back((uint8_t)('a' + rng() % 26));
    }
    v.resize(n);
    return v;
}

// one BGZF block whose payload is deflated in four parts: dynamic, stored (level 0), fixed (Z_FIXED), dynamic
static std::vector<uint8_t> bgzf_mixed(std::mt19937 &rng, std::vector<uint8_t> &payload)
{
    const size_t parts[4] = {6000 + rng() % 8000, 200 + rng() % 3000, 1000 + rng() % 4000, 6000 + rng() % 8000};
    const int level[4] = {6, 0, 6, 6}, strategy[4] = {Z_DEFAULT_STRATEGY, Z_DEFAULT_STRATEGY, Z_FIXED, Z_DEFAULT_STRATEGY};
    std::vector<uint8_t> out(18 + 65536 + 1024);
    static const uint8_t hdr[16] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0};
    memcpy(out.data(), hdr, 16);
    z_stream zs;
    memset(&zs, 0, sizeof zs);
    deflateInit2(&zs, level[0], Z_DEFLATED, -15, 8, strategy[0]);
    zs.next_out = out.data() + 18; zs.avail_out = (uInt)(out.size() - 26);
    payload.clear();
    for (int p = 0; p < 4; p++) {
        std::vector<uint8_t> v = text(rng, parts[p]);
        if (p) deflateParams(&zs, level[p], strategy[p]);   // ends the current deflate block
        const size_t at = payload.size();
        payload.insert(payload.end(), v.begin(), v.end());
        zs.next_in = payload.data() + at; zs.avail_in = (uInt)v.size();
        deflate(&zs, p == 3 ? Z_FINISH : Z_BLOCK);
    }
    const size_t clen = zs.total_out;
    deflateEnd(&zs);
    const size_t bsize = 18 + clen + 8;
    if (bsize > 65536 || payload.size() > 65536) { fprintf(stderr, "synthetic block too large\n"); exit(2); }
    out[16] = (uint8_t)((bsize - 1) & 0xff); out[17] = (uint8_t)((bsize - 1) >> 8);
    const uint32_t crc = (uint32_t)crc32(crc32(0, 0, 0), payload.data(), (uInt)payload.size()), isz = (uint32_t)payload.size();
    for (int i = 0; i < 4; i++) { out[18 + clen + i] = (uint8_t)(crc >> (8 * i)); out[22 + clen + i] = (uint8_t)(isz >> (8 * i)); }
    out.resize(bsize);
    return out;
}

int main()
{
    std::mt19937 rng(7);
    std::vector<uint8_t> file, payload, want;
    for (int b = 0; b < 24; b++) {
        std::vector<uint8_t> blk = bgzf_mixed(rng, payload);
        file.insert(file.end(), blk.begin(), blk.end());
        want.insert(want.end(), payload.begin(), payload.end());
    }
    std::vector<FastfBgzfBlock> blocks;
    size_t consumed = 0;
    if (fastf_bgzf_index(file.data(), file.size(), 0, blocks, &consumed) != FASTF_BGZF_OK) { printf("FAIL index\n"); return 1; }
    const size_t nb = blocks.size();
    std::vector<u64> in_off(nb), out_off(nb);
    std::vector<u32> in_len(nb), isize(nb), status(nb, 0xdeadbeef);
    u64 total = 0;
    for (size_t i = 0; i < nb; i++) { in_off[i] = blocks[i].in_off; in_len[i] = blocks[i].in_len; isize[i] = blocks[i].isize; out_off[i] = total; total += blocks[i].isize; }
    const size_t padded = (file.size() + 3) / 4 * 4 + 16;   // device-like padded copy, 4-byte aligned
    std::vector<u32> comp_words(padded / 4 + 1, 0);
    memcpy(comp_words.data(), file.data(), file.size());
    std::vector<u8> out(total + 64, 0xAA);
    u32 counter = 0;
    std::vector<u16> sorted((size_t)FASTF_TPS_STREAMS * FASTF_TPS_SORTED_U16, 0);
    FastfTpsArgs A;
    A.comp = (const u8 *)comp_words.data(); A.comp_total = padded; A.in_off = in_off.data(); A.in_len = in_len.data(); A.out_off = out_off.data(); A.isize = isize.data();
    A.nblocks = (u32)nb; A.out = out.data(); A.status = status.data(); A.next_block = &counter; A.sorted = sorted.data();
    FASTF_LAUNCH((fastf_bgzf_inflate_tps_kernel<FASTF_TPS_LANES, FASTF_TPS_SVC_WARPS>), 1, FASTF_TPS_THREADS, FASTF_TPS_SMEM_BYTES, 0, A);
    int bad = 0;
    for (size_t i = 0; i < nb; i++) if (status[i] != 0) { printf("FAIL block %zu status=0x%x\n", i, status[i]); bad++; }
    if (total != want.size() || memcmp(out.data(), want.data(), want.size()) != 0) { printf("FAIL output differs from zlib's input\n"); bad++; }
    for (size_t k = total; k < total + 64; k++) if (out[k] != 0xAA) { printf("FAIL wrote past the end\n"); bad++; break; }
    printf("%s blocks=%zu bytes=%llu headers=%llu pending=%llu later=%llu\n", bad ? "FAIL" : "PASS", nb, (unsigned long long)total, g_fastf_tps_prof[18], g_fastf_tps_prof[24], g_fastf_tps_prof[25]);
    return bad ? 1 : 0;
}
