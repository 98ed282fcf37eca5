// TEST INFRASTRUCTURE ONLY: runs the thread-per-stream inflate kernel, built with its role counters (-DFASTF_TPS_PROF=1), under
// the SIMT emulator on one BGZF file, checks every block byte for byte against zlib and prints how many codes longer than the
// primary table were resolved by the canonical walk.  Usage: emu_walk file.bgzf
static inline long long clock64() { return 0; }   // the role counters time the service steps; the emulator has no clock
#include "../../fastf_b200/csrc/bgzf_inflate.cuh"
#include "../../fastf_b200/csrc/bgzf_inflate_tps.cuh"
#include "../../fastf_b200/csrc/bgzf_index.h"
#include <zlib.h>

#if !FASTF_TPS_PROF
#error "build with -DFASTF_TPS_PROF=1"
#endif

int main(int argc, char **argv)
{
    if (argc < 2) { fprintf(stderr, "usage: emu_walk file.bgzf\n"); return 2; }
    FILE *f = fopen(argv[1], "rb");
    if (!f) { perror(argv[1]); return 2; }
    std::vector<uint8_t> file;
    uint8_t buf[65536];
    size_t got;
    while ((got = fread(buf, 1, sizeof buf, f)) > 0) file.insert(file.end(), buf, buf + got);
    fclose(f);
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
    for (size_t i = 0; i < nb; i++) {
        std::vector<u8> ref(isize[i] + 1);
        z_stream zs;
        memset(&zs, 0, sizeof zs);
        inflateInit2(&zs, -15);
        zs.next_in = (Bytef *)file.data() + in_off[i]; zs.avail_in = in_len[i];
        zs.next_out = ref.data(); zs.avail_out = isize[i];
        const int zr = inflate(&zs, Z_FINISH);
        inflateEnd(&zs);
        if (zr != Z_STREAM_END) { printf("FAIL zlib itself failed on block %zu\n", i); bad++; continue; }
        if (status[i] != 0) { printf("FAIL block %zu status=0x%x\n", i, status[i]); bad++; continue; }
        if (memcmp(ref.data(), out.data() + out_off[i], isize[i]) != 0) { printf("FAIL block %zu differs\n", i); bad++; }
    }
    for (size_t k = total; k < total + 64; k++) if (out[k] != 0xAA) { printf("FAIL wrote past the end\n"); bad++; break; }
    printf("%s blocks=%zu bytes=%llu long=%llu walks=%llu\n", bad ? "FAIL" : "PASS", nb, (unsigned long long)total, g_fastf_tps_prof[11], g_fastf_tps_prof[12]);
    return bad ? 1 : 0;
}
