// TEST INFRASTRUCTURE ONLY: the warp-parallel Huffman table build of the thread-per-stream inflate kernel (fastf_tps_build), run
// under the SIMT emulator, against a straightforward serial build on seeded random code-length sets: complete, over-subscribed,
// incomplete, single-code, all-zero and 15-bit codes, for the code-length, literal/length and distance tables.  The verdict must be
// the same; for a valid code the primary table, the sorted symbol list, the walk limits / offsets and the sub-tables must be too.
// Usage: emu_build [cases]
#include "../../fastf_b200/csrc/bgzf_inflate.cuh"
#include "../../fastf_b200/csrc/bgzf_inflate_tps.cuh"
#include <random>

struct Tables {
    u16 lut[1 << FASTF_TPS_LBITS];
    u16 sorted[320];
    u16 lb[32];
    u16 sub[1024];
    u32 bad;
};

// the serial build: count, Kraft check, canonical codes in symbol order, table slots, then the sub-table layout per prefix
static void ref_build(u32 alpha, const u8 *lens, u32 n, u32 tbits, bool walk, u32 sub_cap, Tables &T)
{
    for (u32 i = 0; i < (1u << tbits); i++) T.lut[i] = FASTF_T16_LONG;
    u32 cnt[16] = {0};
    for (u32 s = 0; s < n; s++) cnt[lens[s]]++;
    cnt[0] = 0;
    int left = 1;
    u32 used = 0;
    for (u32 l = 1; l < 16; l++) {
        left = (left << 1) - (int)cnt[l];
        if (left < 0) { T.bad = 1; return; }
        used += cnt[l];
    }
    T.bad = left > 0 && used > 1;
    if (T.bad) return;
    u32 first[17], start[17], code = 0, idx = 0;
    for (u32 l = 1; l < 16; l++) { first[l] = code; start[l] = idx; code = (code + cnt[l]) << 1; idx += cnt[l]; }
    start[16] = idx;
    if (walk) {
        const u32 offs = FASTF_TPS_WALK_OFFS(tbits);
        for (u32 k = 0; k < offs; k++) {
            const u32 l = tbits + 1 + k;
            T.lb[k] = l <= 15 ? (u16)((first[l] + cnt[l]) << (15 - l)) : (u16)0xffff;
            T.lb[offs + k] = l <= 15 ? (u16)(start[l] - first[l]) : (u16)0;
        }
    }
    u32 next[16], sym_code[320];
    for (u32 l = 1; l < 16; l++) next[l] = first[l];
    u32 at[16];
    for (u32 l = 1; l < 16; l++) at[l] = start[l];
    for (u32 s = 0; s < n; s++) {
        const u32 l = lens[s];
        if (!l) continue;
        sym_code[s] = next[l]++;
        T.sorted[at[l]++] = (u16)s;
    }
    auto rev_of = [](u32 c, u32 l) { u32 r = 0; for (u32 i = 0; i < l; i++) r |= ((c >> i) & 1u) << (l - 1 - i); return r; };
    for (u32 s = 0; s < n; s++) {
        const u32 l = lens[s];
        if (!l || l > tbits) continue;
        const u16 e = (u16)(fastf_make16(alpha, s) | l);
        for (u32 j = rev_of(sym_code[s], l); j < (1u << tbits); j += 1u << l) T.lut[j] = e;
    }
    if (!sub_cap || start[tbits + 1] >= used) return;
    // per prefix (table index, stream bit order) the longest code that starts with it; sub-tables in index order, padded to 8
    const u32 nidx = 1u << tbits;
    u32 bits[256] = {0};
    for (u32 s = 0; s < n; s++) {
        const u32 l = lens[s];
        if (l <= tbits) continue;
        const u32 j = rev_of(sym_code[s] >> (l - tbits), tbits);
        if (l - tbits > bits[j]) bits[j] = l - tbits;
    }
    for (u32 j = 0; j < nidx; j++) if (bits[j] > 7) bits[j] = 0;   // 3 bits in the primary entry: longer codes of the prefix take the walk
    u32 total = 0, off[256];
    for (u32 j = 0; j < nidx; j++) { off[j] = total; total += bits[j] ? (bits[j] < 3 ? 8u : 1u << bits[j]) : 0u; }
    if (total > sub_cap) return;
    for (u32 j = 0; j < nidx; j++) if (bits[j]) T.lut[j] = (u16)(FASTF_T16_LONG | (bits[j] << 6) | ((off[j] >> 3) << 9));
    for (u32 s = 0; s < n; s++) {
        const u32 l = lens[s];
        if (l <= tbits) continue;
        const u32 rev = rev_of(sym_code[s], l), j = rev & (nidx - 1u);
        if (!bits[j]) continue;
        const u16 e = (u16)(fastf_make16(alpha, s) | l);
        for (u32 k = rev >> tbits; k < (1u << bits[j]); k += 1u << (l - tbits)) T.sub[off[j] + k] = e;
    }
}

static u8 g_lens[320];
static u16 g_first_start[32];
static u8 g_submax[256];

static void run_build(u32 alpha, u32 n, u32 tbits, bool walk, u32 sub_cap, Tables &T)
{
    FASTF_LAUNCH(([&] {
        const u32 bad = fastf_tps_build(alpha, g_lens, n, walk ? T.lb : nullptr, T.sorted, T.lut, tbits, g_first_start, g_first_start + 16, threadIdx.x,
                                        sub_cap ? T.sub : nullptr, sub_cap, g_submax);
        if (threadIdx.x == 0) T.bad = bad;
    }), 1, 32, 0, 0);
}

// a complete prefix code over k symbols no longer than maxlen: split random leaves of the code tree (deepest first with probability
// `deep`, which makes long chains and 15-bit codes)
static std::vector<u32> complete_lengths(std::mt19937 &rng, u32 k, u32 maxlen, double deep)
{
    std::vector<u32> leaves = {0};
    while (leaves.size() < k) {
        std::vector<u32> can;
        for (u32 i = 0; i < leaves.size(); i++) if (leaves[i] < maxlen) can.push_back(i);
        if (can.empty()) break;
        u32 pick = can[rng() % can.size()];
        if (std::uniform_real_distribution<double>(0, 1)(rng) < deep)
            for (u32 i : can) if (leaves[i] > leaves[pick]) pick = i;
        const u32 d = leaves[pick] + 1;
        leaves[pick] = d;
        leaves.push_back(d);
    }
    return leaves;
}

int main(int argc, char **argv)
{
    const int cases = argc > 1 ? atoi(argv[1]) : 3000;
    std::mt19937 rng(20261022);
    struct Kind { u32 alpha, nmin, nmax, tbits, maxlen; bool walk; u32 sub_cap; const char *name; };
    const Kind kinds[3] = {{FASTF_ALPHA_PLAIN, 19, 19, 7, 7, false, 0, "code-length"},
                           {FASTF_ALPHA_LITLEN, 257, 286, FASTF_TPS_LBITS, 15, true, FASTF_TPS_LITSUB_U16, "lit/len"},
                           {FASTF_ALPHA_DIST, 1, 30, FASTF_TPS_DBITS, 15, true, FASTF_TPS_DISTSUB_U16, "dist"}};
    int bad = 0, seen_bad = 0, seen_15 = 0;
    for (int t = 0; t < cases && bad < 10; t++) {
        const Kind &K = kinds[t % 3];
        const u32 n = K.nmin + rng() % (K.nmax - K.nmin + 1);
        memset(g_lens, 0, sizeof g_lens);
        const u32 shape = (t / 3) % 8;
        if (shape == 7) {
            // arbitrary lengths: mostly over-subscribed
            for (u32 s = 0; s < n; s++) g_lens[s] = (u8)(rng() % 3 ? rng() % (K.maxlen + 1) : 0);
        } else if (shape == 6) {
            // nothing, or a single code of any length
            if (rng() % 2) g_lens[rng() % n] = (u8)(1 + rng() % K.maxlen);
        } else {
            const u32 k = 2 + rng() % (n - 1 > 1 ? n - 1 : 1);
            std::vector<u32> lv = complete_lengths(rng, k < 2 ? 2 : k, K.maxlen, shape == 5 ? 0.9 : 0.2);
            if (shape == 3 && lv.size() > 1) lv.pop_back();                              // incomplete
            if (shape == 4) lv.push_back(1 + rng() % K.maxlen);                            // over-subscribed
            std::vector<u32> syms(n);
            for (u32 s = 0; s < n; s++) syms[s] = s;
            std::shuffle(syms.begin(), syms.end(), rng);
            for (u32 i = 0; i < lv.size() && i < n; i++) g_lens[syms[i]] = (u8)lv[i];
        }
        if (K.alpha == FASTF_ALPHA_LITLEN && shape != 6 && shape != 7 && rng() % 2) { u32 s = rng() % 256; std::swap(g_lens[256], g_lens[s]); }
        Tables want, got;
        memset(&want, 0x5a, sizeof want); memset(&got, 0x5a, sizeof got);
        ref_build(K.alpha, g_lens, n, K.tbits, K.walk, K.sub_cap, want);
        run_build(K.alpha, n, K.tbits, K.walk, K.sub_cap, got);
        u32 used = 0, mx = 0;
        for (u32 s = 0; s < n; s++) { used += g_lens[s] != 0; if (g_lens[s] > mx) mx = g_lens[s]; }
        seen_bad += want.bad != 0;
        seen_15 += !want.bad && mx == 15;
        bool ok = want.bad == got.bad;
        if (ok && !want.bad) {
            ok = !memcmp(want.lut, got.lut, sizeof(u16) << K.tbits) && !memcmp(want.sorted, got.sorted, sizeof(u16) * used);
            if (K.walk) ok = ok && !memcmp(want.lb, got.lb, sizeof(u16) * FASTF_TPS_WALK_U16(K.tbits));
            if (K.sub_cap) ok = ok && !memcmp(want.sub, got.sub, sizeof want.sub);
        }
        if (!ok) { printf("FAIL case %d (%s, n=%u, shape %u): verdict %u / %u\n", t, K.name, n, shape, want.bad, got.bad); bad++; }
    }
    printf("%s cases=%d invalid=%d with-15-bit=%d\n", bad ? "FAIL" : "PASS", cases, seen_bad, seen_15);
    return bad ? 1 : 0;
}
