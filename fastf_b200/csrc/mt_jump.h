// MT19937 jump-ahead: start the reference's single draw sequence (src/mt19937ar.c, one global state) at an arbitrary
// stream index without generating everything in front of it.  Needed by the later ranks of a multi-GPU job: rank g's first
// draw has stream index D0 + (CB-valid reads of ranks < g), which is only known after all ranks have parsed their shard.
//
// The MT19937 recurrence is linear over GF(2): the 624-word window W_t = (x_t .. x_{t+623}) satisfies W_{t+1} = F W_t, and with
// phi the characteristic polynomial of F (degree 19937, minimal polynomial of every output bit sequence),
//      W_{t+J} = g(F) W_t   with   g(x) = x^J mod phi(x)  =  sum_i g_i x^i,        i.e.   W_{t+J}[j] = XOR_{i : g_i = 1} x_{t+i+j}.
// Host side (this header): phi by Berlekamp-Massey over one output bit of the generator, and the table g_k = x^(2^k) mod phi.
// Device side (scan_mt_sample.cuh, fastf_mt_jump_batch_kernel): generate x_t .. x_{t+19936+623} with the normal twist and take the
// XOR.  A jump by J applies g_k for every set bit k of J; each CTA of the kernel makes its own jump.  Published method: Haramoto, Matsumoto,
// Nishimura, Panneton, L'Ecuyer, "Efficient jump ahead for F2-linear random number generators" (2008).
#pragma once
#include <stdint.h>
#include <string.h>
#include <mutex>
#include <vector>

#define FASTF_MT_DEG 19937
#define FASTF_MT_POLY_WORDS 312   // 19968 bits

namespace fastf_mtj {
typedef std::vector<uint64_t> Poly;   // bit i = coefficient of x^i

static inline bool getb(const Poly &p, size_t i) { return (p[i >> 6] >> (i & 63)) & 1u; }
static inline void flipb(Poly &p, size_t i) { p[i >> 6] ^= 1ull << (i & 63); }

// raw MT19937 state words x_0, x_1, ... from init_genrand(seed) (reference src/mt19937ar.c:60-73 and the twist :111-129)
static inline void raw_words(uint32_t seed, size_t n, std::vector<uint32_t> &x)
{
    x.resize(n < 624 ? 624 : n);
    x[0] = seed;
    for (size_t i = 1; i < 624; i++) x[i] = 1812433253u * (x[i - 1] ^ (x[i - 1] >> 30)) + (uint32_t)i;
    for (size_t k = 624; k < n; k++) {
        uint32_t y = (x[k - 624] & 0x80000000u) | (x[k - 623] & 0x7fffffffu);
        x[k] = x[k - 227] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
    }
}

// Berlekamp-Massey over GF(2): connection polynomial C (C_0 = 1) of the shortest LFSR with s_n = XOR_{i=1..L} C_i s_{n-i}
static inline size_t berlekamp_massey(const std::vector<uint8_t> &s, Poly &C)
{
    const size_t N = s.size(), W = (N + 64) / 64 + 1;
    Poly B(W, 0), T;
    C.assign(W, 0);
    C[0] = 1;
    B[0] = 1;
    size_t L = 0, m = 1;
    // the sequence as a reversed bit vector so that the discrepancy is a word-wise AND + parity
    std::vector<uint64_t> rev(W + 1, 0);   // rev bit (N-1-n) = s_n
    for (size_t n = 0; n < N; n++)
        if (s[n]) rev[(N - 1 - n) >> 6] |= 1ull << ((N - 1 - n) & 63);
    for (size_t n = 0; n < N; n++) {
        // d = s_n + sum_{i=1..L} C_i s_{n-i}  = parity over i=0..L of C_i * s_{n-i};  s_{n-i} = rev bit (N-1-n+i)
        const size_t off = N - 1 - n;
        uint64_t acc = 0;
        const size_t words = (L >> 6) + 1;
        const size_t ws = off >> 6, bs = off & 63;
        for (size_t w = 0; w < words; w++) {
            uint64_t r = rev[ws + w] >> bs;
            if (bs) r |= (ws + w + 1 < rev.size() ? rev[ws + w + 1] : 0) << (64 - bs);
            acc ^= C[w] & r;
        }
        // bits of C above L are zero, bits of rev above N-1 are zero: no masking needed
        if (__builtin_parityll(acc)) {
            T = C;
            // C ^= B << m
            const size_t sw = m >> 6, sb = m & 63;
            for (size_t w = 0; w + sw < W; w++) {
                C[w + sw] ^= B[w] << sb;
                if (sb && w + sw + 1 < W) C[w + sw + 1] ^= B[w] >> (64 - sb);
            }
            if (2 * L <= n) { L = n + 1 - L; B = T; m = 1; } else m++;
        } else m++;
    }
    return L;
}

struct Tables {
    bool ok = false;
    Poly phi;                 // characteristic polynomial, degree 19937, bit i = coefficient of x^i
    std::vector<Poly> pow2;   // pow2[k] = x^(2^k) mod phi, FASTF_MT_POLY_WORDS words each
};

// r = a mod phi for deg(a) < 2*19937 (in place, a has >= 2*FASTF_MT_POLY_WORDS words)
static inline void reduce(Poly &a, const Poly &phi)
{
    for (size_t i = 2 * FASTF_MT_DEG; i-- > FASTF_MT_DEG;) {
        if (!getb(a, i)) continue;
        // a ^= phi << (i - DEG)
        const size_t sh = i - FASTF_MT_DEG, sw = sh >> 6, sb = sh & 63;
        for (size_t w = 0; w < FASTF_MT_POLY_WORDS; w++) {
            a[w + sw] ^= phi[w] << sb;
            if (sb) a[w + sw + 1] ^= phi[w] >> (64 - sb);
        }
    }
}

static inline uint64_t spread32(uint32_t v)   // bit i -> bit 2i
{
    uint64_t x = v;
    x = (x | (x << 16)) & 0x0000ffff0000ffffull;
    x = (x | (x << 8)) & 0x00ff00ff00ff00ffull;
    x = (x | (x << 4)) & 0x0f0f0f0f0f0f0f0full;
    x = (x | (x << 2)) & 0x3333333333333333ull;
    x = (x | (x << 1)) & 0x5555555555555555ull;
    return x;
}

static inline const Tables &tables()
{
    // heap objects that are never destroyed: a detached warm-up thread may still be in here when the process exits
    static Tables &T = *new Tables();
    static std::mutex &mu = *new std::mutex();
    std::lock_guard<std::mutex> lock(mu);
    if (T.ok) return T;
    // 1. characteristic polynomial from 2*19937 (+ slack) bits of the most significant bit of x_t
    const size_t N = 2 * FASTF_MT_DEG + 64;
    std::vector<uint32_t> x;
    raw_words(5489u, N + 624, x);
    std::vector<uint8_t> s(N);
    for (size_t n = 0; n < N; n++) s[n] = (uint8_t)(x[n + 624] >> 31);
    Poly C;
    const size_t L = berlekamp_massey(s, C);
    if (L != FASTF_MT_DEG) return T;   // not ok (a bug: the input is a constant); callers report the error
    // C(x) = 1 + C_1 x + .. + C_L x^L is the connection polynomial; the characteristic polynomial is its reciprocal x^L C(1/x)
    T.phi.assign(FASTF_MT_POLY_WORDS + 1, 0);
    for (size_t i = 0; i <= L; i++)
        if (getb(C, i)) flipb(T.phi, L - i);
    // 2. x^(2^k) mod phi by repeated squaring
    Poly g(2 * FASTF_MT_POLY_WORDS + 2, 0);
    flipb(g, 1);   // x
    T.pow2.clear();
    for (int k = 0; k <= 44; k++) {
        T.pow2.push_back(Poly(g.begin(), g.begin() + FASTF_MT_POLY_WORDS));
        Poly sq(2 * FASTF_MT_POLY_WORDS + 2, 0);
        for (size_t w = 0; w < FASTF_MT_POLY_WORDS; w++) {
            sq[2 * w] = spread32((uint32_t)g[w]);
            sq[2 * w + 1] = spread32((uint32_t)(g[w] >> 32));
        }
        reduce(sq, T.phi);
        g = sq;
    }
    T.ok = true;
    return T;
}
}   // namespace fastf_mtj
