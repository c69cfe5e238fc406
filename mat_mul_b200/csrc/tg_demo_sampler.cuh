// tg_demo_sampler.cuh -- the throughput-mode demo sampler (contracts v1 and v2, DESIGN.md; restated by oracle/tg_oracle.c
// orc_demo_philox and orc_demo_philox_v2), shared by tg_demo.cu (the integer generator, tg_demo_gen_philox) and
// tg_gf2_demo.cu (the mod-2 generator, tg_demo_gen_gf2).  Device side: the launch constants, Philox, the group-alias and
// the thresholded draws of one factor triple.  Host side: the alias tables and the per-device table cache.  The
// template flag GF2 turns a contract into its mod-2 reading, "zero" read as "zero mod 2": the "all zero so far" chain
// and the accept test look at the low bit of each entry, and the tilt weighs the all-even outcomes.
#pragma once
#include <cstring>

#include "tg_common.cuh"

namespace tg {

// Launch constants of the sampler (kernel parameter => constant bank operands).
struct Categorical {
    uint32_t cadd[7];   // (0x8000 - thr15[i]) in both 16-bit lanes; thr15[i] = floor(cdf_i * 2^15)
    uint32_t xlut[7];   // (token of bucket i+1) ^ (token of bucket i), in every byte
    uint32_t lut0;      // token (value + shift) of bucket 0, in every byte
    uint32_t zero_pat;  // token of the value 0 in every byte (0xFFFFFFFF if 0 is not in the alphabet)
    uint32_t top_tok;   // token of the last bucket (forced unit triple)
    uint32_t rk[10][2]; // Philox round keys: key + round * (0x9E3779B9, 0xBB67AE85)
    uint32_t sparse_terms; // phase B walks only the terms with v_j != 0 (set by the host when P(0) is large; see there)
};

// one Philox4x32-10 block; IMAD.WIDE gives hi and lo of each product in one instruction
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, const Categorical &cat,
                                              uint32_t out[4]) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        const unsigned long long p0 = (unsigned long long)0xD2511F53u * c0;
        const unsigned long long p1 = (unsigned long long)0xCD9E8D57u * c2;
        c0 = (uint32_t)(p1 >> 32) ^ c1 ^ cat.rk[r][0];
        c1 = (uint32_t)p1;
        c2 = (uint32_t)(p0 >> 32) ^ c3 ^ cat.rk[r][1];
        c3 = (uint32_t)p0;
    }
    out[0] = c0, out[1] = c1, out[2] = c2, out[3] = c3;
}

__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
}

// ---- contract v2: the "group alias" sampler (DESIGN.md; restated by oracle/tg_oracle.c orc_demo_philox_v2).
// An accepted triple of the reference's rejection loop (utils.py:222-232) is three independent factors, each an i.i.d.
// factor conditioned on being non-zero; that conditional distribution is sampled DIRECTLY, group of three entries by group
// of three entries, from alias tables of 128 buckets: one 16-bit draw per group (bucket = draw & 127, keep the bucket's own
// outcome iff draw >> 7 < its 9-bit threshold, else its alias), while all groups so far are zero from the table tilted by
// the probability that the rest of the factor is zero too.  No rejection loop, half the Philox blocks of the thresholded
// contract, and no comparisons per token.
constexpr int ALIAS_BUCKETS = 128;
// the tables in the contract's own terms (host side: built by build_alias, exported by tg_demo_alias_tables)
struct AliasParams {
    uint16_t tab[8][ALIAS_BUCKETS]; // [g] tilted table of group g (g < NG <= 6), [6] plain size 3, [7] plain size 1
    uint32_t lut3[ALIAS_BUCKETS];   // outcome of a size-3 group -> its three tokens (bytes 0..2)
    uint32_t lut1[8];               // outcome of a size-1 group -> its token
    uint32_t zo3, zo1;              // the all-zero outcomes (255 if 0 is not in the alphabet)
    uint32_t rk[10][2];             // Philox round keys
};
// The same tables in the form the kernel reads.  A bucket is ONE word that already holds both of its outcomes as PRMT
// selectors: bits 0..11 its own outcome, bits 12..23 its alias, each three nibbles = the value indices of the group's three
// entries (7 = "no entry": byte 7 of the token LUT is 0), bits 23..31 the 9-bit threshold (bit 23 is shared with the top bit
// of the last alias nibble, which a selector never uses: the kernel masks with 0x777).  The chosen selector turns
// the 8-byte token LUT (two registers) into the group's token bytes with one PRMT -- no outcome -> token table in shared
// memory, and since a factor's groups are drawn in order ("all zero so far" selects the tilted or the plain table by
// ADDRESS), one 4-byte load per group instead of two bucket loads and a LUT load.
// The tables live in a small per-device cache in global memory (alias_device_tables below) and every CTA copies them to
// shared memory with coalesced 16-byte loads; as kernel parameters each CTA paid one SERIALISED constant-bank read per
// word (lanes of a warp read different words): ~23 SM-cycles per 9x9x9 demo.
struct AliasTabs {
    uint32_t tab[8][ALIAS_BUCKETS]; // same table order as AliasParams::tab
};
struct AliasDev {
    const uint32_t *tab;            // device copy of an AliasTabs
    uint32_t lut_lo, lut_hi;        // token (value + shift) of value index 0..3 | 4..7 (unused indices: 0)
    uint32_t zsel3, zsel1;          // selector of the all-zero outcome (0xFFFFFFFF if 0 is not in the alphabet); mod 2: the
                                    // low bits of an all-even group's tokens, (shift & 1) * 0x010101 / shift & 1
    uint32_t rk[10][2];             // Philox round keys
};
template <int S>
struct AliasGeo {
    static constexpr int NG = (S + 2) / 3, LAST = S - 3 * (NG - 1); // groups per factor, size of the last one (1 or 3)
    static constexpr int ND = 3 * NG, NB = (ND + 7) / 8;             // 16-bit draws and Philox blocks per triple
    static constexpr int TAB_WORDS = (NG + 2) * ALIAS_BUCKETS;       // shared-memory copy: tables [0..NG), plain 3, plain 1
    static constexpr int SMEM_BYTES = TAB_WORDS * 4;
    static_assert(LAST == 1 || LAST == 3, "group sizes 3 and 1 only");
    static constexpr __host__ __device__ bool three(int g) { return g < NG - 1 || LAST == 3; }
    // Token word w of the action record (bytes 4w .. 4w+3 of cat(u, v, w)) is one PRMT of the token words of the (at most
    // two) groups it overlaps: group index of its first / last byte and the selector (nibble b: byte of the first group,
    // 4 + byte of the second, 3 = the always-zero top byte of a group's token word for the padding beyond 3S)
    static constexpr __host__ __device__ int group_of(int q) { return (q / S) * NG + ((q % S) / 3 < NG ? (q % S) / 3 : NG - 1); }
    static constexpr __host__ __device__ int group_byte0(int m) { return (m / NG) * S + 3 * (m % NG); }
    static constexpr __host__ __device__ int word_first(int w) { return group_of(4 * w); }
    static constexpr __host__ __device__ int word_last(int w) { return group_of(4 * w + 3 < 3 * S ? 4 * w + 3 : 3 * S - 1); }
    static constexpr __host__ __device__ uint32_t word_sel(int w) {
        uint32_t sel = 0;
        for (int b = 0; b < 4; b++) {
            const int q = 4 * w + b;
            uint32_t nib = 3;
            if (q < 3 * S) nib = group_of(q) == word_first(w) ? (uint32_t)(q - group_byte0(word_first(w))) : 4u + (uint32_t)(q - group_byte0(word_last(w)));
            sel |= nib << (4 * b);
        }
        return sel;
    }
    static constexpr __host__ __device__ bool words_ok() { // every byte of a word belongs to its first or its last group
        for (int q = 0; q < 3 * S; q++)
            if (group_of(q) != word_first(q / 4) && group_of(q) != word_last(q / 4)) return false;
        return true;
    }
};

// CTA-wide copy of the tables from global memory (L2-resident: every CTA reads the same 2-4 KB) to shared memory
template <int S, int NT>
__device__ __forceinline__ void alias_to_smem(const AliasDev &ap, uint32_t *s_alias) {
    using A = AliasGeo<S>;
    const uint4 *src = reinterpret_cast<const uint4 *>(ap.tab);
    uint4 *dst = reinterpret_cast<uint4 *>(s_alias);
    for (int w = threadIdx.x; w < A::NG * (ALIAS_BUCKETS / 4); w += NT) dst[w] = __ldg(src + w);
    for (int w = threadIdx.x; w < 2 * (ALIAS_BUCKETS / 4); w += NT) dst[A::NG * (ALIAS_BUCKETS / 4) + w] = __ldg(src + 6 * (ALIAS_BUCKETS / 4) + w); // plain 3, plain 1
}

// one factor triple (3S tokens) of demo (d_lo, d_hi), term r under contract v2.  GF2: the mod-2 contract, where "zero"
// reads "even" -- a group is "all even" iff the low bits of its token bytes equal ap.zsel3 / zsel1 (shift & 1 in each)
template <int S, bool GF2 = false>
__device__ __forceinline__ void draw_triple_alias(uint32_t words[(3 * S + 3) / 4], uint32_t d_lo, uint32_t d_hi, int r,
                                                  const AliasDev &ap, const uint32_t *s_alias) {
    using A = AliasGeo<S>;
    constexpr int NW = (3 * S + 3) / 4;
    static_assert(A::words_ok(), "a token word overlaps more than two groups");
    uint32_t blk[4 * A::NB];
#pragma unroll
    for (int b = 0; b < A::NB; b++) {
        uint32_t c0 = d_lo, c1 = d_hi, c2 = (uint32_t)r, c3 = (uint32_t)b;
#pragma unroll
        for (int q = 0; q < 10; q++) {
            const unsigned long long p0 = (unsigned long long)0xD2511F53u * c0, p1 = (unsigned long long)0xCD9E8D57u * c2;
            c0 = (uint32_t)(p1 >> 32) ^ c1 ^ ap.rk[q][0], c1 = (uint32_t)p1, c2 = (uint32_t)(p0 >> 32) ^ c3 ^ ap.rk[q][1], c3 = (uint32_t)p0;
        }
        blk[4 * b] = c0, blk[4 * b + 1] = c1, blk[4 * b + 2] = c2, blk[4 * b + 3] = c3;
    }
    // draw m = f * NG + g is half (m & 1) of Philox word m >> 1, moved to the top of a register: bucket = bits 16..22,
    // "draw >> 7 < threshold" is one unsigned compare with the bucket word's threshold bits (the bits below bit 23 of the
    // draw cannot change it).  The three factors are independent chains of NG loads.
    uint32_t tk[A::ND];
    const uint8_t *s_tab = reinterpret_cast<const uint8_t *>(s_alias);
    bool az[3] = {true, true, true}; // every group of the factor so far is all zero
#pragma unroll
    for (int g = 0; g < A::NG; g++) {
#pragma unroll
        for (int f = 0; f < 3; f++) {
            const int m = f * A::NG + g;
            const uint32_t x = (m & 1) ? blk[m >> 1] : (blk[m >> 1] << 16);
            const uint32_t idx4 = (x >> 14) & 0x1FCu;
            const int tilted = g * ALIAS_BUCKETS * 4;
            const int plain = (A::three(g) ? A::NG : A::NG + 1) * ALIAS_BUCKETS * 4;
            uint32_t e;
            if (g == 0 || az[f]) e = *reinterpret_cast<const uint32_t *>(s_tab + tilted + idx4);
            else e = *reinterpret_cast<const uint32_t *>(s_tab + plain + idx4);
            const uint32_t sel = ((x < (e & 0xFF800000u)) ? e : (e >> 12)) & 0x777u;
            tk[m] = prmt(ap.lut_lo, ap.lut_hi, sel); // bytes 0..2 (size 1: byte 0) are tokens, the rest is not used
            if constexpr (GF2) az[f] = az[f] && (tk[m] & (A::three(g) ? 0x010101u : 1u)) == (A::three(g) ? ap.zsel3 : ap.zsel1);
            else az[f] = az[f] && sel == (A::three(g) ? ap.zsel3 : ap.zsel1);
        }
    }
#pragma unroll
    for (int w = 0; w < NW; w++) words[w] = prmt(tk[A::word_first(w)], tk[A::word_last(w)], A::word_sel(w));
    if constexpr ((3 * S) % 4 != 0) words[NW - 1] &= 0xFFFFFFFFu >> (8 * (4 - (3 * S) % 4)); // tape padding stays zero
}

// "is this factor all zero" over packed token words: OR of (word ^ zero_pat) under the factor's byte mask.  GF2 (zero_pat =
// the shift in every byte): "has an odd entry", the same OR on the low bit of each byte only
template <int S, bool GF2 = false>
__device__ __forceinline__ bool factor_nonzero(const uint32_t words[(3 * S + 3) / 4], int f, uint32_t zero_pat) {
    uint32_t acc = 0;
#pragma unroll
    for (int w = 0; w < (3 * S + 3) / 4; w++) {
        uint32_t m = 0;
#pragma unroll
        for (int b = 0; b < 4; b++) {
            const int q = 4 * w + b;
            if (q >= f * S && q < (f + 1) * S) m |= 0xFFu << (8 * b);
        }
        if (m) acc |= (words[w] ^ zero_pat) & m & (GF2 ? ONES4 : 0xFFFFFFFFu);
    }
    return acc != 0;
}

// Draw one factor triple (3S tokens) for demo (d_lo, d_hi), term r, try t; true if accepted.
// Draw q is the 15-bit value in half (q & 1) of word (q >> 1) & 3 of Philox block q >> 3 with
// ctr = (d_lo, d_hi, r | t << 16, q >> 3); bucket = number of thresholds <= draw.  Four draws at a time:
// x + (0x8000 - thr) carries into bit 15 of its 16-bit lane iff x >= thr, PRMT (sign-replicating
// selector) turns the four carries into byte masks, and the token of bucket b is
// lut[0] ^ xlut[0] ^ ... ^ xlut[b-1].  GF2: accepted iff u, v and w each have an odd entry.
template <int S, int NTHR, bool GF2 = false>
__device__ __forceinline__ bool draw_triple(uint32_t words[(3 * S + 3) / 4], uint32_t d_lo, uint32_t d_hi, int r, int t,
                                            const Categorical &cat) {
    constexpr int NB = (3 * S + 7) / 8;
    constexpr int NW = (3 * S + 3) / 4;
#pragma unroll
    for (int bq = 0; bq < NB; bq++) {
        uint32_t blk[4];
        philox4x32_10(d_lo, d_hi, (uint32_t)r | ((uint32_t)t << 16), (uint32_t)bq, cat, blk);
#pragma unroll
        for (int half = 0; half < 2; half++) { // tokens 8bq + 4half .. +3  ->  token word 2bq + half
            if (2 * bq + half < NW) {
                const uint32_t xa = blk[2 * half] & 0x7FFF7FFFu, xb = blk[2 * half + 1] & 0x7FFF7FFFu;
                uint32_t tokw = cat.lut0;
#pragma unroll
                for (int i = 0; i < NTHR; i++)
                    tokw ^= prmt(xa + cat.cadd[i], xb + cat.cadd[i], 0xFDB9u) & cat.xlut[i];
                const int q0 = 8 * bq + 4 * half;
                if (q0 + 4 > 3 * S) tokw &= 0xFFFFFFFFu >> (8 * (q0 + 4 - 3 * S)); // tape padding stays zero
                words[2 * bq + half] = tokw;
            }
        }
    }
    return factor_nonzero<S, GF2>(words, 0, cat.zero_pat) && factor_nonzero<S, GF2>(words, 1, cat.zero_pat) &&
           factor_nonzero<S, GF2>(words, 2, cat.zero_pat);
}

// ---- host side
// the alphabet rules of both generators: every probability >= 0 (NaN refused), a positive sum, values in [-shift, shift]
inline bool alphabet_ok(const int8_t *values, const double *probs, int n, int shift) {
    double total = 0;
    for (int i = 0; i < n; i++) {
        if (!(probs[i] >= 0) || values[i] < -shift || values[i] > shift) return false;
        total += probs[i];
    }
    return total > 0;
}

// contract v1's launch constants: thresholds, token tables and Philox round keys; zero_pat = the token of 0 in every byte
// (0xFFFFFFFF if 0 is not in the alphabet), top_tok = the token of the last value
inline Categorical categorical(const int8_t *values, const double *probs, int n, int shift, uint64_t seed) {
    Categorical cat = {};
    double total = 0, run = 0;
    for (int i = 0; i < n; i++) total += probs[i];
    cat.zero_pat = 0xFFFFFFFFu;
    uint32_t prev = 0;
    for (int i = 0; i < n; i++) {
        const uint32_t tok = (uint32_t)(values[i] + shift) & 0xFFu;
        if (i == 0) cat.lut0 = tok * ONES4;
        if (i > 0) {
            // bucket >= i  <=>  draw >= thr15[i-1] = floor(cdf_{i-1} * 2^15); 32768 is never reached
            const double t = run * 32768.0;
            const uint32_t thr = t >= 32768.0 ? 32768u : (uint32_t)t;
            cat.cadd[i - 1] = (0x8000u - thr) * 0x00010001u;
            cat.xlut[i - 1] = (tok ^ prev) * ONES4;
        }
        run += probs[i] / total;
        prev = tok;
        if (values[i] == 0) cat.zero_pat = (uint32_t)shift * ONES4;
    }
    cat.top_tok = prev;
    for (int r = 0; r < 10; r++) {
        cat.rk[r][0] = (uint32_t)seed + (uint32_t)r * 0x9E3779B9u;
        cat.rk[r][1] = (uint32_t)(seed >> 32) + (uint32_t)r * 0xBB67AE85u;
    }
    return cat;
}

// ---- host side of contract v2: Vose's alias construction, in exactly the order the oracle restates
inline void vose128(const double *P, int count, uint16_t *out) {
    double sc[ALIAS_BUCKETS], prob[ALIAS_BUCKETS];
    int alias[ALIAS_BUCKETS], small[ALIAS_BUCKETS], large[ALIAS_BUCKETS], ns = 0, nl = 0;
    for (int o = 0; o < ALIAS_BUCKETS; o++) sc[o] = (o < count ? P[o] : 0.0) * (double)ALIAS_BUCKETS, alias[o] = o, prob[o] = 1.0;
    for (int o = 0; o < ALIAS_BUCKETS; o++) (sc[o] < 1.0 ? small[ns++] : large[nl++]) = o;
    while (ns > 0 && nl > 0) {
        const int sm = small[--ns], lg = large[--nl];
        prob[sm] = sc[sm], alias[sm] = lg;
        sc[lg] = (sc[lg] + sc[sm]) - 1.0;
        (sc[lg] < 1.0 ? small[ns++] : large[nl++]) = lg;
    }
    for (int o = 0; o < ALIAS_BUCKETS; o++) {
        const double q = prob[o] < 0.0 ? 0.0 : (prob[o] > 1.0 ? 1.0 : prob[o]);
        uint32_t thr = (uint32_t)(q * 512.0 + 0.5);
        int al = alias[o];
        if (thr >= 512u) thr = 511u, al = o; // probability one: either branch gives the bucket's own outcome
        out[o] = (uint16_t)(thr | ((uint32_t)al << 9));
    }
}

// P(value is zero), or modulo 2 P(value is even), of the normalised alphabet
template <bool GF2>
inline double p_null(const int8_t *values, const double *probs, int n) {
    double total = 0, p0 = 0;
    for (int i = 0; i < n; i++) total += probs[i];
    for (int i = 0; i < n; i++)
        if (GF2 ? (values[i] & 1) == 0 : values[i] == 0) p0 += probs[i] / total;
    return p0;
}

// contract v2 applies to alphabets of at most five values whose P(0) (mod 2: P(even)) leaves a non-zero (odd) factor reachable
template <bool GF2 = false>
inline bool alias_applies(const int8_t *values, const double *probs, int n, int S) {
    // AliasParams has room for the tilted tables of six groups (factors of up to 18 entries): 25x25x25 keeps contract v1
    if (n < 1 || n > 5 || !supported_S(S) || (S + 2) / 3 > 6) return false;
    return p_null<GF2>(values, probs, n) <= 0.999;
}

// GF2: the tilt weighs every outcome whose entries are all even by 1 - P(every later entry even) (P(even) = the sum over the
// even values, which is P(0) itself when 0 is the only even value: then the tables are the integer ones)
template <bool GF2 = false>
inline void build_alias(const int8_t *values, const double *probs, int n, int S, int shift, uint64_t seed, AliasParams &A) {
    double p[5], total = 0, p0 = 0;
    int z = -1;
    for (int i = 0; i < n; i++) total += probs[i];
    for (int i = 0; i < n; i++) {
        p[i] = probs[i] / total;
        if (values[i] == 0 && z < 0) z = i, p0 = p[i];
    }
    if constexpr (GF2) p0 = p_null<true>(values, probs, n);
    auto even = [&](int o, int size) { // outcome o of a group of `size` has only even entries
        for (int e = 0, x = o; e < size; e++, x /= n)
            if (values[x % n] & 1) return false;
        return true;
    };
    const int ng = (S + 2) / 3, last = S - 3 * (ng - 1);
    A = AliasParams{};
    A.zo3 = z >= 0 ? (uint32_t)(z + n * z + n * n * z) : 255u;
    A.zo1 = z >= 0 ? (uint32_t)z : 255u;
    double P3[ALIAS_BUCKETS], P1[ALIAS_BUCKETS];
    for (int o = 0; o < n * n * n; o++) {
        P3[o] = (p[o % n] * p[(o / n) % n]) * p[o / (n * n)];
        A.lut3[o] = ((uint32_t)(values[o % n] + shift) & 0xFFu) | (((uint32_t)(values[(o / n) % n] + shift) & 0xFFu) << 8) |
                    (((uint32_t)(values[o / (n * n)] + shift) & 0xFFu) << 16);
    }
    for (int o = 0; o < n; o++) P1[o] = p[o], A.lut1[o] = (uint32_t)(values[o] + shift) & 0xFFu;
    vose128(P3, n * n * n, A.tab[6]);
    vose128(P1, n, A.tab[7]);
    for (int g = 0; g < ng; g++) {
        const int size = (g < ng - 1) ? 3 : last;
        const int count = size == 3 ? n * n * n : n, zo = size == 3 ? (int)A.zo3 : (int)A.zo1;
        double qlater = 1.0; // P(every entry after this group is zero)
        for (int e = 3 * g + size; e < S; e++) qlater *= p0;
        double W[ALIAS_BUCKETS], sum = 0;
        for (int o = 0; o < count; o++) {
            W[o] = size == 3 ? P3[o] : P1[o];
            if (GF2 ? even(o, size) : o == zo) W[o] *= (1.0 - qlater);
            sum += W[o];
        }
        for (int o = 0; o < count; o++) W[o] /= sum;
        vose128(W, count, A.tab[g]);
    }
    for (int r = 0; r < 10; r++) {
        A.rk[r][0] = (uint32_t)seed + (uint32_t)r * 0x9E3779B9u;
        A.rk[r][1] = (uint32_t)(seed >> 32) + (uint32_t)r * 0xBB67AE85u;
    }
}

// the tables as the kernel reads them (AliasDev)
template <bool GF2 = false>
inline void alias_to_dev(const AliasParams &A, const int8_t *values, int n, int S, int shift, AliasTabs &T, AliasDev &D) {
    const int ng = (S + 2) / 3, last = S - 3 * (ng - 1);
    D = AliasDev{};
    T = AliasTabs{};
    auto sel = [&](int o, int size) -> uint32_t {
        if (size == 3) return o < n * n * n ? (uint32_t)(o % n) | ((uint32_t)((o / n) % n) << 4) | ((uint32_t)(o / (n * n)) << 8) : 0x777u;
        return o < n ? (uint32_t)o | 0x770u : 0x777u;
    };
    for (int t = 0; t < 8; t++) {
        const int size = t < 6 ? (t < ng ? (t < ng - 1 ? 3 : last) : 0) : (t == 6 ? 3 : 1);
        if (!size) continue;
        for (int b = 0; b < ALIAS_BUCKETS; b++) {
            const uint32_t thr = A.tab[t][b] & 511u, al = A.tab[t][b] >> 9;
            T.tab[t][b] = sel(b, size) | (sel((int)al, size) << 12) | (thr << 23);
        }
    }
    int z = -1;
    for (int i = 0; i < n; i++) {
        (i < 4 ? D.lut_lo : D.lut_hi) |= ((uint32_t)(values[i] + shift) & 0xFFu) << (8 * (i & 3));
        if (values[i] == 0 && z < 0) z = i;
    }
    D.zsel3 = z >= 0 ? (uint32_t)z * 0x111u : 0xFFFFFFFFu;
    D.zsel1 = z >= 0 ? (uint32_t)z | 0x770u : 0xFFFFFFFFu;
    if constexpr (GF2) D.zsel3 = (uint32_t)(shift & 1) * 0x010101u, D.zsel1 = (uint32_t)(shift & 1);
    memcpy(D.rk, A.rk, sizeof(D.rk));
}

// ---- per-device cache of device-format tables (tg_demo.cu).  A table set is uploaded by a one-CTA kernel on the caller's
// stream the first time it is asked for; a later launch -- on any stream -- waits for that upload's event.  Eight sets
// per device; a ninth distinct set evicts the least recently used one after a cudaDeviceSynchronize (kernels of other
// streams may still be reading it) -- a training run uses one or two.  Both generators use it, and a set is keyed by its
// bytes: the mod-2 tables of an alphabet whose only even value is 0 are the integer ones and share their slot.
int alias_device_tables(const AliasTabs &want, cudaStream_t st, const uint32_t **dptr);

} // namespace tg
