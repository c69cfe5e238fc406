// tg_gf2.cuh -- the bit-slab geometry, the record parities and the term of a record, shared by the mod-2 kernels:
// tg_gf2.cu (the game), tg_gf2_basis.cu (the change of basis), tg_gf2_samples.cu (training samples) and tg_gf2_demo.cu
// (synthetic demonstrations).  Format and formulation: the head of tg_gf2.cu.
#pragma once
#include "tg_common.cuh"

namespace tg {
namespace {

template <int S>
struct GeoB {
    static constexpr int S2 = S * S;
    static constexpr int RW = (S2 + 31) / 32;             // words per row
    static constexpr int GB = (4 * S * RW + 15) & ~15;    // game pitch (bytes)
    static constexpr int NQ = GB / 16;                    // 16-byte chunks per game
    static constexpr int TP = Geo<S>::TP;                 // token pitch (bytes)
    static constexpr int G = S == 16 ? 16 : S == 25 ? 32 : 1; // lanes per game
    static constexpr int NC = (NQ + G - 1) / G;           // chunks per lane
    static constexpr int GPC = 256 / G;                   // games per 256-thread CTA
    static constexpr bool STAGED = G == 1 && NQ > 1;      // 9x9x9: warp-staged global accesses
    static_assert(G == 1 || RW % 4 == 0, "a chunk lies in one row");
    static_assert(G == 1 || GB == 4 * S * RW, "no padding words at 16 and 25");
};

// parity bits of a record's u, v and w (bit m of .u = u_m odd)
struct Par {
    uint32_t u, v, w;
};

template <int S>
__device__ __forceinline__ uint32_t bit_field(const uint32_t (&P)[3], int o) {
    const int w = o / 32, s = o % 32;
    uint32_t r = P[w] >> s;
    if (s + S > 32) r |= P[w + 1] << (32 - s);
    return r & ((1u << S) - 1u);
}

// parities of the 3S tokens in token words rw (word q = tokens 4q .. 4q+3)
template <int S>
__device__ __forceinline__ Par parities_of(const uint32_t *rw, int shift) {
    constexpr int NT = (3 * S + 3) / 4; // token words that hold the 3S tokens
    const uint32_t sh = (uint32_t)shift * ONES4;
    uint32_t P[3] = {0u, 0u, 0u};
#pragma unroll
    for (int q = 0; q < NT; q++) // low bit of each byte of t ^ shift, gathered into bits 28-31 by one multiply
        P[q / 8] |= ((((rw[q] ^ sh) & ONES4) * 0x10204080u) >> 28) << (4 * (q % 8));
    return Par{bit_field<S>(P, 0), bit_field<S>(P, S), bit_field<S>(P, 2 * S)};
}

// parities of the record at rec (global memory)
template <int S>
__device__ __forceinline__ Par parities(const uint8_t *rec, int shift) {
    constexpr int NT = (3 * S + 3) / 4;
    uint32_t rw[4 * ((NT + 3) / 4)];
#pragma unroll
    for (int q = 0; q < (NT + 3) / 4; q++) {
        const uint4 t = __ldg(reinterpret_cast<const uint4 *>(rec) + q);
        rw[4 * q] = t.x, rw[4 * q + 1] = t.y, rw[4 * q + 2] = t.z, rw[4 * q + 3] = t.w;
    }
    return parities_of<S>(rw, shift);
}

// xor the term of a record (parities p) into rows r0 .. r0 + RPT - 1
template <int S, int RPT>
__device__ __forceinline__ void xor_term(uint32_t (&row)[RPT][GeoB<S>::RW], const Par &p, int r0) {
    constexpr int RW = GeoB<S>::RW;
    uint32_t V[RW];
#pragma unroll
    for (int w = 0; w < RW; w++) V[w] = 0;
#pragma unroll
    for (int j = 0; j < S; j++) {
        const uint32_t x = p.w & (0u - ((p.v >> j) & 1u));
        const int o = j * S, q = o / 32, s = o % 32;
        V[q] |= x << s;
        if (s + S > 32) V[q + 1] |= x >> (32 - s);
    }
#pragma unroll
    for (int k = 0; k < RPT; k++) {
        const uint32_t on = 0u - ((p.u >> (r0 + k)) & 1u);
#pragma unroll
        for (int w = 0; w < RW; w++) row[k][w] ^= V[w] & on;
    }
}

// CTAs for n items of `per` per CTA, at most eight resident CTAs of 256 threads per SM (the kernels loop over the rest)
unsigned grid_for(long long n, int per) {
    const long long want = (n + per - 1) / per, cap = 8LL * sm_count();
    return (unsigned)(want < cap ? want : cap);
}

} // namespace
} // namespace tg
