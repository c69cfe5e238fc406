// tg_gf2_basis.cu -- the change of basis over GF(2) on bit slabs: tg_change_of_basis_gf2 (the tensor),
// tg_change_of_basis_factors_gf2 (the factors of a tape) and tg_sample_invertible_gf2 (random bases).
#include "tg_gf2.cuh"

namespace tg {
namespace {

// ------------------------------------------------------------------ change of basis over GF(2)
// A triple (A, B, C) mod 2 is uint32 [3][S]: word r of matrix f is row r, bit c = M[r][c]; bits S..31 are ignored.
__host__ __device__ constexpr uint32_t low_bits(int S) { return (1u << S) - 1u; }

// S-bit chunk j of a row (bits [j S, j S + S) of its RW words) and its inverse (x has no bits above S)
template <int S>
__device__ __forceinline__ uint32_t get_chunk(const uint32_t (&w)[GeoB<S>::RW], int j) {
    const int o = j * S, q = o / 32, s = o % 32;
    uint32_t v = w[q] >> s;
    if (s + S > 32) v |= w[q + 1] << (32 - s);
    return v & low_bits(S);
}
template <int S>
__device__ __forceinline__ void put_chunk(uint32_t (&w)[GeoB<S>::RW], int j, uint32_t x) {
    const int o = j * S, q = o / 32, s = o % 32;
    w[q] |= x << s;
    if (s + S > 32) w[q + 1] |= x >> (32 - s);
}

// One thread per row of a game, GPC games per CTA, staged through shared memory (mode 1 mixes the rows of a game).
template <int S>
struct BasisB {
    static constexpr int GW = GeoB<S>::GB / 4;          // words per game
    static constexpr int GPC = 256 / S;                 // games per CTA
    static constexpr int NT = GPC * S;                  // threads per CTA (256 / 252 / 256 / 250)
    static constexpr int PW = GW % 32 ? GW : GW + 4;    // staged game pitch in words: two games of a warp on other banks
};

// T' = T x1 A x2 B x3 C mod 2.  Thread (game, i) builds row i of T':
//   mode 1   row_i <- xor_{a: A[i][a]} row_a          (RW words per a, read from the staged game)
//   mode 3   chunk_j <- xor_{c in chunk_j} Ccol_c      (Ccol_c = column c of C as an S-bit mask, built once per game)
//   mode 2   chunk'_j <- xor_{b: B[j][b]} chunk_b
// The CTA reads its games whole before it writes them, so bits_out may be bits_in.
template <int S>
__global__ void __launch_bounds__(BasisB<S>::NT) basis_gf2_kernel(const uint4 *__restrict__ in, const uint32_t *__restrict__ mats,
                                                                 long long mat_stride, uint4 *__restrict__ out, long long N) {
    using B = GeoB<S>;
    using P = BasisB<S>;
    constexpr int RW = B::RW;
    constexpr uint32_t MS = low_bits(S);
    __shared__ __align__(16) uint32_t s_game[P::GPC * P::PW];
    __shared__ uint32_t s_b[P::GPC * S], s_c[P::GPC * S], s_ccol[P::GPC * S];
    const int slot = threadIdx.x / S, i = threadIdx.x % S;
    uint32_t *game = s_game + slot * P::PW;
    for (long long g0 = (long long)blockIdx.x * P::GPC; g0 < N; g0 += (long long)gridDim.x * P::GPC) {
        const int ng = N - g0 < P::GPC ? (int)(N - g0) : P::GPC;
        for (int e = threadIdx.x; e < ng * B::NQ; e += P::NT) {
            const int g = e / B::NQ, q = e - g * B::NQ;
            *reinterpret_cast<uint4 *>(s_game + g * P::PW + 4 * q) = in[g0 * B::NQ + e];
        }
        const bool live = slot < ng;
        uint32_t arow = 0;
        if (live) {
            const uint32_t *m = mats + (g0 + slot) * mat_stride;
            arow = m[i] & MS;
            s_b[slot * S + i] = m[S + i] & MS;
            s_c[slot * S + i] = m[2 * S + i] & MS;
        }
        __syncthreads();
        uint32_t ccol = 0;
#pragma unroll
        for (int k = 0; k < S; k++) ccol |= ((s_c[slot * S + k] >> i) & 1u) << k;
        s_ccol[slot * S + i] = ccol;
        uint32_t row[RW];
#pragma unroll
        for (int w = 0; w < RW; w++) row[w] = 0;
#pragma unroll
        for (int a = 0; a < S; a++) {
            const uint32_t on = 0u - ((arow >> a) & 1u);
            if constexpr (RW % 4 == 0) {
#pragma unroll
                for (int w = 0; w < RW; w += 4) {
                    const uint4 v = *reinterpret_cast<const uint4 *>(game + a * RW + w);
                    row[w] ^= v.x & on, row[w + 1] ^= v.y & on, row[w + 2] ^= v.z & on, row[w + 3] ^= v.w & on;
                }
            } else {
#pragma unroll
                for (int w = 0; w < RW; w++) row[w] ^= game[a * RW + w] & on;
            }
        }
        __syncthreads(); // every read of the staged input done, every column of C built
        uint32_t y[S];
#pragma unroll
        for (int j = 0; j < S; j++) y[j] = get_chunk<S>(row, j);
        uint32_t cc[S];
#pragma unroll
        for (int c = 0; c < S; c++) cc[c] = s_ccol[slot * S + c];
#pragma unroll
        for (int j = 0; j < S; j++) {
            uint32_t z = 0;
#pragma unroll
            for (int c = 0; c < S; c++)
                if ((y[j] >> c) & 1u) z ^= cc[c];
            y[j] = z;
        }
#pragma unroll
        for (int w = 0; w < RW; w++) row[w] = 0;
#pragma unroll
        for (int j = 0; j < S; j++) {
            const uint32_t bj = s_b[slot * S + j];
            uint32_t z = 0;
#pragma unroll
            for (int b = 0; b < S; b++)
                if ((bj >> b) & 1u) z ^= y[b];
            put_chunk<S>(row, j, z);
        }
        if constexpr (RW % 4 == 0) {
#pragma unroll
            for (int w = 0; w < RW; w += 4) *reinterpret_cast<uint4 *>(game + i * RW + w) = make_uint4(row[w], row[w + 1], row[w + 2], row[w + 3]);
        } else {
#pragma unroll
            for (int w = 0; w < RW; w++) game[i * RW + w] = row[w];
        }
        if (i == 0) {
#pragma unroll
            for (int w = S * RW; w < P::GW; w++) game[w] = 0; // padding words (9x9x9: word 27)
        }
        __syncthreads();
        for (int e = threadIdx.x; e < ng * B::NQ; e += P::NT) {
            const int g = e / B::NQ, q = e - g * B::NQ;
            out[g0 * B::NQ + e] = *reinterpret_cast<const uint4 *>(s_game + g * P::PW + 4 * q);
        }
        __syncthreads(); // the stage is rewritten by the next batch
    }
}

// u' = A u, v' = B v, w' = C w mod 2 for the R records of a step-major tape: one thread per game, its triple in
// registers for all R records.  A thread reads each record before it writes it, so tape_out may be tape_in.
template <int S>
__global__ void __launch_bounds__(256) basis_factors_gf2_kernel(const uint8_t *__restrict__ tape_in, long long in_stride, int shift_in,
                                                                const uint32_t *__restrict__ mats, long long mat_stride,
                                                                uint8_t *__restrict__ tape_out, long long out_stride, int shift_out,
                                                                long long N, int R) {
    using B = GeoB<S>;
    constexpr uint32_t MS = low_bits(S);
    constexpr int NW = B::TP / 4; // token words of a record
    const uint32_t sh = (uint32_t)shift_out * ONES4;
    for (long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (long long)gridDim.x * blockDim.x) {
        const uint32_t *m = mats + n * mat_stride;
        uint32_t M[3][S];
#pragma unroll
        for (int f = 0; f < 3; f++)
#pragma unroll
            for (int r = 0; r < S; r++) M[f][r] = m[f * S + r] & MS;
        const uint8_t *src = tape_in + n * B::TP;
        uint8_t *dst = tape_out + n * B::TP;
        for (int t = 0; t < R; t++, src += in_stride, dst += out_stride) {
            const Par p = parities<S>(src, shift_in);
            const uint32_t x[3] = {p.u, p.v, p.w};
            uint32_t Q[3] = {0u, 0u, 0u}; // the 3S parity bits of u', v', w' in token order
#pragma unroll
            for (int f = 0; f < 3; f++)
#pragma unroll
                for (int r = 0; r < S; r++) {
                    const int o = f * S + r;
                    Q[o / 32] |= (__popc(M[f][r] & x[f]) & 1u) << (o % 32);
                }
            uint32_t w[NW];
#pragma unroll
            for (int q = 0; q < NW; q++) {
                const int b0 = 4 * q; // first token byte of the word
                if (b0 >= 3 * S) {
                    w[q] = 0;
                } else {
                    const uint32_t nib = (Q[b0 / 32] >> (b0 % 32)) & 15u; // b0 % 32 <= 28: the nibble lies in one word
                    const uint32_t tok = ((nib * 0x00204081u) & ONES4) + sh;  // bit b of the nibble -> bit 0 of byte b
                    w[q] = 3 * S - b0 >= 4 ? tok : tok & ((1u << (8 * (3 * S - b0))) - 1u);
                }
            }
#pragma unroll
            for (int q = 0; q < NW; q += 4) *reinterpret_cast<uint4 *>(dst + 4 * q) = make_uint4(w[q], w[q + 1], w[q + 2], w[q + 3]);
        }
    }
}

// One thread per (game, matrix f): M = L U mod 2 with the draws of tg_sample_unimodular (its matrices mod 2 at S <= 16).
// The draw of entry e = r S + c is byte e % 16 of Philox block e / 16, ctr = (block, f, 0x6D617473, d_lo); it is non-zero
// iff its low 7 bits are below thr_nz.  L: the non-zero draws below the diagonal and a unit diagonal; U: those above it and
// a unit diagonal.  Rows are bit masks, so row r of M is xor_{k <= r: L[r][k]} row k of U.
template <int S>
__global__ void __launch_bounds__(64) invertible_gf2_kernel(unsigned long long seed, unsigned long long first, long long N,
                                                            uint32_t thr_nz, uint32_t *__restrict__ mats) {
    constexpr int NB = (S * S + 15) / 16;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= 3 * N) return;
    const long long n = t / 3;
    const int f = (int)(t - 3 * n);
    const unsigned long long d = first + (unsigned long long)n;
    const uint32_t k0 = (uint32_t)seed ^ ((uint32_t)(d >> 32) * 0x9E3779B9u), k1 = (uint32_t)(seed >> 32);
    const uint32_t cthr = (0x80u - (thr_nz > 0x80u ? 0x80u : thr_nz)) * ONES4; // (draw & 0x7F) + cthr sets bit 7 iff >= thr
    uint32_t nz[GeoB<S>::RW]; // bit e: the draw of entry e is non-zero (S^2 bits, the words of a bit-slab row)
#pragma unroll
    for (int q = 0; q < GeoB<S>::RW; q++) nz[q] = 0;
#pragma unroll
    for (int b = 0; b < NB; b++) {
        uint32_t blk[4];
        philox_block((uint32_t)b, (uint32_t)f, 0x6D617473u, (uint32_t)d, k0, k1, blk);
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int e0 = 16 * b + 4 * q;
            if (e0 >= S * S) continue;
            const uint32_t nzb = ((((blk[q] & 0x7F7F7F7Fu) + cthr) & H4) ^ H4) >> 7; // bit 0 of each byte: non-zero
            nz[e0 / 32] |= ((nzb * 0x10204080u) >> 28) << (e0 % 32);
        }
    }
    uint32_t U[S];
    uint32_t *out = mats + t * S;
#pragma unroll
    for (int r = 0; r < S; r++) {
        const uint32_t rb = get_chunk<S>(nz, r);
        U[r] = (rb & ~((2u << r) - 1u)) | (1u << r);
        const uint32_t L = rb & ((1u << r) - 1u);
        uint32_t m = U[r];
#pragma unroll
        for (int k = 0; k < r; k++)
            if ((L >> k) & 1u) m ^= U[k];
        out[r] = m;
    }
}

} // namespace
} // namespace tg

extern "C" {

int tg_change_of_basis_gf2(const uint32_t *bits_in, const uint32_t *mats, int per_game, uint32_t *bits_out, int64_t N, int S,
                           void *stream) {
    if (const int rc = tg::check_basis(tg::supported_S(S), N, bits_in, mats, 4, bits_out); rc != tg::LAUNCH) return rc;
    return tg::with_S(S, [&](auto s) {
        constexpr int kS = decltype(s)::value;
        using P = tg::BasisB<kS>;
        tg::basis_gf2_kernel<kS><<<tg::grid_for(N, P::GPC), P::NT, 0, (cudaStream_t)stream>>>(
            reinterpret_cast<const uint4 *>(bits_in), mats, per_game ? 3LL * kS : 0LL, reinterpret_cast<uint4 *>(bits_out), N);
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    });
}

int tg_change_of_basis_factors_gf2(const uint8_t *tape_in, int64_t in_step_stride, int shift_in, const uint32_t *mats, int per_game,
                                   uint8_t *tape_out, int64_t out_step_stride, int shift_out, int64_t N, int R, int S, void *stream) {
    if (shift_in < 1 || shift_in > 4 || shift_out < 1 || shift_out > 4) return TG_E_ARG; // the game path's shifts
    const int rc = tg::check_basis_factors(tg::supported_S(S), N, R, tape_in, in_step_stride, mats, 4, tape_out);
    if (rc != tg::LAUNCH) return rc;
    if (tg::misaligned(tape_out, 16) || (out_step_stride & 15)) return TG_E_ARG; // records leave as 16-byte words
    return tg::with_S(S, [&](auto s) {
        constexpr int kS = decltype(s)::value;
        tg::basis_factors_gf2_kernel<kS><<<tg::grid_for(N, 256), 256, 0, (cudaStream_t)stream>>>(
            tape_in, in_step_stride, shift_in, mats, per_game ? 3LL * kS : 0LL, tape_out, out_step_stride, shift_out, N, R);
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    });
}

int tg_sample_invertible_gf2(uint64_t seed, uint64_t first, int64_t N, int S, double p_nonzero, uint32_t *mats, void *stream) {
    if (const int rc = tg::check_sample_bases(tg::supported_S(S), N, p_nonzero, mats, 4); rc != tg::LAUNCH) return rc;
    const uint32_t thr = (uint32_t)(p_nonzero * 128.0);
    return tg::with_S(S, [&](auto s) {
        constexpr int kS = decltype(s)::value;
        tg::invertible_gf2_kernel<kS><<<(unsigned)((3 * N + 63) / 64), 64, 0, (cudaStream_t)stream>>>(seed, first, N, thr, mats);
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    });
}

} // extern "C"
