// tg_basis_inverse.cu -- inverses of change-of-basis triples: tg_invert_bases (over Z, int8 matrices at 4, 9 and 16) and
// tg_invert_bases_gf2 (over GF(2), bit matrices at 4, 9, 16 and 25).  A game solved from T' = T x1 A x2 B x3 C maps its
// factors back to a factorization of T with u = A^-1 u', v = B^-1 v', w = C^-1 w' (tg_change_of_basis_factors with the
// inverse triple).
//
// Over Z: Gauss-Jordan elimination of [M | I] modulo the prime P = 32749 (2^15 - 19: two products of residues and their
// sum fit 32 bits), the result X lifted to the symmetric range (-P/2, P/2), then certified: every entry in [-128, 127]
// and M X = I exactly in int32 (|sum| <= 16 * 128 * 128 = 2^18).  This decides exactly whether M has an integer inverse
// with int8 entries, for any prime P > 256: if such an inverse Y exists, det M = +-1, so M is invertible mod P and
// X = Y mod P, and since |Y| <= 128 < P/2 the lift is Y and the check passes; if the check passes, X is such an inverse.
// The determinant mod P is never taken as evidence (det = 2^31 is 1 mod 2^31 - 1): the product check is the contract.
#include "tg_gf2.cuh"

namespace tg {
namespace {

constexpr uint32_t INV_P = 32749u;

// d^(P-2) = d^-1 mod P for d != 0 (mod P)
__device__ __forceinline__ uint32_t inverse_mod_p(uint32_t d) {
    uint32_t r = 1u, b = d;
#pragma unroll
    for (uint32_t e = INV_P - 2u; e; e >>= 1) {
        if (e & 1u) r = r * b % INV_P;
        b = b * b % INV_P;
    }
    return r;
}

// One group of S lanes per triple, lane r = row r of a matrix (8 / 3 / 2 triples per warp; at 9 lanes 27..31 idle), the
// three matrices one after the other.  Fraction-free elimination as in tg_slice_rank's rank_mod_p: at column c the first
// unused lane with a non-zero entry is the pivot, and every other lane with a non-zero entry takes row <- row * pv -
// mine * pivot row.  Columns < c of the left half are not updated: an unused lane is zero there, and a used lane keeps
// its pivot value d, scaled with its row, in a register.  At the end the lane that pivoted column j holds d * (row j of
// X) in its right half.  A group reads its matrix into registers before it writes it, so inv may be mats.
template <int S>
__global__ void __launch_bounds__(128) invert_bases_kernel(const int8_t *mats, int8_t *inv,
                                                           uint8_t *__restrict__ flags, long long N) {
    constexpr int TPW = 32 / S;
    constexpr uint32_t FULL = 0xFFFFFFFFu;
    const int lane = threadIdx.x & 31, sub = lane / S, r = lane % S;
    const int base = sub * S; // first lane of the group
    const uint32_t gmask = sub < TPW ? ((1u << S) - 1u) << base : 0u;
    const long long warps = (long long)gridDim.x * (blockDim.x / 32);
    // the loop condition is uniform across the warp: every lane takes part in every ballot and shuffle
    for (long long w = (long long)blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32; w * TPW < N; w += warps) {
        const long long n = w * TPW + sub;
        const bool live = sub < TPW && n < N;
        bool bad_any = false;
#pragma unroll 1
        for (int f = 0; f < 3; f++) {
            const long long row0 = ((n * 3 + f) * S + r) * S;
            int m[S];
#pragma unroll
            for (int c = 0; c < S; c++) m[c] = live ? (int)mats[row0 + c] : 0;
            uint32_t a[2 * S]; // row r of [M | I] mod P
#pragma unroll
            for (int c = 0; c < S; c++) {
                a[c] = m[c] >= 0 ? (uint32_t)m[c] : (uint32_t)(m[c] + (int)INV_P);
                a[S + c] = c == r ? 1u : 0u;
            }
            bool used = !live, singular = false;
            uint32_t d = 0;  // pivot value of this lane's row, once it is used
            int src = lane;  // the lane that pivots column r: it ends with row r of X
#pragma unroll
            for (int c = 0; c < S; c++) {
                const uint32_t cand = __ballot_sync(FULL, !used && a[c] != 0) & gmask;
                const bool has = cand != 0; // uniform within the group
                singular |= !has;
                const int pl = has ? __ffs(cand) - 1 : lane;
                const uint32_t pv = __shfl_sync(FULL, a[c], pl);
                const uint32_t mine = a[c], nmine = INV_P - mine;
                const bool elim = has && lane != pl && mine != 0;
#pragma unroll
                for (int k = c + 1; k < 2 * S; k++) {
                    const uint32_t pk = __shfl_sync(FULL, a[k], pl);
                    if (elim) a[k] = (a[k] * pv + nmine * pk) % INV_P; // < 2 (P - 1)^2 < 2^31
                }
                if (elim && used) d = d * pv % INV_P;
                if (has && lane == pl) used = true, d = pv;
                if (has && c == r) src = pl;
            }
            // X = the right halves over their pivots, lifted; lane r fetches row r
            const uint32_t dinv = inverse_mod_p(d);
            int x[S];
#pragma unroll
            for (int k = 0; k < S; k++) {
                const uint32_t v = a[S + k] * dinv % INV_P;
                const int own = v > INV_P / 2 ? (int)v - (int)INV_P : (int)v;
                x[k] = __shfl_sync(FULL, own, src);
            }
            // certificate: row r of X in int8 and row r of M X equal to row r of I
            bool ok = true;
#pragma unroll
            for (int k = 0; k < S; k++) ok &= x[k] >= -128 && x[k] <= 127;
            int acc[S];
#pragma unroll
            for (int j = 0; j < S; j++) acc[j] = 0;
#pragma unroll
            for (int k = 0; k < S; k++)
#pragma unroll
                for (int j = 0; j < S; j++) acc[j] += m[k] * __shfl_sync(FULL, x[j], base + k);
#pragma unroll
            for (int j = 0; j < S; j++) ok &= acc[j] == (j == r ? 1 : 0);
            // every lane votes: a lane without a triple is always `singular`, and a ballot behind `singular ||` would
            // leave it out of a full-warp vote
            const uint32_t failed = __ballot_sync(FULL, !ok) & gmask;
            const bool bad = singular || failed != 0;
            bad_any |= bad;
            if (live) {
#pragma unroll
                for (int c = 0; c < S; c++) inv[row0 + c] = bad ? (int8_t)0 : (int8_t)x[c];
            }
        }
        if (live && r == 0) flags[n] = bad_any ? (uint8_t)TG_FLAG_SINGULAR : (uint8_t)0;
    }
}

// Over GF(2): one thread per triple, the three matrices one after the other, each as S row words of M and S of the
// identity in registers.  Column c: the first row that has bit c and has not pivoted yet is the pivot, and it is xored
// into every other row that has bit c.  Rows are never swapped (the column loop stays rolled and every register index
// static), so at the end the row that pivoted column j holds e_j on the left and row j of the inverse on the right.  A
// thread reads a matrix whole before it writes it, so inv may be mats.
template <int S>
__global__ void __launch_bounds__(256) invert_bases_gf2_kernel(const uint32_t *mats, uint32_t *inv,
                                                               uint8_t *__restrict__ flags, long long N) {
    constexpr uint32_t MS = (1u << S) - 1u;
    for (long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (long long)gridDim.x * blockDim.x) {
        bool bad_any = false;
#pragma unroll 1
        for (int f = 0; f < 3; f++) {
            const uint32_t *src = mats + (n * 3 + f) * S;
            uint32_t L[S], X[S];
#pragma unroll
            for (int r = 0; r < S; r++) L[r] = src[r] & MS, X[r] = 1u << r;
            uint32_t used = 0; // rows that have pivoted a column
            bool singular = false;
#pragma unroll 1
            for (int c = 0; c < S; c++) {
                uint32_t cand = 0;
#pragma unroll
                for (int r = 0; r < S; r++) cand |= ((L[r] >> c) & 1u) << r;
                cand &= ~used;
                if (!cand) {
                    singular = true;
                    break;
                }
                const int p = __ffs(cand) - 1;
                uint32_t pl = 0, px = 0;
#pragma unroll
                for (int r = 0; r < S; r++) {
                    const uint32_t on = 0u - (uint32_t)(r == p);
                    pl |= L[r] & on, px |= X[r] & on;
                }
#pragma unroll
                for (int r = 0; r < S; r++) {
                    const uint32_t on = 0u - (((L[r] >> c) & 1u) & (uint32_t)(r != p));
                    L[r] ^= pl & on, X[r] ^= px & on;
                }
                used |= 1u << p;
            }
            uint32_t *dst = inv + (n * 3 + f) * S;
#pragma unroll
            for (int r = 0; r < S; r++) {
                if (singular) dst[r] = 0u;
                else dst[__ffs(L[r]) - 1] = X[r];
            }
            bad_any |= singular;
        }
        flags[n] = bad_any ? (uint8_t)TG_FLAG_SINGULAR : (uint8_t)0;
    }
}

} // namespace
} // namespace tg

extern "C" {

int tg_invert_bases(const int8_t *mats, int8_t *inv, uint8_t *flags, int64_t N, int S, void *stream) {
    if (const int rc = tg::check_invert_bases(tg::basis_supported_S(S), N, mats, inv, 1, flags); rc != tg::LAUNCH) return rc;
    return tg::with_basis_S(S, [&](auto s) {
        constexpr int kS = decltype(s)::value;
        // four warps of 32 / S triples per CTA
        tg::invert_bases_kernel<kS><<<tg::grid_for(N, 4 * (32 / kS)), 128, 0, (cudaStream_t)stream>>>(mats, inv, flags, N);
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    });
}

int tg_invert_bases_gf2(const uint32_t *mats, uint32_t *inv, uint8_t *flags, int64_t N, int S, void *stream) {
    if (const int rc = tg::check_invert_bases(tg::supported_S(S), N, mats, inv, 4, flags); rc != tg::LAUNCH) return rc;
    return tg::with_S(S, [&](auto s) {
        constexpr int kS = decltype(s)::value;
        tg::invert_bases_gf2_kernel<kS><<<tg::grid_for(N, 256), 256, 0, (cudaStream_t)stream>>>(mats, inv, flags, N);
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    });
}

} // extern "C"
