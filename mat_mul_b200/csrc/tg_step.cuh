// tg_step.cuh -- the rank-1 update of one game held in shared memory, shared
// by the step (K1), rollout (K2) and demo-generation (K3) kernels.
//
// Reference arithmetic restated: new_head = head - u (x) v (x) w
// (act.py:266-275, training.py:253-255, utils.py:69-85), all-zero test
// (utils.py:181-188), null-action test (utils.py:191-194), nnz
// (training.py:259-266).
//
// Formulation.  A game is S rows (index i) of RP bytes; row i holds the S*S
// entries (j,k).  WR = RP/4 threads own one 32-bit word column c each and walk
// the S rows.  With the four int8 of a word in offset-binary (x ^ 0x80), a
// vector of four small integers is the plain integer sum(x_b * 256^b), and the
// whole update of the word is linear in it:
//        T' <- T' - u_i * VW ,   VW = sum_b v[j_b] w[k_b] 256^b
// i.e. ONE 32-bit IMAD per four entries, exact as long as every resulting
// entry stays in [-128,127].  That is guaranteed while residuals are in
// [-64,63] and |u v w| <= 64 (shift <= 4, tokens <= 2 * shift); leaving that
// zone -- or a token above 2 * shift -- raises TG_FLAG_RANGE for the game (a
// step that left the zone with legal tokens is still exact).
#pragma once
#include "tg_common.cuh"

namespace tg {

// Per-thread constants of word column c.
template <int S>
struct Lane {
    int c;
    uint32_t hv;      // 0x80 in every byte that is a real entry (not row padding)
    uint32_t maskA;   // bytes of the word that belong to j = jA
    uint32_t maskB;   // bytes that belong to j = jA + 1 (STRADDLE only)
    int off_vA, off_vB; // token byte offsets of v[jA], v[jA+1]
    int off_w[4];       // token byte offsets of w[k_b]; [0] is word aligned when !STRADDLE
    int tokw;           // the 32-bit word of the game's token record this thread range-checks (tokens_out_of_range)

    __device__ __forceinline__ void init(int c_) {
        using G = Geo<S>;
        c = c_;
        tokw = c_ % (G::TP / 4);
        const int jk0 = 4 * c;
        const int jA = jk0 / S;
        hv = 0, maskA = 0, maskB = 0;
#pragma unroll
        for (int b = 0; b < 4; b++) {
            const int jk = jk0 + b;
            const bool valid = jk < G::S2;
            const int j = valid ? jk / S : jA;
            const int k = valid ? jk % S : 0;
            off_w[b] = 2 * S + k;
            if (valid) {
                hv |= 0x80u << (8 * b);
                if (j == jA)
                    maskA |= 0xFFu << (8 * b);
                else
                    maskB |= 0xFFu << (8 * b);
            }
        }
        off_vA = S + jA;
        off_vB = S + (jA + 1 < S ? jA + 1 : jA);
    }
};

// Packed sum_b v[j_b] w[k_b] 256^b of this thread's word column for the game
// whose tokens start at tok (shared memory).
template <int S>
__device__ __forceinline__ int32_t pack_vw(const uint8_t *tok, const Lane<S> &L, int shift) {
    using G = Geo<S>;
    const int vA = (int)tok[L.off_vA] - shift;
    if constexpr (!G::STRADDLE) {
        const uint32_t wt = *reinterpret_cast<const uint32_t *>(tok + L.off_w[0]);
        return vA * (int32_t)(wt - (uint32_t)shift * ONES4);
    } else {
        const int vB = (int)tok[L.off_vB] - shift;
        const uint32_t wt = (uint32_t)tok[L.off_w[0]] | ((uint32_t)tok[L.off_w[1]] << 8) |
                            ((uint32_t)tok[L.off_w[2]] << 16) | ((uint32_t)tok[L.off_w[3]] << 24);
        // integer form of the valid bytes, ws = wsA + wsB, so vA wsA + vB wsB = vA ws + (vB - vA) wsB
        const uint32_t sh = (uint32_t)shift * ONES4, mv = L.maskA | L.maskB;
        const int32_t ws = (int32_t)((wt & mv) - (sh & mv));
        const int32_t wsB = (int32_t)((wt & L.maskB) - (sh & L.maskB));
        return vA * ws + (vB - vA) * wsB;
    }
}

// Tape contract: every token byte is <= 2 * shift, i.e. |coefficient| <= shift -- the bound the packed arithmetic relies
// on (|u v w| <= shift^3 <= 64 per step).  Thread c tests word c % (TP / 4) of its game's record; the WR >= TP / 4
// threads of a game cover the whole record.  A violation raises TG_FLAG_RANGE for the game.
template <int S>
__device__ __forceinline__ bool tokens_out_of_range(const uint8_t *tok, const Lane<S> &L, int shift) {
    static_assert(Geo<S>::WR >= Geo<S>::TP / 4, "not enough threads per game to cover the token record");
    const uint32_t x = reinterpret_cast<const uint32_t *>(tok)[L.tokw];
    return ((((x & 0x7F7F7F7Fu) + (uint32_t)(0x7F - 2 * shift) * ONES4) | x) & H4) != 0;
}

// The u tokens of a record (bytes 0 .. S-1) as UW<S> words: one 16-byte shared-memory load per 16 tokens (records are
// 16-byte aligned and TP >= 16 * ceil(S / 16) bytes long); words beyond byte S - 1 hold v tokens and are never indexed.
template <int S>
constexpr int UW = 4 * ((S + 15) / 16);
template <int S>
__device__ __forceinline__ void load_u(const uint8_t *tok, uint32_t (&uw)[UW<S>]) {
    static_assert(UW<S> * 4 <= Geo<S>::TP, "u words inside the token record");
#pragma unroll
    for (int q = 0; q < UW<S> / 4; q++) {
        const uint4 ut = reinterpret_cast<const uint4 *>(tok)[q];
        uw[4 * q] = ut.x, uw[4 * q + 1] = ut.y, uw[4 * q + 2] = ut.z, uw[4 * q + 3] = ut.w;
    }
}

// coefficient u_i = token_i - shift from the packed u tokens: one dp4a against a one-hot byte vector
__device__ __forceinline__ int coef_u(const uint32_t *uw, int i, int shift) {
    return (int)__dp4a(uw[i >> 2], 1u << (8 * (i & 3)), (uint32_t)(-shift));
}

// Partial result word of one thread for one game; summing it over the WR
// threads of a game gives nnz (bits 0-15), #threads whose update was non-zero
// (bits 16-23) and #threads that saw an entry outside [-64,63] (bits 24-31).
// The fields cannot carry into each other while S^3 < 2^16 and WR < 2^8 (25x25x25: 15625 entries, 157 threads).
template <int S>
struct PartialFits {
    static constexpr bool value = Geo<S>::S3 < (1 << 16) && Geo<S>::WR < (1 << 8);
};
static_assert(PartialFits<4>::value && PartialFits<9>::value && PartialFits<16>::value && PartialFits<25>::value,
              "partial result word fields");
static_assert(Geo<25>::WR >= Geo<25>::TP / 4, "25x25x25: the threads of a game cover its token record");
__device__ __forceinline__ uint32_t make_partial(uint32_t nnz, bool changed, bool range) {
    return nnz | (changed ? 1u << 16 : 0u) | (range ? 1u << 24 : 0u);
}
__device__ __forceinline__ uint32_t partial_flags(uint32_t sum) {
    return ((sum & 0xFFFFu) == 0 ? TG_FLAG_TERMINAL : 0u) | (((sum >> 16) & 0xFFu) == 0 ? TG_FLAG_NULL : 0u) |
           ((sum >> 24) != 0 ? TG_FLAG_RANGE : 0u);
}

// game <- game + SIGN * u (x) v (x) w for this thread's word column, all S
// rows.  game/tok point into shared memory.  SIGN = -1 for the transition.
template <int S, int SIGN>
__device__ __forceinline__ uint32_t rank1_update(uint8_t *game, const uint8_t *tok, const Lane<S> &L, int shift) {
    using G = Geo<S>;
    const int32_t vw = pack_vw<S>(tok, L, shift);
    uint32_t uw[UW<S>];
    load_u<S>(tok, uw);
    uint32_t cnt = 0, rng = 0;
    int uany = 0;
    uint32_t *col = reinterpret_cast<uint32_t *>(game) + L.c;
    const uint32_t svw = (uint32_t)(SIGN < 0 ? -vw : vw); // SIGN * VW
#pragma unroll
    for (int i = 0; i < S; i++) {
        const int negu = coef_u(uw, i, shift);
        uint32_t t = col[i * G::WR] ^ H4;
        t += (uint32_t)negu * svw;
        t ^= H4;
        col[i * G::WR] = t;
        cnt += ((((t & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | t) & L.hv) >> 7;
        rng |= t ^ (t << 1);
        uany |= negu;
    }
    return make_partial(byte_sum(cnt), vw != 0 && uany != 0, (rng & L.hv) != 0 || tokens_out_of_range<S>(tok, L, shift));
}

// nnz / range of a game without changing it (used for the initial state of a rollout)
template <int S>
__device__ __forceinline__ uint32_t scan_game(const uint8_t *game, const Lane<S> &L) {
    using G = Geo<S>;
    uint32_t cnt = 0, rng = 0;
    const uint32_t *col = reinterpret_cast<const uint32_t *>(game) + L.c;
#pragma unroll
    for (int i = 0; i < S; i++) {
        const uint32_t t = col[i * G::WR];
        cnt += ((((t & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | t) & L.hv) >> 7;
        rng |= t ^ (t << 1);
    }
    return make_partial(byte_sum(cnt), true, (rng & L.hv) != 0);
}

} // namespace tg
