// tg_step.cuh -- the word-column kernels of the int8 and int16 game paths: the rank-1 update of one game held in
// shared memory (K1 step_kernel), the leaf expansion (K8 expand_kernel), and the helpers the rollout (K2) and
// demo-generation (K3) kernels share with them.
//
// Reference arithmetic restated: new_head = head - u (x) v (x) w
// (act.py:266-275, training.py:253-255, utils.py:69-85), all-zero test
// (utils.py:181-188), null-action test (utils.py:191-194), nnz
// (training.py:259-266).
//
// Formulation.  A game is S rows (index i) of RP entries; row i holds the S*S
// entries (j,k).  WR threads own one 32-bit word column c each and walk
// the S rows.  With the lanes of a word in offset-binary (x ^ H), a vector of
// small integers is the plain integer sum(x_b * L^b) (lane base L = 256 for int8, 65536 for int16), and the
// whole update of the word is linear in it:
//        T' <- T' - u_i * VW ,   VW = sum_b v[j_b] w[k_b] L^b
// i.e. ONE 32-bit IMAD per four int8 (two int16) entries, exact as long as every resulting
// entry fits its lane.  That is guaranteed while residuals are in the zone -- [-64,63] for int8, [-16384, 16383]
// for int16: the top two bits of a lane are equal -- and |u v w| <= 64 (shift <= 4, tokens <= 2 * shift); leaving that
// zone -- or a token above 2 * shift -- raises TG_FLAG_RANGE for the game (a
// step that left the zone with legal tokens is still exact).  When S^2 is not a multiple of the lanes per word, a word
// can hold the last entries of row j and the first of row j + 1.
#pragma once
#include "tg_common.cuh"

namespace tg {

// ---------------------------------------------------------------- word formats
// W8: the int8 slab, four entries per word.  W16: the int16 slab, the int8 slab's geometry counted in elements (entry
// (i,j,k) at element i*RP + j*S + k of a game of GP elements), two entries per word.
//
// The partial result word of one thread for one game (make_partial) holds nnz in bits 0 .. NB-1, whether the thread's
// update was non-zero at bit NB and whether it saw an entry outside the zone at bit NB + CB; summed over the WR threads
// of a game the three fields cannot carry into each other while S^3 < 2^NB and WR < 2^CB.
//
// ColumnKey: word column c's share of the state key (key_const), sum_q (B C)[jk_q] * sum_i A_i T[i][jk_q] over its
// entries jk_q, from its S offset-binary row words (unsigned lanes, entry + 2^(8 EB - 1); the offset's share is the
// accumulators' start value).  init(c) takes what depends on the column alone.
struct W8 {
    using T = int8_t;
    static constexpr int EB = 1; // bytes per entry
    static constexpr uint32_t H = H4;
    static constexpr int NB = 16, CB = 8;
    static constexpr bool UNROLL_PASSES = true; // step_kernel's pass loop

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
    static __device__ __forceinline__ int32_t pack_vw(const uint8_t *tok, const Lane<S> &L, int shift) {
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

    // sum of the per-lane counts of a word
    static __device__ __forceinline__ uint32_t lane_sum(uint32_t cnt) { return byte_sum(cnt); }

    template <int S>
    struct ColumnKey {
        unsigned long long kb[4]; // B_j C_k of the column's four entries (0 in the row padding)

        __device__ __forceinline__ void init(int c) {
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const int jk = 4 * c + q;
                kb[q] = jk < Geo<S>::S2 ? key_const(0x2000, jk / S) * key_const(0x3000, jk % S) : 0ull;
            }
        }
        __device__ __forceinline__ unsigned long long operator()(const uint32_t (&row)[S]) const {
            unsigned long long a0 = 0;
#pragma unroll
            for (int i = 0; i < S; i++) a0 -= 128ull * key_const(0x1000, i);
            unsigned long long acc[4] = {a0, a0, a0, a0};
#pragma unroll
            for (int i = 0; i < S; i++) {
#pragma unroll
                for (int q = 0; q < 4; q++) acc[q] += (unsigned long long)((row[i] >> (8 * q)) & 0xFFu) * key_const(0x1000, i);
            }
            return acc[0] * kb[0] + acc[1] * kb[1] + acc[2] * kb[2] + acc[3] * kb[3];
        }
    };
};

struct W16 {
    using T = int16_t;
    static constexpr int EB = 2;
    static constexpr uint32_t H = 0x80008000u;
    static constexpr int NB = 14, CB = 9;
    static constexpr bool UNROLL_PASSES = false; // unrolled, the 9x9x9 step kernel spills

    // Per-thread constants of word column c of an int16 game.
    template <int S>
    struct Lane {
        int c;
        uint32_t hv;            // 0x8000 in every lane that is a real entry (not row padding)
        int off_v[2], off_w[2]; // token byte offsets of v[j_b], w[k_b] (a valid offset for padding lanes too)
        int m1;                 // lane 1 is a real entry
        int tokw;               // the 32-bit word of the game's token record this thread range-checks

        __device__ __forceinline__ void init(int c_) {
            c = c_;
            tokw = c_ % (Geo<S>::TP / 4);
            hv = 0;
#pragma unroll
            for (int b = 0; b < 2; b++) {
                const int jk = 2 * c + b;
                const bool valid = jk < Geo<S>::S2;
                off_v[b] = S + (valid ? jk / S : 0);
                off_w[b] = 2 * S + (valid ? jk % S : 0);
                if (valid) hv |= 0x8000u << (16 * b);
            }
            m1 = (hv >> 31) & 1;
        }
    };

    // VW = v[j_0] w[k_0] + v[j_1] w[k_1] 65536 of this thread's word (0 in padding lanes) for the record at tok
    template <int S>
    static __device__ __forceinline__ uint32_t pack_vw(const uint8_t *tok, const Lane<S> &L, int shift) {
        const int d0 = ((int)tok[L.off_v[0]] - shift) * ((int)tok[L.off_w[0]] - shift);
        const int d1 = ((int)tok[L.off_v[1]] - shift) * ((int)tok[L.off_w[1]] - shift);
        return L.hv ? (uint32_t)d0 + ((uint32_t)(d1 * L.m1) << 16) : 0u;
    }

    static __device__ __forceinline__ uint32_t lane_sum(uint32_t cnt) { return (cnt & 0xFFFFu) + (cnt >> 16); }

    template <int S>
    struct ColumnKey {
        int c;

        __device__ __forceinline__ void init(int c_) { c = c_; }
        __device__ __forceinline__ unsigned long long operator()(const uint32_t (&row)[S]) const {
            unsigned long long a0 = 0;
#pragma unroll
            for (int i = 0; i < S; i++) a0 -= 32768ull * key_const(0x1000, i);
            unsigned long long acc[2] = {a0, a0};
#pragma unroll
            for (int i = 0; i < S; i++) {
                acc[0] += (unsigned long long)(row[i] & 0xFFFFu) * key_const(0x1000, i);
                acc[1] += (unsigned long long)(row[i] >> 16) * key_const(0x1000, i);
            }
            unsigned long long h = 0;
#pragma unroll
            for (int q = 0; q < 2; q++) {
                const int jk = 2 * c + q;
                if (jk < Geo<S>::S2) h += acc[q] * (key_const(0x2000, jk / S) * key_const(0x3000, jk % S));
            }
            return h;
        }
    };
};

template <int S>
using Lane = W8::Lane<S>;

// A game in word format F: Geo<S> in entries, with F's 32-bit words per row and bytes per game
template <int S, class F>
struct GeoW : Geo<S> {
    static constexpr int WR = Geo<S>::RP * F::EB / 4; // 32-bit words per row
    static constexpr int GB = Geo<S>::GP * F::EB;     // game pitch (bytes)
};

// 25x25x25 has the most entries and word columns per game
template <class F>
constexpr bool partial_fits = Geo<25>::S3 < (1 << F::NB) && GeoW<25, F>::WR < (1 << F::CB);
static_assert(partial_fits<W8> && partial_fits<W16>, "partial result word fields");

template <class F = W8>
__device__ __forceinline__ uint32_t make_partial(uint32_t nnz, bool changed, bool range) {
    return nnz | (changed ? 1u << F::NB : 0u) | (range ? 1u << (F::NB + F::CB) : 0u);
}
template <class F = W8>
__device__ __forceinline__ uint32_t partial_nnz(uint32_t sum) { return sum & ((1u << F::NB) - 1u); }
template <class F = W8>
__device__ __forceinline__ uint32_t partial_flags(uint32_t sum) {
    return (partial_nnz<F>(sum) == 0 ? TG_FLAG_TERMINAL : 0u) | (((sum >> F::NB) & ((1u << F::CB) - 1u)) == 0 ? TG_FLAG_NULL : 0u) |
           ((sum >> (F::NB + F::CB)) != 0 ? TG_FLAG_RANGE : 0u);
}

// the lowest bit of every lane of word t that is a non-zero real entry (hv: the top bit of every real lane)
template <class F>
__device__ __forceinline__ uint32_t nonzero_lanes(uint32_t t, uint32_t hv) {
    return ((((t & ~F::H) + ~F::H) | t) & hv) >> (8 * F::EB - 1);
}

// Tape contract: every token byte is <= 2 * shift, i.e. |coefficient| <= shift -- the bound the packed arithmetic relies
// on (|u v w| <= shift^3 <= 64 per step).  Thread c tests word c % (TP / 4) of its game's record; the WR >= TP / 4
// threads of a game cover the whole record.  A violation raises TG_FLAG_RANGE for the game.
template <int S, class F = W8>
__device__ __forceinline__ bool tokens_out_of_range(const uint8_t *tok, const typename F::template Lane<S> &L, int shift) {
    static_assert(GeoW<S, F>::WR >= Geo<S>::TP / 4, "not enough threads per game to cover the token record");
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

// game <- game + SIGN * u (x) v (x) w for this thread's word column, all S
// rows.  game/tok point into shared memory.  SIGN = -1 for the transition.
template <int S, int SIGN, class F = W8>
__device__ __forceinline__ uint32_t rank1_update(uint8_t *game, const uint8_t *tok, const typename F::template Lane<S> &L, int shift) {
    using G = GeoW<S, F>;
    const auto vw = F::template pack_vw<S>(tok, L, shift);
    uint32_t uw[UW<S>];
    load_u<S>(tok, uw);
    uint32_t cnt = 0, rng = 0;
    int uany = 0;
    uint32_t *col = reinterpret_cast<uint32_t *>(game) + L.c;
    const uint32_t svw = (uint32_t)(SIGN < 0 ? -vw : vw); // SIGN * VW
#pragma unroll
    for (int i = 0; i < S; i++) {
        const int negu = coef_u(uw, i, shift);
        uint32_t t = col[i * G::WR] ^ F::H;
        t += (uint32_t)negu * svw;
        t ^= F::H;
        col[i * G::WR] = t;
        cnt += nonzero_lanes<F>(t, L.hv);
        rng |= t ^ (t << 1);
        uany |= negu;
    }
    return make_partial<F>(F::lane_sum(cnt), vw != 0 && uany != 0, (rng & L.hv) != 0 || tokens_out_of_range<S, F>(tok, L, shift));
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

// ---------------------------------------------------------------- K1: batched transition (tg_step, tg_step_i16)
// Persistent, warp-specialised kernel.  Each CTA walks tiles of TG games:
//   producer warp (one elected lane): TMA 1-D bulk copies (cp.async.bulk) of
//     the tile's slab bytes and token bytes into an NSTAGE-deep shared-memory
//     ring, completion on mbarriers; after the compute warps release a stage it
//     bulk-stores the updated slab back to HBM and refills the stage.
//   compute warps: WR threads per game, one IMAD per 32-bit word (rank1_update),
//     per-game nnz/flags reduced through shared memory and written directly.
// HBM traffic per game = 2*GB + TP + 5 bytes, every access a full line.
template <int S, int NT, int NPASS, int NSTAGE, class F>
struct StepCfg {
    using G = GeoW<S, F>;
    static constexpr int GPASS = NT / G::WR;                // games per pass over the compute threads
    static constexpr int TG = GPASS * NPASS;                // games per tile
    static constexpr int ACTIVE = GPASS * G::WR;            // compute threads that own a word column
    static constexpr int SLAB_BYTES = TG * G::GB;
    static constexpr int TOK_BYTES = TG * G::TP;
    static constexpr int STAGE_BYTES = SLAB_BYTES + TOK_BYTES;
    // partial words per game handed to the reducer thread
    static constexpr int PW = (G::WR % 32 == 0) ? G::WR / 32 : ((32 % G::WR == 0) ? 1 : G::WR);
    static constexpr int PART_WORDS = TG * PW;
    static constexpr int SMEM_BYTES = NSTAGE * STAGE_BYTES + 2 * PART_WORDS * 4 + 2 * NSTAGE * 8;
    static constexpr int THREADS = NT + 32;
    static_assert(SMEM_BYTES <= 227 * 1024, "shared memory of one CTA");
};

template <int S, int NT, int NPASS, int NSTAGE, class F>
__global__ void __launch_bounds__(NT + 32)
    step_kernel(const typename F::T *__restrict__ slab_in, const uint8_t *__restrict__ tape, typename F::T *__restrict__ slab_out,
                uint8_t *__restrict__ flags, int32_t *__restrict__ nnz, long long B, int shift) {
    using C = StepCfg<S, NT, NPASS, NSTAGE, F>;
    using G = GeoW<S, F>;
    extern __shared__ __align__(128) uint8_t smem[];
    uint32_t *part = reinterpret_cast<uint32_t *>(smem + NSTAGE * C::STAGE_BYTES);
    uint64_t *full = reinterpret_cast<uint64_t *>(part + 2 * C::PART_WORDS);
    uint64_t *done = full + NSTAGE;

    const int tid = threadIdx.x;
    const long long ntiles = (B + C::TG - 1) / C::TG;

    if (tid == 0) {
        for (int s = 0; s < NSTAGE; s++) {
            mbar_init(&full[s], 1);
            mbar_init(&done[s], 1);
        }
        mbar_fence_init();
    }
    __syncthreads();

    if (tid >= NT) {
        // ------------------------------------------------ producer / storer (one lane)
        if (tid != NT) return;
        auto load = [&](long long tile, int s) {
            const long long g0 = tile * C::TG;
            const int ng = (int)min((long long)C::TG, B - g0);
            uint8_t *st = smem + s * C::STAGE_BYTES;
            mbar_expect_tx(&full[s], (uint32_t)(ng * (G::GB + G::TP)));
            bulk_g2s(st, slab_in + g0 * G::GP, (uint32_t)(ng * G::GB), &full[s]);
            bulk_g2s(st + C::SLAB_BYTES, tape + g0 * G::TP, (uint32_t)(ng * G::TP), &full[s]);
        };
        long long tile = blockIdx.x;
        for (int s = 0; s < NSTAGE && tile + (long long)s * gridDim.x < ntiles; s++) load(tile + (long long)s * gridDim.x, s);
        for (int it = 0; tile < ntiles; tile += gridDim.x, it++) {
            const int s = it % NSTAGE;
            const uint32_t parity = (uint32_t)(it / NSTAGE) & 1u;
            mbar_wait(&done[s], parity); // compute warps have finished this stage
            const long long g0 = tile * C::TG;
            const int ng = (int)min((long long)C::TG, B - g0);
            bulk_s2g(slab_out + g0 * G::GP, smem + s * C::STAGE_BYTES, (uint32_t)(ng * G::GB));
            bulk_commit();
            const long long next = tile + (long long)NSTAGE * gridDim.x;
            if (next < ntiles) {
                bulk_wait_read<0>(); // the store has drained the stage
                load(next, s);
            }
        }
        bulk_wait<0>();
        return;
    }

    // ---------------------------------------------------- compute warps
    typename F::template Lane<S> L;
    const bool active = tid < C::ACTIVE;
    const int gl = tid / G::WR; // game slot within a pass
    L.init(active ? tid % G::WR : 0);

    int it = 0;
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, it++) {
        const int s = it % NSTAGE;
        const uint32_t parity = (uint32_t)(it / NSTAGE) & 1u;
        const long long g0 = tile * C::TG;
        const int ng = (int)min((long long)C::TG, B - g0);
        uint8_t *slab = smem + s * C::STAGE_BYTES;
        const uint8_t *toks = slab + C::SLAB_BYTES;
        uint32_t *pp = part + (it & 1) * C::PART_WORDS;

        mbar_wait(&full[s], parity);
        // the same pass loop twice: unrolled where F allows it (a count after the pragma changes the int8 code)
        if constexpr (F::UNROLL_PASSES) {
#pragma unroll
            for (int p = 0; p < NPASS; p++) {
                const int g = p * C::GPASS + gl;
                uint32_t pr = 0;
                if (active && g < ng) pr = rank1_update<S, -1, F>(slab + g * G::GB, toks + g * G::TP, L, shift);
                if constexpr (G::WR % 32 == 0) { // a game spans whole warps
                    pr = __reduce_add_sync(0xFFFFFFFFu, pr);
                    if ((tid & 31) == 0 && g < ng) pp[g * C::PW + (tid % G::WR) / 32] = pr;
                } else if constexpr (32 % G::WR == 0) { // several games per warp
#pragma unroll
                    for (int o = 1; o < G::WR; o <<= 1) pr += __shfl_xor_sync(0xFFFFFFFFu, pr, o);
                    if (L.c == 0 && g < ng) pp[g] = pr;
                } else {
                    if (active && g < ng) pp[g * C::PW + L.c] = pr;
                }
            }
        } else {
#pragma unroll 1
            for (int p = 0; p < NPASS; p++) {
                const int g = p * C::GPASS + gl;
                uint32_t pr = 0;
                if (active && g < ng) pr = rank1_update<S, -1, F>(slab + g * G::GB, toks + g * G::TP, L, shift);
                if constexpr (G::WR % 32 == 0) { // a game spans whole warps
                    pr = __reduce_add_sync(0xFFFFFFFFu, pr);
                    if ((tid & 31) == 0 && g < ng) pp[g * C::PW + (tid % G::WR) / 32] = pr;
                } else if constexpr (32 % G::WR == 0) { // several games per warp
#pragma unroll
                    for (int o = 1; o < G::WR; o <<= 1) pr += __shfl_xor_sync(0xFFFFFFFFu, pr, o);
                    if (L.c == 0 && g < ng) pp[g] = pr;
                } else {
                    if (active && g < ng) pp[g * C::PW + L.c] = pr;
                }
            }
        }
        fence_proxy_async(); // slab writes -> async proxy, before the producer's bulk store
        asm volatile("bar.sync 1, %0;" ::"n"(NT) : "memory");
        if (tid == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&done[s])) : "memory");
        for (int g = tid; g < ng; g += NT) {
            uint32_t sum = 0;
#pragma unroll
            for (int w = 0; w < C::PW; w++) sum += pp[g * C::PW + w];
            flags[g0 + g] = (uint8_t)partial_flags<F>(sum);
            nnz[g0 + g] = (int32_t)partial_nnz<F>(sum);
        }
    }
}

// ctas_per_sm: CTAs launched per SM at most (the grid is also capped by the number of tiles)
template <int S, int NT, int NPASS, int NSTAGE, class F>
int launch_step(const typename F::T *slab_in, const uint8_t *tape, typename F::T *slab_out, uint8_t *flags, int32_t *nnz,
                long long B, int shift, int ctas_per_sm, cudaStream_t stream) {
    using C = StepCfg<S, NT, NPASS, NSTAGE, F>;
    auto kern = step_kernel<S, NT, NPASS, NSTAGE, F>;
    TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
    const long long ntiles = (B + C::TG - 1) / C::TG;
    const long long cap = (long long)sm_count() * ctas_per_sm;
    const int grid = (int)(ntiles < cap ? ntiles : cap);
    kern<<<grid, C::THREADS, C::SMEM_BYTES, stream>>>(slab_in, tape, slab_out, flags, nnz, B, shift);
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

// ---------------------------------------------------------------- K8: batched leaf expansion (tg_expand_children*)
// The parent is read ONCE: thread (parent, word column) keeps its S row words in registers and produces the k
// children one after the other into a three-stage shared-memory tile; each child game leaves with a TMA bulk store
// while the next ones are computed (three stages so that ONE CTA barrier per child is enough: a stage is rewritten two
// barriers after the threads that issued its stores have seen them drain).  HBM traffic per child: GB * (1 + 1/k) + TP + 13 bytes.
// The state key is the trilinear form of the state at three fixed 64-bit vectors (key_const), so a child's key is the
// parent's key (hashed once per parent) minus (sum u_i A_i)(sum v_j B_j)(sum w_k C_k): 3 S multiply-adds on the
// action's tokens, done for all TG * k children of the block before the child loop -- no pass over the child, no
// per-entry work.
template <int S, int NT, class F>
struct ExpCfg {
    using G = GeoW<S, F>;
    static constexpr int TG = NT / G::WR; // parents per CTA (one word column per thread)
    static constexpr int ACTIVE = TG * G::WR;
    static constexpr int STAGE_BYTES = TG * G::GB;
    static __host__ __device__ constexpr int tok_bytes(int k) { return (TG * k * G::TP + 15) & ~15; }
    static constexpr int NSTAGE = 3;
    // tokens, NSTAGE child stages, per-(stage, game) partial word and key
    static __host__ __device__ constexpr int smem_bytes(int k) {
        return tok_bytes(k) + NSTAGE * STAGE_BYTES + ((NSTAGE * TG * 4 + 7) & ~7) + TG * 8 + 16 + NT * 8;
    }
};

template <int S, int NT, bool KEYS, class F>
__global__ void __launch_bounds__(NT)
    expand_kernel(const typename F::T *__restrict__ parents, const uint8_t *__restrict__ tape, int k,
                  typename F::T *__restrict__ children, uint8_t *__restrict__ flags, int32_t *__restrict__ nnz,
                  unsigned long long *__restrict__ keys, long long B, int shift) {
    using C = ExpCfg<S, NT, F>;
    using G = GeoW<S, F>;
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t *s_tok = smem;                                                            // [TG][k][TP]
    constexpr int NSTAGE = C::NSTAGE;
    uint8_t *s_out = smem + C::tok_bytes(k);                                          // [NSTAGE][TG][GB]
    uint32_t *s_part = reinterpret_cast<uint32_t *>(s_out + NSTAGE * C::STAGE_BYTES); // [NSTAGE][TG]
    unsigned long long *s_pkey = reinterpret_cast<unsigned long long *>(reinterpret_cast<uint8_t *>(s_part) + ((NSTAGE * C::TG * 4 + 7) & ~7)); // [TG] parent keys
    uint64_t *s_bar = reinterpret_cast<uint64_t *>(s_pkey + C::TG);
    unsigned long long *s_ph = reinterpret_cast<unsigned long long *>(s_bar + 2); // [NT] parent key, per word column
    uint8_t *out = reinterpret_cast<uint8_t *>(children);

    const int tid = threadIdx.x;
    const long long g0 = (long long)blockIdx.x * C::TG;
    const int ng = (int)min((long long)C::TG, B - g0);
    const int g = tid / G::WR;
    const bool active = tid < C::ACTIVE && g < ng;
    typename F::template Lane<S> L;
    L.init(tid < C::ACTIVE ? tid % G::WR : 0);

    if (tid == 0) {
        mbar_init(s_bar, 1);
        mbar_fence_init();
    }
    // game padding of the child stages is zero and stays zero (threads only write their word columns of the S rows)
    for (int w = tid; w < NSTAGE * C::STAGE_BYTES / 4; w += NT) reinterpret_cast<uint32_t *>(s_out)[w] = 0;
    for (int i = tid; i < NSTAGE * C::TG; i += NT) s_part[i] = 0;
    typename F::template ColumnKey<S> ck;
    if constexpr (KEYS) ck.init(L.c);
    __syncthreads();
    if (tid == 0) {
        mbar_expect_tx(s_bar, (uint32_t)(ng * k * G::TP));
        bulk_g2s(s_tok, tape + g0 * k * G::TP, (uint32_t)(ng * k * G::TP), s_bar);
    }
    // the parent's rows of this thread's word column, offset-binary
    uint32_t row[S];
    if (active) {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(parents + (g0 + g) * G::GP) + L.c;
#pragma unroll
        for (int i = 0; i < S; i++) row[i] = src[i * G::WR] ^ F::H;
    } else {
#pragma unroll
        for (int i = 0; i < S; i++) row[i] = F::H;
    }
    if constexpr (KEYS) s_ph[tid] = ck(row); // the parent's key, once
    mbar_wait(s_bar, 0);
    if constexpr (KEYS) {
        __syncthreads();
        if (tid < ng) {
            unsigned long long h = 0;
            for (int c = 0; c < G::WR; c++) h += s_ph[tid * G::WR + c];
            s_pkey[tid] = h;
        }
        __syncthreads();
        // child key = parent key - key of its rank-1 action, the latter from the action's tokens alone; one coalesced
        // store of the block's TG * k keys
        for (int x = tid; x < ng * k; x += NT) {
            const uint8_t *tok = s_tok + (size_t)x * G::TP;
            unsigned long long f[3];
#pragma unroll
            for (int m = 0; m < 3; m++) {
                unsigned long long a = 0;
#pragma unroll
                for (int i = 0; i < S; i++) a += (unsigned long long)(long long)((int)tok[m * S + i] - shift) * key_const(0x1000 * (m + 1), i);
                f[m] = a;
            }
            keys[g0 * k + x] = s_pkey[x / k] - f[0] * f[1] * f[2];
        }
    }

    for (int c = 0, st = 0; c < k; c++, st = st + 1 == NSTAGE ? 0 : st + 1) {
        uint8_t *stage = s_out + st * C::STAGE_BYTES;
        // the bulk stores of child c-3 have finished reading this stage: the threads that issued them waited for child c-2's
        // predecessor to drain (bulk_wait_read<1> below, iteration c-2) before they arrived at the barrier of iteration c-1
        if (active) {
            const uint8_t *tok = s_tok + ((size_t)g * k + c) * G::TP;
            const auto vw = F::template pack_vw<S>(tok, L, shift);
            uint32_t uw[UW<S>];
            load_u<S>(tok, uw);
            const uint32_t nvw = (uint32_t)(-vw);
            uint32_t cnt = 0, rng = 0;
            int uany = 0;
            uint32_t *col = reinterpret_cast<uint32_t *>(stage + (size_t)g * G::GB) + L.c;
#pragma unroll
            for (int i = 0; i < S; i++) {
                const int negu = coef_u(uw, i, shift);
                const uint32_t t = (row[i] + (uint32_t)negu * nvw) ^ F::H; // child word, two's complement lanes
                col[i * G::WR] = t;
                cnt += nonzero_lanes<F>(t, L.hv);
                rng |= t ^ (t << 1);
                uany |= negu;
            }
            atomicAdd(&s_part[st * C::TG + g], make_partial<F>(F::lane_sum(cnt), vw != 0 && uany != 0,
                                                               (rng & L.hv) != 0 || tokens_out_of_range<S, F>(tok, L, shift)));
        }
        fence_proxy_async();
        __syncthreads();
        if (tid < ng) {
            const long long child = (g0 + tid) * k + c;
            bulk_s2g(out + child * G::GB, stage + (size_t)tid * G::GB, (uint32_t)G::GB);
            bulk_commit();
            const uint32_t sum = s_part[st * C::TG + tid];
            flags[child] = (uint8_t)partial_flags<F>(sum);
            nnz[child] = (int32_t)partial_nnz<F>(sum);
            s_part[st * C::TG + tid] = 0;
            bulk_wait_read<1>(); // the store of child c-1 has drained; its stage is rewritten at c+2, one barrier from here
        }
        // no second barrier: the partial words of this stage are reset here and next touched at child c+3, two barriers away
    }
    if (tid < ng) bulk_wait<0>();
}

template <int S, int NT, class F>
int launch_expand(const typename F::T *parents, const uint8_t *tape, int k, typename F::T *children, uint8_t *flags, int32_t *nnz,
                  unsigned long long *keys, long long B, int shift, cudaStream_t st) {
    using C = ExpCfg<S, NT, F>;
    // the records of a CTA must fit shared memory; the bound on k is taken before any size in bytes is formed, which
    // could wrap in int
    if (k > (200 * 1024 - C::smem_bytes(0)) / (C::TG * Geo<S>::TP)) return TG_E_ARG;
    const int smem = C::smem_bytes(k);
    const long long grid = (B + C::TG - 1) / C::TG;
    if (grid > 0x7FFFFFFFLL) return TG_E_ARG;
    if (keys) {
        auto kern = expand_kernel<S, NT, true, F>;
        TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        kern<<<(int)grid, NT, smem, st>>>(parents, tape, k, children, flags, nnz, keys, B, shift);
    } else {
        auto kern = expand_kernel<S, NT, false, F>;
        TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        kern<<<(int)grid, NT, smem, st>>>(parents, tape, k, children, flags, nnz, keys, B, shift);
    }
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}
} // namespace tg
