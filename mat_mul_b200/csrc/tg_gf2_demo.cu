// tg_gf2_demo.cu -- K3 modulo 2: synthetic demonstrations with bit-slab targets (C ABI: tg_demo_gen_gf2,
// tg_demo_alias_tables_gf2).
//
// The sampler is tg_demo.cu's (tg_demo_sampler.cuh) with its mod-2 switch: a factor is conditioned on having an odd
// entry, so no term of a demo vanishes mod 2.  The target is the xor of the R terms; a term needs only the parity masks
// of u, v and w, taken from the token words the sampler just built (parities_of, one multiply per word), and is
//     row_i ^= u_i odd ? V : 0,  V = OR_{j: v_j odd} (w bits) << j S     (the formulation of tg_gf2.cu).
// Nothing is read back: the tape is written once and the bit slab once.
//
// Work split (DemoB):
//   4x4x4, 9x9x9  one thread per demo, the S rows (RW words each) in registers; xor_term applies a term.  Consecutive
//                 threads are consecutive demos, so a step's records leave as one coalesced run.  A 4x4x4 target is one
//                 16-byte store; the 32 targets of a warp at 9x9x9 (3584 contiguous bytes) leave through a warp-private
//                 stage in shared memory.
//   16x16x16, 25x25x25  a group of G lanes per demo (8 / 32); lane c owns word c of every row (c < RW = 8 / 20).  The
//                 lanes draw the demo's terms round-robin, so each triple is drawn once, and hand the three masks of
//                 each term to the group by shuffles; lane c builds only word c of V.
#include "tg_demo_sampler.cuh"
#include "tg_gf2.cuh"

namespace tg {
namespace {

template <int S>
struct DemoB {
    static constexpr int G = S == 16 ? 8 : S == 25 ? 32 : 1; // lanes per demo
    static constexpr int NT = 128;                           // threads per CTA
    static constexpr int DPC = NT / G;                       // demos per CTA
};

// word c of V = OR_{j: v_j odd} w << j S (a word meets at most three runs of S bits at 25, two at 16)
template <int S>
__device__ __forceinline__ uint32_t v_word(uint32_t v, uint32_t w, int c) {
    const int j0 = (32 * c) / S;
    uint32_t V = 0;
#pragma unroll
    for (int t = 0; t < 31 / S + 2; t++) {
        const int j = j0 + t, o = j * S - 32 * c; // bit offset of run j in word c: (-S, 32) when it overlaps
        if (j < S && o < 32) {
            const uint32_t x = w & (0u - ((v >> j) & 1u));
            V |= o >= 0 ? x << o : x >> -o;
        }
    }
    return V;
}

// NTHR = 0: contract v2 mod 2 (alias tables ap); NTHR > 0: contract v1 mod 2 with NTHR thresholds (cat, max_tries);
// BOX: contract box v1 mod 2 (tg_demo_gen_box_gf2), v1 with the factors confined to the box
template <int S, int NTHR, bool BOX = false>
__global__ void __launch_bounds__(128) demo_gen_gf2_kernel(unsigned long long first_demo, long long N, int R, int shift,
                                                           const __grid_constant__ Categorical cat, int max_tries,
                                                           uint8_t *__restrict__ tape, long long tape_step_stride,
                                                           uint32_t *__restrict__ bits, uint8_t *__restrict__ flags,
                                                           const __grid_constant__ AliasDev ap, const __grid_constant__ BoxMasks box) {
    using B = GeoB<S>;
    constexpr int G = DemoB<S>::G, RW = B::RW, GW = B::GB / 4, TW = B::TP / 4, NW = (3 * S + 3) / 4;
    constexpr bool ALIAS = NTHR == 0;
    static_assert(!BOX || !ALIAS, "contract box v1 only");
    __shared__ __align__(16) uint32_t s_alias[ALIAS ? AliasGeo<S>::TAB_WORDS : 4];
    __shared__ __align__(16) uint4 s_stage[B::STAGED ? 4 * 32 * (GW / 4) : 1];
    if constexpr (ALIAS) {
        alias_to_smem<S, 128>(ap, s_alias);
        __syncthreads();
    }
    const int lane = threadIdx.x & 31, c = lane % G;
    const long long nw0 = ((long long)blockIdx.x * 128 + (threadIdx.x & ~31)) / G; // first demo of the warp
    if (nw0 >= N) return;
    const long long n0 = ((long long)blockIdx.x * 128 + threadIdx.x) / G;
    const bool real = n0 < N; // lanes past the end draw demo N-1 again (the shuffles need the whole warp) and store nothing
    const long long n = real ? n0 : N - 1;
    const unsigned long long d = first_demo + (unsigned long long)n;
    const uint32_t d_lo = (uint32_t)d, d_hi = (uint32_t)(d >> 32);
    uint32_t fl = 0;

    // draw term r, write its record to the tape, return its parities
    auto term = [&](int r) -> Par {
        uint32_t words[TW];
#pragma unroll
        for (int w = NW; w < TW; w++) words[w] = 0;
        if constexpr (ALIAS) {
            draw_triple_alias<S, true>(words, d_lo, d_hi, r, ap, s_alias);
        } else {
#pragma unroll 1
            for (int t = 0;; t++) {
                if constexpr (BOX) {
                    if (draw_triple_box<S, NTHR, true>(words, d_lo, d_hi, r, t, cat, box)) break;
                } else {
                    if (draw_triple<S, NTHR, true>(words, d_lo, d_hi, r, t, cat)) break;
                }
                if (t + 1 >= max_tries) { // forced: u = v = w = x e_0, x the last odd value (cat.top_tok is its token)
#pragma unroll
                    for (int w = 0; w < NW; w++) words[w] = 0;
#pragma unroll
                    for (int q = 0; q < 3 * S; q++)
                        words[q >> 2] |= (((q % S) == 0 ? cat.top_tok : (uint32_t)shift) & 0xFFu) << (8 * (q & 3));
                    fl = TG_FLAG_EXHAUSTED;
                    break;
                }
            }
        }
        if (real) {
            uint4 *dst = reinterpret_cast<uint4 *>(tape + (size_t)r * tape_step_stride + n * B::TP);
#pragma unroll
            for (int w = 0; w < TW / 4; w++) dst[w] = make_uint4(words[4 * w], words[4 * w + 1], words[4 * w + 2], words[4 * w + 3]);
        }
        return parities_of<S>(words, shift);
    };

    if constexpr (G == 1) {
        uint32_t row[S][RW];
#pragma unroll
        for (int i = 0; i < S; i++)
#pragma unroll
            for (int w = 0; w < RW; w++) row[i][w] = 0;
#pragma unroll 1
        for (int r = 0; r < R; r++) xor_term<S, S>(row, term(r), 0);
        if constexpr (!B::STAGED) {
            static_assert(S * RW == 4 && GW == 4, "4x4x4: one 16-byte target");
            if (real) *reinterpret_cast<uint4 *>(bits + n * GW) = make_uint4(row[0][0], row[1][0], row[2][0], row[3][0]);
        } else {
            // lane l's target goes to 16-byte chunks l*GW/4 .. of the warp's stage (an odd chunk pitch: no bank
            // conflicts), then the warp copies the contiguous run of its targets
            uint4 *stage = s_stage + (threadIdx.x >> 5) * 32 * (GW / 4);
#pragma unroll
            for (int q = 0; q < GW / 4; q++) {
                uint32_t x[4];
#pragma unroll
                for (int e = 0; e < 4; e++) x[e] = 4 * q + e < S * RW ? row[(4 * q + e) / RW][(4 * q + e) % RW] : 0u;
                stage[lane * (GW / 4) + q] = make_uint4(x[0], x[1], x[2], x[3]);
            }
            __syncwarp();
            const int total = (int)min(32LL, N - nw0) * (GW / 4);
            uint4 *out = reinterpret_cast<uint4 *>(bits + nw0 * GW);
            for (int x = lane; x < total; x += 32) out[x] = stage[x];
        }
        if (flags && real) flags[n] = (uint8_t)fl;
    } else {
        uint32_t row[S]; // word c of every row
#pragma unroll
        for (int i = 0; i < S; i++) row[i] = 0;
#pragma unroll 1
        for (int r0 = 0; r0 < R; r0 += G) {
            Par p = {0u, 0u, 0u};
            if (r0 + c < R) p = term(r0 + c);
            const int nk = min(G, R - r0);
#pragma unroll 1
            for (int k = 0; k < nk; k++) {
                const uint32_t u = __shfl_sync(0xFFFFFFFFu, p.u, k, G), v = __shfl_sync(0xFFFFFFFFu, p.v, k, G),
                               w = __shfl_sync(0xFFFFFFFFu, p.w, k, G);
                const uint32_t V = v_word<S>(v, w, c);
#pragma unroll
                for (int i = 0; i < S; i++) row[i] ^= V & (0u - ((u >> i) & 1u));
            }
        }
        if (real && c < RW) {
            uint32_t *dst = bits + n * GW + c;
#pragma unroll
            for (int i = 0; i < S; i++) dst[i * RW] = row[i];
        }
        uint32_t m = __ballot_sync(0xFFFFFFFFu, fl != 0);
        if constexpr (G < 32) m = (m >> (lane & ~(G - 1))) & ((1u << G) - 1u);
        if (flags && real && c == 0) flags[n] = m ? (uint8_t)TG_FLAG_EXHAUSTED : (uint8_t)0;
    }
}

// contract v1 mod 2's launch constants: a factor is "zero" when every entry is even, and the forced triple is the last odd
// value's.  false for an alphabet the generator refuses (alphabet_ok, or no odd value: no factor could be odd)
inline bool categorical_gf2(const int8_t *values, const double *probs, int n, int shift, uint64_t seed, Categorical &cat) {
    if (!alphabet_ok(values, probs, n, shift)) return false;
    int odd = -1;
    for (int i = 0; i < n; i++)
        if (values[i] & 1) odd = i;
    if (odd < 0) return false;
    cat = categorical(values, probs, n, shift, seed);
    cat.zero_pat = (uint32_t)shift * ONES4;
    cat.top_tok = (uint32_t)(values[odd] + shift) & 0xFFu;
    return true;
}

template <int S, int NTHR, bool BOX = false>
int launch_demo_gen_gf2(unsigned long long first, long long N, int R, int shift, const Categorical &cat, int max_tries, const AliasDev &ap,
                        const BoxMasks &box, uint8_t *tape, long long stride, uint32_t *bits, uint8_t *flags, cudaStream_t st) {
    const long long grid = (N + DemoB<S>::DPC - 1) / DemoB<S>::DPC;
    if (grid > 0x7FFFFFFFLL) return TG_E_ARG;
    demo_gen_gf2_kernel<S, NTHR, BOX><<<(unsigned)grid, DemoB<S>::NT, 0, st>>>(first, N, R, shift, cat, max_tries, tape, stride, bits, flags,
                                                                              ap, box);
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

} // namespace
} // namespace tg

extern "C" {

int tg_demo_gen_gf2(uint64_t seed, uint64_t first_demo, int64_t N, int R, int S, int shift, const int8_t *values,
                    const double *probs, int n_values, int max_tries, uint8_t *tape, int64_t tape_step_stride,
                    uint32_t *bits, uint8_t *flags, void *stream) {
    if (const int rc = tg::check_demo_gen(S, N, R, shift, n_values, max_tries, values, probs, tape, tape_step_stride, bits); rc != tg::LAUNCH)
        return rc;
    tg::Categorical cat;
    if (!tg::categorical_gf2(values, probs, n_values, shift, seed, cat)) return TG_E_ARG;
    static const tg::BoxMasks no_box = {};
    cudaStream_t st = (cudaStream_t)stream;
    tg::AliasDev dev = {};
    const bool alias = tg::alias_applies<true>(values, probs, n_values, S);
    if (alias) {
        tg::AliasParams ap;
        tg::build_alias<true>(values, probs, n_values, S, shift, seed, ap);
        tg::AliasTabs tabs;
        tg::alias_to_dev<true>(ap, values, n_values, S, shift, tabs, dev);
        const int rc = tg::alias_device_tables(tabs, st, &dev.tab);
        if (rc != TG_OK) return rc;
    }
    return tg::with_S(S, [&](auto s) {
        constexpr int kS = decltype(s)::value;
        auto go = [&](auto nthr) {
            return tg::launch_demo_gen_gf2<kS, decltype(nthr)::value>(first_demo, N, R, shift, cat, max_tries, dev, no_box, tape,
                                                                      tape_step_stride, bits, flags, st);
        };
        if constexpr (kS != 25) // contract v2 needs at most six groups per factor
            if (alias) return go(std::integral_constant<int, 0>{});
        if (n_values <= 3) return go(std::integral_constant<int, 2>{});
        if (n_values <= 5) return go(std::integral_constant<int, 4>{});
        return go(std::integral_constant<int, 7>{});
    });
}

int tg_demo_gen_box_gf2(uint64_t seed, uint64_t first_demo, int64_t N, int R, int S, int nu, int nv, int nw, int shift,
                        const int8_t *values, const double *probs, int n_values, int max_tries, uint8_t *tape,
                        int64_t tape_step_stride, uint32_t *bits, uint8_t *flags, void *stream) {
    if (const int rc = tg::check_demo_gen_box(S, N, R, nu, nv, nw, shift, n_values, max_tries, values, probs, tape, tape_step_stride, bits);
        rc != tg::LAUNCH)
        return rc;
    tg::Categorical cat;
    if (!tg::categorical_gf2(values, probs, n_values, shift, seed, cat)) return TG_E_ARG;
    const tg::BoxMasks box = tg::box_masks(S, nu, nv, nw, shift);
    static const tg::AliasDev no_alias = {};
    return tg::with_S(S, [&](auto s) {
        constexpr int kS = decltype(s)::value;
        auto go = [&](auto nthr) {
            return tg::launch_demo_gen_gf2<kS, decltype(nthr)::value, true>(first_demo, N, R, shift, cat, max_tries, no_alias, box, tape,
                                                                            tape_step_stride, bits, flags, (cudaStream_t)stream);
        };
        if (n_values <= 3) return go(std::integral_constant<int, 2>{});
        if (n_values <= 5) return go(std::integral_constant<int, 4>{});
        return go(std::integral_constant<int, 7>{});
    });
}

int tg_demo_alias_tables_gf2(const int8_t *values, const double *probs, int n_values, int S, uint16_t *tables_host) {
    return tg::alias_tables_host<true>(values, probs, n_values, S, tables_host);
}

} // extern "C"
