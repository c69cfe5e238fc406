// tg_demo.cu -- K3: synthetic demonstrations (C ABI: tg_demo_gen_philox,
// tg_demo_accumulate, tg_demo_from_ustream, tg_mt19937_fill_f64).
//
// Reference restated: create_synthetic_demo (utils.py:203-233) ==
// SyntheticDemoDataset._create_synthetic_demos (datasets.py:124-142): R
// accepted random factor triples (rejected iff u(x)v(x)w == 0), tokens =
// factors + shift, target = sum of the R rank-1 tensors.
//
// Device formats: multi-step tape uint8 [R][N][TP] (step-major, so step r of
// all games is one contiguous tg_step operand) and the int8 slab [N][GP].
//
// One CTA builds a tile of TG demos:
//   A. (throughput mode) every lane runs a (pair, try) state machine over the
//      (demo, term) pairs of the tile, claimed from a shared counter one
//      warp-aggregated atomic at a time.  A try is ceil(3S/8) Philox4x32-10
//      blocks (round keys are launch constants); four 15-bit draws are turned
//      into four tokens at once: per CDF threshold two IADDs (carry into bit
//      15 of each 16-bit lane), one PRMT that gathers the four carries as byte
//      masks, one LOP3 that XORs the token delta in.  An accepted triple goes
//      straight to the HBM tape and, as an "accumulate record" (packed w
//      coefficients in integer form + u, v coefficient bytes), to shared memory;
//      (replay modes) the records are built from the tape in HBM instead.
//   B. S threads per demo, thread j owning the entries (i, j, 0..S-1) of every
//      row i in registers as packed words: per term  vw = v_j * pack(w) and
//      acc[i][m] += u_i * vw[m]  -- one IMAD per four entries.  The packed sum is
//      exact modulo 2^32 whatever the intermediate values, so only the FINAL
//      entries matter: with R * shift^3 <= 191 a final entry outside int8
//      always decodes outside [-64, 63] and raises TG_FLAG_RANGE; for larger
//      R * shift^3 a per-thread bound shift^2 * sum_r |v_rj| guards the packed
//      path and the (rare) thread above it recomputes its entries one by one.
//   C. the slab tile leaves through one TMA bulk store.
#include <cstring>
#include <mutex>

#include "tg_demo_mma.cuh"
#include "tg_demo_sampler.cuh"
#include "tg_step.cuh"

namespace tg {

template <int S, int NT, int NPASS = 1>
struct DemoCfg {
    using G = Geo<S>;
    static constexpr int GPASS = NT / S;        // demos per pass of phase B: S threads per demo (thread = factor index j)
    static constexpr int TG = GPASS * NPASS;    // demos per CTA: a bigger tile amortises the tail of the sampling phase
    static constexpr int ACTIVE = GPASS * S;
    static constexpr bool TILE = S != 4;         // 4x4x4 games leave straight from the registers: no slab tile
    static constexpr int KW = (S + 3) / 4;       // packed words per run of S entries (one (i, j), k = 0..S-1)
    static constexpr int NCW = (2 * S + 3) / 4;  // words holding the u and v coefficient bytes
    static constexpr int NW = (3 * S + 3) / 4;   // token words of one action
    static constexpr int REC = G::TP;            // accumulate record: KW words pack(w) + NCW words coefficient bytes
    static_assert(4 * (KW + NCW) <= REC, "record does not fit the token pitch");
    // pitch of a game in the shared-memory tile: padded so that the lanes of neighbouring demos in a warp store to
    // different banks (768 B and 64 B pitches are 0 mod 128 / alias every other demo); each game leaves with its
    // own bulk store
    static constexpr int PITCH = G::GP + (S == 9 ? 32 : (S == 4 ? 16 : 0));
    static constexpr int PASS_SLAB = TILE ? GPASS * PITCH : 0;
    static __host__ __device__ constexpr int rec_bytes(int R) { return R * TG * REC; }
    static __host__ __device__ constexpr int rec_region(int R) { return (rec_bytes(R) + 15) & ~15; } // tensor-core variants: [TG][R][TP]
    // Integer variants: one region per pass of phase B.  It holds the accumulate records of the pass's GPASS demos and,
    // once the pass has consumed them, its part of the slab tile IN THE SAME BYTES (one CTA barrier per pass), so a CTA
    // needs max(records, tile) instead of records + tile: 22.4 instead of 43 KB at 9x9x9, NPASS = 2.
    // 9x9x9: the three pieces a phase-B thread reads per term are arrays of their own, X = {pack(w) x 3, u0..u3} at a pitch of
    // 16 bytes, Y = {u4..u7, u8 v0 v1 v2} at 8 and V = {u8 v0..v2, v3..v6, v7 v8} at 12, so that the records the lanes of a
    // warp gather (every lane walks its own list of terms) spread over 8 / 16 / 32 bank classes instead of the 4 of one 32-byte
    // record (ncu: 7.4 + 6.1 + 3.4 shared-memory wavefronts per warp and term against 2.8 + 1.6 + 1.0 without conflicts)
    static constexpr bool SPLIT = S == 9;
    static constexpr int REC_SMEM = SPLIT ? 36 : REC; // shared-memory bytes of one accumulate record
    static __host__ __device__ constexpr int pass_rec(int R) { return GPASS * R * REC_SMEM; }
    static __host__ __device__ constexpr int pass_stride(int R) { return ((pass_rec(R) > PASS_SLAB ? pass_rec(R) : PASS_SLAB) + 15) & ~15; }
    static __host__ __device__ constexpr int main_bytes(int R) { return NPASS * pass_stride(R); }
    // record of (demo g of the tile, term r): byte offset of its pass region and its index in there
    static __device__ __forceinline__ void rec_pos(int g, int r, int R, int &region, int &k) {
        const int pass = NPASS == 1 ? 0 : g / GPASS;
        region = pass * pass_stride(R), k = (g - pass * GPASS) * R + r;
    }
    static __device__ __forceinline__ int slab_off(int g, int R) { // tile bytes of demo g
        if constexpr (NPASS == 1) return g * PITCH;
        const int pass = g / GPASS;
        return pass * pass_stride(R) + (g - pass * GPASS) * PITCH;
    }
    // regions, per-demo flags, work counter + 2 retry-list counters, 2 retry lists of NT entries
    static constexpr int FLAG_BYTES = ((TG + 3) & ~3) * 4; // per-demo flags, rounded so that what follows stays 16-byte aligned
    static __host__ __device__ constexpr int smem_bytes(int R) { return main_bytes(R) + FLAG_BYTES + 16 + 2 * NT * 4; }
};

// token words of one action -> accumulate record: pack(w) in integer form (sum_b (w_b - shift) 256^b per word,
// bytes beyond S contribute 0) followed by the u, v coefficient bytes (token - shift as int8)
// SMALL: every token is below 128 + shift (sampled tokens are <= 2 * shift): the per-byte subtraction needs no guard bit
template <int S, int NT, int NPASS, bool SMALL>
__device__ __forceinline__ void emit_record(const uint32_t words[(3 * S + 3) / 4], int shift, uint8_t *region, int k, int R) {
    using C = DemoCfg<S, NT, NPASS>;
    constexpr int o = 2 * S;
    constexpr uint32_t WLAST = (S % 4) ? (0xFFFFFFFFu >> (8 * (4 - S % 4))) : 0xFFFFFFFFu;
    const uint32_t sh4 = (uint32_t)shift * ONES4;
    uint32_t out[C::REC / 4];
#pragma unroll
    for (int m = 0; m < C::REC / 4; m++) out[m] = 0;
#pragma unroll
    for (int m = 0; m < C::KW; m++) {
        const uint32_t lo = words[(o >> 2) + m];
        uint32_t wt = lo;
        if constexpr ((o & 3) != 0) {
            const uint32_t hi = ((o >> 2) + m + 1 < C::NW) ? words[(o >> 2) + m + 1] : 0u;
            wt = __funnelshift_r(lo, hi, 8 * (o & 3));
        }
        const uint32_t msk = (m == C::KW - 1) ? WLAST : 0xFFFFFFFFu;
        out[m] = (wt & msk) - (sh4 & msk);
    }
#pragma unroll
    for (int m = 0; m < C::NCW; m++) out[C::KW + m] = SMALL ? (words[m] + (H4 - sh4)) ^ H4 : ((words[m] | H4) - sh4) ^ H4;
    if constexpr (C::SPLIT) {
        static_assert(!C::SPLIT || (C::KW == 3 && C::NCW == 5), "split records: 9x9x9");
        const int n = C::GPASS * R;
        *reinterpret_cast<uint4 *>(region + k * 16) = make_uint4(out[0], out[1], out[2], out[3]);
        *reinterpret_cast<uint2 *>(region + n * 16 + k * 8) = make_uint2(out[4], out[5]);
        uint32_t *v = reinterpret_cast<uint32_t *>(region + n * 24 + k * 12);
        v[0] = out[5], v[1] = out[6], v[2] = out[7];
    } else {
        static_assert(C::REC % 16 == 0, "record pitch");
        uint8_t *rec = region + k * C::REC;
#pragma unroll
        for (int m = 0; m < C::REC / 16; m++)
            reinterpret_cast<uint4 *>(rec)[m] = make_uint4(out[4 * m], out[4 * m + 1], out[4 * m + 2], out[4 * m + 3]);
    }
}

// sign-extended byte b of a coefficient word
template <int B>
__device__ __forceinline__ int coef_byte(uint32_t w) {
    constexpr uint32_t sel = (uint32_t)B | ((uint32_t)(B | 8) << 4) | ((uint32_t)(B | 8) << 8) | ((uint32_t)(B | 8) << 12);
    return (int)prmt(w, 0u, sel);
}

// MMA = 0: phases A, B, C as described above.  MMA = -1: sample only (phase A writes the tape, nothing else).
// MMA = KS > 0 (16x16x16, R <= 16 KS): phase A also leaves the raw 48-byte action records in shared memory and every warp
// then sums the targets of its demos on the tensor cores (tg_demo_mma.cuh) -- CTAs of one SM are in different phases, so
// the sampler's integer work and the MMAs overlap.
// ALIAS: phase A draws under contract v2 (group alias tables, no rejection loop); the categorical thresholds are unused.
// OR_FLAGS (replay only): OR the flags into the caller's (the EXHAUSTED flags of a sampler that ran before) instead of
// overwriting them.
template <int S, int NT, int NPASS, bool SAMPLE, int NTHR, bool GUARD, int MMA = 0, bool ALIAS = false, bool OR_FLAGS = false>
__global__ void __launch_bounds__(NT, S == 16 ? (NT <= 128 ? 4 : 2) : (S == 9 ? (NT == 128 ? 8 : NT == 64 ? 16 : 3) : 4))
    demo_kernel(unsigned long long first_demo, long long N, int R, uint32_t magic_r, int shift,
                const __grid_constant__ Categorical cat, int max_tries, uint8_t *__restrict__ tape,
                long long tape_step_stride, int8_t *__restrict__ slab, uint8_t *__restrict__ flags,
                const __grid_constant__ AliasDev ap) {
    using C = DemoCfg<S, NT, NPASS>;
    using G = Geo<S>;
    static_assert(!OR_FLAGS || (!SAMPLE && MMA == 0), "OR_FLAGS: the replay mode");
    extern __shared__ __align__(128) uint8_t smem[];
    // integer variants: per pass of phase B one region, first the accumulate records [GPASS][R][REC] (phases A, B), then the
    // pass's slab tile [GPASS][PITCH] in the same bytes (C::rec_off / C::slab_off); tensor-core variants: records [TG][R][TP]
    uint8_t *s_rec = smem;
    constexpr int MMA_SCRATCH = MMA > 0 ? (NT / 32) * acc16::WARP_WORDS * 4 : 0; // per-warp H and U2 tables
    uint32_t *s_flag = reinterpret_cast<uint32_t *>(smem + (MMA == 0 ? C::main_bytes(R) : MMA > 0 ? C::rec_region(R) + MMA_SCRATCH : 0)); // [TG]
    uint32_t *s_work = s_flag + C::FLAG_BYTES / 4; // [0] next fresh pair, [1], [2] sizes of the two retry lists
    uint32_t *s_list = s_work + 4;       // [2][NT]  pending (pair | try << 16); ALIAS: the tables live here instead
    uint32_t *s_alias = MMA > 0 ? reinterpret_cast<uint32_t *>(smem + C::rec_region(R)) : s_list; // fused kernels: the (not yet used) MMA scratch

    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const long long g0 = (long long)blockIdx.x * C::TG;
    const int ng = (int)min((long long)C::TG, N - g0);
    const int npairs = ng * R;

    for (int g = tid; g < C::TG; g += NT) s_flag[g] = 0;
    if (tid < 3) s_work[tid] = 0;
    if constexpr (ALIAS) alias_to_smem<S, NT>(ap, s_alias);
    __syncthreads();

    if constexpr (SAMPLE && ALIAS) {
        // ---------------- A (contract v2). every (demo, term) pair is one draw: no tries, no retry lists
        for (int p = tid; p < npairs; p += NT) {
            const int g = magic_r ? (int)__umulhi((uint32_t)p, magic_r) : p; // p / R
            const int r = p - g * R;
            const unsigned long long d = first_demo + (unsigned long long)(g0 + g);
            uint32_t words[G::TP / 4];
#pragma unroll
            for (int w = C::NW; w < G::TP / 4; w++) words[w] = 0;
            draw_triple_alias<S>(words, (uint32_t)d, (uint32_t)(d >> 32), r, ap, s_alias);
            uint4 *dst = reinterpret_cast<uint4 *>(tape + (size_t)r * tape_step_stride + (g0 + g) * G::TP);
#pragma unroll
            for (int w = 0; w < G::TP / 16; w++) dst[w] = make_uint4(words[4 * w], words[4 * w + 1], words[4 * w + 2], words[4 * w + 3]);
            if constexpr (MMA == 0) {
                {
                    int region, k;
                    C::rec_pos(g, r, R, region, k);
                    emit_record<S, NT, NPASS, true>(words, shift, smem + region, k, R);
                }
            } else if constexpr (MMA > 0) {
                uint4 *rdst = reinterpret_cast<uint4 *>(s_rec + ((size_t)g * R + r) * G::TP);
#pragma unroll
                for (int w = 0; w < G::TP / 16; w++) rdst[w] = make_uint4(words[4 * w], words[4 * w + 1], words[4 * w + 2], words[4 * w + 3]);
            }
        }
    } else if constexpr (SAMPLE) {
        // ---------------- A. draw the factor triples of the tile.
        // A1: every lane runs a (pair, try) state machine: a rejected triple just bumps the lane's try, an accepted
        // one is stored and the lane takes the next fresh pair (one atomic per warp and round) -- all 32 lanes draw in
        // every round.  When the fresh pairs run out the warp parks its pending retries in a shared list, and
        // A2: the CTA works the retry lists off densely, 32 retries per warp-round, until none is left.
        auto decode = [&](int p, int &g, int &r, uint32_t &d_lo, uint32_t &d_hi) {
            g = magic_r ? (int)__umulhi((uint32_t)p, magic_r) : p; // p / R  (p * R < 2^32; magic 0 <=> R == 1)
            r = p - g * R;
            const unsigned long long d = first_demo + (unsigned long long)(g0 + g);
            d_lo = (uint32_t)d, d_hi = (uint32_t)(d >> 32);
        };
        // one try of pair (g, r); returns true when the pair is finished (accepted or forced)
        auto attempt = [&](int g, int r, uint32_t d_lo, uint32_t d_hi, int t) -> bool {
            uint32_t words[G::TP / 4];
#pragma unroll
            for (int w = C::NW; w < G::TP / 4; w++) words[w] = 0;
            bool ok = draw_triple<S, NTHR>(words, d_lo, d_hi, r, t, cat);
            if (!ok && t + 1 >= max_tries) { // bounded retries: forced unit triple (the reference would loop forever, Q11)
#pragma unroll
                for (int w = 0; w < C::NW; w++) words[w] = 0;
#pragma unroll
                for (int q = 0; q < 3 * S; q++)
                    words[q >> 2] |= (((q % S) == 0 ? cat.top_tok : (uint32_t)shift) & 0xFFu) << (8 * (q & 3));
                atomicOr(&s_flag[g], (uint32_t)TG_FLAG_EXHAUSTED);
                ok = true;
            }
            if (ok) {
                uint4 *dst = reinterpret_cast<uint4 *>(tape + (size_t)r * tape_step_stride + (g0 + g) * G::TP);
#pragma unroll
                for (int w = 0; w < G::TP / 16; w++)
                    dst[w] = make_uint4(words[4 * w], words[4 * w + 1], words[4 * w + 2], words[4 * w + 3]);
                if constexpr (MMA == 0) {
                    {
                    int region, k;
                    C::rec_pos(g, r, R, region, k);
                    emit_record<S, NT, NPASS, false>(words, shift, smem + region, k, R);
                }
                } else if constexpr (MMA > 0) {
                    uint4 *rdst = reinterpret_cast<uint4 *>(s_rec + ((size_t)g * R + r) * G::TP);
#pragma unroll
                    for (int w = 0; w < G::TP / 16; w++)
                        rdst[w] = make_uint4(words[4 * w], words[4 * w + 1], words[4 * w + 2], words[4 * w + 3]);
                }
            }
            return ok;
        };
        // park (pair | try << 16) of the lanes with `pending` in retry list `which`
        auto park = [&](bool pending, int p, int t, int which) {
            const uint32_t m = __ballot_sync(0xFFFFFFFFu, pending);
            if (m) {
                const int leader = __ffs(m) - 1;
                int base = 0;
                if (lane == leader) base = (int)atomicAdd(&s_work[1 + which], (uint32_t)__popc(m));
                base = __shfl_sync(0xFFFFFFFFu, base, leader);
                if (pending) s_list[which * NT + base + __popc(m & ((1u << lane) - 1u))] = (uint32_t)p | ((uint32_t)t << 16);
            }
        };
        {
            int p = npairs, t = 0, g = 0, r = 0;
            uint32_t d_lo = 0, d_hi = 0;
            bool need = true;
            while (true) {
                const uint32_t m = __ballot_sync(0xFFFFFFFFu, need);
                if (m) {
                    const int leader = __ffs(m) - 1;
                    int base = 0;
                    if (lane == leader) base = (int)atomicAdd(&s_work[0], (uint32_t)__popc(m));
                    base = __shfl_sync(0xFFFFFFFFu, base, leader);
                    if (need) {
                        p = base + __popc(m & ((1u << lane) - 1u));
                        t = 0, need = false;
                        if (p < npairs) decode(p, g, r, d_lo, d_hi);
                    }
                }
                if (__ballot_sync(0xFFFFFFFFu, p >= npairs) != 0) { // fresh pairs ran out for this warp
                    park(p < npairs, p, t, 0);
                    break;
                }
                if (attempt(g, r, d_lo, d_hi, t))
                    need = true;
                else
                    t++;
            }
        }
        __syncthreads();
        for (int cur = 0;; cur ^= 1) {
            const int n = (int)s_work[1 + cur];
            if (n == 0) break;
            __syncthreads(); // everybody has read the size of list cur before anybody refills the other one
            if (tid == 0) s_work[1 + (cur ^ 1)] = 0;
            __syncthreads();
            const bool have = tid < n;
            int p = 0, t = 0, g = 0, r = 0;
            uint32_t d_lo = 0, d_hi = 0;
            bool pending = false;
            if (have) {
                const uint32_t it = s_list[cur * NT + tid];
                p = (int)(it & 0xFFFFu), t = (int)(it >> 16);
                decode(p, g, r, d_lo, d_hi);
                pending = true;
            }
            // up to three tries per round: the rounds (and their CTA barriers) shrink geometrically faster
#pragma unroll 1
            for (int k = 0; k < 3; k++) {
                if (pending) {
                    pending = !attempt(g, r, d_lo, d_hi, t);
                    t++;
                }
                if (__ballot_sync(0xFFFFFFFFu, pending) == 0) break;
            }
            park(pending, p, t, cur ^ 1);
            __syncthreads();
        }
    } else {
        // ---------------- A'. replay: build the records from the tape in HBM
        for (int p = tid; p < npairs; p += NT) {
            const int g = magic_r ? (int)__umulhi((uint32_t)p, magic_r) : p;
            const int r = p - g * R;
            const uint4 *src = reinterpret_cast<const uint4 *>(tape + (size_t)r * tape_step_stride + (g0 + g) * G::TP);
            uint32_t words[G::TP / 4];
#pragma unroll
            for (int w = 0; w < G::TP / 16; w++) {
                const uint4 q = src[w];
                words[4 * w] = q.x, words[4 * w + 1] = q.y, words[4 * w + 2] = q.z, words[4 * w + 3] = q.w;
            }
            {
                    int region, k;
                    C::rec_pos(g, r, R, region, k);
                    emit_record<S, NT, NPASS, false>(words, shift, smem + region, k, R);
                }
        }
    }
    __syncthreads();
    if constexpr (MMA != 0) {
        if constexpr (MMA > 0) {
            static_assert(MMA <= 0 || (S == 16 && G::TP == 48), "tensor-core accumulation: 16x16x16 only");
            const int warp = tid >> 5;
            uint32_t *sH = reinterpret_cast<uint32_t *>(smem + C::rec_region(R)) + warp * acc16::WARP_WORDS, *sU = sH + acc16::H_WORDS;
            for (int g = warp; g < ng; g += NT / 32) {
#pragma unroll
                for (int pass = 0; pass < (MMA + 1) / 2; pass++) {
                    const int r = 32 * pass + lane;
                    if (r < 16 * MMA) {
                        const uint32_t z = (uint32_t)shift * ONES4; // coefficient 0
                        uint4 raw[3] = {make_uint4(z, z, z, z), make_uint4(z, z, z, z), make_uint4(z, z, z, z)};
                        if (r < R) {
                            const uint4 *src = reinterpret_cast<const uint4 *>(s_rec + ((size_t)g * R + r) * G::TP);
                            raw[0] = src[0], raw[1] = src[1], raw[2] = src[2];
                        }
                        acc16::record_to_halves(raw, shift, sH + r * acc16::HP);
                    }
                }
                __syncwarp();
                const bool bad = acc16::gemms_from_halves<MMA>(sH, sU, slab + (g0 + g) * G::GP, lane);
                if (bad && lane == 0) s_flag[g] |= (uint32_t)TG_FLAG_RANGE; // this warp is the only writer of s_flag[g] now
            }
            __syncthreads();
        }
        if (flags)
            for (int gg = tid; gg < ng; gg += NT) flags[g0 + gg] = (uint8_t)s_flag[gg];
        return;
    }

    // ---------------- B. accumulate the R rank-1 terms in registers
    constexpr int KW = C::KW;
    const bool sparse = cat.sparse_terms && R <= 32;
#pragma unroll 1
    for (int pass = 0; pass < NPASS; pass++) {
    int gl = tid / S, j = tid % S; // the thread's row: demo gl of the pass, factor index j
    bool worker = tid < C::ACTIVE && pass * C::GPASS + gl < ng;
    uint32_t tmask = 0; // sparse: the terms r with v_j != 0
    if (sparse) {
        // most coefficients are zero (P(0) = 0.7 in the reference's distributions): a term with v_j = 0 adds nothing to
        // this thread's entries, so every lane walks only ITS non-zero terms (a bit mask over r, built from the v_j
        // bytes of the records): ~7 of 23, the warp as many as its busiest lane (~12).  Measured and not kept: loading the
        // record of the next term before applying the current one (0.792 vs 0.772 ms per 2^20 demos); handing the rows of a
        // pass to the threads in the order of their term counts (counting sort with match.any + shuffles: 25 % fewer loop
        // instructions, but the warp with the long rows keeps the CTA's other warps at the pass barrier: 0.805 vs 0.700 ms)
        if (worker) {
            const uint8_t *region = smem + pass * C::pass_stride(R);
            const int8_t *vb = reinterpret_cast<const int8_t *>(
                C::SPLIT ? region + C::GPASS * R * 24 + gl * R * 12 + 1 + j : region + gl * R * C::REC + 4 * C::KW + S + j);
            uint32_t bit = 1;
#pragma unroll 4
            for (int r = 0; r < R; r++, bit <<= 1)
                if (vb[r * (C::SPLIT ? 12 : C::REC)] != 0) tmask |= bit;
        }
    }
    const int g = pass * C::GPASS + gl;
    // the sums start at 128 per byte: integer form + H4 = offset-binary bytes, which is what the end of the pass wants
    int32_t acc[S][KW];
#pragma unroll
    for (int i = 0; i < S; i++)
#pragma unroll
        for (int m = 0; m < KW; m++) acc[i][m] = (int32_t)H4;
    uint32_t bad = 0;
    if (worker) {
        int bound = 0;
        const uint8_t *region = smem + pass * C::pass_stride(R);
        const int k0 = gl * R, nrec = C::GPASS * R; // index of the demo's first record in the region
        const uint8_t *rec0 = region + k0 * C::REC;                                     // one-piece records
        const int voff = 4 * KW + S + j;                                                // byte offset of v_j in there
        const uint8_t *recx = region + k0 * 16, *recy = region + nrec * 16 + k0 * 8;    // split records (C::SPLIT)
        const int8_t *recv = reinterpret_cast<const int8_t *>(region + nrec * 24 + k0 * 12 + 1 + j);
        auto v_of = [&](int r) -> int { // v_j of term r
            if constexpr (C::SPLIT) return (int)recv[r * 12];
            else return (int)reinterpret_cast<const int8_t *>(rec0 + (size_t)r * C::REC)[voff];
        };
        // one term: acc[i][.] += u_i * (v_j * pack(w))
        auto load_rec = [&](int r, uint32_t (&q)[C::REC / 4], int &vj) {
            if constexpr (C::SPLIT) {
                const uint4 x = *reinterpret_cast<const uint4 *>(recx + r * 16);
                const uint2 y = *reinterpret_cast<const uint2 *>(recy + r * 8);
                q[0] = x.x, q[1] = x.y, q[2] = x.z, q[3] = x.w, q[4] = y.x, q[5] = y.y;
            } else {
                const uint8_t *rec = rec0 + (size_t)r * C::REC;
#pragma unroll
                for (int m = 0; m < C::REC / 16; m++) {
                    const uint4 v4 = reinterpret_cast<const uint4 *>(rec)[m];
                    q[4 * m] = v4.x, q[4 * m + 1] = v4.y, q[4 * m + 2] = v4.z, q[4 * m + 3] = v4.w;
                }
            }
            vj = v_of(r);
        };
        auto apply_rec = [&](const uint32_t (&q)[C::REC / 4], int vj) {
            if constexpr (GUARD) bound += abs(vj);
            int32_t vw[KW];
#pragma unroll
            for (int m = 0; m < KW; m++) vw[m] = vj * (int32_t)q[m];
#pragma unroll
            for (int i = 0; i < S; i++) {
                int ui;
                switch (i & 3) {
                case 0: ui = coef_byte<0>(q[KW + (i >> 2)]); break;
                case 1: ui = coef_byte<1>(q[KW + (i >> 2)]); break;
                case 2: ui = coef_byte<2>(q[KW + (i >> 2)]); break;
                default: ui = coef_byte<3>(q[KW + (i >> 2)]); break;
                }
#pragma unroll
                for (int m = 0; m < KW; m++) acc[i][m] += ui * vw[m];
            }
        };
        if (sparse) {
            while (tmask) {
                uint32_t q[C::REC / 4];
                int vj;
                const int t = 31 - __clz((int)tmask); // the terms in any order: the highest set bit is one FLO
                load_rec(t, q, vj);
                tmask ^= 1u << t;
                apply_rec(q, vj);
            }
        } else {
#pragma unroll 2
            for (int r = 0; r < R; r++) {
                uint32_t q[C::REC / 4];
                int vj;
                load_rec(r, q, vj);
                apply_rec(q, vj);
            }
        }
        if (GUARD && bound * shift * shift > 191) {
            // a final entry might alias inside the packed words: recompute this thread's entries one by one
#pragma unroll
            for (int i = 0; i < S; i++)
#pragma unroll
                for (int m = 0; m < KW; m++) {
                    uint32_t word = 0;
#pragma unroll 1
                    for (int kk = 0; kk < 4; kk++) {
                        const int k = 4 * m + kk;
                        if (k >= S) break;
                        int e = 0;
#pragma unroll 1
                        for (int r = 0; r < R; r++) {
                            uint32_t q[C::REC / 4];
                            int vj;
                            load_rec(r, q, vj);
                            const uint32_t wb = (q[m] + H4) ^ H4; // integer form -> bytes
                            const int ui = (int)(int8_t)((q[KW + (i >> 2)] >> (8 * (i & 3))) & 0xFFu);
                            e += ui * vj * (int)(int8_t)((wb >> (8 * kk)) & 0xFFu);
                        }
                        if (e < -64 || e > 63) bad = 1;
                        word |= ((uint32_t)e & 0xFFu) << (8 * kk);
                    }
                    acc[i][m] = (int32_t)word;
                }
        } else {
            // offset-binary byte b holds entry + 128: in [-64, 63] <=> bits 7 and 6 differ (padding bytes hold 128: fine);
            // one LOP3 per word keeps the AND of (bit 7 ^ bit 6) over all bytes, another turns the word into two's complement
            uint32_t ok = H4;
#pragma unroll
            for (int i = 0; i < S; i++)
#pragma unroll
                for (int m = 0; m < KW; m++) {
                    const uint32_t o = (uint32_t)acc[i][m];
                    ok &= o ^ (o << 1);
                    acc[i][m] = (int32_t)(o ^ H4);
                }
            bad = ~ok & H4;
        }
    }
    if constexpr (C::TILE) __syncthreads(); // every record of the pass has been consumed: its slab tile takes over the same bytes
    if constexpr (S == 4) {
        // 4x4x4: a game is 64 bytes and thread j holds one aligned word of each of its four rows: straight to HBM (the four
        // threads of a game fill 16 contiguous bytes per store; a bulk store per 64-byte game costs ~10 warp-instructions)
        if (worker) {
            uint32_t *gdst = reinterpret_cast<uint32_t *>(slab + (g0 + g) * G::GP) + j;
#pragma unroll
            for (int i = 0; i < S; i++) gdst[i * (G::RP / 4)] = (uint32_t)acc[i][0];
            if (bad) atomicOr(&s_flag[g], (uint32_t)TG_FLAG_RANGE);
        }
    } else if (worker) {
        // registers -> slab tile: entry (i, j, k) is byte i*RP + j*S + k; the last j also zeroes the row padding,
        // j = 0 the game padding
        uint8_t *gbase = smem + pass * C::pass_stride(R) + gl * C::PITCH + j * S;
#pragma unroll
        for (int i = 0; i < S; i++) {
            if constexpr (S == 9) {
                // the 9-byte run starts at byte 9j of the row: parity j & 1.  Four aligned halfwords (bytes sj .. sj+7 of the
                // run, funnel-shifted into place) and one single byte (the first for odd j, the last for even j) instead of
                // nine byte stores
                const int sj = j & 1;
                const uint32_t w0 = (uint32_t)acc[i][0], w1 = (uint32_t)acc[i][1], w2 = (uint32_t)acc[i][2];
                const uint32_t x0 = __funnelshift_r(w0, w1, 8 * sj), x1 = __funnelshift_r(w1, w2, 8 * sj);
                uint8_t *rowp = gbase + i * G::RP;
                uint16_t *hp = reinterpret_cast<uint16_t *>(rowp + sj);
                hp[0] = (uint16_t)x0, hp[1] = (uint16_t)(x0 >> 16), hp[2] = (uint16_t)x1, hp[3] = (uint16_t)(x1 >> 16);
                rowp[sj ? 0 : 8] = (uint8_t)(sj ? w0 : w2);
            } else {
#pragma unroll
                for (int m = 0; m < KW; m++) {
                    const uint32_t t = (uint32_t)acc[i][m];
                    if constexpr (S % 4 == 0) {
                        reinterpret_cast<uint32_t *>(gbase + i * G::RP)[m] = t;
                    } else {
#pragma unroll
                        for (int k = 4 * m; k < S && k < 4 * m + 4; k++) gbase[i * G::RP + k] = (uint8_t)(t >> (8 * (k & 3)));
                    }
                }
            }
            if constexpr (G::RP != G::S2) {
                if (j == S - 1)
#pragma unroll
                    for (int x = S; x < S + G::RP - G::S2; x++) gbase[i * G::RP + x] = 0;
            }
        }
        if constexpr (G::GP != S * G::RP) {
            if (j == 0)
#pragma unroll
                for (int x = S * G::RP; x < G::GP; x += 4) *reinterpret_cast<uint32_t *>(gbase + x) = 0u;
        }
        if (bad) atomicOr(&s_flag[g], (uint32_t)TG_FLAG_RANGE);
    }
    } // pass
    fence_proxy_async();
    __syncthreads();

    // ---------------- C. tile out: one bulk store per game (S = 4 wrote its games from registers)
    if constexpr (S != 4) {
        for (int gg = tid; gg < ng; gg += NT) bulk_s2g(slab + (g0 + gg) * G::GP, smem + C::slab_off(gg, R), (uint32_t)G::GP);
        if (tid < ng) bulk_commit();
    }
    if (flags)
        for (int gg = tid; gg < ng; gg += NT) flags[g0 + gg] = (uint8_t)(OR_FLAGS ? flags[g0 + gg] | s_flag[gg] : s_flag[gg]);
    if constexpr (S != 4) {
        if (tid < ng) bulk_wait<0>();
    }
}

template <int S, int NT, int NPASS, bool SAMPLE, int NTHR, bool OR_FLAGS = false>
static int launch_demo(unsigned long long first, long long N, int R, int shift, const Categorical &cat, int max_tries,
                       uint8_t *tape, long long stride, int8_t *slab, uint8_t *flags, cudaStream_t st) {
    using C = DemoCfg<S, NT, NPASS>;
    const int smem = C::smem_bytes(R);
    if (smem > 227 * 1024 || R > 65535 || (long long)C::TG * R >= (1LL << 16)) return TG_E_ARG;
    const bool guard = (long long)R * shift * shift * shift > 191;
    const uint32_t magic = R == 1 ? 0u : (uint32_t)((0x100000000ULL + (unsigned)R - 1) / (unsigned)R); // ceil(2^32 / R)
    const long long grid = (N + C::TG - 1) / C::TG;
    if (grid > 0x7FFFFFFFLL) return TG_E_ARG;
    static const AliasDev no_alias = {};
    if (guard) {
        auto kern = demo_kernel<S, NT, NPASS, SAMPLE, NTHR, true, 0, false, OR_FLAGS>;
        TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        kern<<<(int)grid, NT, smem, st>>>(first, N, R, magic, shift, cat, max_tries, tape, stride, slab, flags, no_alias);
    } else {
        auto kern = demo_kernel<S, NT, NPASS, SAMPLE, NTHR, false, 0, false, OR_FLAGS>;
        TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        kern<<<(int)grid, NT, smem, st>>>(first, N, R, magic, shift, cat, max_tries, tape, stride, slab, flags, no_alias);
    }
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

// 16x16x16, R <= 64: sampling fused with the tensor-core accumulation (KS = K-steps of 16 actions), or sampling only
template <int NTHR, int NT, int NPASS, int MMA>
static int launch_demo16_mma(unsigned long long first, long long N, int R, int shift, const Categorical &cat, int max_tries,
                             uint8_t *tape, long long stride, int8_t *slab, uint8_t *flags, cudaStream_t st) {
    using C = DemoCfg<16, NT, NPASS>;
    const int smem = (MMA > 0 ? C::rec_region(R) + (NT / 32) * acc16::WARP_WORDS * 4 : 0) + C::FLAG_BYTES + 16 + 2 * NT * 4;
    if (smem > 227 * 1024 || R > 65535 || (long long)C::TG * R >= (1LL << 16)) return TG_E_ARG;
    const uint32_t magic = R == 1 ? 0u : (uint32_t)((0x100000000ULL + (unsigned)R - 1) / (unsigned)R);
    const long long grid = (N + C::TG - 1) / C::TG;
    if (grid > 0x7FFFFFFFLL) return TG_E_ARG;
    static const AliasDev no_alias = {};
    auto kern = demo_kernel<16, NT, NPASS, true, NTHR, false, MMA>;
    TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    kern<<<(int)grid, NT, smem, st>>>(first, N, R, magic, shift, cat, max_tries, tape, stride, slab, flags, no_alias);
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

// ---- contract v2 launches (the measured-best tile shapes of each size, phase A on the alias tables)
template <int S, int NT, int NPASS, int MMA>
static int launch_demo_alias(unsigned long long first, long long N, int R, int shift, const Categorical &cat, const AliasDev &ap,
                             uint8_t *tape, long long stride, int8_t *slab, uint8_t *flags, cudaStream_t st) {
    using C = DemoCfg<S, NT, NPASS>;
    constexpr int TAIL = MMA > 0 ? 2 * NT * 4 : (2 * NT * 4 > AliasGeo<S>::SMEM_BYTES ? 2 * NT * 4 : AliasGeo<S>::SMEM_BYTES);
    static_assert(MMA <= 0 || AliasGeo<S>::SMEM_BYTES <= acc16::WARP_WORDS * 4, "the alias tables overlay one warp's MMA scratch");
    const int smem = (MMA > 0 ? C::rec_region(R) + (NT / 32) * acc16::WARP_WORDS * 4 : C::main_bytes(R)) + C::FLAG_BYTES + 16 + TAIL;
    if (smem > 227 * 1024 || R > 65535 || (long long)C::TG * R >= (1LL << 16)) return TG_E_ARG;
    const uint32_t magic = R == 1 ? 0u : (uint32_t)((0x100000000ULL + (unsigned)R - 1) / (unsigned)R);
    const long long grid = (N + C::TG - 1) / C::TG;
    if (grid > 0x7FFFFFFFLL) return TG_E_ARG;
    const bool guard = MMA == 0 && (long long)R * shift * shift * shift > 191;
    if (guard) {
        auto kern = demo_kernel<S, NT, NPASS, true, 2, true, MMA, true>;
        TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        kern<<<(int)grid, NT, smem, st>>>(first, N, R, magic, shift, cat, 1, tape, stride, slab, flags, ap);
    } else {
        auto kern = demo_kernel<S, NT, NPASS, true, 2, false, MMA, true>;
        TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        kern<<<(int)grid, NT, smem, st>>>(first, N, R, magic, shift, cat, 1, tape, stride, slab, flags, ap);
    }
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

// ---- 4x4x4, contract v2: one THREAD per demo.  A 4x4x4 target is 16 words: it stays in the registers of the thread that
// draws the demo's R triples one after the other (one Philox block and six table loads each) -- a term is written to the
// tape with one coalesced 16-byte store (consecutive threads, consecutive demos of the step-major tape) and added with four
// products v_j pack(w) and sixteen IMADs; no accumulate records in shared memory, no CTA barrier after the table copy.  The
// 32 targets of a warp are one contiguous block of the slab: they leave through a warp-private stage so that a store
// instruction writes 512 contiguous bytes.  Taken when R * shift^3 <= 191 (a final entry outside int8 then always decodes
// outside [-64, 63]); larger R keeps the guarded tile kernel.
// SAMPLE = false (tg_demo_accumulate): the records come from the tape instead (any token: the guarded coefficient form);
// OR_FLAGS: OR the RANGE flags into the caller's, as demo_kernel does.
template <bool SAMPLE, bool OR_FLAGS = false>
__global__ void __launch_bounds__(128)
    demo4_thread_kernel(unsigned long long first_demo, long long N, int R, int shift, uint8_t *__restrict__ tape, long long tape_step_stride,
                        int8_t *__restrict__ slab, uint8_t *__restrict__ flags, const __grid_constant__ AliasDev ap) {
    constexpr int S = 4, PITCH = 64 + 16;
    __shared__ __align__(16) uint32_t s_alias[SAMPLE ? AliasGeo<S>::TAB_WORDS : 4];
    __shared__ __align__(16) uint8_t s_stage[4][32 * PITCH];
    if constexpr (SAMPLE) {
        alias_to_smem<S, 128>(ap, s_alias);
        __syncthreads();
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long nw0 = (long long)blockIdx.x * 128 + warp * 32; // first demo of the warp
    if (nw0 >= N) return;
    const bool real = nw0 + lane < N;
    const long long n = min(nw0 + lane, N - 1);
    const unsigned long long d = first_demo + (unsigned long long)n;
    uint32_t acc[16]; // word 4 i + j = entries (i, j, 0..3), offset-binary
#pragma unroll
    for (int e = 0; e < 16; e++) acc[e] = H4;
    const uint32_t sh4 = (uint32_t)shift * ONES4;
    uint4 *rec = reinterpret_cast<uint4 *>(tape + n * 16);
    const long long stride16 = tape_step_stride / 16;
    uint4 nextq = (!SAMPLE && R > 0) ? __ldg(reinterpret_cast<const uint4 *>(rec)) : make_uint4(0, 0, 0, 0);
    for (int r = 0; r < R; r++) {
        uint32_t words[3];
        uint32_t cu, cv;
        if constexpr (SAMPLE) {
            draw_triple_alias<S>(words, (uint32_t)d, (uint32_t)(d >> 32), r, ap, s_alias);
            if (real) rec[(long long)r * stride16] = make_uint4(words[0], words[1], words[2], 0u);
            cu = (words[0] + (H4 - sh4)) ^ H4, cv = (words[1] + (H4 - sh4)) ^ H4; // int8 coefficients (tokens <= 2 shift)
        } else {
            words[0] = nextq.x, words[1] = nextq.y, words[2] = nextq.z;
            if (r + 1 < R) nextq = __ldg(reinterpret_cast<const uint4 *>(rec) + (long long)(r + 1) * stride16); // next record in flight
            cu = ((words[0] | H4) - sh4) ^ H4, cv = ((words[1] | H4) - sh4) ^ H4;
        }
        const int wi = (int)(words[2] - sh4); // integer form of pack(w)
        const int vw[4] = {coef_byte<0>(cv) * wi, coef_byte<1>(cv) * wi, coef_byte<2>(cv) * wi, coef_byte<3>(cv) * wi};
        const int u[4] = {coef_byte<0>(cu), coef_byte<1>(cu), coef_byte<2>(cu), coef_byte<3>(cu)};
#pragma unroll
        for (int i = 0; i < 4; i++)
#pragma unroll
            for (int j = 0; j < 4; j++) acc[4 * i + j] += (uint32_t)(u[i] * vw[j]);
    }
    // offset-binary byte in [-64, 63] + 128 <=> bits 7 and 6 differ
    uint32_t ok = H4;
    uint4 *mine = reinterpret_cast<uint4 *>(s_stage[warp] + lane * PITCH);
#pragma unroll
    for (int i = 0; i < 4; i++) {
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const uint32_t o = acc[4 * i + j];
            ok &= o ^ (o << 1);
            acc[4 * i + j] = o ^ H4;
        }
        mine[i] = make_uint4(acc[4 * i], acc[4 * i + 1], acc[4 * i + 2], acc[4 * i + 3]);
    }
    if (flags && real) flags[n] = (uint8_t)((OR_FLAGS ? flags[n] : 0) | ((~ok & H4) ? TG_FLAG_RANGE : 0));
    __syncwarp();
    const int total = (int)min(32LL, N - nw0) * 4;
    uint4 *out = reinterpret_cast<uint4 *>(slab + nw0 * 64);
    for (int x = lane; x < total; x += 32) out[x] = *reinterpret_cast<const uint4 *>(s_stage[warp] + (x >> 2) * PITCH + (x & 3) * 16);
}

static int dispatch_demo_alias(unsigned long long first, long long N, int R, int S, int shift, const Categorical &cat,
                               const AliasDev &ap, uint8_t *tape, long long stride, int8_t *slab, uint8_t *flags, cudaStream_t st) {
    switch (S) {
    case 4:
#ifdef TG_TUNING
        if (tuning_env("TG_DEMO_VARIANT", 0) == 0)
#endif
        if ((long long)R * shift * shift * shift <= 191 && R <= 65535) { // one thread per demo
            const long long grid = (N + 127) / 128;
            if (grid > 0x7FFFFFFFLL) return TG_E_ARG;
            demo4_thread_kernel<true><<<(int)grid, 128, 0, st>>>(first, N, R, shift, tape, stride, slab, flags, ap);
            TG_CUDA(cudaGetLastError());
            return TG_OK;
        }
        if (DemoCfg<4, 256, 4>::smem_bytes(R) <= 160 * 1024)
            return launch_demo_alias<4, 256, 4, 0>(first, N, R, shift, cat, ap, tape, stride, slab, flags, st);
        return launch_demo_alias<4, 256, 1, 0>(first, N, R, shift, cat, ap, tape, stride, slab, flags, st);
    case 9:
#ifdef TG_TUNING
        switch (tuning_env("TG_DEMO_VARIANT", 0)) {
        case 1: return launch_demo_alias<9, 256, 1, 0>(first, N, R, shift, cat, ap, tape, stride, slab, flags, st);
        case 2: return launch_demo_alias<9, 128, 1, 0>(first, N, R, shift, cat, ap, tape, stride, slab, flags, st);
        case 3: return launch_demo_alias<9, 256, 2, 0>(first, N, R, shift, cat, ap, tape, stride, slab, flags, st);
        case 4: return launch_demo_alias<9, 64, 2, 0>(first, N, R, shift, cat, ap, tape, stride, slab, flags, st);
        case 5: return launch_demo_alias<9, 64, 1, 0>(first, N, R, shift, cat, ap, tape, stride, slab, flags, st);
        default: break;
        }
#endif
        return launch_demo_alias<9, 128, 2, 0>(first, N, R, shift, cat, ap, tape, stride, slab, flags, st);
    case 16:
        if (demo_acc16_mma_applies(R)) {
            if (R <= 32) return launch_demo_alias<16, 128, 2, 2>(first, N, R, shift, cat, ap, tape, stride, slab, flags, st);
            return launch_demo_alias<16, 128, 2, 4>(first, N, R, shift, cat, ap, tape, stride, slab, flags, st);
        }
        return launch_demo_alias<16, 128, 1, 0>(first, N, R, shift, cat, ap, tape, stride, slab, flags, st);
    }
    return TG_E_ARG;
}

// ---- the per-device cache of device-format tables (tg_demo_sampler.cuh), in static device memory: the library still
// allocates nothing
constexpr int ALIAS_SLOTS = 8, ALIAS_MAXDEV = 64;
__device__ __align__(16) uint32_t g_alias_tab[ALIAS_SLOTS][8 * ALIAS_BUCKETS];
__global__ void alias_upload_kernel(const __grid_constant__ AliasTabs t, int slot) {
    for (int w = threadIdx.x; w < 8 * ALIAS_BUCKETS; w += blockDim.x) g_alias_tab[slot][w] = (&t.tab[0][0])[w];
}
struct AliasSlot {
    bool valid = false;
    AliasTabs host;
    cudaEvent_t ready = nullptr;
    unsigned long long stamp = 0;
};
static AliasSlot g_alias_slots[ALIAS_MAXDEV][ALIAS_SLOTS];
static std::mutex g_alias_mu;
static unsigned long long g_alias_stamp = 0;

int alias_device_tables(const AliasTabs &want, cudaStream_t st, const uint32_t **dptr) {
    int dev = 0;
    TG_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= ALIAS_MAXDEV) return TG_E_ARG;
    uint32_t *base = nullptr;
    TG_CUDA(cudaGetSymbolAddress(reinterpret_cast<void **>(&base), g_alias_tab));
    std::lock_guard<std::mutex> lock(g_alias_mu);
    AliasSlot *slots = g_alias_slots[dev];
    int hit = -1, lru = -1; // lru: the first free slot, else the least recently used one
    for (int i = 0; i < ALIAS_SLOTS; i++) {
        if (slots[i].valid && memcmp(&slots[i].host, &want, sizeof(AliasTabs)) == 0) hit = i;
        if (lru < 0 || (slots[lru].valid && (!slots[i].valid || slots[i].stamp < slots[lru].stamp))) lru = i;
    }
    if (hit < 0) {
        AliasSlot &sl = slots[lru];
        if (sl.valid) TG_CUDA(cudaDeviceSynchronize()); // eviction: nobody may still be reading the old tables
        if (!sl.ready) TG_CUDA(cudaEventCreateWithFlags(&sl.ready, cudaEventDisableTiming));
        sl.valid = false;
        alias_upload_kernel<<<1, 256, 0, st>>>(want, lru);
        TG_CUDA(cudaGetLastError());
        TG_CUDA(cudaEventRecord(sl.ready, st));
        sl.host = want, sl.valid = true;
        hit = lru;
    } else {
        TG_CUDA(cudaStreamWaitEvent(st, slots[hit].ready, 0));
    }
    slots[hit].stamp = ++g_alias_stamp;
    *dptr = base + (size_t)hit * 8 * ALIAS_BUCKETS;
    return TG_OK;
}

template <int NTHR>
static int dispatch_demo16_mma(unsigned long long first, long long N, int R, int shift, const Categorical &cat, int max_tries,
                               uint8_t *tape, long long stride, int8_t *slab, uint8_t *flags, cudaStream_t st) {
#ifdef TG_TUNING
    static const int variant = tuning_env("TG_DEMO_VARIANT", 0);
    if (variant == 9) { // two kernels: sample, then sum from the tape
        const int rc = launch_demo16_mma<NTHR, 128, 4, -1>(first, N, R, shift, cat, max_tries, tape, stride, nullptr, flags, st);
        return rc != TG_OK ? rc : launch_demo_acc16_mma(tape, stride, N, R, shift, slab, flags, 1, st);
    }
    if (variant == 8) return launch_demo16_mma<NTHR, 128, 1, 4>(first, N, R, shift, cat, max_tries, tape, stride, slab, flags, st);
#endif
    if (R <= 32) return launch_demo16_mma<NTHR, 128, 2, 2>(first, N, R, shift, cat, max_tries, tape, stride, slab, flags, st);
    // measured (profiles/README.md): 16-demo tiles 0.504 ms per 2^17 demos, 8-demo tiles 0.535, 256-thread CTAs 0.534
    return launch_demo16_mma<NTHR, 128, 2, 4>(first, N, R, shift, cat, max_tries, tape, stride, slab, flags, st);
}

// ---- 25x25x25.  Phase B of demo_kernel (thread j holds the S x KW packed words of its runs (i, j, .)) would need 175
// accumulator registers here.  Instead the sampler runs alone (MMA = -1: phase A writes the tape and the EXHAUSTED flags)
// and demo_acc_cols_kernel sums the targets from the tape: thread (demo, word column c) holds the four entries
// (i, 4c .. 4c+3) of every row as plain int32 (100 registers, exact for any tape), the CTA stages its demo's R records in
// shared memory first.  Stored bytes are the entries modulo 256 and TG_FLAG_RANGE marks an entry outside [-64, 63] -- the
// contract of the packed kernels.  or_flags: OR into flags (after the sampler) instead of overwriting them.
template <int S>
__global__ void __launch_bounds__(160)
    demo_acc_cols_kernel(const uint8_t *__restrict__ tape, long long tape_step_stride, long long N, int R, int shift,
                         int8_t *__restrict__ slab, uint8_t *__restrict__ flags, int or_flags) {
    using G = Geo<S>;
    static_assert(G::WR <= 160, "one demo per CTA");
    extern __shared__ __align__(16) uint8_t s_tok[]; // [R][TP]
    __shared__ uint32_t s_bad;
    const int tid = threadIdx.x;
    const long long n = blockIdx.x;
    if (tid == 0) s_bad = 0;
    for (int w = tid; w < R * (G::TP / 16); w += 160) {
        const int r = w / (G::TP / 16), q = w - r * (G::TP / 16);
        reinterpret_cast<uint4 *>(s_tok)[w] = __ldg(reinterpret_cast<const uint4 *>(tape + (size_t)r * tape_step_stride + n * G::TP) + q);
    }
    __syncthreads();
    if (tid < G::WR) {
        Lane<S> L;
        L.init(tid);
        int acc[S][4];
#pragma unroll
        for (int i = 0; i < S; i++)
#pragma unroll
            for (int q = 0; q < 4; q++) acc[i][q] = 0;
#pragma unroll 1
        for (int r = 0; r < R; r++) {
            const uint8_t *tok = s_tok + (size_t)r * G::TP;
            const int vA = (int)tok[L.off_vA] - shift, vB = (int)tok[L.off_vB] - shift;
            int vw[4];
#pragma unroll
            for (int b = 0; b < 4; b++) {
                const bool inA = (L.maskA >> (8 * b)) & 1u, inB = (L.maskB >> (8 * b)) & 1u;
                vw[b] = inA ? vA * ((int)tok[L.off_w[b]] - shift) : (inB ? vB * ((int)tok[L.off_w[b]] - shift) : 0);
            }
#pragma unroll
            for (int i = 0; i < S; i++) {
                const int u = (int)tok[i] - shift;
#pragma unroll
                for (int q = 0; q < 4; q++) acc[i][q] += u * vw[q];
            }
        }
        bool bad = false;
        uint32_t *dst = reinterpret_cast<uint32_t *>(slab + n * G::GP) + L.c;
#pragma unroll
        for (int i = 0; i < S; i++) {
            uint32_t word = 0;
#pragma unroll
            for (int q = 0; q < 4; q++) {
                bad |= acc[i][q] < -64 || acc[i][q] > 63;
                word |= ((uint32_t)acc[i][q] & 0xFFu) << (8 * q);
            }
            dst[i * G::WR] = word;
        }
        if constexpr (G::GP != S * G::RP) {
            if (L.c == 0)
                for (int x = S * G::RP; x < G::GP; x += 4) *reinterpret_cast<uint32_t *>(slab + n * G::GP + x) = 0u;
        }
        if (bad) atomicOr(&s_bad, (uint32_t)TG_FLAG_RANGE);
    }
    __syncthreads();
    if (flags && tid == 0) flags[n] = (uint8_t)((or_flags ? flags[n] : 0) | s_bad);
}

template <int S>
static int launch_demo_acc_cols(const uint8_t *tape, long long stride, long long N, int R, int shift, int8_t *slab, uint8_t *flags,
                                int or_flags, cudaStream_t st) {
    const long long smem = (long long)R * Geo<S>::TP;
    if (smem > 227 * 1024 || N > 0x7FFFFFFFLL) return TG_E_ARG;
    auto kern = demo_acc_cols_kernel<S>;
    TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<(unsigned)N, 160, (size_t)smem, st>>>(tape, stride, N, R, shift, slab, flags, or_flags);
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

// 25x25x25 throughput mode (contract v1): the sampler alone, then the column sum from the tape
template <int NTHR>
static int launch_demo25(unsigned long long first, long long N, int R, int shift, const Categorical &cat, int max_tries, uint8_t *tape,
                         long long stride, int8_t *slab, uint8_t *flags, cudaStream_t st) {
    constexpr int NT = 128;
    using C = DemoCfg<25, NT, 1>;
    const int smem = C::FLAG_BYTES + 16 + 2 * NT * 4;
    if (R > 65535 || (long long)C::TG * R >= (1LL << 16)) return TG_E_ARG;
    const uint32_t magic = R == 1 ? 0u : (uint32_t)((0x100000000ULL + (unsigned)R - 1) / (unsigned)R);
    const long long grid = (N + C::TG - 1) / C::TG;
    if (grid > 0x7FFFFFFFLL) return TG_E_ARG;
    static const AliasDev no_alias = {};
    demo_kernel<25, NT, 1, true, NTHR, false, -1><<<(int)grid, NT, smem, st>>>(first, N, R, magic, shift, cat, max_tries, tape, stride,
                                                                              nullptr, flags, no_alias);
    TG_CUDA(cudaGetLastError());
    return launch_demo_acc_cols<25>(tape, stride, N, R, shift, slab, flags, 1, st);
}

template <bool SAMPLE, int NTHR, bool OR_FLAGS = false>
static int dispatch_demo(unsigned long long first, long long N, int R, int S, int shift, const Categorical &cat,
                         int max_tries, uint8_t *tape, long long stride, int8_t *slab, uint8_t *flags, cudaStream_t st) {
    switch (S) {
    case 4: { // big tiles (several passes of phase B) amortise the retry tail of the sampler; long action lists fall back
#ifdef TG_TUNING
        static const int variant = tuning_env("TG_DEMO_VARIANT", 0);
        if (variant == 1 && DemoCfg<4, 128, 8>::smem_bytes(R) <= 160 * 1024)
            return launch_demo<4, 128, 8, SAMPLE, NTHR, OR_FLAGS>(first, N, R, shift, cat, max_tries, tape, stride, slab, flags, st);
        if (variant == 2 && DemoCfg<4, 128, 4>::smem_bytes(R) <= 160 * 1024)
            return launch_demo<4, 128, 4, SAMPLE, NTHR, OR_FLAGS>(first, N, R, shift, cat, max_tries, tape, stride, slab, flags, st);
        if (variant == 3 && DemoCfg<4, 512, 2>::smem_bytes(R) <= 160 * 1024)
            return launch_demo<4, 512, 2, SAMPLE, NTHR, OR_FLAGS>(first, N, R, shift, cat, max_tries, tape, stride, slab, flags, st);
#endif
        if (DemoCfg<4, 256, 4>::smem_bytes(R) <= 160 * 1024)
            return launch_demo<4, 256, 4, SAMPLE, NTHR, OR_FLAGS>(first, N, R, shift, cat, max_tries, tape, stride, slab, flags, st);
        return launch_demo<4, 256, 1, SAMPLE, NTHR, OR_FLAGS>(first, N, R, shift, cat, max_tries, tape, stride, slab, flags, st);
    }
    case 9: {
#ifdef TG_TUNING
        switch (tuning_env("TG_DEMO_VARIANT", 0)) {
        case 1: return launch_demo<9, 256, 1, SAMPLE, NTHR, OR_FLAGS>(first, N, R, shift, cat, max_tries, tape, stride, slab, flags, st);
        case 3: return launch_demo<9, 128, 3, SAMPLE, NTHR, OR_FLAGS>(first, N, R, shift, cat, max_tries, tape, stride, slab, flags, st);
        case 4: return launch_demo<9, 192, 2, SAMPLE, NTHR, OR_FLAGS>(first, N, R, shift, cat, max_tries, tape, stride, slab, flags, st);
        case 5: return launch_demo<9, 64, 4, SAMPLE, NTHR, OR_FLAGS>(first, N, R, shift, cat, max_tries, tape, stride, slab, flags, st);
        default: break;
        }
#endif
        // measured best (profiles/README.md): 128-thread CTAs; 28-demo tiles when sampling, 14-demo tiles (slab tile
        // overlaid on the records) when only accumulating
        if (SAMPLE) return launch_demo<9, 128, 2, SAMPLE, NTHR, OR_FLAGS>(first, N, R, shift, cat, max_tries, tape, stride, slab, flags, st);
        return launch_demo<9, 128, 1, SAMPLE, NTHR, OR_FLAGS>(first, N, R, shift, cat, max_tries, tape, stride, slab, flags, st);
    }
    case 16: {
#ifdef TG_TUNING
        static const int variant = tuning_env("TG_DEMO_VARIANT", 0);
        if (variant == 1) return launch_demo<16, 256, 1, SAMPLE, NTHR, OR_FLAGS>(first, N, R, shift, cat, max_tries, tape, stride, slab, flags, st);
        if (variant == 2) return launch_demo<16, 64, 1, SAMPLE, NTHR, OR_FLAGS>(first, N, R, shift, cat, max_tries, tape, stride, slab, flags, st);
        if (variant == 3) return launch_demo<16, 128, 2, SAMPLE, NTHR, OR_FLAGS>(first, N, R, shift, cat, max_tries, tape, stride, slab, flags, st);
#endif
        return launch_demo<16, 128, 1, SAMPLE, NTHR, OR_FLAGS>(first, N, R, shift, cat, max_tries, tape, stride, slab, flags, st); // measured best
    }
    }
    return TG_E_ARG;
}

// tg_demo_accumulate's choice of sum for (S, R, shift).  OR_FLAGS: OR the flags into the caller's (tg_demo_gen_box, after
// its sampler wrote the EXHAUSTED flags) instead of overwriting them.
template <bool OR_FLAGS>
static int accumulate(const uint8_t *tape, long long stride, long long N, int R, int S, int shift, int8_t *slab, uint8_t *flags,
                      cudaStream_t st) {
    // 16x16x16: tensor cores (tg_demo_mma.cu); TG_DEMO_MMA=0 keeps the packed-IMAD kernel (A/B timing only)
#ifdef TG_TUNING
    static const int use_mma = tuning_env("TG_DEMO_MMA", 1);
#else
    constexpr int use_mma = 1;
#endif
    if (S == 25) return launch_demo_acc_cols<25>(tape, stride, N, R, shift, slab, flags, OR_FLAGS, st);
    if (S == 16 && use_mma && demo_acc16_mma_applies(R)) return launch_demo_acc16_mma(tape, stride, N, R, shift, slab, flags, OR_FLAGS, st);
    if (S == 4 && (long long)R * shift * shift * shift <= 191 && R <= 65535 && N <= 0x7FFFFFFFLL * 128) { // one thread per demo
        static const AliasDev no_tables = {};
        demo4_thread_kernel<false, OR_FLAGS><<<(int)((N + 127) / 128), 128, 0, st>>>(0, N, R, shift, const_cast<uint8_t *>(tape), stride,
                                                                                   slab, flags, no_tables);
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    }
    Categorical cat = {};
    // 9x9x9: walk only the terms with a non-zero v_j (the masks are built from the tape itself, so this is exact for any tape;
    // with the reference's distributions 70 % of the coefficients are zero: 0.62 -> 0.55 ms per 2^20 demos; a tape without zeros
    // pays ~15 % in the term loop)
    cat.sparse_terms = S == 9 ? 1u : 0u;
    return dispatch_demo<false, 2, OR_FLAGS>(0, N, R, S, shift, cat, 1, const_cast<uint8_t *>(tape), stride, slab, flags, st);
}

// ---- contract box v1 (tg_demo_gen_box): the sampler alone, one thread per demo -- consecutive threads write consecutive
// records of a step, so a warp stores 32 TP contiguous bytes per term -- then tg_demo_accumulate's sum with the flags OR-ed
template <int S, int NTHR>
__global__ void __launch_bounds__(128)
    demo_box_sample_kernel(unsigned long long first_demo, long long N, int R, int shift, const __grid_constant__ Categorical cat,
                           int max_tries, const __grid_constant__ BoxMasks box, uint8_t *__restrict__ tape, long long tape_step_stride,
                           uint8_t *__restrict__ flags) {
    constexpr int TP = Geo<S>::TP, NW = (3 * S + 3) / 4;
    const long long n = (long long)blockIdx.x * 128 + threadIdx.x;
    if (n >= N) return;
    const unsigned long long d = first_demo + (unsigned long long)n;
    const uint32_t d_lo = (uint32_t)d, d_hi = (uint32_t)(d >> 32);
    uint32_t fl = 0;
#pragma unroll 1
    for (int r = 0; r < R; r++) {
        uint32_t words[TP / 4];
#pragma unroll
        for (int w = NW; w < TP / 4; w++) words[w] = 0;
#pragma unroll 1
        for (int t = 0;; t++) {
            if (draw_triple_box<S, NTHR>(words, d_lo, d_hi, r, t, cat, box)) break;
            if (t + 1 >= max_tries) { // forced: u = v = w = x e_0 (e_0 lies inside every box), x the last value
#pragma unroll
                for (int w = 0; w < NW; w++) words[w] = 0;
#pragma unroll
                for (int q = 0; q < 3 * S; q++)
                    words[q >> 2] |= (((q % S) == 0 ? cat.top_tok : (uint32_t)shift) & 0xFFu) << (8 * (q & 3));
                fl = TG_FLAG_EXHAUSTED;
                break;
            }
        }
        uint4 *dst = reinterpret_cast<uint4 *>(tape + (size_t)r * tape_step_stride + n * TP);
#pragma unroll
        for (int w = 0; w < TP / 16; w++) dst[w] = make_uint4(words[4 * w], words[4 * w + 1], words[4 * w + 2], words[4 * w + 3]);
    }
    if (flags) flags[n] = (uint8_t)fl;
}

template <int S, int NTHR>
static int launch_demo_box_sample(unsigned long long first, long long N, int R, int shift, const Categorical &cat, int max_tries,
                                  const BoxMasks &box, uint8_t *tape, long long stride, uint8_t *flags, cudaStream_t st) {
    const long long grid = (N + 127) / 128;
    if (grid > 0x7FFFFFFFLL) return TG_E_ARG;
    demo_box_sample_kernel<S, NTHR><<<(unsigned)grid, 128, 0, st>>>(first, N, R, shift, cat, max_tries, box, tape, stride, flags);
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

} // namespace tg

extern "C" {

int tg_demo_gen_philox(uint64_t seed, uint64_t first_demo, int64_t N, int R, int S, int shift, const int8_t *values,
                       const double *probs, int n_values, int max_tries, uint8_t *tape, int64_t tape_step_stride,
                       int8_t *slab, uint8_t *flags, void *stream) {
    if (const int rc = tg::check_demo_gen(S, N, R, shift, n_values, max_tries, values, probs, tape, tape_step_stride, slab); rc != tg::LAUNCH)
        return rc;
    if (!tg::alphabet_ok(values, probs, n_values, shift)) return TG_E_ARG;
    tg::Categorical cat = tg::categorical(values, probs, n_values, shift, seed);
    // measured (profiles/README.md): skipping the zero-coefficient terms in the accumulation pays at 9x9x9 (+10 %) when most
    // coefficients are zero, not at 4x4x4 (R = 7: too few terms per lane) and not when replaying a tape
    cat.sparse_terms = (S == 9 && tg::p_null<false>(values, probs, n_values) >= 0.5) ? 1u : 0u;
    cudaStream_t st = (cudaStream_t)stream;
    // contract v2 (group alias tables, no rejection loop) for alphabets of at most five values; max_tries does not apply
    if (tg::alias_applies(values, probs, n_values, S)) {
        tg::AliasParams ap;
        tg::build_alias(values, probs, n_values, S, shift, seed, ap);
        tg::AliasTabs tabs;
        tg::AliasDev dev;
        tg::alias_to_dev(ap, values, n_values, S, shift, tabs, dev);
        const int rc = tg::alias_device_tables(tabs, st, &dev.tab);
        if (rc != TG_OK) return rc;
        return tg::dispatch_demo_alias(first_demo, N, R, S, shift, cat, dev, tape, tape_step_stride, slab, flags, st);
    }
    // 16x16x16, R <= 64: the targets are summed on the tensor cores (tg_demo_mma.cuh) inside the sampling kernel;
    // TG_DEMO_MMA=0 keeps the packed-IMAD accumulation (A/B timing only)
#ifdef TG_TUNING
    static const int use_mma = tg::tuning_env("TG_DEMO_MMA", 1);
#else
    constexpr int use_mma = 1;
#endif
    if (S == 25) {
        if (n_values <= 3) return tg::launch_demo25<2>(first_demo, N, R, shift, cat, max_tries, tape, tape_step_stride, slab, flags, st);
        if (n_values <= 5) return tg::launch_demo25<4>(first_demo, N, R, shift, cat, max_tries, tape, tape_step_stride, slab, flags, st);
        return tg::launch_demo25<7>(first_demo, N, R, shift, cat, max_tries, tape, tape_step_stride, slab, flags, st);
    }
    if (S == 16 && use_mma && tg::demo_acc16_mma_applies(R)) {
        if (n_values <= 3) return tg::dispatch_demo16_mma<2>(first_demo, N, R, shift, cat, max_tries, tape, tape_step_stride, slab, flags, st);
        if (n_values <= 5) return tg::dispatch_demo16_mma<4>(first_demo, N, R, shift, cat, max_tries, tape, tape_step_stride, slab, flags, st);
        return tg::dispatch_demo16_mma<7>(first_demo, N, R, shift, cat, max_tries, tape, tape_step_stride, slab, flags, st);
    }
    if (n_values <= 3)
        return tg::dispatch_demo<true, 2>(first_demo, N, R, S, shift, cat, max_tries, tape, tape_step_stride, slab, flags, st);
    if (n_values <= 5)
        return tg::dispatch_demo<true, 4>(first_demo, N, R, S, shift, cat, max_tries, tape, tape_step_stride, slab, flags, st);
    return tg::dispatch_demo<true, 7>(first_demo, N, R, S, shift, cat, max_tries, tape, tape_step_stride, slab, flags, st);
}

int tg_demo_alias_tables(const int8_t *values, const double *probs, int n_values, int S, uint16_t *tables_host) {
    return tg::alias_tables_host<false>(values, probs, n_values, S, tables_host);
}

int tg_demo_accumulate(const uint8_t *tape, int64_t tape_step_stride, int64_t N, int R, int S, int shift, int8_t *slab,
                       uint8_t *flags, void *stream) {
    if (const int rc = tg::check_accumulate(tg::supported_S(S), N, R, shift, 1, 4, tape, tape_step_stride, slab); rc != tg::LAUNCH)
        return rc;
    return tg::accumulate<false>(tape, tape_step_stride, N, R, S, shift, slab, flags, (cudaStream_t)stream);
}

int tg_demo_gen_box(uint64_t seed, uint64_t first_demo, int64_t N, int R, int S, int nu, int nv, int nw, int shift,
                    const int8_t *values, const double *probs, int n_values, int max_tries, uint8_t *tape, int64_t tape_step_stride,
                    int8_t *slab, uint8_t *flags, void *stream) {
    if (const int rc = tg::check_demo_gen_box(S, N, R, nu, nv, nw, shift, n_values, max_tries, values, probs, tape, tape_step_stride, slab);
        rc != tg::LAUNCH)
        return rc;
    if (!tg::alphabet_ok(values, probs, n_values, shift)) return TG_E_ARG;
    const tg::Categorical cat = tg::categorical(values, probs, n_values, shift, seed);
    const tg::BoxMasks box = tg::box_masks(S, nu, nv, nw, shift);
    cudaStream_t st = (cudaStream_t)stream;
    const int rc = tg::with_S(S, [&](auto s) {
        constexpr int kS = decltype(s)::value;
        if (n_values <= 3) return tg::launch_demo_box_sample<kS, 2>(first_demo, N, R, shift, cat, max_tries, box, tape, tape_step_stride, flags, st);
        if (n_values <= 5) return tg::launch_demo_box_sample<kS, 4>(first_demo, N, R, shift, cat, max_tries, box, tape, tape_step_stride, flags, st);
        return tg::launch_demo_box_sample<kS, 7>(first_demo, N, R, shift, cat, max_tries, box, tape, tape_step_stride, flags, st);
    });
    if (rc != TG_OK) return rc;
    return tg::accumulate<true>(tape, tape_step_stride, N, R, S, shift, slab, flags, st);
}

} // extern "C"
