// tg_i16.cu -- the game path on int16 slabs: K1 tg_step_i16, K8 tg_expand_children_i16, K2 tg_rollout_i16 /
// tg_replay_i16, K7 tg_state_key_i16, K6 tg_slice_rank_i16.
//
// Residuals the int8 slab cannot hold (change-of-basis outputs, demo targets beyond int8, start tensors with large
// entries) are played here.  The int16 slab has the int8 slab's geometry counted in elements: entry (i,j,k) at element
// i*RP + j*S + k of a game of GP elements (2 GP bytes), padding zero.
//
// Formulation (tg_step.cuh, with 16-bit lanes).  A 32-bit word holds two consecutive (j,k) entries of one i-row; with
// both lanes in offset-binary (x ^ 0x8000) the word is the plain integer sum_b (x_b + 2^15) 65536^b, so the rank-1
// update of the word is
//        T' <- T' - u_i * VW ,   VW = v[j_0] w[k_0] + v[j_1] w[k_1] 65536
// ONE IMAD per two entries, exact as long as every resulting entry fits int16.  That is guaranteed while residuals are
// in [-16384, 16383] (the top two bits of a lane are equal: one SWAR test on the word) and |u v w| <= 64 (shift <= 4,
// tokens <= 2 * shift).  Leaving that zone -- or a token above 2 * shift -- raises TG_FLAG_RANGE for the game; a step
// that left the zone with legal tokens is still exact.  At S = 9 and 25 a row has an odd number of entries, so a word
// can hold the last entry of row j and the first of row j + 1, as the int8 words do.
//
// Rank (K6) is exact over Q for every int16 slab: the elimination of tg_aux.cu's slice_rank_kernel with 16-bit rows,
// whose Hadamard bound (|row|^2 <= 25 * 2^30 at 25x25x25) needs up to fifteen 31-bit primes instead of eight.
#include "tg_step.cuh"

namespace tg {

constexpr uint32_t H16 = 0x80008000u;

// int16 slab geometry in elements (the int8 slab's) and per-game byte sizes
template <int S>
struct Geo16 {
    using G = Geo<S>;
    static constexpr int RP = G::RP;       // row pitch (elements)
    static constexpr int WR = RP / 2;      // 32-bit words per row
    static constexpr int GP = G::GP;       // game pitch (elements)
    static constexpr int GB = 2 * G::GP;   // game pitch (bytes)
    static constexpr int TP = G::TP;       // token pitch (bytes)
};

// Partial result word of one thread for one game; summed over the WR threads of a game it gives nnz (bits 0-13),
// #threads whose update was non-zero (bits 14-22) and #threads that saw an entry outside [-16384, 16383] (bits 23-31).
// The fields cannot carry into each other while S^3 < 2^14 and WR < 2^9 (25x25x25: 15625 entries, 314 threads).
static_assert(Geo<25>::S3 < (1 << 14) && Geo16<25>::WR < (1 << 9), "partial result word fields");
static_assert(Geo16<4>::WR >= Geo16<4>::TP / 4, "the threads of a game cover its token record");
__device__ __forceinline__ uint32_t make_partial16(uint32_t nnz, bool changed, bool range) {
    return nnz | (changed ? 1u << 14 : 0u) | (range ? 1u << 23 : 0u);
}
__device__ __forceinline__ uint32_t partial_flags16(uint32_t sum) {
    return ((sum & 0x3FFFu) == 0 ? TG_FLAG_TERMINAL : 0u) | (((sum >> 14) & 0x1FFu) == 0 ? TG_FLAG_NULL : 0u) |
           ((sum >> 23) != 0 ? TG_FLAG_RANGE : 0u);
}

// bit 15 / 31 set iff that lane is non-zero; count of such lanes of a word with (lanes & hv) >> 15 summed
__device__ __forceinline__ uint32_t nonzero16(uint32_t x) { return (((x & 0x7FFF7FFFu) + 0x7FFF7FFFu) | x) & H16; }
__device__ __forceinline__ uint32_t lane_sum16(uint32_t cnt) { return (cnt & 0xFFFFu) + (cnt >> 16); }

// Per-thread constants of word column c of an int16 game.
template <int S>
struct Lane16 {
    int c;
    uint32_t hv;         // 0x8000 in every lane that is a real entry (not row padding)
    int off_v[2], off_w[2]; // token byte offsets of v[j_b], w[k_b] (a valid offset for padding lanes too)
    int m1;              // lane 1 is a real entry
    int tokw;            // the 32-bit word of the game's token record this thread range-checks

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
template <int S, typename TB>
__device__ __forceinline__ uint32_t pack_vw16(const TB *tok, const Lane16<S> &L, int shift) {
    const int d0 = ((int)tok[L.off_v[0]] - shift) * ((int)tok[L.off_w[0]] - shift);
    const int d1 = ((int)tok[L.off_v[1]] - shift) * ((int)tok[L.off_w[1]] - shift);
    return L.hv ? (uint32_t)d0 + ((uint32_t)(d1 * L.m1) << 16) : 0u;
}

// tape contract (tg_step.cuh): every token byte <= 2 * shift; thread c tests word c % (TP / 4) of its game's record
__device__ __forceinline__ bool token_word_over(uint32_t x, int shift) {
    return ((((x & 0x7F7F7F7Fu) + (uint32_t)(0x7F - 2 * shift) * ONES4) | x) & H4) != 0;
}

// game <- game - u (x) v (x) w for this thread's word column, all S rows (game/tok in shared memory)
template <int S>
__device__ __forceinline__ uint32_t rank1_update16(uint8_t *game, const uint8_t *tok, const Lane16<S> &L, int shift) {
    const uint32_t vw = pack_vw16<S>(tok, L, shift);
    uint32_t uw[UW<S>];
    load_u<S>(tok, uw);
    uint32_t cnt = 0, rng = 0;
    int uany = 0;
    uint32_t *col = reinterpret_cast<uint32_t *>(game) + L.c;
    const uint32_t nvw = 0u - vw;
#pragma unroll
    for (int i = 0; i < S; i++) {
        const int u = coef_u(uw, i, shift);
        const uint32_t t = ((col[i * Geo16<S>::WR] ^ H16) + (uint32_t)u * nvw) ^ H16;
        col[i * Geo16<S>::WR] = t;
        cnt += (nonzero16(t) & L.hv) >> 15;
        rng |= t ^ (t << 1);
        uany |= u;
    }
    const bool over = token_word_over(reinterpret_cast<const uint32_t *>(tok)[L.tokw], shift);
    return make_partial16(lane_sum16(cnt), vw != 0 && uany != 0, (rng & L.hv) != 0 || over);
}

// ------------------------------------------------------------------ K1: the step kernel of tg_step.cu on int16 games
template <int S, int NT, int NPASS, int NSTAGE>
struct Step16Cfg {
    using G = Geo16<S>;
    static constexpr int GPASS = NT / G::WR;
    static constexpr int TG = GPASS * NPASS;
    static constexpr int ACTIVE = GPASS * G::WR;
    static constexpr int SLAB_BYTES = TG * G::GB;
    static constexpr int TOK_BYTES = TG * G::TP;
    static constexpr int STAGE_BYTES = SLAB_BYTES + TOK_BYTES;
    static constexpr int PW = (G::WR % 32 == 0) ? G::WR / 32 : ((32 % G::WR == 0) ? 1 : G::WR);
    static constexpr int PART_WORDS = TG * PW;
    static constexpr int SMEM_BYTES = NSTAGE * STAGE_BYTES + 2 * PART_WORDS * 4 + 2 * NSTAGE * 8;
    static constexpr int THREADS = NT + 32;
    static_assert(SMEM_BYTES <= 227 * 1024, "shared memory of one CTA");
};

template <int S, int NT, int NPASS, int NSTAGE>
__global__ void __launch_bounds__(NT + 32)
    step16_kernel(const int16_t *__restrict__ slab_in, const uint8_t *__restrict__ tape, int16_t *__restrict__ slab_out,
                  uint8_t *__restrict__ flags, int32_t *__restrict__ nnz, long long B, int shift) {
    using C = Step16Cfg<S, NT, NPASS, NSTAGE>;
    using G = Geo16<S>;
    extern __shared__ __align__(128) uint8_t smem[];
    uint32_t *part = reinterpret_cast<uint32_t *>(smem + NSTAGE * C::STAGE_BYTES);
    uint64_t *full = reinterpret_cast<uint64_t *>(part + 2 * C::PART_WORDS);
    uint64_t *done = full + NSTAGE;
    const uint8_t *in = reinterpret_cast<const uint8_t *>(slab_in);
    uint8_t *out = reinterpret_cast<uint8_t *>(slab_out);

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
        // producer / storer (one lane): TMA bulk copies of the tile's games and records, bulk store of the results
        if (tid != NT) return;
        auto load = [&](long long tile, int s) {
            const long long g0 = tile * C::TG;
            const int ng = (int)min((long long)C::TG, B - g0);
            uint8_t *st = smem + s * C::STAGE_BYTES;
            mbar_expect_tx(&full[s], (uint32_t)(ng * (G::GB + G::TP)));
            bulk_g2s(st, in + g0 * G::GB, (uint32_t)(ng * G::GB), &full[s]);
            bulk_g2s(st + C::SLAB_BYTES, tape + g0 * G::TP, (uint32_t)(ng * G::TP), &full[s]);
        };
        long long tile = blockIdx.x;
        for (int s = 0; s < NSTAGE && tile + (long long)s * gridDim.x < ntiles; s++) load(tile + (long long)s * gridDim.x, s);
        for (int it = 0; tile < ntiles; tile += gridDim.x, it++) {
            const int s = it % NSTAGE;
            const uint32_t parity = (uint32_t)(it / NSTAGE) & 1u;
            mbar_wait(&done[s], parity);
            const long long g0 = tile * C::TG;
            const int ng = (int)min((long long)C::TG, B - g0);
            bulk_s2g(out + g0 * G::GB, smem + s * C::STAGE_BYTES, (uint32_t)(ng * G::GB));
            bulk_commit();
            const long long next = tile + (long long)NSTAGE * gridDim.x;
            if (next < ntiles) {
                bulk_wait_read<0>();
                load(next, s);
            }
        }
        bulk_wait<0>();
        return;
    }

    Lane16<S> L;
    const bool active = tid < C::ACTIVE;
    const int gl = tid / G::WR;
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
#pragma unroll 1 // unrolled, the 9x9x9 instantiation spills
        for (int p = 0; p < NPASS; p++) {
            const int g = p * C::GPASS + gl;
            uint32_t pr = 0;
            if (active && g < ng) pr = rank1_update16<S>(slab + g * G::GB, toks + g * G::TP, L, shift);
            if constexpr (G::WR % 32 == 0) {
                pr = __reduce_add_sync(0xFFFFFFFFu, pr);
                if ((tid & 31) == 0 && g < ng) pp[g * C::PW + (tid % G::WR) / 32] = pr;
            } else if constexpr (32 % G::WR == 0) {
#pragma unroll
                for (int o = 1; o < G::WR; o <<= 1) pr += __shfl_xor_sync(0xFFFFFFFFu, pr, o);
                if (L.c == 0 && g < ng) pp[g] = pr;
            } else {
                if (active && g < ng) pp[g * C::PW + L.c] = pr;
            }
        }
        fence_proxy_async();
        asm volatile("bar.sync 1, %0;" ::"n"(NT) : "memory");
        if (tid == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&done[s])) : "memory");
        for (int g = tid; g < ng; g += NT) {
            uint32_t sum = 0;
            for (int w = 0; w < C::PW; w++) sum += pp[g * C::PW + w];
            flags[g0 + g] = (uint8_t)partial_flags16(sum);
            nnz[g0 + g] = (int32_t)(sum & 0x3FFFu);
        }
    }
}

template <int S, int NT, int NPASS, int NSTAGE>
static int launch_step16(const int16_t *slab_in, const uint8_t *tape, int16_t *slab_out, uint8_t *flags, int32_t *nnz, long long B,
                         int shift, cudaStream_t stream) {
    using C = Step16Cfg<S, NT, NPASS, NSTAGE>;
    auto kern = step16_kernel<S, NT, NPASS, NSTAGE>;
    TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
    const long long ntiles = (B + C::TG - 1) / C::TG;
    const long long cap = (long long)sm_count() * 32;
    const int grid = (int)(ntiles < cap ? ntiles : cap);
    kern<<<grid, C::THREADS, C::SMEM_BYTES, stream>>>(slab_in, tape, slab_out, flags, nnz, B, shift);
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

// ------------------------------------------------------------------ K7 key constants (tg_state_key)
__device__ __forceinline__ unsigned long long splitmix64_16(unsigned long long z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
// A_i / B_j / C_k of the state key: base 0x1000 / 0x2000 / 0x3000
__device__ __forceinline__ unsigned long long key_const16(unsigned base, int i) { return splitmix64_16((unsigned long long)(base + i)) | 1ull; }

// sum_q (B C)[2c + q] * sum_i A_i T[i][2c + q] of one word column from its S offset-binary row words (lane = entry + 2^15,
// the offset's share -2^15 sum_i A_i is the accumulators' start value): this column's share of the state key
template <int S>
__device__ __forceinline__ unsigned long long column_key16(const uint32_t (&row)[S], int c) {
    unsigned long long a0 = 0;
#pragma unroll
    for (int i = 0; i < S; i++) a0 -= 32768ull * key_const16(0x1000, i);
    unsigned long long acc[2] = {a0, a0};
#pragma unroll
    for (int i = 0; i < S; i++) {
        acc[0] += (unsigned long long)(row[i] & 0xFFFFu) * key_const16(0x1000, i);
        acc[1] += (unsigned long long)(row[i] >> 16) * key_const16(0x1000, i);
    }
    unsigned long long h = 0;
#pragma unroll
    for (int q = 0; q < 2; q++) {
        const int jk = 2 * c + q;
        if (jk < Geo<S>::S2) h += acc[q] * (key_const16(0x2000, jk / S) * key_const16(0x3000, jk % S));
    }
    return h;
}

// ------------------------------------------------------------------ K8: expand_kernel of tg_expand.cu on int16 games
template <int S, int NT>
struct Exp16Cfg {
    using G = Geo16<S>;
    static constexpr int TG = NT / G::WR;
    static constexpr int ACTIVE = TG * G::WR;
    static constexpr int STAGE_BYTES = TG * G::GB;
    static __host__ __device__ constexpr int tok_bytes(int k) { return (TG * k * G::TP + 15) & ~15; }
    static constexpr int NSTAGE = 3;
    static __host__ __device__ constexpr int smem_bytes(int k) {
        return tok_bytes(k) + NSTAGE * STAGE_BYTES + ((NSTAGE * TG * 4 + 7) & ~7) + TG * 8 + 16 + NT * 8;
    }
};

template <int S, int NT, bool KEYS>
__global__ void __launch_bounds__(NT)
    expand16_kernel(const int16_t *__restrict__ parents, const uint8_t *__restrict__ tape, int k, int16_t *__restrict__ children,
                    uint8_t *__restrict__ flags, int32_t *__restrict__ nnz, unsigned long long *__restrict__ keys, long long B,
                    int shift) {
    using C = Exp16Cfg<S, NT>;
    using G = Geo16<S>;
    extern __shared__ __align__(128) uint8_t smem[];
    constexpr int NSTAGE = C::NSTAGE;
    uint8_t *s_tok = smem;                                                            // [TG][k][TP]
    uint8_t *s_out = smem + C::tok_bytes(k);                                          // [NSTAGE][TG][GB]
    uint32_t *s_part = reinterpret_cast<uint32_t *>(s_out + NSTAGE * C::STAGE_BYTES); // [NSTAGE][TG]
    unsigned long long *s_pkey = reinterpret_cast<unsigned long long *>(reinterpret_cast<uint8_t *>(s_part) + ((NSTAGE * C::TG * 4 + 7) & ~7));
    uint64_t *s_bar = reinterpret_cast<uint64_t *>(s_pkey + C::TG);
    unsigned long long *s_ph = reinterpret_cast<unsigned long long *>(s_bar + 2); // [NT] parent key, per word column
    uint8_t *out = reinterpret_cast<uint8_t *>(children);

    const int tid = threadIdx.x;
    const long long g0 = (long long)blockIdx.x * C::TG;
    const int ng = (int)min((long long)C::TG, B - g0);
    const int g = tid / G::WR;
    const bool active = tid < C::ACTIVE && g < ng;
    Lane16<S> L;
    L.init(tid < C::ACTIVE ? tid % G::WR : 0);

    if (tid == 0) {
        mbar_init(s_bar, 1);
        mbar_fence_init();
    }
    // game padding of the child stages is zero and stays zero (threads only write their word columns of the S rows)
    for (int w = tid; w < NSTAGE * C::STAGE_BYTES / 4; w += NT) reinterpret_cast<uint32_t *>(s_out)[w] = 0;
    for (int i = tid; i < NSTAGE * C::TG; i += NT) s_part[i] = 0;
    __syncthreads();
    if (tid == 0) {
        mbar_expect_tx(s_bar, (uint32_t)(ng * k * G::TP));
        bulk_g2s(s_tok, tape + g0 * k * G::TP, (uint32_t)(ng * k * G::TP), s_bar);
    }
    // the parent's rows of this thread's word column, offset-binary, read once
    uint32_t row[S];
    if (active) {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(parents + (g0 + g) * G::GP) + L.c;
#pragma unroll
        for (int i = 0; i < S; i++) row[i] = src[i * G::WR] ^ H16;
    } else {
#pragma unroll
        for (int i = 0; i < S; i++) row[i] = H16;
    }
    if constexpr (KEYS) s_ph[tid] = column_key16<S>(row, L.c);
    mbar_wait(s_bar, 0);
    if constexpr (KEYS) {
        __syncthreads();
        if (tid < ng) {
            unsigned long long h = 0;
            for (int c = 0; c < G::WR; c++) h += s_ph[tid * G::WR + c];
            s_pkey[tid] = h;
        }
        __syncthreads();
        // child key = parent key - key of its rank-1 action (tg_expand.cu)
        for (int x = tid; x < ng * k; x += NT) {
            const uint8_t *tok = s_tok + (size_t)x * G::TP;
            unsigned long long f[3];
#pragma unroll
            for (int m = 0; m < 3; m++) {
                unsigned long long a = 0;
#pragma unroll
                for (int i = 0; i < S; i++) a += (unsigned long long)(long long)((int)tok[m * S + i] - shift) * key_const16(0x1000 * (m + 1), i);
                f[m] = a;
            }
            keys[g0 * k + x] = s_pkey[x / k] - f[0] * f[1] * f[2];
        }
    }

    for (int c = 0, st = 0; c < k; c++, st = st + 1 == NSTAGE ? 0 : st + 1) {
        uint8_t *stage = s_out + st * C::STAGE_BYTES;
        if (active) {
            const uint8_t *tok = s_tok + ((size_t)g * k + c) * G::TP;
            const uint32_t vw = pack_vw16<S>(tok, L, shift);
            uint32_t uw[UW<S>];
            load_u<S>(tok, uw);
            const uint32_t nvw = 0u - vw;
            uint32_t cnt = 0, rng = 0;
            int uany = 0;
            uint32_t *col = reinterpret_cast<uint32_t *>(stage + (size_t)g * G::GB) + L.c;
#pragma unroll
            for (int i = 0; i < S; i++) {
                const int u = coef_u(uw, i, shift);
                const uint32_t t = (row[i] + (uint32_t)u * nvw) ^ H16; // child word, two's complement lanes
                col[i * G::WR] = t;
                cnt += (nonzero16(t) & L.hv) >> 15;
                rng |= t ^ (t << 1);
                uany |= u;
            }
            const bool over = token_word_over(reinterpret_cast<const uint32_t *>(tok)[L.tokw], shift);
            atomicAdd(&s_part[st * C::TG + g], make_partial16(lane_sum16(cnt), vw != 0 && uany != 0, (rng & L.hv) != 0 || over));
        }
        fence_proxy_async();
        __syncthreads();
        if (tid < ng) {
            const long long child = (g0 + tid) * k + c;
            bulk_s2g(out + child * G::GB, stage + (size_t)tid * G::GB, (uint32_t)G::GB);
            bulk_commit();
            const uint32_t sum = s_part[st * C::TG + tid];
            flags[child] = (uint8_t)partial_flags16(sum);
            nnz[child] = (int32_t)(sum & 0x3FFFu);
            s_part[st * C::TG + tid] = 0;
            bulk_wait_read<1>(); // three stages, one barrier per child: see expand_kernel
        }
    }
    if (tid < ng) bulk_wait<0>();
}

template <int S, int NT>
static int launch_expand16(const int16_t *parents, const uint8_t *tape, int k, int16_t *children, uint8_t *flags, int32_t *nnz,
                           unsigned long long *keys, long long B, int shift, cudaStream_t st) {
    using C = Exp16Cfg<S, NT>;
    if (k > (200 * 1024 - C::smem_bytes(0)) / (C::TG * Geo<S>::TP)) return TG_E_ARG; // the records of a CTA exceed shared memory
    const int smem = C::smem_bytes(k);
    const long long grid = (B + C::TG - 1) / C::TG;
    if (grid > 0x7FFFFFFFLL) return TG_E_ARG;
    if (keys) {
        auto kern = expand16_kernel<S, NT, true>;
        TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        kern<<<(int)grid, NT, smem, st>>>(parents, tape, k, children, flags, nnz, keys, B, shift);
    } else {
        auto kern = expand16_kernel<S, NT, false>;
        TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        kern<<<(int)grid, NT, smem, st>>>(parents, tape, k, children, flags, nnz, keys, B, shift);
    }
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

// ------------------------------------------------------------------ K2: word-column rollout / replay on int16 games
// Thread (game, word column) keeps its S row words in registers for all K steps and reads each step's record straight
// from the tape (the threads of a game read the same record: L1 broadcasts).  The zone is tested after every applied
// step (one SWAR test per word), so TG_FLAG_RANGE means: the start state or the state after some applied step had an
// entry outside [-16384, 16383], or an applied step's record broke the token bound.  FREEZE: a game stops at the first
// all-zero state (the break at act.py:49), decided by one vote per step in shared memory (three buffers, so one CTA
// barrier per step is enough: a buffer is cleared one barrier after its last read and rewritten one barrier later).
template <int S, int NT>
struct Roll16Cfg {
    using G = Geo16<S>;
    static constexpr int TG = NT / G::WR;
    static constexpr int ACTIVE = TG * G::WR;
};

template <int S, int NT, bool FREEZE>
__global__ void __launch_bounds__(NT)
    rollout16_kernel(const int16_t *__restrict__ slab_in, const uint8_t *__restrict__ tape, long long tape_step_stride, int K,
                     int16_t *__restrict__ slab_out, uint8_t *__restrict__ flags, int32_t *__restrict__ nnz,
                     int32_t *__restrict__ steps, long long B, int shift) {
    using C = Roll16Cfg<S, NT>;
    using G = Geo16<S>;
    __shared__ uint32_t s_nz[3][C::TG]; // per step: the game is non-zero after it ([2]: the start state)
    __shared__ uint32_t s_sum[C::TG];
    __shared__ uint32_t s_steps[C::TG];

    const int tid = threadIdx.x;
    const long long g0 = (long long)blockIdx.x * C::TG;
    const int ng = (int)min((long long)C::TG, B - g0);
    const int g = tid / G::WR;
    const bool active = tid < C::ACTIVE && g < ng;
    Lane16<S> L;
    L.init(tid < C::ACTIVE ? tid % G::WR : 0);
    const uint32_t vmask = (L.hv >> 15) * 0xFFFFu; // lanes that are real entries

    for (int i = tid; i < 3 * C::TG; i += NT) (&s_nz[0][0])[i] = 0;
    for (int i = tid; i < C::TG; i += NT) s_sum[i] = 0, s_steps[i] = 0;
    __syncthreads();

    uint32_t row[S];
    uint32_t nzw = 0, bad = 0;
    bool tok_over = false; // an applied step's record broke the token bound
    if (active) {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(slab_in + (g0 + g) * G::GP) + L.c;
#pragma unroll
        for (int i = 0; i < S; i++) {
            const uint32_t t = src[i * G::WR];
            nzw |= t & vmask;
            row[i] = t ^ H16;
            bad |= ~(row[i] ^ (row[i] << 1)); // offset-binary: bits 15 / 31 equal to bits 14 / 30 <=> outside the zone
        }
    } else {
#pragma unroll
        for (int i = 0; i < S; i++) row[i] = H16;
    }
    if (active && nzw) s_nz[2][g] = 1;
    __syncthreads();
    bool alive = active && (!FREEZE || s_nz[2][g] != 0);
    int my_steps = 0;
    const uint8_t *rec = tape + (g0 + g) * G::TP;

    for (int t = 0; t < K; t++, rec += tape_step_stride) {
        if (alive) {
            const uint32_t vw = pack_vw16<S>(rec, L, shift);
            uint32_t uw[UW<S>];
#pragma unroll
            for (int q = 0; q < UW<S> / 4; q++) {
                const uint4 ut = __ldg(reinterpret_cast<const uint4 *>(rec) + q);
                uw[4 * q] = ut.x, uw[4 * q + 1] = ut.y, uw[4 * q + 2] = ut.z, uw[4 * q + 3] = ut.w;
            }
            const uint32_t nvw = 0u - vw;
            uint32_t any = 0;
#pragma unroll
            for (int i = 0; i < S; i++) {
                row[i] += (uint32_t)coef_u(uw, i, shift) * nvw;
                any |= row[i] ^ H16;
                bad |= ~(row[i] ^ (row[i] << 1));
            }
            tok_over = tok_over || token_word_over(__ldg(reinterpret_cast<const uint32_t *>(rec) + L.tokw), shift);
            my_steps = t + 1;
            if (FREEZE && (any & vmask) != 0) s_nz[t % 3][g] = 1;
        }
        if constexpr (FREEZE) {
            const int live = __syncthreads_or(alive);
            if (alive && s_nz[t % 3][g] == 0) alive = false; // solved at step t: frozen at the zero tensor
            if (tid < C::TG) s_nz[(t + 2) % 3][tid] = 0;
            if (!live) break;
        }
    }

    if (active) {
        uint32_t cnt = 0;
        uint32_t *dst = reinterpret_cast<uint32_t *>(slab_out + (g0 + g) * G::GP) + L.c;
#pragma unroll
        for (int i = 0; i < S; i++) {
            const uint32_t t = row[i] ^ H16;
            dst[i * G::WR] = t;
            cnt += (nonzero16(t) & L.hv) >> 15;
        }
        atomicAdd(&s_sum[g], make_partial16(lane_sum16(cnt), true, (bad & L.hv) != 0 || tok_over));
        if (L.c == 0) s_steps[g] = (uint32_t)my_steps;
    }
    __syncthreads();
    for (int q = tid; q < ng; q += NT) {
        const uint32_t sum = s_sum[q];
        flags[g0 + q] = (uint8_t)(partial_flags16(sum) & ~TG_FLAG_NULL);
        nnz[g0 + q] = (int32_t)(sum & 0x3FFFu);
        if (steps) steps[g0 + q] = (int32_t)s_steps[q];
    }
    if constexpr (G::GP > S * G::RP) { // keep the slab tail padding of out-of-place results zero
        constexpr int TAILW = (G::GP - S * G::RP) / 2;
        if (slab_out != slab_in)
            for (int q = tid; q < ng * TAILW; q += NT)
                reinterpret_cast<uint32_t *>(slab_out + (g0 + q / TAILW) * G::GP + S * G::RP)[q % TAILW] = 0;
    }
}

template <int S, int NT>
static int launch_rollout16(const int16_t *slab_in, const uint8_t *tape, long long stride, int K, int16_t *slab_out, uint8_t *flags,
                            int32_t *nnz, int32_t *steps, long long B, int shift, int freeze, cudaStream_t st) {
    using C = Roll16Cfg<S, NT>;
    const long long grid = (B + C::TG - 1) / C::TG;
    if (grid > 0x7FFFFFFFLL) return TG_E_ARG;
    if (freeze) rollout16_kernel<S, NT, true><<<(int)grid, NT, 0, st>>>(slab_in, tape, stride, K, slab_out, flags, nnz, steps, B, shift);
    else rollout16_kernel<S, NT, false><<<(int)grid, NT, 0, st>>>(slab_in, tape, stride, K, slab_out, flags, nnz, steps, B, shift);
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

// ------------------------------------------------------------------ K7: state key of int16 games
// The trilinear form of tg_state_key over the int16 values, so a state whose values fit int8 has the same key in both
// formats.  One thread per word column (column_key16), the WR partial sums of a game reduced by one warp.
template <int S, int NT>
__global__ void __launch_bounds__(NT) state_key16_kernel(const int16_t *__restrict__ slab, unsigned long long *__restrict__ keys,
                                                         long long B) {
    using G = Geo16<S>;
    constexpr int TG = NT / G::WR;
    static_assert(TG >= 1, "one game per pass at least");
    __shared__ unsigned long long s_ph[NT];
    const int tid = threadIdx.x;
    const int gl = tid / G::WR, c = tid % G::WR;
    const int wp = tid >> 5, ln = tid & 31;
    for (long long g0 = (long long)blockIdx.x * TG; g0 < B; g0 += (long long)gridDim.x * TG) {
        const long long g = g0 + gl;
        uint32_t w[S];
        if (gl < TG && g < B) {
            const uint32_t *col = reinterpret_cast<const uint32_t *>(slab + g * G::GP) + c;
#pragma unroll
            for (int i = 0; i < S; i++) w[i] = __ldg(col + i * G::WR) ^ H16;
        } else {
#pragma unroll
            for (int i = 0; i < S; i++) w[i] = H16;
        }
        s_ph[tid] = column_key16<S>(w, c);
        __syncthreads();
        for (int q = wp; q < TG; q += NT / 32) { // warp wp sums games wp, wp + NT/32, ...
            unsigned long long k = 0;
            for (int x = ln; x < G::WR; x += 32) k += s_ph[q * G::WR + x];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) k += __shfl_xor_sync(0xFFFFFFFFu, k, o);
            if (ln == 0 && g0 + q < B) keys[g0 + q] = k;
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------ K6: slice rank of int16 games
// slice_rank_kernel (tg_aux.cu) with 16-bit rows: |row|^2 <= 25 * 2^30 < 2^35, so the r+1 largest e of a 25x25 slice
// sum to at most 875 and fifteen primes 2^31 - c (a product above 2^900) always settle the rank.  The reduction of
// rank16_mod_p holds for c < 2^9 (the second fold stays below 2^19).
__constant__ uint32_t c_rank16_c[15] = {1, 19, 61, 69, 85, 99, 105, 151, 159, 171, 225, 249, 295, 325, 379}; // all prime
constexpr int RANK16_PRIMES = 15;

template <int S>
__device__ __forceinline__ int rank16_mod_p(const int16_t *__restrict__ src, bool live, int lane, uint32_t gmask, uint32_t P, uint32_t C) {
    uint32_t row[S];
#pragma unroll
    for (int c = 0; c < S; c++) {
        const int v = live ? src[c] : 0;
        row[c] = v >= 0 ? (uint32_t)v : P - (uint32_t)(-v);
    }
    bool used = !live;
    int rank = 0;
#pragma unroll
    for (int c = 0; c < S; c++) {
        const uint32_t cand = __ballot_sync(0xFFFFFFFFu, !used && row[c] != 0) & gmask;
        const bool has = cand != 0;
        const int pl = has ? __ffs(cand) - 1 : lane;
        const uint32_t pv = __shfl_sync(0xFFFFFFFFu, row[c], pl);
        const uint32_t mine = row[c];
        const bool elim = has && !used && lane != pl && mine != 0;
        const uint32_t nmine = P - mine;
#pragma unroll
        for (int k = c + 1; k < S; k++) {
            const uint32_t pk = __shfl_sync(0xFFFFFFFFu, row[k], pl);
            if (elim) {
                const unsigned long long z = (unsigned long long)row[k] * pv + (unsigned long long)nmine * pk; // < 2^63
                unsigned long long r = (z & 0x7FFFFFFFull) + (z >> 31) * C;                                    // < 2^41
                uint32_t q = (uint32_t)(r & 0x7FFFFFFFull) + (uint32_t)(r >> 31) * C;                          // < P + 2^19
                row[k] = q >= P ? q - P : q;
            }
        }
        if (has && lane == pl) used = true;
        rank += has ? 1 : 0;
    }
    return rank;
}

template <int S>
__global__ void slice_rank16_kernel(const int16_t *__restrict__ slab, int32_t *__restrict__ ranks, long long B) {
    using G = Geo16<S>;
    constexpr int LG = S;
    constexpr int MPW = 32 / LG;
    const int lane = threadIdx.x & 31;
    const int sub = lane / LG, r = lane % LG;
    const long long warp = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    const long long mat = warp * MPW + sub;
    const long long game = mat / S;
    const int slice = (int)(mat - game * S);
    const bool live = sub < MPW && game < B && r < S;
    const int16_t *src = slab + (live ? game * G::GP + slice * G::RP + r * S : 0);
    const uint32_t gmask = sub < MPW ? (((1u << LG) - 1u) << (sub * LG)) : 0u;
    int rank = rank16_mod_p<S>(src, live, lane, gmask, 0x7FFFFFFFu, 1u);
    unsigned long long n2 = 0; // |row|^2 <= 25 * 2^30
#pragma unroll
    for (int c = 0; c < S; c++) {
        const long long v = live ? src[c] : 0;
        n2 += (unsigned long long)(v * v);
    }
    const int e = n2 <= 1 ? 0 : 64 - __clzll((long long)(n2 - 1)); // |row|^2 <= 2^e
    const int emax = (int)__reduce_max_sync(0xFFFFFFFFu, (unsigned)e);
    const int nzrows = __popc(__ballot_sync(0xFFFFFFFFu, n2 != 0) & gmask);
    auto top_e = [&](int m) {
        int E = 0;
        for (int t = 1; t <= emax; t++) E += min(m, __popc(__ballot_sync(0xFFFFFFFFu, e >= t) & gmask));
        return E;
    };
    bool fin = rank == nzrows;
    if (!__all_sync(0xFFFFFFFFu, fin)) {
        const int E = top_e(rank + 1);
        fin = fin || E <= 60;
    }
#pragma unroll 1
    for (int j = 1; j < RANK16_PRIMES && !__all_sync(0xFFFFFFFFu, fin); j++) {
        const int rj = rank16_mod_p<S>(src, live, lane, gmask, 0x80000000u - c_rank16_c[j], c_rank16_c[j]);
        if (!fin) rank = max(rank, rj);
        const int E = top_e(rank + 1);
        fin = fin || rank == nzrows || E <= 60 * (j + 1);
    }
    if (live && r == 0) atomicAdd(&ranks[game], rank);
}

} // namespace tg

static int rollout16_dispatch(const int16_t *slab_in, const uint8_t *tape, int64_t tape_step_stride, int K, int16_t *slab_out,
                              uint8_t *flags, int32_t *nnz, int32_t *steps, int64_t B, int S, int shift, int freeze, void *stream) {
    const int rc = tg::check_rollout(S, B, K, shift, slab_in, tape, tape_step_stride, slab_out, flags, nnz, steps, freeze);
    if (rc != tg::LAUNCH) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    switch (S) {
    case 4: return tg::launch_rollout16<4, 128>(slab_in, tape, tape_step_stride, K, slab_out, flags, nnz, steps, B, shift, freeze, st);
    case 9: return tg::launch_rollout16<9, 256>(slab_in, tape, tape_step_stride, K, slab_out, flags, nnz, steps, B, shift, freeze, st);
    case 16: return tg::launch_rollout16<16, 256>(slab_in, tape, tape_step_stride, K, slab_out, flags, nnz, steps, B, shift, freeze, st);
    case 25: return tg::launch_rollout16<25, 320>(slab_in, tape, tape_step_stride, K, slab_out, flags, nnz, steps, B, shift, freeze, st);
    }
    return TG_E_ARG;
}

extern "C" {

int tg_step_i16(const int16_t *slab_in, const uint8_t *tape, int16_t *slab_out, uint8_t *flags, int32_t *nnz, int64_t B, int S,
                int shift, void *stream) {
    if (const int rc = tg::check_step(S, B, shift, slab_in, tape, slab_out, flags, nnz); rc != tg::LAUNCH) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    // the int8 configurations' stage sizes (about 16-20 KB per stage, two stages), with half the games per stage
    switch (S) {
    case 4: return tg::launch_step16<4, 256, 4, 2>(slab_in, tape, slab_out, flags, nnz, B, shift, st);
    case 9: return tg::launch_step16<9, 256, 2, 2>(slab_in, tape, slab_out, flags, nnz, B, shift, st);
    case 16: return tg::launch_step16<16, 256, 1, 2>(slab_in, tape, slab_out, flags, nnz, B, shift, st);
    // 25x25x25: 314 word columns per game, ten compute warps hold one game; two 31.5 KB stages
    case 25: return tg::launch_step16<25, 320, 1, 2>(slab_in, tape, slab_out, flags, nnz, B, shift, st);
    }
    return TG_E_ARG;
}

int tg_expand_children_i16(const int16_t *parents, const uint8_t *tape, int k, int16_t *children, uint8_t *flags, int32_t *nnz,
                           uint64_t *keys, int64_t B, int S, int shift, void *stream) {
    if (const int rc = tg::check_expand(S, B, k, shift, parents, tape, children, flags, nnz); rc != tg::LAUNCH) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    unsigned long long *kp = (unsigned long long *)keys;
    switch (S) {
    case 4: return tg::launch_expand16<4, 128>(parents, tape, k, children, flags, nnz, kp, B, shift, st);
    case 9: return tg::launch_expand16<9, 256>(parents, tape, k, children, flags, nnz, kp, B, shift, st);
    case 16: return tg::launch_expand16<16, 256>(parents, tape, k, children, flags, nnz, kp, B, shift, st);
    case 25: return tg::launch_expand16<25, 320>(parents, tape, k, children, flags, nnz, kp, B, shift, st); // one parent per CTA
    }
    return TG_E_ARG;
}

int tg_rollout_i16(const int16_t *slab_in, const uint8_t *tape, int64_t tape_step_stride, int K, int16_t *slab_out, uint8_t *flags,
                   int32_t *nnz, int32_t *steps, int64_t B, int S, int shift, void *stream) {
    return rollout16_dispatch(slab_in, tape, tape_step_stride, K, slab_out, flags, nnz, steps, B, S, shift, 1, stream);
}

int tg_replay_i16(const int16_t *slab_in, const uint8_t *tape, int64_t tape_step_stride, int K, int16_t *slab_out, uint8_t *flags,
                  int32_t *nnz, int64_t B, int S, int shift, void *stream) {
    return rollout16_dispatch(slab_in, tape, tape_step_stride, K, slab_out, flags, nnz, nullptr, B, S, shift, 0, stream);
}

int tg_state_key_i16(const int16_t *slab16, uint64_t *keys, int64_t B, int S, void *stream) {
    if (const int rc = tg::check_pair(S, B, slab16, 16, keys, 1); rc != tg::LAUNCH) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    unsigned long long *kp = (unsigned long long *)keys;
    auto grid = [B](int tg_) { const long long t = (B + tg_ - 1) / tg_; return (unsigned)(t < 148 * 16 ? t : 148 * 16); };
    switch (S) {
    case 4: tg::state_key16_kernel<4, 256><<<grid(256 / tg::Geo16<4>::WR), 256, 0, st>>>(slab16, kp, B); break;
    case 9: tg::state_key16_kernel<9, 256><<<grid(256 / tg::Geo16<9>::WR), 256, 0, st>>>(slab16, kp, B); break;
    case 16: tg::state_key16_kernel<16, 256><<<grid(256 / tg::Geo16<16>::WR), 256, 0, st>>>(slab16, kp, B); break;
    case 25: tg::state_key16_kernel<25, 320><<<grid(1), 320, 0, st>>>(slab16, kp, B); break;
    default: return TG_E_ARG;
    }
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

int tg_slice_rank_i16(const int16_t *slab16, int32_t *ranks, int64_t B, int S, void *stream) {
    if (const int rc = tg::check_pair(S, B, slab16, 16, ranks, 1); rc != tg::LAUNCH) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    TG_CUDA(cudaMemsetAsync(ranks, 0, (size_t)B * 4, st));
    return tg::with_S(S, [&](auto s) {
        constexpr int kS = decltype(s)::value;
        const long long warps = (B * kS + (32 / kS) - 1) / (32 / kS);
        tg::slice_rank16_kernel<kS><<<(unsigned)((warps * 32 + 127) / 128), 128, 0, st>>>(slab16, ranks, B);
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    });
}

} // extern "C"
