// tg_rollout.cu -- K2: fused K-step rollout from an action tape (C ABI: tg_rollout).
//
// Reference restated: SyntheticDemoDataset._take_actions (datasets.py:144-153)
// and the greedy loop of training.py:336-342 around _take_action: K successive
// transitions T <- T - u(x)v(x)w with the game frozen once its head is all
// zero (the break at act.py:49), one -1 reward per applied action
// (act.py:60-62).
//
// The residual never leaves the SM: thread (game, word column c) keeps its S
// row words in REGISTERS (offset-binary, see tg_step.cuh) for all K steps, so a
// step costs one pack(v w) and S IMADs per thread.  Only the tokens stream
// from HBM (TP bytes per game-step) through a small shared-memory ring that a
// dedicated producer warp keeps full with TMA bulk copies (full/empty
// mbarriers).  "Is the game solved" is decided lazily: a thread notes, per step,
// whether ITS words are all zero (one bit), and only every SEG = 8 steps the bit
// masks of a game's threads are AND-ed through shared memory (three named
// barriers of the compute warps per 8 steps instead of one per step, so the
// warps drift freely inside a segment).  A game solved at step t of a segment
// keeps computing until the segment ends; that is harmless: frozen at the zero
// tensor means its result IS the zero tensor, `steps` comes from the first set
// bit, and range checks made after t are discarded.  HBM traffic per game:
// 2*GP + K*TP + 9 bytes.
#include "tg_step.cuh"

namespace tg {

// sign-extended byte B of a word of int8 coefficients
template <int B>
__device__ __forceinline__ int sext_byte4(uint32_t w) {
    constexpr uint32_t sel = (uint32_t)B | ((uint32_t)(B | 8) << 4) | ((uint32_t)(B | 8) << 8) | ((uint32_t)(B | 8) << 12);
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(w), "r"(0u), "r"(sel));
    return (int)d;
}

template <int S, int NT, int NST>
struct RollCfg {
    using G = Geo<S>;
    static constexpr int TG = NT / G::WR;      // games per CTA (one word column per thread)
    static constexpr int ACTIVE = TG * G::WR;
    static constexpr int TOK_BYTES = TG * G::TP;
    static constexpr int SEG = 8;              // steps between two game-level "solved?" reductions
    static constexpr int SMEM_BYTES = NST * TOK_BYTES + 4 * TG * 4 + 2 * TG * 4 + 2 * NST * 8;
    static_assert((NST & (NST - 1)) == 0, "ring depth must be a power of two");
};

template <int S, int NT, int NST>
__global__ void __launch_bounds__(NT + 32)
    rollout_kernel(const int8_t *__restrict__ slab_in, const uint8_t *__restrict__ tape, long long tape_step_stride, int K,
                   int8_t *__restrict__ slab_out, uint8_t *__restrict__ flags, int32_t *__restrict__ nnz,
                   int32_t *__restrict__ steps, long long B, int shift, int chk, int freeze) {
    using C = RollCfg<S, NT, NST>;
    using G = Geo<S>;
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t *s_tok = smem;                                                     // [NST][TG][TP]
    uint32_t *s_any = reinterpret_cast<uint32_t *>(smem + NST * C::TOK_BYTES); // [4][TG] votes "still non-zero"
    uint32_t *s_sum = s_any + 4 * C::TG;                                       // [TG] final partial sums
    uint32_t *s_steps = s_sum + C::TG;                                         // [TG]
    uint64_t *s_full = reinterpret_cast<uint64_t *>(s_steps + C::TG);          // [NST] tokens of a step have landed
    uint64_t *s_empty = s_full + NST;                                          // [NST] ... have been consumed

    const int tid = threadIdx.x;
    const long long g0 = (long long)blockIdx.x * C::TG;
    const int ng = (int)min((long long)C::TG, B - g0);
    const bool compute = tid < NT;
    const bool active = tid < C::ACTIVE && (tid / G::WR) < ng;
    const int g = tid / G::WR;
    Lane<S> L;
    L.init(tid < C::ACTIVE ? tid % G::WR : 0);

    // s_any[0][g]: AND of the per-thread "my words are zero" step masks of game g; s_any[3][g]: initial state non-zero
    for (int i = tid; i < 4 * C::TG; i += NT + 32) s_any[i] = i < C::TG ? 0xFFFFFFFFu : 0u;
    for (int i = tid; i < C::TG; i += NT + 32) s_sum[i] = 0, s_steps[i] = 0;
    if (tid == 0) {
        for (int s = 0; s < NST; s++) mbar_init(&s_full[s], 1), mbar_init(&s_empty[s], NT / 32);
        mbar_fence_init();
    }
    __syncthreads();

    // residual rows of this thread's word column, offset-binary
    uint32_t row[S];
    uint32_t nzw = 0, bad = 0;
    const uint32_t vmask = (L.hv >> 7) * 0xFFu; // bytes that are real entries
    if (active) {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(slab_in + (g0 + g) * G::GP) + L.c;
#pragma unroll
        for (int i = 0; i < S; i++) {
            const uint32_t t = src[i * G::WR];
            nzw |= t & vmask;
            row[i] = t ^ H4;
            bad |= ~(row[i] ^ (row[i] << 1)); // the start state must already be inside [-64,63]
        }
    } else {
#pragma unroll
        for (int i = 0; i < S; i++) row[i] = H4;
    }
    // vote on the initial state (slot 3 is the "step -1" slot)
    if (active && nzw) s_any[3 * C::TG + g] = 1;
    __syncthreads();
    bool alive = active && (!freeze || s_any[3 * C::TG + g] != 0);
    int until = chk;
    int my_steps = 0;

    if (!compute) {
        // ---------------- producer warp: one lane streams the tokens of step t into ring stage t % NST
        if (tid == NT) {
            const uint8_t *src = tape + g0 * G::TP;
            for (int t = 0; t < K; t++, src += tape_step_stride) {
                const int st = t & (NST - 1);
                if (t >= NST) mbar_wait(&s_empty[st], (uint32_t)(t / NST - 1) & 1u); // every compute warp has read it
                mbar_expect_tx(&s_full[st], (uint32_t)(ng * G::TP));
                bulk_g2s(s_tok + st * C::TOK_BYTES, src, (uint32_t)(ng * G::TP), &s_full[st]);
            }
        }
    } else {
        const uint8_t *tok0 = s_tok + g * G::TP;
        uint32_t zmask = 0, bmask = 0; // per step of the current segment: my words all zero / my range check failed
        // one step; `st` is a literal in the unrolled main loop, so every shared-memory address of the step is
        // (per-thread register + immediate)
        auto step = [&](int t, int st, uint32_t parity) {
            mbar_wait(&s_full[st], parity);
            if (alive) {
                const uint8_t *tok = tok0 + st * C::TOK_BYTES;
                const int32_t vw = W8::pack_vw<S>(tok, L, shift);
                uint32_t uw[UW<S>];
                load_u<S>(tok, uw);
                uint32_t any = 0;
                const uint32_t nvw = (uint32_t)(-vw);
#pragma unroll
                for (int i = 0; i < S; i++) {
                    row[i] += (uint32_t)coef_u(uw, i, shift) * nvw;
                    any |= row[i] ^ H4;
                }
                if (--until == 0) { // all entries still in [-64,63]? then chk more steps cannot alias the packed form
                    until = chk;
                    uint32_t b = 0;
#pragma unroll
                    for (int i = 0; i < S; i++) b |= ~(row[i] ^ (row[i] << 1));
                    if (freeze)
                        bmask |= ((b & L.hv) != 0 ? 1u : 0u) << (t & (C::SEG - 1));
                    else
                        bad |= b;
                }
                if (tokens_out_of_range<S>(tok, L, shift)) { // tape contract (tg_step.cuh): the packed update may have aliased
                    if (freeze)
                        bmask |= 1u << (t & (C::SEG - 1));
                    else
                        bad = 0xFFFFFFFFu;
                }
                my_steps = t + 1;
                if ((any & vmask) == 0) zmask |= 1u << (t & (C::SEG - 1));
            }
            __syncwarp();
            if ((tid & 31) == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&s_empty[st])) : "memory");
        };
        // segment end after step t: has the game been all zero at some step of the segment?
        auto segment_end = [&](int t) {
            asm volatile("bar.sync 1, %0;" ::"n"(NT) : "memory"); // the masks of the previous segment have been re-armed
            if (alive) atomicAnd(&s_any[g], zmask);
            asm volatile("bar.sync 1, %0;" ::"n"(NT) : "memory");
            const uint32_t solved = alive ? (s_any[g] & (0xFFFFFFFFu >> (31 - (t & (C::SEG - 1))))) : 0u;
            asm volatile("bar.sync 1, %0;" ::"n"(NT) : "memory");
            if (tid < C::TG) s_any[tid] = 0xFFFFFFFFu;
            if (alive) {
                if (solved) {
                    const int first = __ffs(solved) - 1; // frozen from this step on: the zero tensor
                    my_steps = (t & ~(C::SEG - 1)) + first + 1;
                    alive = false;
#pragma unroll
                    for (int i = 0; i < S; i++) row[i] = H4;
                    if (bmask & (0xFFFFFFFFu >> (31 - first))) bad = 0xFFFFFFFFu;
                } else if (bmask) {
                    bad = 0xFFFFFFFFu;
                }
            }
            zmask = 0, bmask = 0;
        };
        static_assert(C::SEG % NST == 0, "a segment is a whole number of ring turns");
        int t = 0;
        for (; t + NST <= K; t += NST) {
            const uint32_t parity = (uint32_t)(t / NST) & 1u;
#pragma unroll
            for (int q = 0; q < NST; q++) step(t + q, q, parity);
            if (freeze && ((t + NST) & (C::SEG - 1)) == 0) segment_end(t + NST - 1);
        }
        for (; t < K; t++) step(t, t & (NST - 1), (uint32_t)(t / NST) & 1u);
        if (freeze && (K & (C::SEG - 1)) != 0) segment_end(K - 1);
    }

    // final state out, per-game nnz / flags / steps
    if (active) {
        uint32_t cnt = 0;
        uint32_t *dst = reinterpret_cast<uint32_t *>(slab_out + (g0 + g) * G::GP) + L.c;
#pragma unroll
        for (int i = 0; i < S; i++) {
            bad |= ~(row[i] ^ (row[i] << 1));
            const uint32_t t = row[i] ^ H4;
            dst[i * G::WR] = t;
            cnt += ((((t & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | t) & L.hv) >> 7;
        }
        atomicAdd(&s_sum[g], make_partial(byte_sum(cnt), true, (bad & L.hv) != 0));
        if (L.c == 0) s_steps[g] = (uint32_t)my_steps;
    }
    __syncthreads();
    for (int q = tid; q < ng; q += NT + 32) {
        const uint32_t sum = s_sum[q];
        flags[g0 + q] = (uint8_t)(partial_flags(sum) & ~TG_FLAG_NULL);
        nnz[g0 + q] = (int32_t)(sum & 0xFFFFu);
        if (steps) steps[g0 + q] = (int32_t)s_steps[q];
    }
    if constexpr (G::GP > S * G::RP) { // keep the slab tail padding of out-of-place results zero
        if (slab_out != slab_in)
            for (int q = tid; q < ng * ((G::GP - S * G::RP) / 4); q += NT + 32) {
                const int gg = q / ((G::GP - S * G::RP) / 4), w = q % ((G::GP - S * G::RP) / 4);
                reinterpret_cast<uint32_t *>(slab_out + (g0 + gg) * G::GP + S * G::RP)[w] = 0;
            }
    }
}

// ------------------------------------------------------------------ 4x4x4: one THREAD per game
// A 4x4x4 game is 16 words: it lives in the registers of one thread for all K steps (offset-binary, tg_step.cuh).  A step is
// one 16-byte load of the game's record (coalesced: consecutive threads, consecutive records of the step-major tape), the
// twelve coefficients with three packed subtractions and eight sign-extending PRMTs, sixteen products u_i v_j and sixteen
// IMADs with the integer form of pack(w): ~80 instructions per game-step and THREAD (2.5 per warp and game-step against
// ~12 for the word-column kernel), no shared memory, no barrier, "solved" is a register test.  Same contract as
// rollout_kernel (freeze at the zero tensor, steps, nnz, TERMINAL / RANGE flags, token bound).
template <bool FREEZE>
__global__ void __launch_bounds__(128)
    rollout4_thread_kernel(const int8_t *__restrict__ slab_in, const uint8_t *__restrict__ tape, long long tape_step_stride, int K,
                           int8_t *__restrict__ slab_out, uint8_t *__restrict__ flags, int32_t *__restrict__ nnz,
                           int32_t *__restrict__ steps, long long B, int shift, int chk) {
    const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= B) return;
    uint32_t row[16]; // word 4 i + j = entries (i, j, 0..3)
    uint32_t bad = 0, nzw = 0;
    {
        const uint4 *src = reinterpret_cast<const uint4 *>(slab_in + n * 64);
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const uint4 t = __ldg(src + i);
            row[4 * i] = t.x, row[4 * i + 1] = t.y, row[4 * i + 2] = t.z, row[4 * i + 3] = t.w;
        }
#pragma unroll
        for (int e = 0; e < 16; e++) {
            nzw |= row[e];
            row[e] ^= H4;
            bad |= ~(row[e] ^ (row[e] << 1)); // the start state must already be inside [-64,63]
        }
    }
    bool alive = !FREEZE || nzw != 0;
    int until = chk, my_steps = 0;
    const uint32_t sh4 = (uint32_t)shift * ONES4, tokmax = (uint32_t)(0x7F - 2 * shift) * ONES4;
    const uint4 *rec = reinterpret_cast<const uint4 *>(tape + n * 16);
    const long long stride16 = tape_step_stride / 16;
    uint4 q = K > 0 ? __ldg(rec) : make_uint4(0, 0, 0, 0);
    for (int t = 0; t < K; t++) {
        const uint4 cur = q;
        if (t + 1 < K) q = __ldg(rec + (long long)(t + 1) * stride16); // next step's record in flight
        if (!alive) {
            if (FREEZE) break; // frozen at the zero tensor: nothing left to do for this game
            continue;
        }
        // tape contract (tg_step.cuh): every token <= 2 * shift, else the packed update may have aliased
        const uint32_t over = ((((cur.x & 0x7F7F7F7Fu) + tokmax) | cur.x) | (((cur.y & 0x7F7F7F7Fu) + tokmax) | cur.y) |
                               (((cur.z & 0x7F7F7F7Fu) + tokmax) | cur.z)) & H4;
        if (over) bad = 0xFFFFFFFFu;
        const uint32_t cu = ((cur.x | H4) - sh4) ^ H4, cv = ((cur.y | H4) - sh4) ^ H4; // int8 coefficients
        const int wi = (int)(cur.z - sh4);                                             // integer form of pack(w)
        const int u[4] = {sext_byte4<0>(cu), sext_byte4<1>(cu), sext_byte4<2>(cu), sext_byte4<3>(cu)};
        const int v[4] = {sext_byte4<0>(cv), sext_byte4<1>(cv), sext_byte4<2>(cv), sext_byte4<3>(cv)};
        uint32_t sum = 0;
#pragma unroll
        for (int i = 0; i < 4; i++)
#pragma unroll
            for (int j = 0; j < 4; j++) {
                row[4 * i + j] -= (uint32_t)(u[i] * v[j] * wi);
                sum += row[4 * i + j];
            }
        if (--until == 0) { // all entries still in [-64,63]? then chk more steps cannot alias the packed form
            until = chk;
#pragma unroll
            for (int e = 0; e < 16; e++) bad |= ~(row[e] ^ (row[e] << 1));
        }
        my_steps = t + 1;
        if (FREEZE && sum == (uint32_t)(16ull * H4)) { // checksum of the zero tensor: confirm word by word
            bool zero = true;
#pragma unroll
            for (int e = 0; e < 16; e++) zero = zero && row[e] == H4;
            if (zero) alive = false;
        }
    }
    uint32_t cnt = 0;
    uint4 *dst = reinterpret_cast<uint4 *>(slab_out + n * 64);
#pragma unroll
    for (int e = 0; e < 16; e++) {
        bad |= ~(row[e] ^ (row[e] << 1));
        row[e] ^= H4;
        cnt += (uint32_t)__popc(nonzero_mask(row[e]));
    }
#pragma unroll
    for (int i = 0; i < 4; i++) dst[i] = make_uint4(row[4 * i], row[4 * i + 1], row[4 * i + 2], row[4 * i + 3]);
    flags[n] = (uint8_t)((cnt == 0 ? TG_FLAG_TERMINAL : 0u) | ((bad & H4) != 0 ? TG_FLAG_RANGE : 0u));
    nnz[n] = (int32_t)cnt;
    if (steps) steps[n] = my_steps;
}

template <int S, int NT, int NST>
static int launch_rollout(const int8_t *slab_in, const uint8_t *tape, long long stride, int K, int8_t *slab_out,
                          uint8_t *flags, int32_t *nnz, int32_t *steps, long long B, int shift, int freeze, cudaStream_t st) {
    using C = RollCfg<S, NT, NST>;
    const long long grid = (B + C::TG - 1) / C::TG;
    if (grid > 0x7FFFFFFFLL) return TG_E_ARG;
    const int s3 = shift * shift * shift;
    const int chk = s3 >= 64 ? 1 : 64 / s3;
    rollout_kernel<S, NT, NST><<<(int)grid, NT + 32, C::SMEM_BYTES, st>>>(slab_in, tape, stride, K, slab_out, flags, nnz, steps, B,
                                                                     shift, chk, freeze);
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

} // namespace tg

static int rollout_dispatch(const int8_t *slab_in, const uint8_t *tape, int64_t tape_step_stride, int K, int8_t *slab_out,
                            uint8_t *flags, int32_t *nnz, int32_t *steps, int64_t B, int S, int shift, int freeze,
                            void *stream) {
    const int rc = tg::check_rollout(S, B, K, shift, slab_in, tape, tape_step_stride, slab_out, flags, nnz, steps, freeze);
    if (rc != tg::LAUNCH) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    switch (S) {
    case 4: {
#ifdef TG_TUNING
        if (tg::tuning_env("TG_ROLLOUT_COLUMNS", 0)) // A/B: the word-column kernel
            return tg::launch_rollout<4, 256, 4>(slab_in, tape, tape_step_stride, K, slab_out, flags, nnz, steps, B, shift, freeze, st);
#endif
        const int s3 = shift * shift * shift;
        const int chk = s3 >= 64 ? 1 : 64 / s3;
        const long long grid = (B + 127) / 128;
        if (grid > 0x7FFFFFFFLL) return TG_E_ARG;
        if (freeze) tg::rollout4_thread_kernel<true><<<(int)grid, 128, 0, st>>>(slab_in, tape, tape_step_stride, K, slab_out, flags, nnz, steps, B, shift, chk);
        else tg::rollout4_thread_kernel<false><<<(int)grid, 128, 0, st>>>(slab_in, tape, tape_step_stride, K, slab_out, flags, nnz, steps, B, shift, chk);
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    }
    case 9:
#ifdef TG_TUNING
        if (tg::tuning_env("TG_ROLLOUT_COLUMNS", 0)) // A/B: the word-column kernel of this file
            return tg::launch_rollout<9, 256, 4>(slab_in, tape, tape_step_stride, K, slab_out, flags, nnz, steps, B, shift, freeze, st);
#endif
        return tg::launch_rollout_rows(slab_in, tape, tape_step_stride, K, slab_out, flags, nnz, steps, B, 9, shift, freeze, st);
    case 16:
#ifdef TG_TUNING
        if (tg::tuning_env("TG_ROLLOUT_COLUMNS", 0))
            return tg::launch_rollout<16, 256, 4>(slab_in, tape, tape_step_stride, K, slab_out, flags, nnz, steps, B, shift, freeze, st);
#endif
        return tg::launch_rollout_rows(slab_in, tape, tape_step_stride, K, slab_out, flags, nnz, steps, B, 16, shift, freeze, st);
    case 25: // the word-column kernel: 25 row words per thread, two games (314 of 320 compute threads) per CTA
        return tg::launch_rollout<25, 320, 4>(slab_in, tape, tape_step_stride, K, slab_out, flags, nnz, steps, B, shift, freeze, st);
    }
    return TG_E_ARG;
}

extern "C" {

int tg_rollout(const int8_t *slab_in, const uint8_t *tape, int64_t tape_step_stride, int K, int8_t *slab_out, uint8_t *flags,
               int32_t *nnz, int32_t *steps, int64_t B, int S, int shift, void *stream) {
    return rollout_dispatch(slab_in, tape, tape_step_stride, K, slab_out, flags, nnz, steps, B, S, shift, 1, stream);
}

int tg_replay(const int8_t *slab_in, const uint8_t *tape, int64_t tape_step_stride, int K, int8_t *slab_out, uint8_t *flags,
              int32_t *nnz, int64_t B, int S, int shift, void *stream) {
    return rollout_dispatch(slab_in, tape, tape_step_stride, K, slab_out, flags, nnz, nullptr, B, S, shift, 0, stream);
}

} // extern "C"
