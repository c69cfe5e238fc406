// tg_i16.cu -- the game path on int16 slabs: the entry points tg_step_i16, tg_expand_children_i16 (step_kernel and
// expand_kernel of tg_step.cuh on W16), K2 tg_rollout_i16 / tg_replay_i16 (rollout16_kernel) and K7 tg_state_key_i16
// (state_key16_kernel).  K6 tg_slice_rank_i16 is slice_rank_kernel in tg_aux.cu.
//
// Residuals the int8 slab cannot hold (change-of-basis outputs, demo targets beyond int8, start tensors with large
// entries) are played here.  The int16 slab has the int8 slab's geometry counted in elements (W16, tg_step.cuh).
#include "tg_step.cuh"

namespace tg {

// ------------------------------------------------------------------ K2: word-column rollout / replay on int16 games
// Thread (game, word column) keeps its S row words in registers for all K steps and reads each step's record straight
// from the tape (the threads of a game read the same record: L1 broadcasts).  The zone is tested after every applied
// step (one SWAR test per word), so TG_FLAG_RANGE means: the start state or the state after some applied step had an
// entry outside [-16384, 16383], or an applied step's record broke the token bound.  FREEZE: a game stops at the first
// all-zero state (the break at act.py:49), decided by one vote per step in shared memory (three buffers, so one CTA
// barrier per step is enough: a buffer is cleared one barrier after its last read and rewritten one barrier later).
template <int S, int NT>
struct Roll16Cfg {
    using G = GeoW<S, W16>;
    static constexpr int TG = NT / G::WR;
    static constexpr int ACTIVE = TG * G::WR;
};

template <int S, int NT, bool FREEZE>
__global__ void __launch_bounds__(NT)
    rollout16_kernel(const int16_t *__restrict__ slab_in, const uint8_t *__restrict__ tape, long long tape_step_stride, int K,
                     int16_t *__restrict__ slab_out, uint8_t *__restrict__ flags, int32_t *__restrict__ nnz,
                     int32_t *__restrict__ steps, long long B, int shift) {
    using C = Roll16Cfg<S, NT>;
    using G = GeoW<S, W16>;
    __shared__ uint32_t s_nz[3][C::TG]; // per step: the game is non-zero after it ([2]: the start state)
    __shared__ uint32_t s_sum[C::TG];
    __shared__ uint32_t s_steps[C::TG];

    const int tid = threadIdx.x;
    const long long g0 = (long long)blockIdx.x * C::TG;
    const int ng = (int)min((long long)C::TG, B - g0);
    const int g = tid / G::WR;
    const bool active = tid < C::ACTIVE && g < ng;
    W16::Lane<S> L;
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
            row[i] = t ^ W16::H;
            bad |= ~(row[i] ^ (row[i] << 1)); // offset-binary: bits 15 / 31 equal to bits 14 / 30 <=> outside the zone
        }
    } else {
#pragma unroll
        for (int i = 0; i < S; i++) row[i] = W16::H;
    }
    if (active && nzw) s_nz[2][g] = 1;
    __syncthreads();
    bool alive = active && (!FREEZE || s_nz[2][g] != 0);
    int my_steps = 0;
    const uint8_t *rec = tape + (g0 + g) * G::TP;

    for (int t = 0; t < K; t++, rec += tape_step_stride) {
        if (alive) {
            const uint32_t vw = W16::pack_vw<S>(rec, L, shift);
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
                any |= row[i] ^ W16::H;
                bad |= ~(row[i] ^ (row[i] << 1));
            }
            tok_over = tok_over || tokens_out_of_range<S, W16>(rec, L, shift);
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
            const uint32_t t = row[i] ^ W16::H;
            dst[i * G::WR] = t;
            cnt += nonzero_lanes<W16>(t, L.hv);
        }
        atomicAdd(&s_sum[g], make_partial<W16>(W16::lane_sum(cnt), true, (bad & L.hv) != 0 || tok_over));
        if (L.c == 0) s_steps[g] = (uint32_t)my_steps;
    }
    __syncthreads();
    for (int q = tid; q < ng; q += NT) {
        const uint32_t sum = s_sum[q];
        flags[g0 + q] = (uint8_t)(partial_flags<W16>(sum) & ~TG_FLAG_NULL);
        nnz[g0 + q] = (int32_t)partial_nnz<W16>(sum);
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
// formats.  One thread per word column (W16::ColumnKey), the WR partial sums of a game reduced by one warp.
template <int S, int NT>
__global__ void __launch_bounds__(NT) state_key16_kernel(const int16_t *__restrict__ slab, unsigned long long *__restrict__ keys,
                                                         long long B) {
    using G = GeoW<S, W16>;
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
            for (int i = 0; i < S; i++) w[i] = __ldg(col + i * G::WR) ^ W16::H;
        } else {
#pragma unroll
            for (int i = 0; i < S; i++) w[i] = W16::H;
        }
        W16::ColumnKey<S> ck;
        ck.init(c);
        s_ph[tid] = ck(w);
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
    case 4: return tg::launch_step<4, 256, 4, 2, tg::W16>(slab_in, tape, slab_out, flags, nnz, B, shift, 32, st);
    case 9: return tg::launch_step<9, 256, 2, 2, tg::W16>(slab_in, tape, slab_out, flags, nnz, B, shift, 32, st);
    case 16: return tg::launch_step<16, 256, 1, 2, tg::W16>(slab_in, tape, slab_out, flags, nnz, B, shift, 32, st);
    // 25x25x25: 314 word columns per game, ten compute warps hold one game; two 31.5 KB stages
    case 25: return tg::launch_step<25, 320, 1, 2, tg::W16>(slab_in, tape, slab_out, flags, nnz, B, shift, 32, st);
    }
    return TG_E_ARG;
}

int tg_expand_children_i16(const int16_t *parents, const uint8_t *tape, int k, int16_t *children, uint8_t *flags, int32_t *nnz,
                           uint64_t *keys, int64_t B, int S, int shift, void *stream) {
    if (const int rc = tg::check_expand(S, B, k, shift, parents, tape, children, flags, nnz); rc != tg::LAUNCH) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    unsigned long long *kp = (unsigned long long *)keys;
    switch (S) {
    case 4: return tg::launch_expand<4, 128, tg::W16>(parents, tape, k, children, flags, nnz, kp, B, shift, st);
    case 9: return tg::launch_expand<9, 256, tg::W16>(parents, tape, k, children, flags, nnz, kp, B, shift, st);
    case 16: return tg::launch_expand<16, 256, tg::W16>(parents, tape, k, children, flags, nnz, kp, B, shift, st);
    case 25: return tg::launch_expand<25, 320, tg::W16>(parents, tape, k, children, flags, nnz, kp, B, shift, st); // one parent per CTA
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
    case 4: tg::state_key16_kernel<4, 256><<<grid(256 / tg::GeoW<4, tg::W16>::WR), 256, 0, st>>>(slab16, kp, B); break;
    case 9: tg::state_key16_kernel<9, 256><<<grid(256 / tg::GeoW<9, tg::W16>::WR), 256, 0, st>>>(slab16, kp, B); break;
    case 16: tg::state_key16_kernel<16, 256><<<grid(256 / tg::GeoW<16, tg::W16>::WR), 256, 0, st>>>(slab16, kp, B); break;
    case 25: tg::state_key16_kernel<25, 320><<<grid(1), 320, 0, st>>>(slab16, kp, B); break;
    default: return TG_E_ARG;
    }
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

} // extern "C"
