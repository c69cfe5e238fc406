// tg_step.cu -- K1: batched TensorGame transition (C ABI: tg_step).
//
// Persistent, warp-specialised kernel.  Each CTA walks tiles of TG games:
//   producer warp (one elected lane): TMA 1-D bulk copies (cp.async.bulk) of
//     the tile's slab bytes and token bytes into an NSTAGE-deep shared-memory
//     ring, completion on mbarriers; after the compute warps release a stage it
//     bulk-stores the updated slab back to HBM and refills the stage.
//   compute warps: WR threads per game, one IMAD per 32-bit word (tg_step.cuh),
//     per-game nnz/flags reduced through shared memory and written directly.
// HBM traffic per game = 2*GP + TP + 5 bytes, every access a full line.
#include "tg_step.cuh"

namespace tg {

int g_last_cuda_error = 0;

template <int S, int NT, int NPASS, int NSTAGE>
struct StepCfg {
    using G = Geo<S>;
    static constexpr int GPASS = NT / G::WR;                // games per pass over the compute threads
    static constexpr int TG = GPASS * NPASS;                // games per tile
    static constexpr int ACTIVE = GPASS * G::WR;            // compute threads that own a word column
    static constexpr int SLAB_BYTES = TG * G::GP;
    static constexpr int TOK_BYTES = TG * G::TP;
    static constexpr int STAGE_BYTES = SLAB_BYTES + TOK_BYTES;
    // partial words per game handed to the reducer thread
    static constexpr int PW = (G::WR % 32 == 0) ? G::WR / 32 : ((32 % G::WR == 0) ? 1 : G::WR);
    static constexpr int PART_WORDS = TG * PW;
    static constexpr int SMEM_BYTES = NSTAGE * STAGE_BYTES + 2 * PART_WORDS * 4 + 2 * NSTAGE * 8;
    static constexpr int THREADS = NT + 32;
};

template <int S, int NT, int NPASS, int NSTAGE>
__global__ void __launch_bounds__(NT + 32)
    step_kernel(const int8_t *__restrict__ slab_in, const uint8_t *__restrict__ tape, int8_t *__restrict__ slab_out,
                uint8_t *__restrict__ flags, int32_t *__restrict__ nnz, long long B, int shift) {
    using C = StepCfg<S, NT, NPASS, NSTAGE>;
    using G = Geo<S>;
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
            mbar_expect_tx(&full[s], (uint32_t)(ng * (G::GP + G::TP)));
            bulk_g2s(st, slab_in + g0 * G::GP, (uint32_t)(ng * G::GP), &full[s]);
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
            bulk_s2g(slab_out + g0 * G::GP, smem + s * C::STAGE_BYTES, (uint32_t)(ng * G::GP));
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
    Lane<S> L;
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
#pragma unroll
        for (int p = 0; p < NPASS; p++) {
            const int g = p * C::GPASS + gl;
            uint32_t pr = 0;
            if (active && g < ng) pr = rank1_update<S, -1>(slab + g * G::GP, toks + g * G::TP, L, shift);
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
        fence_proxy_async(); // slab writes -> async proxy, before the producer's bulk store
        asm volatile("bar.sync 1, %0;" ::"n"(NT) : "memory");
        if (tid == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&done[s])) : "memory");
        for (int g = tid; g < ng; g += NT) {
            uint32_t sum = 0;
#pragma unroll
            for (int w = 0; w < C::PW; w++) sum += pp[g * C::PW + w];
            flags[g0 + g] = (uint8_t)partial_flags(sum);
            nnz[g0 + g] = (int32_t)(sum & 0xFFFFu);
        }
    }
}

// ---------------------------------------------------------------- host side
int sm_count() {
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (!cached[dev]) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached[dev] = n;
    }
    return cached[dev];
}

#ifdef TG_TUNING
static int g_step_ctas_per_sm = 0; // 0 = per-size default
static int g_step_variant = 0;     // tuning sweeps only
#endif

template <int S, int NT, int NPASS, int NSTAGE>
static int launch_step(const int8_t *slab_in, const uint8_t *tape, int8_t *slab_out, uint8_t *flags, int32_t *nnz,
                       long long B, int shift, int ctas_per_sm, cudaStream_t stream) {
    using C = StepCfg<S, NT, NPASS, NSTAGE>;
    auto kern = step_kernel<S, NT, NPASS, NSTAGE>;
    TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
    const long long ntiles = (B + C::TG - 1) / C::TG;
#ifdef TG_TUNING
    if (g_step_ctas_per_sm > 0) ctas_per_sm = g_step_ctas_per_sm;
#endif
    const long long cap = (long long)sm_count() * ctas_per_sm;
    const int grid = (int)(ntiles < cap ? ntiles : cap);
    kern<<<grid, C::THREADS, C::SMEM_BYTES, stream>>>(slab_in, tape, slab_out, flags, nnz, B, shift);
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

} // namespace tg

extern "C" {

int tg_version(void) { return TG_VERSION; }
int tg_last_cuda_error(void) { return tg::g_last_cuda_error; }

const char *tg_error_string(int code) {
    switch (code) {
    case TG_OK: return "ok";
    case TG_E_ARG: return "bad argument";
    case TG_E_CUDA: return "CUDA runtime error (see tg_last_cuda_error)";
    case TG_E_RANGE: return "value does not fit the device format";
    default: return "unknown error";
    }
}

int tg_layout(int S, int *row_pitch, int *game_pitch, int *token_pitch) {
    if (!tg::supported_S(S)) return TG_E_ARG;
    const int rp = (S * S + 3) & ~3;
    if (row_pitch) *row_pitch = rp;
    if (game_pitch) *game_pitch = (S * rp + 15) & ~15;
    if (token_pitch) *token_pitch = (3 * S + 15) & ~15;
    return TG_OK;
}

#ifdef TG_TUNING
// tuning knobs for bench sweeps: CTAs launched per SM (0 = default) and kernel variant
int tg_tune_step_ctas_per_sm(int n) {
    tg::g_step_ctas_per_sm = n;
    return TG_OK;
}
int tg_tune_step_variant(int v) {
    tg::g_step_variant = v;
    return TG_OK;
}
#endif

int tg_step(const int8_t *slab_in, const uint8_t *tape, int8_t *slab_out, uint8_t *flags, int32_t *nnz, int64_t B, int S,
            int shift, void *stream) {
    if (const int rc = tg::check_step(S, B, shift, slab_in, tape, slab_out, flags, nnz); rc != tg::LAUNCH) return rc;
    cudaStream_t st = (cudaStream_t)stream;
#ifdef TG_TUNING
    switch (S * 10 + tg::g_step_variant) { // sweep-only instantiations
    case 41: return tg::launch_step<4, 256, 2, 2>(slab_in, tape, slab_out, flags, nnz, B, shift, 32, st);
    case 42: return tg::launch_step<4, 256, 4, 3>(slab_in, tape, slab_out, flags, nnz, B, shift, 32, st);
    case 43: return tg::launch_step<4, 256, 8, 2>(slab_in, tape, slab_out, flags, nnz, B, shift, 32, st);
    case 91: return tg::launch_step<9, 256, 1, 3>(slab_in, tape, slab_out, flags, nnz, B, shift, 5, st);
    case 92: return tg::launch_step<9, 256, 1, 4>(slab_in, tape, slab_out, flags, nnz, B, shift, 5, st);
    case 93: return tg::launch_step<9, 256, 4, 2>(slab_in, tape, slab_out, flags, nnz, B, shift, 32, st);
    case 94: return tg::launch_step<9, 512, 1, 3>(slab_in, tape, slab_out, flags, nnz, B, shift, 3, st);
    case 95: return tg::launch_step<9, 128, 2, 3>(slab_in, tape, slab_out, flags, nnz, B, shift, 7, st);
    case 96: return tg::launch_step<9, 128, 4, 3>(slab_in, tape, slab_out, flags, nnz, B, shift, 5, st);
    case 97: return tg::launch_step<9, 256, 2, 3>(slab_in, tape, slab_out, flags, nnz, B, shift, 32, st);
    case 161: return tg::launch_step<16, 256, 1, 3>(slab_in, tape, slab_out, flags, nnz, B, shift, 32, st);
    case 162: return tg::launch_step<16, 256, 2, 2>(slab_in, tape, slab_out, flags, nnz, B, shift, 32, st);
    case 163: return tg::launch_step<16, 512, 1, 2>(slab_in, tape, slab_out, flags, nnz, B, shift, 32, st);
    default: break;
    }
#endif
    // measured best (profiles/r01_sweep_step_S9.txt): 32 short CTAs per SM, two-stage ring
    switch (S) {
    case 4: return tg::launch_step<4, 256, 4, 2>(slab_in, tape, slab_out, flags, nnz, B, shift, 32, st);
    case 9: return tg::launch_step<9, 256, 2, 2>(slab_in, tape, slab_out, flags, nnz, B, shift, 32, st);
    case 16: return tg::launch_step<16, 256, 1, 2>(slab_in, tape, slab_out, flags, nnz, B, shift, 32, st);
    // 25x25x25: 157 word columns per game, so five compute warps hold one game with three threads idle (256 would leave 99);
    // shared memory (two 15.8 KB stages) allows seven such CTAs per SM
    case 25: return tg::launch_step<25, 160, 1, 2>(slab_in, tape, slab_out, flags, nnz, B, shift, 32, st);
    }
    return TG_E_ARG;
}

} // extern "C"
