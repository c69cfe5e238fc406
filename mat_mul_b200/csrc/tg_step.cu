// tg_step.cu -- K1: batched TensorGame transition (C ABI: tg_step), step_kernel (tg_step.cuh) on int8 slabs.
#include "tg_step.cuh"

namespace tg {

int g_last_cuda_error = 0;

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

// CTAs per SM of an int8 step launch: the per-size default n, or the tuning sweeps' override
static int step_ctas_per_sm(int n) {
#ifdef TG_TUNING
    if (g_step_ctas_per_sm > 0) return g_step_ctas_per_sm;
#endif
    return n;
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
    case 41: return tg::launch_step<4, 256, 2, 2, tg::W8>(slab_in, tape, slab_out, flags, nnz, B, shift, tg::step_ctas_per_sm(32), st);
    case 42: return tg::launch_step<4, 256, 4, 3, tg::W8>(slab_in, tape, slab_out, flags, nnz, B, shift, tg::step_ctas_per_sm(32), st);
    case 43: return tg::launch_step<4, 256, 8, 2, tg::W8>(slab_in, tape, slab_out, flags, nnz, B, shift, tg::step_ctas_per_sm(32), st);
    case 91: return tg::launch_step<9, 256, 1, 3, tg::W8>(slab_in, tape, slab_out, flags, nnz, B, shift, tg::step_ctas_per_sm(5), st);
    case 92: return tg::launch_step<9, 256, 1, 4, tg::W8>(slab_in, tape, slab_out, flags, nnz, B, shift, tg::step_ctas_per_sm(5), st);
    case 93: return tg::launch_step<9, 256, 4, 2, tg::W8>(slab_in, tape, slab_out, flags, nnz, B, shift, tg::step_ctas_per_sm(32), st);
    case 94: return tg::launch_step<9, 512, 1, 3, tg::W8>(slab_in, tape, slab_out, flags, nnz, B, shift, tg::step_ctas_per_sm(3), st);
    case 95: return tg::launch_step<9, 128, 2, 3, tg::W8>(slab_in, tape, slab_out, flags, nnz, B, shift, tg::step_ctas_per_sm(7), st);
    case 96: return tg::launch_step<9, 128, 4, 3, tg::W8>(slab_in, tape, slab_out, flags, nnz, B, shift, tg::step_ctas_per_sm(5), st);
    case 97: return tg::launch_step<9, 256, 2, 3, tg::W8>(slab_in, tape, slab_out, flags, nnz, B, shift, tg::step_ctas_per_sm(32), st);
    case 161: return tg::launch_step<16, 256, 1, 3, tg::W8>(slab_in, tape, slab_out, flags, nnz, B, shift, tg::step_ctas_per_sm(32), st);
    case 162: return tg::launch_step<16, 256, 2, 2, tg::W8>(slab_in, tape, slab_out, flags, nnz, B, shift, tg::step_ctas_per_sm(32), st);
    case 163: return tg::launch_step<16, 512, 1, 2, tg::W8>(slab_in, tape, slab_out, flags, nnz, B, shift, tg::step_ctas_per_sm(32), st);
    default: break;
    }
#endif
    // measured best (profiles/r01_sweep_step_S9.txt): 32 short CTAs per SM, two-stage ring
    switch (S) {
    case 4: return tg::launch_step<4, 256, 4, 2, tg::W8>(slab_in, tape, slab_out, flags, nnz, B, shift, tg::step_ctas_per_sm(32), st);
    case 9: return tg::launch_step<9, 256, 2, 2, tg::W8>(slab_in, tape, slab_out, flags, nnz, B, shift, tg::step_ctas_per_sm(32), st);
    case 16: return tg::launch_step<16, 256, 1, 2, tg::W8>(slab_in, tape, slab_out, flags, nnz, B, shift, tg::step_ctas_per_sm(32), st);
    // 25x25x25: 157 word columns per game, so five compute warps hold one game with three threads idle (256 would leave 99);
    // shared memory (two 15.8 KB stages) allows seven such CTAs per SM
    case 25: return tg::launch_step<25, 160, 1, 2, tg::W8>(slab_in, tape, slab_out, flags, nnz, B, shift, tg::step_ctas_per_sm(32), st);
    }
    return TG_E_ARG;
}

} // extern "C"
