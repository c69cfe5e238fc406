// tg_convert.cu -- boundary conversions between the reference's dtypes
// (float32 residual tensors, int64 action tokens) and the device formats.
// Pure streaming kernels; they run only where the Python API hands data to or
// from reference-typed code (model.py consumes float32 states).
#include "tg_common.cuh"

namespace tg {

// one thread per 32-bit slab word: four floats in with the widest loads their address allows (load_run)
template <int S>
__global__ void pack_f32_kernel(const float *__restrict__ src, long long src_stride, uint32_t *__restrict__ slab,
                                long long B, int32_t *range_flag) {
    using G = Geo<S>;
    constexpr int WG = G::GP / 4; // words per game
    const long long total = B * WG;
    bool bad = false;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long b = idx / WG;
        const int wg = (int)(idx % WG);
        const int i = wg / G::WR, c = wg % G::WR;
        uint32_t word = 0;
        if (i < S) {
            const int nv = min(4, G::S2 - 4 * c);
            float f[4];
            load_run<S>(src + b * src_stride + i * G::S2 + 4 * c, nv, f);
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const int v = __float2int_rn(f[q]); // entries beyond nv are 0.f
                bad |= ((float)v != f[q]) | (v < -128) | (v > 127);
                word |= ((uint32_t)v & 0xFFu) << (8 * q);
            }
        }
        slab[idx] = word;
    }
    if (bad && range_flag) atomicOr(range_flag, 1);
}

// one thread per 32-bit slab word: four floats out with the widest stores their address allows (store_run)
template <int S>
__global__ void expand_f32_kernel(const int8_t *__restrict__ slab, float *__restrict__ dst, long long dst_stride,
                                  long long B) {
    using G = Geo<S>;
    constexpr int WG = S * G::WR; // words of the S rows (the game padding is not read)
    const long long total = B * WG;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long b = idx / WG;
        const int wg = (int)(idx % WG);
        const int i = wg / G::WR, c = wg % G::WR;
        const uint32_t w = __ldg(reinterpret_cast<const uint32_t *>(slab + b * G::GP + i * G::RP) + c);
        store_run<S>(dst + b * dst_stride + i * G::S2 + 4 * c, min(4, G::S2 - 4 * c), (float)(int8_t)(w & 0xFFu),
                     (float)(int8_t)((w >> 8) & 0xFFu), (float)(int8_t)((w >> 16) & 0xFFu), (float)(int8_t)(w >> 24));
    }
}

template <int S>
__global__ void pack_actions_kernel(const int64_t *__restrict__ actions, uint8_t *__restrict__ tape, long long B,
                                    int32_t *range_flag) {
    using G = Geo<S>;
    const long long total = B * G::TP;
    bool bad = false;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long b = idx / G::TP;
        const int q = (int)(idx % G::TP);
        uint8_t t = 0;
        if (q < 3 * S) {
            const int64_t a = actions[b * 3 * S + q];
            bad |= (a < 0) | (a > 255);
            t = (uint8_t)a;
        }
        tape[idx] = t;
    }
    if (bad && range_flag) atomicOr(range_flag, 1);
}

template <int S>
__global__ void unpack_actions_kernel(const uint8_t *__restrict__ tape, int64_t *__restrict__ actions, long long B) {
    using G = Geo<S>;
    const long long total = B * 3 * S;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long b = idx / (3 * S);
        const int q = (int)(idx % (3 * S));
        actions[idx] = (int64_t)tape[b * G::TP + q];
    }
}

static inline int grid_for(long long total, int block) {
    long long g = (total + block - 1) / block;
    const long long cap = 148LL * 16;
    return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

} // namespace tg

extern "C" {

int tg_pack_f32(const float *src, int64_t src_stride, int8_t *slab, int64_t B, int S, int32_t *range_flag, void *stream) {
    if (const int rc = tg::check_pair(S, B, src, 4, slab, 16); rc != tg::LAUNCH) return rc;
    return tg::with_S(S, [&](auto s) {
        constexpr int kS = decltype(s)::value;
        tg::pack_f32_kernel<kS><<<tg::grid_for(B * (tg::Geo<kS>::GP / 4), 256), 256, 0, (cudaStream_t)stream>>>(
            src, src_stride, reinterpret_cast<uint32_t *>(slab), B, range_flag);
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    });
}

int tg_expand_f32(const int8_t *slab, float *dst, int64_t dst_stride, int64_t B, int S, void *stream) {
    if (const int rc = tg::check_pair(S, B, slab, 16, dst, 4); rc != tg::LAUNCH) return rc;
    return tg::with_S(S, [&](auto s) {
        constexpr int kS = decltype(s)::value;
        tg::expand_f32_kernel<kS><<<tg::grid_for(B * kS * tg::Geo<kS>::WR, 256), 256, 0, (cudaStream_t)stream>>>(slab, dst, dst_stride, B);
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    });
}

int tg_pack_actions_i64(const int64_t *actions, uint8_t *tape, int64_t B, int S, int32_t *range_flag, void *stream) {
    if (const int rc = tg::check_pair(S, B, actions, 8, tape, 16); rc != tg::LAUNCH) return rc;
    return tg::with_S(S, [&](auto s) {
        constexpr int kS = decltype(s)::value;
        tg::pack_actions_kernel<kS><<<tg::grid_for(B * tg::Geo<kS>::TP, 256), 256, 0, (cudaStream_t)stream>>>(actions, tape, B, range_flag);
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    });
}

int tg_unpack_actions_i64(const uint8_t *tape, int64_t *actions, int64_t B, int S, void *stream) {
    if (const int rc = tg::check_pair(S, B, tape, 16, actions, 8); rc != tg::LAUNCH) return rc;
    return tg::with_S(S, [&](auto s) {
        constexpr int kS = decltype(s)::value;
        tg::unpack_actions_kernel<kS><<<tg::grid_for(B * 3 * kS, 256), 256, 0, (cudaStream_t)stream>>>(tape, actions, B);
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    });
}

} // extern "C"
