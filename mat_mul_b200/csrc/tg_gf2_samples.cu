// tg_gf2_samples.cu -- float32 states from bit slabs: K4 tg_demo_sample_gf2 (training samples modulo 2 from a demo-major
// store with bit-slab targets) and tg_expand_f32_gf2 (a bit slab to the float32 states the model consumes).
//
// Both kernels build the bits of a run of consecutive states in a warp-private image in shared memory -- the rows of the
// states one after the other, RW words each, as in a bit slab -- and then write the run's floats with one shared store
// routine (store_run_bits): lane l writes floats 4 l, 4 l + 1, ... of each 128-float stretch, so one store instruction of
// the warp covers 512 contiguous bytes, with 16-byte stores wherever the run's alignment allows them.  A float is
// __int_as_float(0x3F800000 & -bit): 0.0f or 1.0f.
//
// Sampler work split: a unit is one state slot (sample b, slot s) of the output, flat index b * dim_t + s, and its S^3
// floats follow those of the unit before it in `states`.  A warp takes UPW consecutive units at a time (one run), one
// thread per row of a unit at 9, 16 and 25 (27 / 32 / 25 lanes busy) and one thread per unit at 4 (its four 16-bit rows
// in four registers).  A thread builds its rows in registers, in the formulation of tg_gf2.cu: the term of a record is
// V = OR_{j: v_j odd} (w bits) << (j S) in every row i with u_i odd.  Slot 0 is the target's rows with the terms of
// records a+1 .. R-1 xored in; a history slot is one term.  Records are read straight from the store, so no R is too
// long for shared memory.
#include "tg_gf2.cuh"

namespace tg {
namespace {

template <int S>
struct SampB {
    using B = GeoB<S>;
    static constexpr int RPT = S == 4 ? 4 : 1;             // rows per thread
    static constexpr int TPU = S / RPT;                    // threads per unit (state slot)
    static constexpr int UPW = 32 / TPU;                   // units per warp and run: 32 / 3 / 2 / 1
    static constexpr int IMG = UPW * S * B::RW;            // words of a run's rows
    static constexpr int PITCH = (IMG + 1 + 3) & ~3;       // warp image pitch: one word beyond the rows for the funnel shift
    static constexpr int WARPS = 8;                        // warps per 256-thread CTA
};

// bit e of the run (float e: row e / S^2, entry e % S^2 of that row)
template <int S>
__device__ __forceinline__ uint32_t run_bit(const uint32_t *img, int e) {
    constexpr int S2 = S * S, RW = GeoB<S>::RW;
    const int r = e / S2, jk = e - r * S2;
    return (img[r * RW + (jk >> 5)] >> (jk & 31)) & 1u;
}

// bits e .. e+3 of the run in bits 0..3 (a row ends inside the four at 9 and 25, and at every size for runs that start
// off a 16-byte boundary)
template <int S>
__device__ __forceinline__ uint32_t run_bits4(const uint32_t *img, int e) {
    constexpr int S2 = S * S, RW = GeoB<S>::RW;
    const int r = e / S2, jk = e - r * S2, p = r * RW * 32 + jk;
    uint32_t x = __funnelshift_r(img[p >> 5], img[(p >> 5) + 1], p & 31);
    if (jk > S2 - 4) { // the next row supplies the last 4 - n bits
        const int n = S2 - jk;
        x = (x & ((1u << n) - 1u)) | (img[(r + 1) * RW] << n);
    }
    return x;
}

__device__ __forceinline__ float bit_float(uint32_t x, int q) { return __int_as_float(0x3F800000 & -(int)((x >> q) & 1u)); }

// The warp writes floats 0 .. n-1 of a run to dst (any float address): the floats before the first 16-byte boundary and
// after the last one singly, the rest as 16-byte stores, lane l on the l-th four of every 128 floats.
template <int S>
__device__ __forceinline__ void store_run_bits(const uint32_t *img, float *dst, int n, int lane) {
    const int h = min((int)((16u - ((uint32_t)reinterpret_cast<uintptr_t>(dst) & 15u)) & 15u) >> 2, n);
    if (lane < h) st_f32(dst + lane, bit_float(run_bit<S>(img, lane), 0));
    const int body = (n - h) & ~3;
    for (int e = h + 4 * lane; e < h + body; e += 128) {
        const uint32_t x = run_bits4<S>(img, e);
        st_f32x4(dst + e, bit_float(x, 0), bit_float(x, 1), bit_float(x, 2), bit_float(x, 3));
    }
    const int t = h + body + lane;
    if (t < n) st_f32(dst + t, bit_float(run_bit<S>(img, t), 0));
}

// x = q d + r for x >= 0; a 32-bit division below 2^32 (every realistic batch and store)
__device__ __forceinline__ void split(long long x, int d, long long &q, int &r) {
    if ((unsigned long long)x < 0x100000000ULL) {
        const uint32_t q32 = (uint32_t)x / (uint32_t)d;
        q = (long long)q32, r = (int)((uint32_t)x - q32 * (uint32_t)d);
    } else {
        q = x / d, r = (int)(x - q * d);
    }
}

template <int S>
__global__ void __launch_bounds__(256) demo_sample_gf2_kernel(const uint8_t *__restrict__ tape_dm, const uint32_t *__restrict__ targets,
                                                              long long N, int R, int dim_t, int shift, const long long *__restrict__ idx,
                                                              long long nb, float *__restrict__ states, float *__restrict__ scalars,
                                                              long long *__restrict__ actions, float *__restrict__ rewards) {
    using B = GeoB<S>;
    using P = SampB<S>;
    constexpr int RW = B::RW, RPT = P::RPT, GW = B::GB / 4, S3 = S * S * S;
    __shared__ __align__(16) uint32_t s_img[P::WARPS * P::PITCH];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t *img = s_img + warp * P::PITCH;
    if (lane == 0) img[P::IMG] = 0;
    const int slot = lane / P::TPU, r0 = (lane - slot * P::TPU) * RPT;
    const long long units = nb * dim_t;
    for (long long u0 = ((long long)blockIdx.x * P::WARPS + warp) * P::UPW; u0 < units; u0 += (long long)gridDim.x * P::WARPS * P::UPW) {
        const long long u = u0 + slot;
        uint32_t row[RPT][RW];
#pragma unroll
        for (int k = 0; k < RPT; k++)
#pragma unroll
            for (int w = 0; w < RW; w++) row[k][w] = 0;
        if (slot < P::UPW && u < units) {
            long long b, demo = -1;
            int s, a = 0;
            split(u, dim_t, b, s);
            const long long id = idx[b];
            if (id >= 0) split(id, R, demo, a);
            if (demo >= 0 && demo < N) {
                const uint8_t *rec = tape_dm + (size_t)demo * R * B::TP;
                if (s == 0) {
                    const uint32_t *t = targets + (size_t)demo * GW + r0 * RW;
#pragma unroll
                    for (int k = 0; k < RPT; k++)
#pragma unroll
                        for (int w = 0; w < RW; w += RW % 4 ? 1 : 4) {
                            if constexpr (RW % 4 == 0) { // 16 and 25: rows of 32 and 80 bytes
                                const uint4 v = __ldg(reinterpret_cast<const uint4 *>(t + k * RW + w));
                                row[k][w] = v.x, row[k][w + 1] = v.y, row[k][w + 2] = v.z, row[k][w + 3] = v.w;
                            } else {
                                row[k][w] = __ldg(t + k * RW + w);
                            }
                        }
#pragma unroll 2
                    for (int j = a + 1; j < R; j++) xor_term<S, RPT>(row, parities<S>(rec + (size_t)j * B::TP, shift), r0);
                    if (r0 == 0) {
                        scalars[b] = (float)(R - a);
                        rewards[b] = -(float)(a + 1);
                    }
                    const uint8_t *ta = rec + (size_t)a * B::TP; // the sample's own action: raw tokens
                    for (int q = r0 / RPT; q < 3 * S; q += P::TPU) actions[b * 3 * S + q] = (long long)ta[q];
                } else {
                    const int j = min(a + dim_t, R) - s;
                    if (j > a) xor_term<S, RPT>(row, parities<S>(rec + (size_t)j * B::TP, shift), r0);
                }
            }
        }
        if (slot < P::UPW) {
#pragma unroll
            for (int k = 0; k < RPT; k++)
#pragma unroll
                for (int w = 0; w < RW; w++) img[(slot * S + r0 + k) * RW + w] = row[k][w];
        }
        __syncwarp();
        const long long nu = units - u0 < P::UPW ? units - u0 : P::UPW;
        store_run_bits<S>(img, states + u0 * S3, (int)nu * S3, lane);
        __syncwarp();
    }
}

// bit slab -> float32: a warp stages UPW games' rows (the padding word of a 9x9x9 game dropped) and writes each game's S^3
// floats at dst + b * dst_stride, the UPW games as one run when they are contiguous (dst_stride == S^3)
template <int S>
__global__ void __launch_bounds__(256) expand_f32_gf2_kernel(const uint32_t *__restrict__ bits, float *__restrict__ dst,
                                                             long long dst_stride, long long nG) {
    using B = GeoB<S>;
    using P = SampB<S>;
    constexpr int GW = B::GB / 4, SW = S * B::RW, S3 = S * S * S;
    __shared__ __align__(16) uint32_t s_img[P::WARPS * P::PITCH];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t *img = s_img + warp * P::PITCH;
    if (lane == 0) img[P::IMG] = 0;
    for (long long g0 = ((long long)blockIdx.x * P::WARPS + warp) * P::UPW; g0 < nG; g0 += (long long)gridDim.x * P::WARPS * P::UPW) {
        const int ng = nG - g0 < P::UPW ? (int)(nG - g0) : P::UPW;
        for (int t = lane; t < ng * SW; t += 32) {
            const int g = t / SW;
            img[t] = __ldg(bits + (g0 + g) * GW + (t - g * SW));
        }
        __syncwarp();
        if (dst_stride == S3) {
            store_run_bits<S>(img, dst + g0 * S3, ng * S3, lane);
        } else {
            for (int g = 0; g < ng; g++) store_run_bits<S>(img + g * SW, dst + (g0 + g) * dst_stride, S3, lane);
        }
        __syncwarp();
    }
}

template <int S>
unsigned grid_for_runs(long long n) {
    return grid_for((n + SampB<S>::UPW - 1) / SampB<S>::UPW, SampB<S>::WARPS);
}

} // namespace
} // namespace tg

extern "C" {

int tg_demo_sample_gf2(const uint8_t *tape_dm, const uint32_t *targets_bits, int64_t N, int R, int S, int dim_t, int replay_shift,
                       const int64_t *idx, int64_t nb, float *states, float *scalars, int64_t *actions, float *rewards, void *stream) {
    const int rc = tg::check_demo_sample_gf2(S, N, R, dim_t, replay_shift, nb, tape_dm, targets_bits, idx, states, scalars, actions, rewards);
    if (rc != tg::LAUNCH) return rc;
    return tg::with_S(S, [&](auto s) {
        constexpr int kS = decltype(s)::value;
        tg::demo_sample_gf2_kernel<kS><<<tg::grid_for_runs<kS>(nb * dim_t), 256, 0, (cudaStream_t)stream>>>(
            tape_dm, targets_bits, N, R, dim_t, replay_shift, (const long long *)idx, nb, states, scalars, (long long *)actions, rewards);
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    });
}

int tg_expand_f32_gf2(const uint32_t *bits, float *dst, int64_t dst_stride, int64_t B, int S, void *stream) {
    if (const int rc = tg::check_pair(S, B, bits, 16, dst, 4); rc != tg::LAUNCH) return rc;
    return tg::with_S(S, [&](auto s) {
        constexpr int kS = decltype(s)::value;
        tg::expand_f32_gf2_kernel<kS><<<tg::grid_for_runs<kS>(B), 256, 0, (cudaStream_t)stream>>>(bits, dst, dst_stride, B);
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    });
}

} // extern "C"
