// tg_wide.cu -- the int16 residual format ("slab16") for values the int8 slab cannot hold
// (C ABI: tg_demo_accumulate_i16, tg_expand_f32_i16, tg_pack_f32_i16).
//
// The reference keeps every residual as float32 and never overflows (utils.py:218-232 accumulates targets without
// limit; uniform coefficient probabilities reach |T| = 86 at 9x9x9 rank 23 and 174 at 16x16x16, SURVEY 7.3), and the
// change of basis multiplies magnitudes by the matrix norms (SURVEY 8(d): int8 in, int16 out).  slab16 is the same
// geometry as the int8 slab with two bytes per entry: int16 [B][GP], entry (i,j,k) at ELEMENT i*RP + j*S + k, padding
// elements zero.  Producers: tg_demo_accumulate_i16 (targets of any action list), tg_change_of_basis_i16; consumers:
// tg_demo_sample_dm (training samples from int16 targets), tg_expand_f32_i16 (float32 states for the model).
#include "tg_step.cuh"

namespace tg {

// slab16[n] = sum_r rank1(tape[r][n]) in plain int32 arithmetic per entry, stored as int16.  Exact while R * cmax^3 fits
// int32 (cmax = max(shift, 255 - shift), the largest |token - shift| of a byte); longer tapes go to the kernel below.
// Thread (demo, word column c) owns the entries (i, 4c .. 4c+3) of every row; the CTA stages the records of its demos for
// one step at a time in shared memory.
template <int S>
__global__ void __launch_bounds__(256)
    demo_accumulate_i16_kernel(const uint8_t *__restrict__ tape, long long tape_step_stride, long long N, int R, int shift,
                               int16_t *__restrict__ slab16, uint8_t *__restrict__ flags) {
    using G = Geo<S>;
    constexpr int NT = 256, DPC = NT / G::WR; // demos per CTA
    __shared__ __align__(16) uint8_t s_tok[DPC * G::TP];
    __shared__ uint32_t s_bad[DPC];
    const int tid = threadIdx.x;
    const long long g0 = (long long)blockIdx.x * DPC;
    const int ng = (int)min((long long)DPC, N - g0);
    const int g = tid / G::WR;
    const bool worker = tid < DPC * G::WR && g < ng;
    Lane<S> L;
    L.init(tid < DPC * G::WR ? tid % G::WR : 0);
    if (tid < DPC) s_bad[tid] = 0;
    int acc[S][4];
#pragma unroll
    for (int i = 0; i < S; i++)
#pragma unroll
        for (int q = 0; q < 4; q++) acc[i][q] = 0;
    for (int r = 0; r < R; r++) {
        __syncthreads();
        const uint4 *src = reinterpret_cast<const uint4 *>(tape + (size_t)r * tape_step_stride + g0 * G::TP);
        for (int w = tid; w < ng * (G::TP / 16); w += NT) reinterpret_cast<uint4 *>(s_tok)[w] = __ldg(src + w);
        __syncthreads();
        if (worker) {
            const uint8_t *tok = s_tok + g * G::TP;
            const int vA = (int)tok[L.off_vA] - shift, vB = (int)tok[L.off_vB] - shift;
            int vw[4];
#pragma unroll
            for (int b = 0; b < 4; b++) {
                const bool inA = (L.maskA >> (8 * b)) & 1u, inB = (L.maskB >> (8 * b)) & 1u;
                const int w = (int)tok[L.off_w[b]] - shift;
                vw[b] = inA ? vA * w : (inB ? vB * w : 0);
            }
#pragma unroll
            for (int i = 0; i < S; i++) {
                const int u = (int)tok[i] - shift;
#pragma unroll
                for (int q = 0; q < 4; q++) acc[i][q] += u * vw[q];
            }
        }
    }
    if (worker) {
        bool bad = false;
        int16_t *dst = slab16 + (g0 + g) * G::GP;
#pragma unroll
        for (int i = 0; i < S; i++) {
#pragma unroll
            for (int q = 0; q < 4; q++) bad |= acc[i][q] < -32768 || acc[i][q] > 32767;
            const uint32_t lo = ((uint32_t)acc[i][0] & 0xFFFFu) | ((uint32_t)acc[i][1] << 16);
            const uint32_t hi = ((uint32_t)acc[i][2] & 0xFFFFu) | ((uint32_t)acc[i][3] << 16);
            *reinterpret_cast<uint2 *>(dst + i * G::RP + 4 * L.c) = make_uint2(lo, hi);
        }
        if constexpr (G::GP != S * G::RP) {
            if (L.c == 0)
                for (int x = S * G::RP; x < G::GP; x += 2) *reinterpret_cast<uint32_t *>(dst + x) = 0u;
        }
        if (bad) atomicOr(&s_bad[g], (uint32_t)TG_FLAG_RANGE);
    }
    __syncthreads();
    if (flags && tid < ng) flags[g0 + tid] = (uint8_t)s_bad[tid];
}

// The same sum in 64 bit, one thread per entry: for tapes whose terms could carry an int32 sum past 2^31 (R >= 130 at
// shift 0, R >= 1024 at shift 127).
template <int S>
__global__ void __launch_bounds__(256)
    demo_accumulate_i16_wide_kernel(const uint8_t *__restrict__ tape, long long tape_step_stride, long long N, int R, int shift,
                                    int16_t *__restrict__ slab16, uint8_t *__restrict__ flags) {
    using G = Geo<S>;
    for (long long x = blockIdx.x * (long long)blockDim.x + threadIdx.x; x < N * G::GP; x += (long long)gridDim.x * blockDim.x) {
        const long long n = x / G::GP;
        const int e = (int)(x % G::GP), i = e / G::RP, jk = e % G::RP, j = jk / S, k = jk % S;
        long long v = 0;
        if (i < S && jk < G::S2) {
            const uint8_t *tok = tape + n * G::TP;
            for (int r = 0; r < R; r++, tok += tape_step_stride)
                v += (long long)(((int)__ldg(tok + i) - shift) * ((int)__ldg(tok + S + j) - shift)) * ((int)__ldg(tok + 2 * S + k) - shift);
        }
        slab16[x] = (int16_t)v;
        if (flags && (v < -32768 || v > 32767)) flags[n] = (uint8_t)TG_FLAG_RANGE; // same value from every writer
    }
}

// slab16 -> float32 dense (S,S,S) at dst + b*dst_stride; one thread per pair of entries
template <int S>
__global__ void expand_f32_i16_kernel(const int16_t *__restrict__ slab16, float *__restrict__ dst, long long dst_stride, long long B) {
    using G = Geo<S>;
    const long long total = B * G::S3;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const long long b = idx / G::S3;
        const int e = (int)(idx % G::S3);
        const int i = e / G::S2, jk = e % G::S2;
        dst[b * dst_stride + e] = (float)slab16[b * G::GP + i * G::RP + jk];
    }
}

// float32 dense -> slab16; range_flag |= 1 if a value is non-integral or outside int16
template <int S>
__global__ void pack_f32_i16_kernel(const float *__restrict__ src, long long src_stride, int16_t *__restrict__ slab16, long long B,
                                    int32_t *range_flag) {
    using G = Geo<S>;
    const long long total = B * G::GP;
    bool bad = false;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const long long b = idx / G::GP;
        const int x = (int)(idx % G::GP);
        const int i = x / G::RP, jk = x % G::RP;
        int v = 0;
        if (i < S && jk < G::S2) {
            const float f = src[b * src_stride + i * G::S2 + jk];
            v = __float2int_rn(f);
            bad |= ((float)v != f) | (v < -32768) | (v > 32767);
        }
        slab16[idx] = (int16_t)v;
    }
    if (bad && range_flag) atomicOr(range_flag, 1);
}

} // namespace tg

extern "C" {

int tg_demo_accumulate_i16(const uint8_t *tape, int64_t tape_step_stride, int64_t N, int R, int S, int shift, int16_t *slab16,
                           uint8_t *flags, void *stream) {
    if (const int rc = tg::check_accumulate(tg::supported_S(S), N, R, shift, 0, 127, tape, tape_step_stride, slab16); rc != tg::LAUNCH)
        return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const long long cmax = shift > 255 - shift ? shift : 255 - shift;
    if ((long long)R * cmax * cmax * cmax > 0x7FFFFFFFLL) {
        if (flags) TG_CUDA(cudaMemsetAsync(flags, 0, (size_t)N, st));
        return tg::with_S(S, [&](auto s) {
            constexpr int kS = decltype(s)::value;
            const long long blocks = (N * tg::Geo<kS>::GP + 255) / 256;
            tg::demo_accumulate_i16_wide_kernel<kS><<<(unsigned)(blocks < 148 * 32 ? blocks : 148 * 32), 256, 0, st>>>(
                tape, tape_step_stride, N, R, shift, slab16, flags);
            TG_CUDA(cudaGetLastError());
            return TG_OK;
        });
    }
    return tg::with_S(S, [&](auto s) {
        constexpr int kS = decltype(s)::value, DPC = 256 / tg::Geo<kS>::WR;
        const long long grid = (N + DPC - 1) / DPC;
        if (grid > 0x7FFFFFFFLL) return TG_E_ARG;
        tg::demo_accumulate_i16_kernel<kS><<<(unsigned)grid, 256, 0, st>>>(tape, tape_step_stride, N, R, shift, slab16, flags);
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    });
}

int tg_expand_f32_i16(const int16_t *slab16, float *dst, int64_t dst_stride, int64_t B, int S, void *stream) {
    if (const int rc = tg::check_pair(S, B, slab16, 16, dst, 4); rc != tg::LAUNCH) return rc;
    return tg::with_S(S, [&](auto s) {
        constexpr int kS = decltype(s)::value;
        const long long blocks = (B * tg::Geo<kS>::S3 + 255) / 256;
        tg::expand_f32_i16_kernel<kS><<<(unsigned)(blocks < 148 * 64 ? blocks : 148 * 64), 256, 0, (cudaStream_t)stream>>>(
            slab16, dst, dst_stride, B);
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    });
}

int tg_pack_f32_i16(const float *src, int64_t src_stride, int16_t *slab16, int64_t B, int S, int32_t *range_flag, void *stream) {
    if (const int rc = tg::check_pair(S, B, src, 4, slab16, 16); rc != tg::LAUNCH) return rc;
    return tg::with_S(S, [&](auto s) {
        constexpr int kS = decltype(s)::value;
        const long long blocks = (B * tg::Geo<kS>::GP + 255) / 256;
        tg::pack_f32_i16_kernel<kS><<<(unsigned)(blocks < 148 * 64 ? blocks : 148 * 64), 256, 0, (cudaStream_t)stream>>>(
            src, src_stride, slab16, B, range_flag);
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    });
}

} // extern "C"
