// tg_ustream.cu -- K3 parity mode: same-seed synthetic demos.
//
// The reference draws every factor with a fresh Categorical(probs).sample([S])
// (utils.py:197-200, datasets.py:155-158), i.e. torch.multinomial on the CPU
// generator: MT19937 -> 53-bit doubles -> first CDF bucket >= u, with the CDF a
// float32 running sum of probs/sum(probs).  Tries are consumed strictly in
// stream order (u, v, w; S doubles each) and rejected iff one factor is all
// zero (utils.py:229).  Hence the i-th ACCEPTED try of the stream is term
// i % R of demo i / R: the sequential rejection loop is a stream compaction.
//
//   host : tg_mt19937_fill_f64   (the torch CPU uniform stream for a seed)
//   map  : one thread per try -> tokens + accepted flag
//   scan : exclusive prefix sum of the flags (3 small kernels)
//   scatter: accepted try i -> tape[i % R][i / R]
//   tg_demo_accumulate builds the target tensors from the tape.
#include "tg_common.cuh"

namespace tg {

struct CdfF32 {
    float cdf[8];
    int8_t values[8];
    int n;
};

// one thread per try
template <int S>
__global__ void ustream_map_kernel(const double *__restrict__ u, long long n_tries, CdfF32 cat, int shift,
                                   uint32_t *__restrict__ tok, uint32_t *__restrict__ valid) {
    using G = Geo<S>;
    const long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (t >= n_tries) return;
    const double *src = u + t * 3 * S;
    uint32_t words[G::TP / 4];
#pragma unroll
    for (int w = 0; w < G::TP / 4; w++) words[w] = 0;
    uint32_t nz[3] = {0, 0, 0};
#pragma unroll
    for (int q = 0; q < 3 * S; q++) {
        const double x = src[q];
        int lo = 0, hi = cat.n; // the multinomial kernel's binary search: first bucket with cdf >= x
        while (hi - lo > 0) {
            const int mid = lo + (hi - lo) / 2;
            float c = 0.f;
#pragma unroll
            for (int i = 0; i < 8; i++) c = (mid == i) ? cat.cdf[i] : c;
            if ((double)c < x)
                lo = mid + 1;
            else
                hi = mid;
        }
        if (lo >= cat.n) lo = cat.n - 1;
        int val = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) val = (lo == i) ? (int)cat.values[i] : val;
        nz[q / S] |= (uint32_t)(val != 0);
        words[q >> 2] |= (uint32_t)((val + shift) & 0xFF) << (8 * (q & 3));
    }
    uint32_t *dst = tok + t * (G::TP / 4);
#pragma unroll
    for (int w = 0; w < G::TP / 4; w++) dst[w] = words[w];
    valid[t] = nz[0] & nz[1] & nz[2];
}

constexpr int SCAN_BLOCK = 1024;

__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t *total) {
    __shared__ uint32_t warp_sums[32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) warp_sums[wid] = x;
    __syncthreads();
    if (wid == 0) {
        uint32_t s = warp_sums[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, s, o);
            if (lane >= o) s += y;
        }
        warp_sums[lane] = s;
    }
    __syncthreads();
    const uint32_t base = wid ? warp_sums[wid - 1] : 0;
    if (total) *total = warp_sums[31];
    __syncthreads();
    return base + x - v;
}

__global__ void scan_block_sums_kernel(const uint32_t *__restrict__ valid, long long n, uint32_t *__restrict__ sums) {
    const long long i = blockIdx.x * (long long)SCAN_BLOCK + threadIdx.x;
    uint32_t tot;
    block_exclusive_scan(i < n ? valid[i] : 0u, &tot);
    if (threadIdx.x == 0) sums[blockIdx.x] = tot;
}

// single block: sums[b] <- exclusive prefix; sums[nb] <- grand total
__global__ void scan_sums_kernel(uint32_t *sums, int nb) {
    __shared__ uint32_t carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < nb; base += SCAN_BLOCK) {
        const int i = base + threadIdx.x;
        const uint32_t v = i < nb ? sums[i] : 0u;
        uint32_t tot;
        const uint32_t ex = block_exclusive_scan(v, &tot);
        if (i < nb) sums[i] = carry + ex;
        __syncthreads();
        if (threadIdx.x == 0) carry += tot;
        __syncthreads();
    }
    if (threadIdx.x == 0) sums[nb] = carry;
}

template <int S>
__global__ void ustream_scatter_kernel(const uint32_t *__restrict__ tok, const uint32_t *__restrict__ valid,
                                       const uint32_t *__restrict__ sums, long long n_tries, int nb, int R, long long N,
                                       uint8_t *__restrict__ tape, long long tape_step_stride,
                                       long long *__restrict__ result) {
    using G = Geo<S>;
    const long long t = blockIdx.x * (long long)SCAN_BLOCK + threadIdx.x;
    const uint32_t v = t < n_tries ? valid[t] : 0u;
    const uint32_t ex = block_exclusive_scan(v, nullptr);
    const long long total = sums[nb];
    const long long done = min(N, total / R);
    if (t == 0 && result) {
        result[0] = done;
        if (done == 0) result[1] = 0;
    }
    if (!v) return;
    const long long pos = (long long)sums[blockIdx.x] + ex;
    if (pos >= done * R) return;
    const long long demo = pos / R;
    const int term = (int)(pos - demo * R);
    const uint4 *src = reinterpret_cast<const uint4 *>(tok + t * (G::TP / 4));
    uint4 *dst = reinterpret_cast<uint4 *>(tape + (size_t)term * tape_step_stride + demo * G::TP);
#pragma unroll
    for (int w = 0; w < G::TP / 16; w++) dst[w] = src[w];
    if (pos == done * R - 1 && result) result[1] = (t + 1) * 3 * S;
}

} // namespace tg

extern "C" {

int tg_mt19937_fill_f64_state(const uint32_t *state624, int pos, int64_t skip, int64_t n, double *out) {
    if (n < 0 || skip < 0 || !state624 || pos < 0 || (n > 0 && !out)) return TG_E_ARG;
    uint32_t s[624];
    for (int i = 0; i < 624; i++) s[i] = state624[i];
    auto next = [&]() -> uint32_t {
        if (pos >= 624) {
            for (int i = 0; i < 624; i++) {
                const uint32_t y = (s[i] & 0x80000000u) | (s[(i + 1) % 624] & 0x7fffffffu);
                s[i] = s[(i + 397) % 624] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
            }
            pos = 0;
        }
        uint32_t y = s[pos++];
        y ^= y >> 11;
        y ^= (y << 7) & 0x9d2c5680u;
        y ^= (y << 15) & 0xefc60000u;
        y ^= y >> 18;
        return y;
    };
    for (int64_t i = 0; i < skip + n; i++) {
        const uint64_t hi = next(), lo = next();
        if (i >= skip) out[i - skip] = (double)(((hi << 32) | lo) & ((1ull << 53) - 1)) * (1.0 / 9007199254740992.0);
    }
    return TG_OK;
}

int tg_mt19937_fill_f64(uint32_t seed, int64_t skip, int64_t n, double *out) {
    uint32_t s[624];
    s[0] = seed;
    for (int i = 1; i < 624; i++) s[i] = 1812433253u * (s[i - 1] ^ (s[i - 1] >> 30)) + (uint32_t)i;
    return tg_mt19937_fill_f64_state(s, 624, skip, n, out);
}

int64_t tg_demo_from_ustream_workspace(int64_t n_u, int S) {
    if (!tg::supported_S(S) || n_u < 0) return TG_E_ARG;
    const int64_t n_tries = n_u / (3 * S);
    const int64_t nb = (n_tries + tg::SCAN_BLOCK - 1) / tg::SCAN_BLOCK;
    const int tp = (3 * S + 15) & ~15;
    return n_tries * tp + n_tries * 4 + (nb + 1) * 4 + 64;
}

int tg_demo_from_ustream(const double *u, int64_t n_u, const int8_t *values, const float *probs, int n_values, int R, int S,
                         int shift, int64_t N, uint8_t *tape, int64_t tape_step_stride, int8_t *slab, uint8_t *flags,
                         int64_t *result, void *workspace, int64_t workspace_bytes, void *stream) {
    if (!tg::supported_S(S) || N < 0 || R < 1 || shift < 1 || shift > 4 || n_values < 1 || n_values > 8 || n_u < 0)
        return TG_E_ARG;
    if (!u || !values || !probs || !tape || !slab || !result || !workspace) return TG_E_ARG;
    if (((uintptr_t)tape | (uintptr_t)slab | (uintptr_t)tape_step_stride | (uintptr_t)workspace) & 15) return TG_E_ARG;
    const int64_t n_tries = n_u / (3 * S);
    if (n_tries >= (1LL << 31) || workspace_bytes < tg_demo_from_ustream_workspace(n_u, S)) return TG_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    // the CDF exactly as Categorical + the multinomial CPU kernel build it (float32)
    tg::CdfF32 cat;
    float total = 0.f, run = 0.f;
    for (int i = 0; i < n_values; i++) total += probs[i];
    for (int i = 0; i < 8; i++) cat.cdf[i] = 1.f, cat.values[i] = 0;
    for (int i = 0; i < n_values; i++) {
        run += probs[i] / total;
        cat.cdf[i] = run;
        cat.values[i] = values[i];
    }
    const float last = run;
    for (int i = 0; i < n_values; i++) cat.cdf[i] /= last;
    cat.cdf[n_values - 1] = 1.f;
    cat.n = n_values;

    const int tp = (3 * S + 15) & ~15;
    uint32_t *tok = reinterpret_cast<uint32_t *>(workspace);
    uint32_t *valid = reinterpret_cast<uint32_t *>(reinterpret_cast<uint8_t *>(workspace) + n_tries * tp);
    uint32_t *sums = valid + n_tries;
    const int nb = (int)((n_tries + tg::SCAN_BLOCK - 1) / tg::SCAN_BLOCK);
    if (n_tries == 0) {
        TG_CUDA(cudaMemsetAsync(result, 0, 16, st));
        return TG_OK;
    }
    const int mb = (int)((n_tries + 127) / 128);
    const int rc = tg::with_S(S, [&](auto s) {
        constexpr int kS = decltype(s)::value;
        tg::ustream_map_kernel<kS><<<mb, 128, 0, st>>>(u, n_tries, cat, shift, tok, valid);
        TG_CUDA(cudaGetLastError());
        tg::scan_block_sums_kernel<<<nb, tg::SCAN_BLOCK, 0, st>>>(valid, n_tries, sums);
        tg::scan_sums_kernel<<<1, tg::SCAN_BLOCK, 0, st>>>(sums, nb);
        tg::ustream_scatter_kernel<kS><<<nb, tg::SCAN_BLOCK, 0, st>>>(tok, valid, sums, n_tries, nb, R, N, tape, tape_step_stride,
                                                                     (long long *)result);
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    });
    if (rc != TG_OK) return rc;
    return tg_demo_accumulate(tape, tape_step_stride, N, R, S, shift, slab, flags, stream);
}

} // extern "C"
