// tg_expand.cu -- K8: batched leaf expansion (C ABI: tg_expand_children).
//
// Reference restated: get_child_states (act.py:266-275) -- for each of the k sampled actions of a state,
// new_head = head - u (x) v (x) w -- together with what extend_tree does with the children right away:
// remove_null_actions (utils.py:191-194), tensor_factorized on the head (utils.py:181-188, act.py:177) and the
// "already in the tree" lookup by state key (act.py:185-195; key = tg_state_key instead of utils.py:164-169 strings).
// The reference does this for one state at a time; here B states expand at once:
//     children[b][c] = parents[b] - rank1(tape[b][c]),  c < k,
// with per-child flags (terminal / null action / range), non-zero count and 64-bit state key.
//
// The word-column kernel expand_kernel (tg_step.cuh) serves 9x9x9, 16x16x16 and 25x25x25; 4x4x4 has a row kernel here.
#include "tg_step.cuh"

namespace tg {

// ------------------------------------------------------------------ 4x4x4: four threads per parent, rows in registers
// A 4x4x4 parent is 16 words: thread (parent, i) keeps ROW i (4 words, offset-binary) in registers while the k children are
// produced one after the other -- a child is one 16-byte record load (the four threads of a parent read the same one),
// the coefficients with three packed subtractions and sign-extending PRMTs, four products u_i v_j and four IMADs with the
// integer form of pack(w), and ONE 16-byte store per thread: the four threads of a parent write the 64 contiguous bytes of
// the child (one thread per parent with four stores each was measured: 20 G children/s against 29 for the word-column
// kernel -- 16-byte pieces of 32 different lines per store instruction).  nnz / range / key partials meet by two xor-
// shuffles; no shared memory, no barrier, no atomics.  Same outputs as expand_kernel.
template <int B>
__device__ __forceinline__ int sext_byte_e(uint32_t w) {
    constexpr uint32_t sel = (uint32_t)B | ((uint32_t)(B | 8) << 4) | ((uint32_t)(B | 8) << 8) | ((uint32_t)(B | 8) << 12);
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(w), "r"(0u), "r"(sel));
    return (int)d;
}
__device__ __forceinline__ unsigned long long quad_sum64(unsigned long long x) { // sum over the four lanes of a quad
    x += __shfl_xor_sync(0xFFFFFFFFu, x, 1);
    x += __shfl_xor_sync(0xFFFFFFFFu, x, 2);
    return x;
}

template <bool KEYS>
__global__ void __launch_bounds__(128)
    expand4_rows_kernel(const int8_t *__restrict__ parents, const uint8_t *__restrict__ tape, int k, int8_t *__restrict__ children,
                        uint8_t *__restrict__ flags, int32_t *__restrict__ nnz, unsigned long long *__restrict__ keys, long long B,
                        int shift) {
    constexpr int S = 4;
    const long long gt = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long b = min(gt >> 2, B - 1); // the last warp's spare quads repeat the last parent (shuffles need every lane)
    const bool real = (gt >> 2) < B;
    const int i = (int)(gt & 3);
    uint32_t row[4]; // entries (i, j, 0..3), offset-binary
    {
        const uint4 t = __ldg(reinterpret_cast<const uint4 *>(parents + b * 64) + i);
        row[0] = t.x ^ H4, row[1] = t.y ^ H4, row[2] = t.z ^ H4, row[3] = t.w ^ H4;
    }
    unsigned long long pkey = 0;
    const unsigned long long Ai = i == 0 ? key_const(0x1000, 0) : i == 1 ? key_const(0x1000, 1) : i == 2 ? key_const(0x1000, 2) : key_const(0x1000, 3);
    if constexpr (KEYS) { // sum T[i][j][k] A_i B_j C_k mod 2^64 (tg_state_key): this row's share, then the quad's sum
        unsigned long long ti = 0;
#pragma unroll
        for (int j = 0; j < S; j++) {
            const uint32_t w = row[j] ^ H4; // two's complement bytes
            unsigned long long sij = 0;
#pragma unroll
            for (int kk = 0; kk < S; kk++) sij += (unsigned long long)(long long)(int8_t)(w >> (8 * kk)) * key_const(0x3000, kk);
            ti += sij * key_const(0x2000, j);
        }
        pkey = quad_sum64(ti * Ai);
    }
    const uint32_t sh4 = (uint32_t)shift * ONES4, tokmax = (uint32_t)(0x7F - 2 * shift) * ONES4;
    const uint4 *rec = reinterpret_cast<const uint4 *>(tape + b * k * 16);
    uint4 *dst = reinterpret_cast<uint4 *>(children + b * k * 64) + i;
    const int ush = 8 * i;
    unsigned long long kc[S] = {0, 0, 0, 0}; // lane i < 3: the constants of factor i of an action's key
    if constexpr (KEYS) {
#pragma unroll
        for (int x = 0; x < S; x++) kc[x] = key_const(0x1000u * (unsigned)(i + 1), x);
    }
    uint4 q = __ldg(rec);
    for (int c = 0; c < k; c++) {
        const uint4 cur = q;
        if (c + 1 < k) q = __ldg(rec + c + 1);
        const uint32_t over = ((((cur.x & 0x7F7F7F7Fu) + tokmax) | cur.x) | (((cur.y & 0x7F7F7F7Fu) + tokmax) | cur.y) |
                               (((cur.z & 0x7F7F7F7Fu) + tokmax) | cur.z)) & H4;
        const uint32_t cu = ((cur.x | H4) - sh4) ^ H4, cv = ((cur.y | H4) - sh4) ^ H4, cw = ((cur.z | H4) - sh4) ^ H4;
        const int wi = (int)(cur.z - sh4); // integer form of pack(w)
        const int ui = (int)(int8_t)(cu >> ush);
        const int v[4] = {sext_byte_e<0>(cv), sext_byte_e<1>(cv), sext_byte_e<2>(cv), sext_byte_e<3>(cv)};
        uint32_t part = 0, rng = 0; // nnz of this row | range flag << 16
        uint32_t t[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const uint32_t x = (row[j] - (uint32_t)(ui * v[j] * wi)) ^ H4; // child word, two's complement bytes
            t[j] = x;
            part += (uint32_t)__popc(nonzero_mask(x));
            rng |= x ^ (x << 1);
        }
        if (real) dst[4 * c] = make_uint4(t[0], t[1], t[2], t[3]);
        part |= (rng & H4) != 0 ? 1u << 16 : 0u;
        part += __shfl_xor_sync(0xFFFFFFFFu, part, 1);
        part += __shfl_xor_sync(0xFFFFFFFFu, part, 2);
        unsigned long long fkey = 0;
        if constexpr (KEYS) { // lane i < 3 of the quad: factor i of the action's key, sum_x coef_x * const(i, x)
            const uint32_t cm = i == 0 ? cu : (i == 1 ? cv : cw);
            unsigned long long f = 0;
#pragma unroll
            for (int x = 0; x < S; x++) f += (unsigned long long)(long long)(int8_t)(cm >> (8 * x)) * kc[x];
            const unsigned long long f1 = __shfl_sync(0xFFFFFFFFu, f, (threadIdx.x & 28) | 1);
            const unsigned long long f2 = __shfl_sync(0xFFFFFFFFu, f, (threadIdx.x & 28) | 2);
            fkey = f * f1 * f2; // meaningful in lane 0 of the quad
        }
        if (real && i == 0) {
            const uint32_t cntv = part & 0xFFFFu;
            const bool changed = cu != 0 && cv != 0 && cw != 0; // u (x) v (x) w != 0
            const long long child = b * k + c;
            flags[child] = (uint8_t)((cntv == 0 ? TG_FLAG_TERMINAL : 0u) | (changed ? 0u : TG_FLAG_NULL) |
                                     (((part >> 16) != 0 || over != 0) ? TG_FLAG_RANGE : 0u));
            nnz[child] = (int32_t)cntv;
            if constexpr (KEYS) keys[child] = pkey - fkey;
        }
    }
}

} // namespace tg

extern "C" int tg_expand_children(const int8_t *parents, const uint8_t *tape, int k, int8_t *children, uint8_t *flags,
                                  int32_t *nnz, uint64_t *keys, int64_t B, int S, int shift, void *stream) {
    if (const int rc = tg::check_expand(S, B, k, shift, parents, tape, children, flags, nnz); rc != tg::LAUNCH) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    switch (S) {
    case 4: {
#ifdef TG_TUNING
        if (tg::tuning_env("TG_EXPAND_COLUMNS", 0)) // A/B: the word-column kernel
            return tg::launch_expand<4, 256, tg::W8>(parents, tape, k, children, flags, nnz, (unsigned long long *)keys, B, shift, st);
#endif
        const long long grid = (B * 4 + 127) / 128;
        if (grid > 0x7FFFFFFFLL) return TG_E_ARG;
        if (keys) tg::expand4_rows_kernel<true><<<(int)grid, 128, 0, st>>>(parents, tape, k, children, flags, nnz, (unsigned long long *)keys, B, shift);
        else tg::expand4_rows_kernel<false><<<(int)grid, 128, 0, st>>>(parents, tape, k, children, flags, nnz, nullptr, B, shift);
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    }
    case 9: return tg::launch_expand<9, 128, tg::W8>(parents, tape, k, children, flags, nnz, (unsigned long long *)keys, B, shift, st);
    case 16: return tg::launch_expand<16, 128, tg::W8>(parents, tape, k, children, flags, nnz, (unsigned long long *)keys, B, shift, st);
    case 25: return tg::launch_expand<25, 160, tg::W8>(parents, tape, k, children, flags, nnz, (unsigned long long *)keys, B, shift, st); // one parent per CTA
    }
    return TG_E_ARG;
}
