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
// The parent is read ONCE: thread (parent, word column) keeps its S row words in registers and produces the k
// children one after the other into a three-stage shared-memory tile; each child game leaves with a TMA bulk store
// while the next ones are computed (three stages so that ONE CTA barrier per child is enough: a stage is rewritten two
// barriers after the threads that issued its stores have seen them drain).  HBM traffic per child: GP * (1 + 1/k) + TP + 13 bytes.
// The state key is the trilinear form of the state at three fixed 64-bit vectors (sum T[i][j][k] A_i B_j C_k mod 2^64,
// tg_state_key), so a child's key is the parent's key (hashed once per parent) minus
// (sum u_i A_i)(sum v_j B_j)(sum w_k C_k): 3 S multiply-adds on the action's tokens, done for all TG * k children of the
// block before the child loop -- no pass over the child, no per-entry work.
#include "tg_step.cuh"

namespace tg {

template <int S, int NT>
struct ExpCfg {
    using G = Geo<S>;
    static constexpr int TG = NT / G::WR; // parents per CTA (one word column per thread)
    static constexpr int ACTIVE = TG * G::WR;
    static constexpr int STAGE_BYTES = TG * G::GP;
    static __host__ __device__ constexpr int tok_bytes(int k) { return (TG * k * G::TP + 15) & ~15; }
    static constexpr int NSTAGE = 3;
    // tokens, NSTAGE child stages, per-(stage, game) partial word and key
    static __host__ __device__ constexpr int smem_bytes(int k) {
        return tok_bytes(k) + NSTAGE * STAGE_BYTES + ((NSTAGE * TG * 4 + 7) & ~7) + TG * 8 + 16 + NT * 8;
    }
};

__device__ __forceinline__ unsigned long long splitmix64_e(unsigned long long z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
// A_i / B_j / C_k of the state key (tg_state_key): base 0x1000 / 0x2000 / 0x3000
__device__ __forceinline__ unsigned long long key_const(unsigned base, int i) { return splitmix64_e((unsigned long long)(base + i)) | 1ull; }
__device__ __forceinline__ unsigned long long splitmix_or1(unsigned x) { return splitmix64_e((unsigned long long)x) | 1ull; } // the same constant from a run-time index

template <int S, int NT, bool KEYS>
__global__ void __launch_bounds__(NT)
    expand_kernel(const int8_t *__restrict__ parents, const uint8_t *__restrict__ tape, int k, int8_t *__restrict__ children,
                  uint8_t *__restrict__ flags, int32_t *__restrict__ nnz, unsigned long long *__restrict__ keys, long long B,
                  int shift) {
    using C = ExpCfg<S, NT>;
    using G = Geo<S>;
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t *s_tok = smem;                                                            // [TG][k][TP]
    constexpr int NSTAGE = C::NSTAGE;
    uint8_t *s_out = smem + C::tok_bytes(k);                                          // [NSTAGE][TG][GP]
    uint32_t *s_part = reinterpret_cast<uint32_t *>(s_out + NSTAGE * C::STAGE_BYTES); // [NSTAGE][TG]
    unsigned long long *s_pkey = reinterpret_cast<unsigned long long *>(reinterpret_cast<uint8_t *>(s_part) + ((NSTAGE * C::TG * 4 + 7) & ~7)); // [TG] parent keys
    uint64_t *s_bar = reinterpret_cast<uint64_t *>(s_pkey + C::TG);
    unsigned long long *s_ph = reinterpret_cast<unsigned long long *>(s_bar + 2); // [NT] parent key, per word column

    const int tid = threadIdx.x;
    const long long g0 = (long long)blockIdx.x * C::TG;
    const int ng = (int)min((long long)C::TG, B - g0);
    const int g = tid / G::WR;
    const bool active = tid < C::ACTIVE && g < ng;
    Lane<S> L;
    L.init(tid < C::ACTIVE ? tid % G::WR : 0);

    if (tid == 0) {
        mbar_init(s_bar, 1);
        mbar_fence_init();
    }
    // game padding of the child stages is zero and stays zero (threads only write their word columns of the S rows)
    for (int w = tid; w < NSTAGE * C::STAGE_BYTES / 4; w += NT) reinterpret_cast<uint32_t *>(s_out)[w] = 0;
    for (int i = tid; i < NSTAGE * C::TG; i += NT) s_part[i] = 0;
    // key constants of this thread's word column: B_j C_k of its four entries (0 in the row padding)
    unsigned long long kb[4] = {0, 0, 0, 0};
    if constexpr (KEYS) {
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int jk = 4 * L.c + q;
            kb[q] = jk < G::S2 ? key_const(0x2000, jk / S) * key_const(0x3000, jk % S) : 0ull;
        }
    }
    __syncthreads();
    if (tid == 0) {
        mbar_expect_tx(s_bar, (uint32_t)(ng * k * G::TP));
        bulk_g2s(s_tok, tape + g0 * k * G::TP, (uint32_t)(ng * k * G::TP), s_bar);
    }
    // the parent's rows of this thread's word column, offset-binary
    uint32_t row[S];
    if (active) {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(parents + (g0 + g) * G::GP) + L.c;
#pragma unroll
        for (int i = 0; i < S; i++) row[i] = src[i * G::WR] ^ H4;
    } else {
#pragma unroll
        for (int i = 0; i < S; i++) row[i] = H4;
    }
    if constexpr (KEYS) {
        // the parent's key, once: this thread's word column gives sum_q (B C)[4c + q] * sum_i A_i T[i][4c + q]; the rows
        // are offset-binary bytes (entry + 128, unsigned: one wide multiply-add and one 32-bit one per entry), the
        // offset's share -128 sum_i A_i is the accumulators' start value
        unsigned long long a0 = 0;
#pragma unroll
        for (int i = 0; i < S; i++) a0 -= 128ull * key_const(0x1000, i);
        unsigned long long acc[4] = {a0, a0, a0, a0};
#pragma unroll
        for (int i = 0; i < S; i++) {
#pragma unroll
            for (int q = 0; q < 4; q++) acc[q] += (unsigned long long)((row[i] >> (8 * q)) & 0xFFu) * key_const(0x1000, i);
        }
        s_ph[tid] = acc[0] * kb[0] + acc[1] * kb[1] + acc[2] * kb[2] + acc[3] * kb[3];
    }
    mbar_wait(s_bar, 0);
    if constexpr (KEYS) {
        __syncthreads();
        if (tid < ng) {
            unsigned long long h = 0;
            for (int c = 0; c < G::WR; c++) h += s_ph[tid * G::WR + c];
            s_pkey[tid] = h;
        }
        __syncthreads();
        // child key = parent key - key of its rank-1 action, the latter from the action's tokens alone; one coalesced
        // store of the block's TG * k keys
        for (int x = tid; x < ng * k; x += NT) {
            const uint8_t *tok = s_tok + (size_t)x * G::TP;
            unsigned long long f[3];
#pragma unroll
            for (int m = 0; m < 3; m++) {
                unsigned long long a = 0;
#pragma unroll
                for (int i = 0; i < S; i++) a += (unsigned long long)(long long)((int)tok[m * S + i] - shift) * key_const(0x1000 * (m + 1), i);
                f[m] = a;
            }
            keys[g0 * k + x] = s_pkey[x / k] - f[0] * f[1] * f[2];
        }
    }

    for (int c = 0, st = 0; c < k; c++, st = st + 1 == NSTAGE ? 0 : st + 1) {
        uint8_t *stage = s_out + st * C::STAGE_BYTES;
        // the bulk stores of child c-3 have finished reading this stage: the threads that issued them waited for child c-2's
        // predecessor to drain (bulk_wait_read<1> below, iteration c-2) before they arrived at the barrier of iteration c-1
        if (active) {
            const uint8_t *tok = s_tok + ((size_t)g * k + c) * G::TP;
            const int32_t vw = pack_vw<S>(tok, L, shift);
            uint32_t uw[UW<S>];
            load_u<S>(tok, uw);
            const uint32_t nvw = (uint32_t)(-vw);
            uint32_t cnt = 0, rng = 0;
            int uany = 0;
            uint32_t *col = reinterpret_cast<uint32_t *>(stage + (size_t)g * G::GP) + L.c;
#pragma unroll
            for (int i = 0; i < S; i++) {
                const int negu = coef_u(uw, i, shift);
                const uint32_t t = (row[i] + (uint32_t)negu * nvw) ^ H4; // child word, two's complement bytes
                col[i * G::WR] = t;
                cnt += ((((t & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | t) & L.hv) >> 7;
                rng |= t ^ (t << 1);
                uany |= negu;
            }
            atomicAdd(&s_part[st * C::TG + g], make_partial(byte_sum(cnt), vw != 0 && uany != 0,
                                                            (rng & L.hv) != 0 || tokens_out_of_range<S>(tok, L, shift)));
        }
        fence_proxy_async();
        __syncthreads();
        if (tid < ng) {
            const long long child = (g0 + tid) * k + c;
            bulk_s2g(children + child * G::GP, stage + (size_t)tid * G::GP, (uint32_t)G::GP);
            bulk_commit();
            const uint32_t sum = s_part[st * C::TG + tid];
            flags[child] = (uint8_t)partial_flags(sum);
            nnz[child] = (int32_t)(sum & 0xFFFFu);
            s_part[st * C::TG + tid] = 0;
            bulk_wait_read<1>(); // the store of child c-1 has drained; its stage is rewritten at c+2, one barrier from here
        }
        // no second barrier: the partial words of this stage are reset here and next touched at child c+3, two barriers away
    }
    if (tid < ng) bulk_wait<0>();
}

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
        for (int x = 0; x < S; x++) kc[x] = splitmix_or1(0x1000u * (unsigned)(i + 1) + (unsigned)x);
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

template <int S, int NT>
static int launch_expand(const int8_t *parents, const uint8_t *tape, int k, int8_t *children, uint8_t *flags, int32_t *nnz,
                         unsigned long long *keys, long long B, int shift, cudaStream_t st) {
    using C = ExpCfg<S, NT>;
    const int smem = C::smem_bytes(k);
    if (smem > 200 * 1024) return TG_E_ARG;
    const long long grid = (B + C::TG - 1) / C::TG;
    if (grid > 0x7FFFFFFFLL) return TG_E_ARG;
    if (keys) {
        auto kern = expand_kernel<S, NT, true>;
        TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        kern<<<(int)grid, NT, smem, st>>>(parents, tape, k, children, flags, nnz, keys, B, shift);
    } else {
        auto kern = expand_kernel<S, NT, false>;
        TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        kern<<<(int)grid, NT, smem, st>>>(parents, tape, k, children, flags, nnz, keys, B, shift);
    }
    TG_CUDA(cudaGetLastError());
    return TG_OK;
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
            return tg::launch_expand<4, 256>(parents, tape, k, children, flags, nnz, (unsigned long long *)keys, B, shift, st);
#endif
        const long long grid = (B * 4 + 127) / 128;
        if (grid > 0x7FFFFFFFLL) return TG_E_ARG;
        if (keys) tg::expand4_rows_kernel<true><<<(int)grid, 128, 0, st>>>(parents, tape, k, children, flags, nnz, (unsigned long long *)keys, B, shift);
        else tg::expand4_rows_kernel<false><<<(int)grid, 128, 0, st>>>(parents, tape, k, children, flags, nnz, nullptr, B, shift);
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    }
    case 9: return tg::launch_expand<9, 128>(parents, tape, k, children, flags, nnz, (unsigned long long *)keys, B, shift, st);
    case 16: return tg::launch_expand<16, 128>(parents, tape, k, children, flags, nnz, (unsigned long long *)keys, B, shift, st);
    case 25: return tg::launch_expand<25, 160>(parents, tape, k, children, flags, nnz, (unsigned long long *)keys, B, shift, st); // one parent per CTA
    }
    return TG_E_ARG;
}
