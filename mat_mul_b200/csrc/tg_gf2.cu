// tg_gf2.cu -- the game path modulo 2 on bit slabs: tg_pack_gf2(_i16) / tg_unpack_gf2, K1 tg_step_gf2, K8
// tg_expand_children_gf2, K2 tg_rollout_gf2 / tg_replay_gf2, K7 tg_state_key_gf2, K6 tg_slice_rank_gf2.
//
// AlphaTensor plays the game over Z (standard) and over Z_2 (modular); its 47-multiplication 4x4 factorization is a
// mod-2 one.  Mod 2 an entry is one bit: row i of a game is the S^2 bits (j,k) in RW = ceil(S^2 / 32) little-endian
// words, bit (j S + k) % 32 of word i RW + (j S + k) / 32, padding bits and words zero, games 16-byte aligned at a pitch
// of GB = roundup16(4 S RW) bytes (16 / 112 / 512 / 2000).
//
// Formulation.  A token t stands for the coefficient t - shift, whose residue is the low bit of t ^ shift, so every byte
// is a valid token (no TG_FLAG_RANGE).  The rank-1 term u (x) v (x) w mod 2 is, in row i, either nothing (u_i even) or
// the mask V = OR_{j: v_j odd} (w bits) << (j S) of S^2 bits, so a step is   row_i ^= u_i ? V : 0   word by word.
// V is built once per game and step from the parity bits of v and w (mask_word).
//
// Work split: a group of G lanes per game -- one thread per game at 4x4x4 (the game is one uint4) and 9x9x9 (27 words in
// registers; the 112-byte games of a warp move through shared memory so that global accesses are coalesced), 16 lanes
// at 16x16x16 and a warp at 25x25x25, each lane holding NC of the game's 16-byte chunks (chunk q = lane + G m).  A chunk
// of those two sizes lies in one row (RW is a multiple of four), and lane r of the group builds word r of V, which the
// lanes read with a shuffle.
#include <type_traits>

#include "tg_gf2.cuh"

namespace tg {
namespace {

constexpr uint32_t FULL = 0xFFFFFFFFu;

// word r of V = OR_{j: v_j odd} w << (j S): bits [32 r, 32 r + 32) of the S^2-bit row mask
template <int S>
__device__ __forceinline__ uint32_t mask_word(uint32_t vb, uint32_t wb, int r) {
    uint32_t m = 0;
    const int j0 = (32 * r) / S;
#pragma unroll
    for (int t = 0; t < 32 / S + 2; t++) {
        const int j = j0 + t;
        const int o = j * S - 32 * r;
        if (j < S && o < 32 && ((vb >> j) & 1u)) m |= o >= 0 ? wb << o : wb >> -o;
    }
    return m;
}

// sum over the lanes of a game's group
template <int G, typename T>
__device__ __forceinline__ T group_sum(T x) {
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) x += __shfl_xor_sync(FULL, x, o);
    return x;
}

// ------------------------------------------------------------------ state key tables
// key(T) = sum T[i][j][k] A_i B_j C_k (mod 2^64) over the 0/1 values (tg_state_key).  A word r of row i adds
// A_i * sum_{bits b} (B C)[32 r + b]; that sum is read from nibble tables tab[r][n][16] of the (B C) products.
template <int S>
struct KeyTab {
    unsigned long long a[S];
    unsigned long long tab[GeoB<S>::RW * 128];

    __device__ __forceinline__ void build() {
        for (int i = threadIdx.x; i < S; i += blockDim.x) a[i] = key_const(0x1000, i);
        for (int e = threadIdx.x; e < GeoB<S>::RW * 128; e += blockDim.x) {
            const int r = e / 128, n = (e / 16) % 8, v = e % 16;
            unsigned long long s = 0;
            for (int b = 0; b < 4; b++) {
                const int jk = 32 * r + 4 * n + b;
                if (((v >> b) & 1) && jk < GeoB<S>::S2) s += key_const(0x2000, jk / S) * key_const(0x3000, jk % S);
            }
            tab[e] = s;
        }
    }
    // sum of (B C) over the set bits of word r of a row
    __device__ __forceinline__ unsigned long long word(uint32_t x, int r) const {
        unsigned long long s = 0;
#pragma unroll
        for (int n = 0; n < 8; n++) s += tab[(r * 8 + n) * 16 + ((x >> (4 * n)) & 15u)];
        return s;
    }
};

// ------------------------------------------------------------------ game loads and stores
// Chunks c[m] = chunk gl + G m of game `game` (zero where absent).  STAGED (9x9x9, one thread per game): the warp's 32
// consecutive games are one contiguous run, copied through the warp's shared buffer with coalesced 16-byte accesses.
template <int S>
struct Games {
    using B = GeoB<S>;
    uint4 *buf; // STAGED: this warp's buffer [32][NQ]

    __device__ __forceinline__ void load_direct(const uint4 *src, long long game, bool live, int gl, uint4 (&c)[B::NC]) const {
#pragma unroll
        for (int m = 0; m < B::NC; m++) {
            const int q = gl + B::G * m;
            c[m] = live && q < B::NQ ? src[game * B::NQ + q] : make_uint4(0, 0, 0, 0);
        }
    }
    // games w0 .. w0 + 31 of n (w0 = the warp's first game)
    __device__ __forceinline__ void load_staged(const uint4 *src, long long w0, long long n, uint4 (&c)[B::NC]) const {
        const int lane = threadIdx.x & 31;
        const long long end = (n - w0 < 32 ? n - w0 : 32) * B::NQ;
        for (int e = lane; e < end; e += 32) buf[e] = src[w0 * B::NQ + e];
        __syncwarp();
#pragma unroll
        for (int m = 0; m < B::NC; m++) c[m] = buf[lane * B::NQ + m];
        __syncwarp();
    }
    __device__ __forceinline__ void store_staged(uint4 *dst, long long w0, long long n, const uint4 (&c)[B::NC]) const {
        const int lane = threadIdx.x & 31;
#pragma unroll
        for (int m = 0; m < B::NC; m++) buf[lane * B::NQ + m] = c[m];
        __syncwarp();
        const long long end = (n - w0 < 32 ? n - w0 : 32) * B::NQ;
        for (int e = lane; e < end; e += 32) dst[w0 * B::NQ + e] = buf[e];
        __syncwarp();
    }
    __device__ __forceinline__ void store_direct(uint4 *dst, long long game, bool live, int gl, const uint4 (&c)[B::NC]) const {
#pragma unroll
        for (int m = 0; m < B::NC; m++) {
            const int q = gl + B::G * m;
            if (live && q < B::NQ) dst[game * B::NQ + q] = c[m];
        }
    }
};

__device__ __forceinline__ uint32_t &cw(uint4 &c, int k) { return k == 0 ? c.x : k == 1 ? c.y : k == 2 ? c.z : c.w; }

// The row of word k of chunk m of lane gl, and the word's index in its row; -1 for padding words (9x9x9: word 27).
template <int S>
__device__ __forceinline__ int chunk_row(int gl, int m) {
    using B = GeoB<S>;
    if constexpr (B::G == 1) return 0; // rows of single-thread games are per word (word_row)
    else return (gl + B::G * m) / (B::RW / 4);
}
template <int S>
__device__ __forceinline__ int word_row(int m, int k) { return (4 * m + k) / GeoB<S>::RW; }

// Applies the rank-1 term (parities p) to the chunks, returns the popcount of the result; KEYS: adds the key of the
// result to *key.  All lanes of the warp must call it (shuffles).
template <int S, bool KEYS>
__device__ __forceinline__ int apply(uint4 (&c)[GeoB<S>::NC], const Par &p, bool on, int gl, const KeyTab<S> *kt,
                                     unsigned long long *key) {
    using B = GeoB<S>;
    int cnt = 0;
    if constexpr (B::G == 1) {
        uint32_t M[B::RW];
#pragma unroll
        for (int r = 0; r < B::RW; r++) M[r] = on ? mask_word<S>(p.v, p.w, r) : 0u;
        unsigned long long ks = 0;
#pragma unroll
        for (int m = 0; m < B::NC; m++) {
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const int wg = 4 * m + k;
                if (wg >= S * B::RW) continue; // padding word
                const int i = wg / B::RW, r = wg % B::RW;
                uint32_t &x = cw(c[m], k);
                x ^= M[r] & (0u - ((p.u >> i) & 1u));
                cnt += __popc(x);
                if constexpr (KEYS) ks += kt->a[i] * kt->word(x, r);
            }
        }
        if constexpr (KEYS) *key += ks;
    } else {
        const int lane = threadIdx.x & 31;
        const uint32_t Mw = on ? mask_word<S>(p.v, p.w, gl < B::RW ? gl : 0) : 0u;
        const int base = lane & ~(B::G - 1);
#pragma unroll
        for (int m = 0; m < B::NC; m++) {
            const int q = gl + B::G * m;
            const int i = chunk_row<S>(gl, m), r0 = 4 * (q % (B::RW / 4));
            const uint32_t ui = 0u - ((p.u >> i) & 1u); // 0 for the absent chunks (i = S)
            unsigned long long ks = 0;
#pragma unroll
            for (int k = 0; k < 4; k++) {
                uint32_t &x = cw(c[m], k);
                x ^= __shfl_sync(FULL, Mw, base + r0 + k) & ui;
                cnt += __popc(x);
                if constexpr (KEYS) ks += kt->word(x, r0 + k);
            }
            if constexpr (KEYS) {
                if (i < S) *key += kt->a[i] * ks;
            }
        }
    }
    return cnt;
}

// ------------------------------------------------------------------ K1 / K8: step and leaf expansion
// Game x < N of the output is game x / k of the input plus the rank-1 term of record x: k = 1 is the step (in place
// allowed: a game is read whole before it is written), k > 1 the k children of every parent (parents are re-read by
// the k groups of their children, which run side by side, so each is fetched from memory about once).
template <int S, bool KEYS>
__global__ void __launch_bounds__(256) step_gf2_kernel(const uint4 *__restrict__ in, const uint8_t *__restrict__ tape, int k,
                                                       uint4 *__restrict__ out, uint8_t *__restrict__ flags, int32_t *__restrict__ nnz,
                                                       unsigned long long *__restrict__ keys, long long N, int shift) {
    using B = GeoB<S>;
    __shared__ __align__(16) uint4 s_stage[B::STAGED ? 8 * 32 * B::NQ : 1];
    __shared__ typename std::conditional<KEYS, KeyTab<S>, char>::type s_key; // the key tables only where keys are asked for
    const KeyTab<S> *kt = nullptr;
    if constexpr (KEYS) {
        s_key.build();
        __syncthreads();
        kt = &s_key;
    }
    Games<S> io{s_stage + (threadIdx.x >> 5) * 32 * B::NQ};
    const int gl = threadIdx.x % B::G, slot = threadIdx.x / B::G;
    for (long long x0 = (long long)blockIdx.x * B::GPC; x0 < N; x0 += (long long)gridDim.x * B::GPC) {
        const long long x = x0 + slot;
        const bool live = x < N;
        uint4 c[B::NC];
        if constexpr (B::STAGED) {
            if (k == 1) io.load_staged(in, x0 + (threadIdx.x & ~31), N, c);
            else io.load_direct(in, x / k, live, gl, c);
        } else {
            io.load_direct(in, x / k, live, gl, c);
        }
        const Par p = live ? parities<S>(tape + x * B::TP, shift) : Par{0u, 0u, 0u};
        unsigned long long key = 0;
        int cnt = apply<S, KEYS>(c, p, true, gl, kt, &key);
        if constexpr (B::STAGED) io.store_staged(out, x0 + (threadIdx.x & ~31), N, c);
        else io.store_direct(out, x, live, gl, c);
        cnt = group_sum<B::G>(cnt);
        if constexpr (KEYS) key = group_sum<B::G>(key);
        if (live && gl == 0) {
            flags[x] = (uint8_t)((cnt == 0 ? TG_FLAG_TERMINAL : 0u) | (p.u == 0 || p.v == 0 || p.w == 0 ? TG_FLAG_NULL : 0u));
            nnz[x] = cnt;
            if constexpr (KEYS) keys[x] = key;
        }
    }
}

// ------------------------------------------------------------------ K2: rollout / replay
// The game stays in registers for all K steps; each step's record is read straight from the tape.  FREEZE: a game stops
// at its first all-zero state (the break at act.py:49).  A warp leaves the loop once none of its games is alive.
template <int S, bool FREEZE>
__global__ void __launch_bounds__(256) rollout_gf2_kernel(const uint4 *__restrict__ in, const uint8_t *__restrict__ tape,
                                                          long long stride, int K, uint4 *__restrict__ out, uint8_t *__restrict__ flags,
                                                          int32_t *__restrict__ nnz, int32_t *__restrict__ steps, long long N, int shift) {
    using B = GeoB<S>;
    __shared__ __align__(16) uint4 s_stage[B::STAGED ? 8 * 32 * B::NQ : 1];
    Games<S> io{s_stage + (threadIdx.x >> 5) * 32 * B::NQ};
    const int gl = threadIdx.x % B::G, slot = threadIdx.x / B::G;
    for (long long x0 = (long long)blockIdx.x * B::GPC; x0 < N; x0 += (long long)gridDim.x * B::GPC) {
        const long long x = x0 + slot;
        const bool live = x < N;
        uint4 c[B::NC];
        if constexpr (B::STAGED) io.load_staged(in, x0 + (threadIdx.x & ~31), N, c);
        else io.load_direct(in, x, live, gl, c);
        int cnt = 0;
#pragma unroll
        for (int m = 0; m < B::NC; m++) cnt += __popc(c[m].x) + __popc(c[m].y) + __popc(c[m].z) + __popc(c[m].w);
        cnt = group_sum<B::G>(cnt);
        bool alive = live && (!FREEZE || cnt != 0);
        int my_steps = 0;
        const uint8_t *rec = tape + x * B::TP;
        for (int t = 0; t < K; t++, rec += stride) {
            if (!__any_sync(FULL, alive)) break;
            const Par p = alive ? parities<S>(rec, shift) : Par{0u, 0u, 0u};
            cnt = group_sum<B::G>(apply<S, false>(c, p, alive, gl, nullptr, nullptr));
            if (alive) my_steps = t + 1;
            if (FREEZE && cnt == 0) alive = false;
        }
        if constexpr (B::STAGED) io.store_staged(out, x0 + (threadIdx.x & ~31), N, c);
        else io.store_direct(out, x, live, gl, c);
        cnt = 0;
#pragma unroll
        for (int m = 0; m < B::NC; m++) cnt += __popc(c[m].x) + __popc(c[m].y) + __popc(c[m].z) + __popc(c[m].w);
        cnt = group_sum<B::G>(cnt);
        if (live && gl == 0) {
            flags[x] = (uint8_t)(cnt == 0 ? TG_FLAG_TERMINAL : 0u);
            nnz[x] = cnt;
            if (FREEZE) steps[x] = my_steps;
        }
    }
}

// ------------------------------------------------------------------ K7: state key
template <int S>
__global__ void __launch_bounds__(256) state_key_gf2_kernel(const uint4 *__restrict__ in, unsigned long long *__restrict__ keys, long long N) {
    using B = GeoB<S>;
    __shared__ __align__(16) uint4 s_stage[B::STAGED ? 8 * 32 * B::NQ : 1];
    __shared__ KeyTab<S> s_key;
    s_key.build();
    __syncthreads();
    Games<S> io{s_stage + (threadIdx.x >> 5) * 32 * B::NQ};
    const int gl = threadIdx.x % B::G, slot = threadIdx.x / B::G;
    for (long long x0 = (long long)blockIdx.x * B::GPC; x0 < N; x0 += (long long)gridDim.x * B::GPC) {
        const long long x = x0 + slot;
        const bool live = x < N;
        uint4 c[B::NC];
        if constexpr (B::STAGED) io.load_staged(in, x0 + (threadIdx.x & ~31), N, c);
        else io.load_direct(in, x, live, gl, c);
        unsigned long long key = 0;
        apply<S, true>(c, Par{0u, 0u, 0u}, false, gl, &s_key, &key);
        key = group_sum<B::G>(key);
        if (live && gl == 0) keys[x] = key;
    }
}

// ------------------------------------------------------------------ K6: slice rank over GF(2)
// Slice i is the S x S bit matrix T[i,:,:]: its row j is bits [j S, j S + S) of row i, at most 25 bits, one register.
// Elimination: the lowest set bit of each non-zero row is its pivot, cleared from the rows below by XOR.
template <int S>
__device__ __forceinline__ int rank_gf2(const uint32_t (&w)[GeoB<S>::RW]) {
    uint32_t r[S];
#pragma unroll
    for (int j = 0; j < S; j++) {
        const int o = j * S, q = o / 32, s = o % 32;
        uint32_t v = w[q] >> s;
        if (s + S > 32) v |= w[q + 1] << (32 - s);
        r[j] = v & ((1u << S) - 1u);
    }
    int rank = 0;
#pragma unroll
    for (int j = 0; j < S; j++) {
        const uint32_t x = r[j];
        rank += x != 0;
        const uint32_t piv = x & (0u - x);
#pragma unroll
        for (int q = j + 1; q < S; q++) r[q] ^= (r[q] & piv) ? x : 0u;
    }
    return rank;
}

template <int S>
__global__ void __launch_bounds__(256) slice_rank_gf2_kernel(const uint4 *__restrict__ in, int32_t *__restrict__ ranks, long long N) {
    using B = GeoB<S>;
    __shared__ __align__(16) uint4 s_stage[B::STAGED ? 8 * 32 * B::NQ : 1];
    Games<S> io{s_stage + (threadIdx.x >> 5) * 32 * B::NQ};
    const int gl = threadIdx.x % B::G, slot = threadIdx.x / B::G;
    for (long long x0 = (long long)blockIdx.x * B::GPC; x0 < N; x0 += (long long)gridDim.x * B::GPC) {
        const long long x = x0 + slot;
        const bool live = x < N;
        int rank = 0;
        if constexpr (B::G == 1) { // one thread per game, all S slices
            uint4 c[B::NC];
            if constexpr (B::STAGED) io.load_staged(in, x0 + (threadIdx.x & ~31), N, c);
            else io.load_direct(in, x, live, 0, c);
#pragma unroll
            for (int i = 0; i < S; i++) {
                uint32_t w[B::RW];
#pragma unroll
                for (int r = 0; r < B::RW; r++) w[r] = cw(c[(i * B::RW + r) / 4], (i * B::RW + r) % 4);
                rank += rank_gf2<S>(w);
            }
        } else { // lane i of the group: slice i
            uint32_t w[B::RW];
            const bool mine = live && gl < S;
#pragma unroll
            for (int q = 0; q < B::RW / 4; q++) {
                const uint4 t = mine ? in[x * B::NQ + gl * (B::RW / 4) + q] : make_uint4(0, 0, 0, 0);
                w[4 * q] = t.x, w[4 * q + 1] = t.y, w[4 * q + 2] = t.z, w[4 * q + 3] = t.w;
            }
            rank = group_sum<B::G>(rank_gf2<S>(w));
        }
        if (live && gl == 0) ranks[x] = rank;
    }
}

// ------------------------------------------------------------------ boundary conversions
// int8 / int16 slab -> bit slab: the low bit of each two's-complement entry; one thread per output word
template <int S, typename E>
__global__ void __launch_bounds__(256) pack_gf2_kernel(const E *__restrict__ slab, uint32_t *__restrict__ bits, long long nwords) {
    using B = GeoB<S>;
    using G = Geo<S>; // element geometry of the int8 / int16 slab
    constexpr int GW = B::GB / 4;
    for (long long o = blockIdx.x * (long long)blockDim.x + threadIdx.x; o < nwords; o += (long long)gridDim.x * blockDim.x) {
        const long long g = o / GW;
        const int wg = (int)(o - g * GW);
        uint32_t x = 0;
        if (wg < S * B::RW) {
            const int i = wg / B::RW, r = wg % B::RW;
            const E *row = slab + g * G::GP + i * G::RP + 32 * r;
            const int nb = B::S2 - 32 * r < 32 ? B::S2 - 32 * r : 32;
            for (int b = 0; b < nb; b++) x |= ((uint32_t)row[b] & 1u) << b;
        }
        bits[o] = x;
    }
}

// bit slab -> int8 slab of 0/1; one thread per output word (four entries)
template <int S>
__global__ void __launch_bounds__(256) unpack_gf2_kernel(const uint32_t *__restrict__ bits, uint32_t *__restrict__ slab, long long nwords) {
    using B = GeoB<S>;
    using G = Geo<S>;
    constexpr int GW = G::GP / 4;
    for (long long o = blockIdx.x * (long long)blockDim.x + threadIdx.x; o < nwords; o += (long long)gridDim.x * blockDim.x) {
        const long long g = o / GW;
        const int e = 4 * (int)(o - g * GW); // byte offset in the int8 game
        const int i = e / G::RP, jk = e % G::RP;
        uint32_t x = 0;
        if (i < S) {
            const uint32_t *row = bits + g * (B::GB / 4) + i * B::RW;
#pragma unroll
            for (int b = 0; b < 4; b++)
                if (jk + b < B::S2) x |= ((row[(jk + b) / 32] >> ((jk + b) % 32)) & 1u) << (8 * b);
        }
        slab[o] = x;
    }
}

template <int S>
int launch_step_gf2(const uint32_t *in, const uint8_t *tape, int k, uint32_t *out, uint8_t *flags, int32_t *nnz, uint64_t *keys,
                    long long N, int shift, cudaStream_t st) {
    const unsigned grid = grid_for(N, GeoB<S>::GPC);
    const uint4 *i4 = reinterpret_cast<const uint4 *>(in);
    uint4 *o4 = reinterpret_cast<uint4 *>(out);
    unsigned long long *kp = reinterpret_cast<unsigned long long *>(keys);
    if (keys) step_gf2_kernel<S, true><<<grid, 256, 0, st>>>(i4, tape, k, o4, flags, nnz, kp, N, shift);
    else step_gf2_kernel<S, false><<<grid, 256, 0, st>>>(i4, tape, k, o4, flags, nnz, kp, N, shift);
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

template <int S>
int launch_rollout_gf2(const uint32_t *in, const uint8_t *tape, long long stride, int K, uint32_t *out, uint8_t *flags, int32_t *nnz,
                       int32_t *steps, long long B, int shift, int freeze, cudaStream_t st) {
    const unsigned grid = grid_for(B, GeoB<S>::GPC);
    const uint4 *i4 = reinterpret_cast<const uint4 *>(in);
    uint4 *o4 = reinterpret_cast<uint4 *>(out);
    if (freeze) rollout_gf2_kernel<S, true><<<grid, 256, 0, st>>>(i4, tape, stride, K, o4, flags, nnz, steps, B, shift);
    else rollout_gf2_kernel<S, false><<<grid, 256, 0, st>>>(i4, tape, stride, K, o4, flags, nnz, steps, B, shift);
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

template <typename E>
int pack_gf2_any(const E *slab, uint32_t *bits, int64_t B, int S, void *stream) {
    if (const int rc = check_pair(S, B, slab, 16, bits, 16); rc != LAUNCH) return rc;
    return with_S(S, [&](auto s) {
        constexpr int kS = decltype(s)::value;
        pack_gf2_kernel<kS, E><<<grid_for(B * (GeoB<kS>::GB / 4), 256), 256, 0, (cudaStream_t)stream>>>(slab, bits, B * (GeoB<kS>::GB / 4));
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    });
}

int rollout_gf2_dispatch(const uint32_t *in, const uint8_t *tape, int64_t stride, int K, uint32_t *out, uint8_t *flags, int32_t *nnz,
                         int32_t *steps, int64_t B, int S, int shift, int freeze, void *stream) {
    const int rc = check_rollout(S, B, K, shift, in, tape, stride, out, flags, nnz, steps, freeze);
    if (rc != LAUNCH) return rc;
    return with_S(S, [&](auto s) {
        return launch_rollout_gf2<decltype(s)::value>(in, tape, stride, K, out, flags, nnz, steps, B, shift, freeze, (cudaStream_t)stream);
    });
}

} // namespace
} // namespace tg

extern "C" {

int tg_layout_gf2(int S, int *row_words, int *game_bytes) {
    if (!tg::supported_S(S)) return TG_E_ARG;
    const int rw = (S * S + 31) / 32;
    if (row_words) *row_words = rw;
    if (game_bytes) *game_bytes = (4 * S * rw + 15) & ~15;
    return TG_OK;
}

int tg_pack_gf2(const int8_t *slab, uint32_t *bits, int64_t B, int S, void *stream) { return tg::pack_gf2_any(slab, bits, B, S, stream); }

int tg_pack_gf2_i16(const int16_t *slab16, uint32_t *bits, int64_t B, int S, void *stream) {
    return tg::pack_gf2_any(slab16, bits, B, S, stream);
}

int tg_unpack_gf2(const uint32_t *bits, int8_t *slab, int64_t B, int S, void *stream) {
    if (const int rc = tg::check_pair(S, B, bits, 16, slab, 16); rc != tg::LAUNCH) return rc;
    return tg::with_S(S, [&](auto s) {
        constexpr int kS = decltype(s)::value;
        tg::unpack_gf2_kernel<kS><<<tg::grid_for(B * (tg::Geo<kS>::GP / 4), 256), 256, 0, (cudaStream_t)stream>>>(
            bits, reinterpret_cast<uint32_t *>(slab), B * (tg::Geo<kS>::GP / 4));
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    });
}

int tg_step_gf2(const uint32_t *bits_in, const uint8_t *tape, uint32_t *bits_out, uint8_t *flags, int32_t *nnz, int64_t B, int S,
                int shift, void *stream) {
    if (const int rc = tg::check_step(S, B, shift, bits_in, tape, bits_out, flags, nnz); rc != tg::LAUNCH) return rc;
    return tg::with_S(S, [&](auto s) {
        return tg::launch_step_gf2<decltype(s)::value>(bits_in, tape, 1, bits_out, flags, nnz, nullptr, B, shift, (cudaStream_t)stream);
    });
}

int tg_expand_children_gf2(const uint32_t *parents, const uint8_t *tape, int k, uint32_t *children, uint8_t *flags, int32_t *nnz,
                           uint64_t *keys, int64_t B, int S, int shift, void *stream) {
    if (const int rc = tg::check_expand(S, B, k, shift, parents, tape, children, flags, nnz); rc != tg::LAUNCH) return rc;
    const long long N = (long long)B * k;
    return tg::with_S(S, [&](auto s) {
        return tg::launch_step_gf2<decltype(s)::value>(parents, tape, k, children, flags, nnz, keys, N, shift, (cudaStream_t)stream);
    });
}

int tg_rollout_gf2(const uint32_t *bits_in, const uint8_t *tape, int64_t tape_step_stride, int K, uint32_t *bits_out, uint8_t *flags,
                   int32_t *nnz, int32_t *steps, int64_t B, int S, int shift, void *stream) {
    return tg::rollout_gf2_dispatch(bits_in, tape, tape_step_stride, K, bits_out, flags, nnz, steps, B, S, shift, 1, stream);
}

int tg_replay_gf2(const uint32_t *bits_in, const uint8_t *tape, int64_t tape_step_stride, int K, uint32_t *bits_out, uint8_t *flags,
                  int32_t *nnz, int64_t B, int S, int shift, void *stream) {
    return tg::rollout_gf2_dispatch(bits_in, tape, tape_step_stride, K, bits_out, flags, nnz, nullptr, B, S, shift, 0, stream);
}

int tg_state_key_gf2(const uint32_t *bits, uint64_t *keys, int64_t B, int S, void *stream) {
    if (const int rc = tg::check_pair(S, B, bits, 16, keys, 1); rc != tg::LAUNCH) return rc;
    return tg::with_S(S, [&](auto s) {
        constexpr int kS = decltype(s)::value;
        tg::state_key_gf2_kernel<kS><<<tg::grid_for(B, tg::GeoB<kS>::GPC), 256, 0, (cudaStream_t)stream>>>(
            reinterpret_cast<const uint4 *>(bits), reinterpret_cast<unsigned long long *>(keys), B);
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    });
}

int tg_slice_rank_gf2(const uint32_t *bits, int32_t *ranks, int64_t B, int S, void *stream) {
    if (const int rc = tg::check_pair(S, B, bits, 16, ranks, 1); rc != tg::LAUNCH) return rc;
    return tg::with_S(S, [&](auto s) {
        constexpr int kS = decltype(s)::value;
        tg::slice_rank_gf2_kernel<kS><<<tg::grid_for(B, tg::GeoB<kS>::GPC), 256, 0, (cudaStream_t)stream>>>(
            reinterpret_cast<const uint4 *>(bits), ranks, B);
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    });
}

} // extern "C"
