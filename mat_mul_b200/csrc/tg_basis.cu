// tg_basis.cu -- K5: change-of-basis augmentation (C ABI: tg_change_of_basis,
// tg_change_of_basis_factors, tg_sample_unimodular).
//
// ABSENT from the reference (grep finds no basis/einsum code); specified from
// the AlphaTensor paper (Fawzi et al. 2022, Methods "Change of basis"):
//     T'[i][j][k] = sum_abc A[i][a] B[j][b] C[k][c] T[a][b][c]
//     u' = A u,  v' = B v,  w' = C w      (so sum u'(x)v'(x)w' = T')
// with A, B, C integer and unimodular.  Parity is pinned by our own int64
// oracle (oracle/tg_oracle.c orc_change_of_basis) and algebraic invariants.
//
// Fast path (basis_fast_kernel): a group of S*W threads per game, several games
// per CTA, three passes through shared memory:
//   C. Y[a][b][k'] = sum_k C[k'][k] T[a][b][k]   -- the contracted axis is the packed
//      one: DP4A over 4 consecutive k, exact int32 results, their maximum tracked;
//   A. Z[i][b][.]  = sum_a A[i][a] Y[a][b][.]    -- one IMAD per LPW entries: the
//   B. T'[i][j][.] = sum_b B[j][b] Z[i][b][.]       k' axis is packed LPW entries per
//      word (3 x 10 bit for S = 9, 2 x 16 bit otherwise) in integer form
//      sum_l y_l 2^(LB l), linear in the scalar matrix entry.
// The packed passes are exact while every entry fits its lane; that is
// guaranteed up front by  max|Y| * ||A||_inf * ||B||_inf <= 2^(LB-1) - 1.  A game
// that fails the test (large matrices) is marked and redone by the exact int32
// kernel below -- results are identical either way.
//
// Exact path (basis_kernel): one CTA per game, three passes of the SAME routine
// "contract the slowest axis, write the result rotated":
//     X[b][c][i] = sum_a A[i][a] T[a][b][c]
//     Y[c][i][j] = sum_b B[j][b] X[b][c][i]
//     Z[i][j][k] = sum_c C[k][c] Y[c][i][j]
// X and Y live in shared memory as int32 (|Y| <= S^2 * 2^21 <= 2^29 for int8
// input and int8 matrices); the last pass accumulates in 64 bit, because |T'|
// reaches S^3 * 2^28 = 2^34 .. 2^40.  A thread owns one column of the
// contracted axis in registers and produces its S outputs.  TG_FLAG_RANGE marks
// games whose T' leaves the int8 slab's guaranteed zone [-64,63].
#include "tg_common.cuh"

namespace tg {

template <int S>
struct BasisCfg {
    using G = Geo<S>;
    static constexpr int S2 = S * S, S3 = S2 * S;
    static constexpr int NT = S2 >= 256 ? 256 : (S2 >= 64 ? 96 : 32);
    static constexpr int SMEM_BYTES = G::GP + 2 * S3 * 4 + 3 * S2 * 4 + 16;
};

// out[rest][a'] = sum_a M[a'][a] in[a][rest]; `rest` has S*S entries.  Acc = long long: the sums are formed in 64 bit,
// stored as their low 32 bits, and TG_FLAG_RANGE is OR-ed into *s_flag where one does not fit int32.
template <int S, int NT, typename Acc = int32_t>
__device__ __forceinline__ void mode_pass(const int32_t *__restrict__ in, int32_t *__restrict__ out,
                                          const int32_t *__restrict__ M, uint32_t *s_flag = nullptr) {
    constexpr int S2 = S * S;
    bool wide = false;
    for (int r = threadIdx.x; r < S2; r += NT) {
        int32_t col[S];
#pragma unroll
        for (int a = 0; a < S; a++) col[a] = in[a * S2 + r];
#pragma unroll
        for (int ap = 0; ap < S; ap++) {
            Acc acc = 0;
#pragma unroll
            for (int a = 0; a < S; a++) acc += (Acc)M[ap * S + a] * col[a];
            out[r * S + ap] = (int32_t)acc;
            if constexpr (sizeof(Acc) > 4) wide |= acc != (Acc)(int32_t)acc;
        }
    }
    if (wide) atomicOr(s_flag, (uint32_t)TG_FLAG_RANGE);
}


// only_marked: visit every game, redo those the fast kernel marked with BASIS_REDO (they leave with TG_FLAG_PATH_EXACT).
// OUT16: the result is written as an int16 slab (TG_FLAG_RANGE: an entry does not fit int16) instead of an int8 slab
// (TG_FLAG_RANGE: an entry left [-64, 63]).
template <int S, bool OUT16>
__global__ void __launch_bounds__(BasisCfg<S>::NT)
    basis_kernel(const int8_t *__restrict__ slab_in, const int8_t *__restrict__ mats, long long mat_stride,
                 void *__restrict__ slab_out_v, uint8_t *__restrict__ flags, long long N, int only_marked) {
    using C = BasisCfg<S>;
    using G = Geo<S>;
    constexpr int NT = C::NT;
    extern __shared__ __align__(128) uint8_t smem[];
    int8_t *s_in = reinterpret_cast<int8_t *>(smem);
    int32_t *s_a = reinterpret_cast<int32_t *>(smem + G::GP);
    int32_t *s_b = s_a + C::S3;
    int32_t *s_m = s_b + C::S3; // A, B, C as int32 [3][S][S]
    uint32_t *s_flag = reinterpret_cast<uint32_t *>(s_m + 3 * C::S2);

    const int tid = threadIdx.x;
    // all games (grid-stride), or only the marked ones of this CTA's contiguous chunk of the flags array
    __shared__ int s_list[1024];
    __shared__ int s_cnt;
    const long long chunk = only_marked ? (N + gridDim.x - 1) / gridDim.x : 0;
    const long long lo = only_marked ? chunk * blockIdx.x : blockIdx.x, hi = only_marked ? min(N, lo + chunk) : N;
    for (long long base = lo; base < hi; base += only_marked ? 1024 : (long long)gridDim.x) {
    int cnt = 1;
    if (only_marked) {
        if (tid == 0) s_cnt = 0;
        __syncthreads();
        for (long long q = base + tid; q < min(hi, base + 1024); q += NT)
            if (flags[q] & BASIS_REDO) s_list[atomicAdd(&s_cnt, 1)] = (int)(q - base);
        __syncthreads();
        cnt = s_cnt;
    }
    for (int it = 0; it < cnt; it++) {
    const long long n = only_marked ? base + s_list[it] : base;
    __syncthreads();
    const uint32_t *src = reinterpret_cast<const uint32_t *>(slab_in + n * G::GP);
    for (int w = tid; w < G::GP / 4; w += NT) reinterpret_cast<uint32_t *>(s_in)[w] = src[w];
    const int8_t *m = mats + n * mat_stride;
    for (int q = tid; q < 3 * C::S2; q += NT) s_m[q] = (int32_t)m[q];
    if (tid == 0) *s_flag = 0;
    __syncthreads();
    for (int e = tid; e < C::S3; e += NT) { // dense copy T[a][b][c]
        const int i = e / C::S2, jk = e % C::S2;
        s_a[e] = (int32_t)s_in[i * G::RP + jk];
    }
    __syncthreads();
    mode_pass<S, NT>(s_a, s_b, s_m); // contract a with A
    __syncthreads();
    mode_pass<S, NT>(s_b, s_a, s_m + C::S2); // contract b with B
    __syncthreads();
    mode_pass<S, NT, long long>(s_a, s_b, s_m + 2 * C::S2, s_flag); // contract c with C -> Z[i][j][k]
    __syncthreads();
    uint32_t bad = 0;
    if constexpr (OUT16) {
        uint32_t *dst = reinterpret_cast<uint32_t *>(reinterpret_cast<int16_t *>(slab_out_v) + n * G::GP);
        for (int w = tid; w < G::GP / 2; w += NT) { // two int16 per word
            const int i = (2 * w) / G::RP, x = (2 * w) % G::RP;
            uint32_t word = 0;
            if (i < S) {
#pragma unroll
                for (int q = 0; q < 2; q++) {
                    const int jk = x + q;
                    if (jk < C::S2) {
                        const int v = s_b[i * C::S2 + jk];
                        if (v < -32768 || v > 32767) bad = TG_FLAG_RANGE;
                        word |= ((uint32_t)v & 0xFFFFu) << (16 * q);
                    }
                }
            }
            dst[w] = word;
        }
    } else {
        uint32_t *dst = reinterpret_cast<uint32_t *>(reinterpret_cast<int8_t *>(slab_out_v) + n * G::GP);
        for (int w = tid; w < G::GP / 4; w += NT) {
            const int i = w / G::WR, c = w % G::WR;
            uint32_t word = 0;
            if (i < S) {
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    const int jk = 4 * c + q;
                    if (jk < C::S2) {
                        const int v = s_b[i * C::S2 + jk];
                        if (v < -64 || v > 63) bad = TG_FLAG_RANGE;
                        word |= ((uint32_t)v & 0xFFu) << (8 * q);
                    }
                }
            }
            dst[w] = word;
        }
    }
    if (bad) atomicOr(s_flag, bad);
    __syncthreads();
    if (tid == 0 && flags) flags[n] = (uint8_t)(*s_flag | (only_marked ? TG_FLAG_PATH_EXACT : 0u));
    }
    }
}

// ------------------------------------------------------------------ fast path
template <int S, bool OUT16 = false>
struct BasisFast {
    using G = Geo<S>;
    static constexpr int EB = OUT16 ? 2 : 1;            // bytes per entry of the OUTPUT tile
    static constexpr int LPW = (S == 9) ? 3 : 2;        // entries per packed word
    static constexpr int LB = (S == 9) ? 10 : 16;       // bits per lane
    static constexpr int LMAX = (1 << (LB - 1)) - 1;    // every entry must stay in [-LMAX, LMAX]
    static constexpr int W = (S + LPW - 1) / LPW;       // packed words per run of S entries: 3 / 8 / 2
    static constexpr int CB = S == 9 ? 3 : (S == 16 ? 4 : 2); // words (columns) of a run owned by one thread
    static constexpr int VEC = S == 4 ? 2 : 4;          // words per vector access of a thread's columns
    static constexpr int NSPLIT = W / CB;               // threads sharing a run: 1 / 2 / 1
    static constexpr int WP = NSPLIT * VEC;             // padded words per run: 4 / 8 / 2
    static constexpr int TPG = S * NSPLIT;              // threads per game: 9 / 32 / 4
    static constexpr int RPT = S / NSPLIT;              // runs per thread in pass C: 9 / 8 / 4
    static constexpr int BB = S == 9 ? 3 : (S == 16 ? 2 : 4); // ... worked off BB at a time
    static constexpr int KW4 = (S + 3) / 4;             // byte words per run (DP4A operands)
    static constexpr int GPC = S == 9 ? 24 : (S == 16 ? 4 : 64); // games per CTA
    static constexpr int NT = GPC * TPG;                // 216 / 128 / 256
    static constexpr int RW = (S + 3) & ~3;             // int32 per (padded) matrix row: rows are read as int4
    static constexpr int YROW = S * WP + (S == 16 ? 8 : 0); // words between Y[a][.][.] and Y[a+1][.][.], padded so that
                                                        // lanes that differ in the first index hit different banks
    static constexpr int YB = S * YROW * 4;             // bytes of Y (Z is written over it in place)
    static constexpr int OROW = G::RP + (S == 16 ? 16 : 0); // row pitch (entries) of the OUTPUT tile (same reason); a
                                                        // padded tile leaves row by row
    static constexpr int TILE_BYTES = ((EB * (S * OROW > G::GP ? S * OROW : G::GP) + (S == 9 ? 32 : (S == 4 ? 16 : 0))) + 15) & ~15;
    // per game, every part 16-byte aligned: tile, Y/Z, A and B as int32 [S][RW], C as packed bytes [S][4 words],
    // {max|Y|, normA, normB, flag}
    static constexpr int GAME_BYTES = TILE_BYTES + YB + 2 * S * RW * 4 + S * 16 + 16;
    static constexpr int SMEM_BYTES = GPC * GAME_BYTES + 16;
    static_assert(W % CB == 0 && S % NSPLIT == 0 && RPT % BB == 0 && KW4 <= 4 && GAME_BYTES % 16 == 0, "layout");
};

template <int N>
struct VecW;
template <>
struct VecW<2> { using T = int2; };
template <>
struct VecW<4> { using T = int4; };

template <int VEC>
__device__ __forceinline__ void ld_vec(const int32_t *p, int out[VEC]) {
    const typename VecW<VEC>::T v = *reinterpret_cast<const typename VecW<VEC>::T *>(p);
    out[0] = v.x, out[1] = v.y;
    if constexpr (VEC == 4) out[2] = v.z, out[3] = v.w;
}
template <int VEC>
__device__ __forceinline__ void st_vec(int32_t *p, const int in[VEC]) {
    typename VecW<VEC>::T v;
    v.x = in[0], v.y = in[1];
    if constexpr (VEC == 4) v.z = in[2], v.w = in[3];
    *reinterpret_cast<typename VecW<VEC>::T *>(p) = v;
}

template <int S, bool OUT16>
__global__ void __launch_bounds__(BasisFast<S, OUT16>::NT)
    basis_fast_kernel(const int8_t *__restrict__ slab_in, const int8_t *__restrict__ mats, long long mat_stride,
                      void *__restrict__ slab_out_v, uint8_t *__restrict__ flags, long long N) {
    using F = BasisFast<S, OUT16>;
    uint8_t *slab_out = reinterpret_cast<uint8_t *>(slab_out_v);
    using G = Geo<S>;
    constexpr int W = F::W, LPW = F::LPW, LB = F::LB, KW4 = F::KW4, S2 = S * S, RW = F::RW, CB = F::CB, VEC = F::VEC,
                  WP = F::WP, BB = F::BB, YROW = F::YROW, OROW = F::OROW;
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t *s_bar = reinterpret_cast<uint64_t *>(smem);
    const int tid = threadIdx.x;
    const int gl = tid / F::TPG, t = tid % F::TPG; // game slot, thread within the game
    const int rr = t / F::NSPLIT, h = t % F::NSPLIT; // the row index this thread owns in a pass, its column split
    const long long g0 = (long long)blockIdx.x * F::GPC;
    const int ng = (int)min((long long)F::GPC, N - g0);
    uint8_t *gbase = smem + 16 + (size_t)gl * F::GAME_BYTES;
    uint8_t *s_tile = gbase;
    int32_t *s_y = reinterpret_cast<int32_t *>(gbase + F::TILE_BYTES);
    int32_t *s_ma = reinterpret_cast<int32_t *>(gbase + F::TILE_BYTES + F::YB);
    int32_t *s_mb = s_ma + S * RW;
    uint32_t *s_cp = reinterpret_cast<uint32_t *>(s_mb + S * RW);
    int32_t *s_st = reinterpret_cast<int32_t *>(s_cp + S * 4); // {max|Y|, normA, normB, bad}
    const bool live = gl < ng;

    int32_t *s_nrm = s_st + 1;
    if (live && t < 4) s_st[t] = 0;
    if (tid == 0) {
        mbar_init(s_bar, 1);
        mbar_fence_init();
    }
    __syncthreads();
    if (tid == 0) {
        mbar_expect_tx(s_bar, (uint32_t)(ng * G::GP));
        for (int g = 0; g < ng; g++)
            bulk_g2s(smem + 16 + (size_t)g * F::GAME_BYTES, slab_in + (g0 + g) * G::GP, (uint32_t)G::GP, s_bar);
    }
    if (live) {
        const int8_t *m = mats + (g0 + gl) * mat_stride;
        // one matrix row per thread and step: A and B rows -> int32 (padded to RW, read as int4 later) and their
        // 1-norms, C rows -> bytes packed four to a word
        // TPG == S (S = 4, 9): thread t takes row t of A, of B and of C -- f and row are compile-time after unrolling, and the
        // 3 S byte loads of a thread are all in flight before the first is used
        constexpr int RSTEPS = F::TPG == S ? 3 : (3 * S + F::TPG - 1) / F::TPG;
#pragma unroll
        for (int rs = 0; rs < RSTEPS; rs++) {
            const int r = t + rs * F::TPG;
            if (F::TPG != S && r >= 3 * S) break;
            const int f = F::TPG == S ? rs : r / S, row = F::TPG == S ? t : r % S;
            int v[RW];
#pragma unroll
            for (int a = 0; a < RW; a++) v[a] = a < S ? (int)m[f * S2 + row * S + a] : 0;
            if (f < 2) {
                int nrm = 0;
#pragma unroll
                for (int a = 0; a < S; a++) nrm += abs(v[a]);
#pragma unroll
                for (int q = 0; q < RW / 4; q++) st_vec<4>((f == 0 ? s_ma : s_mb) + row * RW + 4 * q, v + 4 * q);
                atomicMax(&s_nrm[f], nrm);
            } else {
                int words[4] = {0, 0, 0, 0};
#pragma unroll
                for (int a = 0; a < S; a++) words[a >> 2] |= (v[a] & 0xFF) << (8 * (a & 3));
                st_vec<4>(reinterpret_cast<int32_t *>(s_cp) + row * 4, words);
            }
        }
    }
    __syncthreads();
    mbar_wait(s_bar, 0);

    // ---------------- pass C: Y[a][b][k'] = sum_k C[k'][k] T[a][b][k]  (DP4A), packed LPW per word.
    // thread (b = t % S, t / S) owns the runs (a, b), a = (t/S)*RPT .. +RPT-1, BB at a time (one load of a C row
    // serves BB runs); lanes differ in b, i.e. read neighbouring runs of the tile
    if (live) {
        int mx = 0;
        const int bfix = t % S;
#pragma unroll 1
        for (int a0 = (t / S) * F::RPT; a0 < (t / S + 1) * F::RPT; a0 += BB) {
            uint32_t x[BB][KW4];
#pragma unroll
            for (int bb = 0; bb < BB; bb++) {
                const int off = (a0 + bb) * G::RP + bfix * S;
                if constexpr (S % 4 == 0) {
#pragma unroll
                    for (int mw = 0; mw < KW4; mw++) x[bb][mw] = *reinterpret_cast<const uint32_t *>(s_tile + off + 4 * mw);
                } else {
                    const uint32_t *wp = reinterpret_cast<const uint32_t *>(s_tile + (off & ~3));
                    const int sh = 8 * (off & 3);
                    uint32_t raw[KW4 + 1];
#pragma unroll
                    for (int mw = 0; mw <= KW4; mw++) raw[mw] = wp[mw]; // stays inside the (padded) tile
#pragma unroll
                    for (int mw = 0; mw < KW4; mw++) x[bb][mw] = __funnelshift_r(raw[mw], raw[mw + 1], sh);
                    x[bb][KW4 - 1] &= 0xFFFFFFFFu >> (8 * (4 - S % 4));
                }
            }
            int y[BB][S];
#pragma unroll
            for (int kp = 0; kp < S; kp++) {
                const uint4 c4 = reinterpret_cast<const uint4 *>(s_cp)[kp];
                const uint32_t cw4[4] = {c4.x, c4.y, c4.z, c4.w};
#pragma unroll
                for (int bb = 0; bb < BB; bb++) {
                    int acc = 0;
#pragma unroll
                    for (int mw = 0; mw < KW4; mw++) acc = __dp4a((int)x[bb][mw], (int)cw4[mw], acc);
                    y[bb][kp] = acc;
                    mx = max(mx, abs(acc));
                }
            }
#pragma unroll
            for (int bb = 0; bb < BB; bb++) {
                int words[F::NSPLIT * VEC];
#pragma unroll
                for (int q = 0; q < F::NSPLIT * VEC; q++) words[q] = 0;
#pragma unroll
                for (int cw = 0; cw < W; cw++) {
                    int word = 0;
#pragma unroll
                    for (int l = LPW - 1; l >= 0; l--)
                        if (cw * LPW + l < S) word = word * (1 << LB) + y[bb][cw * LPW + l];
                    words[(cw / CB) * VEC + cw % CB] = word;
                }
#pragma unroll
                for (int q = 0; q < F::NSPLIT; q++) st_vec<VEC>(s_y + (a0 + bb) * YROW + bfix * WP + q * VEC, words + q * VEC);
            }
        }
        atomicMax(&s_st[0], mx);
    }
    __syncthreads();
    // packed passes are exact iff max|Y| * ||A|| <= LMAX and max|Y| * ||A|| * ||B|| <= LMAX
    bool fast = false;
    if (live) {
        const long long za = (long long)s_st[0] * s_st[1];
        fast = za <= F::LMAX && za * s_st[2] <= F::LMAX;
    }
    // ---------------- pass A: Z[i][b][.] = sum_a A[i][a] Y[a][b][.], thread (b = rr, h) works on its CB columns of
    // every row, in place
    if (fast) {
        int y[S][VEC];
#pragma unroll
        for (int a = 0; a < S; a++) ld_vec<VEC>(s_y + a * YROW + rr * WP + h * VEC, y[a]);
#pragma unroll
        for (int i = 0; i < S; i++) {
            int mrow[RW];
#pragma unroll
            for (int q = 0; q < RW / 4; q++) ld_vec<4>(s_ma + i * RW + 4 * q, mrow + 4 * q);
            int acc[VEC];
#pragma unroll
            for (int c = 0; c < VEC; c++) acc[c] = 0;
#pragma unroll
            for (int a = 0; a < S; a++)
#pragma unroll
                for (int c = 0; c < CB; c++) acc[c] += mrow[a] * y[a][c];
            st_vec<VEC>(s_y + i * YROW + rr * WP + h * VEC, acc);
        }
    }
    __syncthreads();
    // ---------------- pass B: T'[i][j][.] = sum_b B[j][b] Z[i][b][.], thread (i = rr, h); range test on the packed
    // words, low bytes of the lanes into the tile
    if (fast) {
        int z[S][VEC];
#pragma unroll
        for (int b = 0; b < S; b++) ld_vec<VEC>(s_y + rr * YROW + b * WP + h * VEC, z[b]);
        constexpr uint32_t HALF = 1u << (LB - 1);
        constexpr uint32_t ONE = LPW == 3 ? (1u | (1u << LB) | (1u << (2 * LB))) : (1u | (1u << LB));
        constexpr uint32_t LMASK = (1u << LB) - 1u;
        uint32_t over = 0;
#pragma unroll
        for (int j = 0; j < S; j++) {
            int mrow[RW];
#pragma unroll
            for (int q = 0; q < RW / 4; q++) ld_vec<4>(s_mb + j * RW + 4 * q, mrow + 4 * q);
            uint32_t u[CB];
#pragma unroll
            for (int c = 0; c < CB; c++) {
                int acc = 0;
#pragma unroll
                for (int b = 0; b < S; b++) acc += mrow[b] * z[b][c];
                u[c] = (uint32_t)acc + HALF * ONE; // lanes biased to [0, 2^LB)
                // every lane in [HALF-64, HALF+63]  <=>  (lane - (HALF-64)) < 128 in every lane
                over |= (u[c] - (HALF - 64u) * ONE) & ((LMASK & ~127u) * ONE);
            }
            if constexpr (OUT16) {
                // int16 out: the lanes ARE the results (exact under the guard, |entry| <= LMAX <= 32767)
                int16_t *d16 = reinterpret_cast<int16_t *>(s_tile) + rr * OROW + j * S + h * CB * LPW;
#pragma unroll
                for (int c = 0; c < CB; c++)
#pragma unroll
                    for (int l = 0; l < LPW; l++)
                        if (h * CB * LPW + c * LPW + l < S) d16[c * LPW + l] = (int16_t)((int)((u[c] >> (LB * l)) & LMASK) - (int)HALF);
                continue;
            }
            uint8_t *dst = s_tile + rr * OROW + j * S + h * CB * LPW;
            if constexpr (S == 9) {
#pragma unroll
                for (int c = 0; c < CB; c++)
#pragma unroll
                    for (int l = 0; l < LPW; l++) dst[c * LPW + l] = (uint8_t)(u[c] >> (LB * l)); // HALF = 0 mod 256
            } else {
                // 16-bit lanes: bytes 0 and 2 of each word are the int8 entries
#pragma unroll
                for (int c = 0; c < CB; c += 2)
                    *reinterpret_cast<uint32_t *>(dst + 2 * c) = __byte_perm(u[c], u[c + 1], 0x6420);
            }
        }
        if (over && !OUT16) s_st[3] = TG_FLAG_RANGE;
        if constexpr (OUT16 && (G::RP != S2 || G::GP != S * G::RP)) {
            // the int16 tile does not inherit zero padding from the input game: row and game padding written here
            int16_t *t16 = reinterpret_cast<int16_t *>(s_tile);
            if (h == 0) {
#pragma unroll
                for (int x = S2; x < G::RP; x++) t16[rr * OROW + x] = 0;
                if (rr == 0)
                    for (int x = S * G::RP; x < G::GP; x++) t16[x] = 0;
            }
        }
    }
    fence_proxy_async();
    __syncthreads();
    constexpr int EB = F::EB;
    if constexpr (OROW == G::RP) {
        if (live && t == 0 && fast) {
            bulk_s2g(slab_out + (g0 + gl) * G::GP * EB, s_tile, (uint32_t)(G::GP * EB));
            bulk_commit();
            bulk_wait<0>();
        }
    } else { // padded output tile: one bulk store per row
        if (live && t < S && fast) {
            bulk_s2g(slab_out + ((g0 + gl) * G::GP + t * G::RP) * EB, s_tile + t * OROW * EB, (uint32_t)(G::RP * EB));
            bulk_commit();
            bulk_wait<0>();
        }
    }
    if (live && t == 0) flags[g0 + gl] = fast ? (uint8_t)s_st[3] : BASIS_REDO;
}

// unsigned bytes of a  x  signed bytes of b, accumulated
__device__ __forceinline__ int dp4a_us(uint32_t a, uint32_t b, int c) {
    int d;
    asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

// factors follow the change of basis: coef' = M coef for the three factors of every action; token' = coef' + shift_out.
// Thread (game n, row i) keeps row i of A, B and C as packed bytes in registers for all R actions of the game; per
// action it reads the token record once (128-bit loads), takes each factor's S tokens with static funnel shifts and
// needs ceil(S/4) DP4A (unsigned tokens x signed matrix row; the input shift is folded in through the row sum).
template <int S>
__global__ void __launch_bounds__(256)
    basis_factors_kernel(const uint8_t *__restrict__ tape_in, long long in_step_stride, int shift_in,
                         const int8_t *__restrict__ mats, long long mat_stride, uint8_t *__restrict__ tape_out,
                         long long out_step_stride, int shift_out, uint8_t *__restrict__ flags, long long N, int R) {
    using G = Geo<S>;
    constexpr int GPB = 256 / S, KW4 = (S + 3) / 4, NWT = G::TP / 4;
    constexpr uint32_t WLAST = (S % 4) ? (0xFFFFFFFFu >> (8 * (4 - S % 4))) : 0xFFFFFFFFu;
    const int gl = threadIdx.x / S, i = threadIdx.x % S;
    if (gl >= GPB) return;
    for (long long n = (long long)blockIdx.x * GPB + gl; n < N; n += (long long)gridDim.x * GPB) {
        uint32_t mrow[3][KW4];
        int rowsum[3];
#pragma unroll
        for (int f = 0; f < 3; f++) {
            const int8_t *M = mats + n * mat_stride + f * S * S + i * S;
            rowsum[f] = 0;
#pragma unroll
            for (int m = 0; m < KW4; m++) mrow[f][m] = 0;
#pragma unroll
            for (int a = 0; a < S; a++) {
                const int v = (int)M[a];
                rowsum[f] += v;
                mrow[f][a >> 2] |= ((uint32_t)v & 0xFFu) << (8 * (a & 3));
            }
        }
        bool bad = false;
        // the record of action r+1 is in flight while action r is transformed
        uint4 nxt[NWT / 4];
        {
            const uint4 *src0 = reinterpret_cast<const uint4 *>(tape_in + n * G::TP);
#pragma unroll
            for (int q = 0; q < NWT / 4; q++) nxt[q] = src0[q];
        }
        for (int r = 0; r < R; r++) {
            uint32_t w[NWT + 1];
#pragma unroll
            for (int q = 0; q < NWT / 4; q++)
                w[4 * q] = nxt[q].x, w[4 * q + 1] = nxt[q].y, w[4 * q + 2] = nxt[q].z, w[4 * q + 3] = nxt[q].w;
            w[NWT] = 0;
            if (r + 1 < R) {
                const uint4 *src = reinterpret_cast<const uint4 *>(tape_in + (size_t)(r + 1) * in_step_stride + n * G::TP);
#pragma unroll
                for (int q = 0; q < NWT / 4; q++) nxt[q] = src[q];
            }
            uint8_t *dst = tape_out + (size_t)r * out_step_stride + n * G::TP;
#pragma unroll
            for (int f = 0; f < 3; f++) {
                constexpr int dummy = 0;
                (void)dummy;
                const int o = f * S; // byte offset of the factor's tokens in the record (compile time after unrolling)
                int acc = -shift_in * rowsum[f];
#pragma unroll
                for (int m = 0; m < KW4; m++) {
                    uint32_t tw = w[(o >> 2) + m];
                    if ((o & 3) != 0) tw = __funnelshift_r(tw, w[(o >> 2) + m + 1], 8 * (o & 3));
                    if (m == KW4 - 1) tw &= WLAST;
                    acc = dp4a_us(tw, mrow[f][m], acc);
                }
                bad |= (acc < -shift_out) | (acc > shift_out);
                dst[o + i] = (uint8_t)(acc + shift_out);
            }
            if (3 * S + i < G::TP) dst[3 * S + i] = 0; // tape padding stays zero
        }
        if (bad) flags[n] |= (uint8_t)TG_FLAG_TOKEN_RANGE; // same bit from every writer
    }
}

// S = 16: a factor's 16 tokens are one aligned 16-byte block, so a thread can own FOUR consecutive rows of one
// factor's matrix (16 registers), read just that block per action and store its four output tokens as one word.
__global__ void __launch_bounds__(252)
    basis_factors16_kernel(const uint8_t *__restrict__ tape_in, long long in_step_stride, int shift_in,
                           const int8_t *__restrict__ mats, long long mat_stride, uint8_t *__restrict__ tape_out,
                           long long out_step_stride, int shift_out, uint8_t *__restrict__ flags, long long N, int R) {
    constexpr int S = 16, TPG = 12, GPB = 252 / TPG, TP = 48;
    const int gl = threadIdx.x / TPG, t = threadIdx.x % TPG;
    const int f = t >> 2, i0 = 4 * (t & 3); // factor, first of the four rows
    for (long long n = (long long)blockIdx.x * GPB + gl; n < N; n += (long long)gridDim.x * GPB) {
        uint32_t mrow[4][4];
        int rowsum[4];
        const int8_t *M = mats + n * mat_stride + f * S * S + i0 * S; // four consecutive rows = 64 contiguous bytes
        if ((((uintptr_t)mats | (uintptr_t)mat_stride) & 15) == 0) {
#pragma unroll
            for (int ii = 0; ii < 4; ii++) {
                const uint4 v4 = reinterpret_cast<const uint4 *>(M)[ii];
                mrow[ii][0] = v4.x, mrow[ii][1] = v4.y, mrow[ii][2] = v4.z, mrow[ii][3] = v4.w;
            }
        } else {
#pragma unroll
            for (int ii = 0; ii < 4; ii++)
#pragma unroll
                for (int m = 0; m < 4; m++) {
                    uint32_t word = 0;
#pragma unroll
                    for (int b = 0; b < 4; b++) word |= ((uint32_t)(uint8_t)M[ii * S + 4 * m + b]) << (8 * b);
                    mrow[ii][m] = word;
                }
        }
#pragma unroll
        for (int ii = 0; ii < 4; ii++) {
            int rs = 0;
#pragma unroll
            for (int m = 0; m < 4; m++) rs = __dp4a((int)mrow[ii][m], 0x01010101, rs);
            rowsum[ii] = rs;
        }
        bool bad = false;
        // the steps of a game are N*TP bytes apart (step-major tape): every load is a fresh DRAM page, so the loop keeps
        // PF of them in flight per thread (bytes in flight, not instructions, bound this kernel)
        constexpr int PF = 4;
        const uint8_t *src = tape_in + n * TP + 16 * f;
        uint4 ring[PF];
#pragma unroll
        for (int q = 0; q < PF; q++)
            ring[q] = q < R ? *reinterpret_cast<const uint4 *>(src + (size_t)q * in_step_stride) : make_uint4(0, 0, 0, 0);
        for (int r0 = 0; r0 < R; r0 += PF) {
#pragma unroll
            for (int q = 0; q < PF; q++) {
                const int r = r0 + q;
                if (r < R) {
                    const uint4 cur = ring[q];
                    if (r + PF < R) ring[q] = *reinterpret_cast<const uint4 *>(src + (size_t)(r + PF) * in_step_stride);
                    uint32_t outw = 0;
#pragma unroll
                    for (int ii = 0; ii < 4; ii++) {
                        int acc = -shift_in * rowsum[ii];
                        acc = dp4a_us(cur.x, mrow[ii][0], acc);
                        acc = dp4a_us(cur.y, mrow[ii][1], acc);
                        acc = dp4a_us(cur.z, mrow[ii][2], acc);
                        acc = dp4a_us(cur.w, mrow[ii][3], acc);
                        bad |= (acc < -shift_out) | (acc > shift_out);
                        outw |= ((uint32_t)(acc + shift_out) & 0xFFu) << (8 * ii);
                    }
                    *reinterpret_cast<uint32_t *>(tape_out + (size_t)r * out_step_stride + n * TP + 16 * f + i0) = outw;
                }
            }
        }
        if (bad) flags[n] |= (uint8_t)TG_FLAG_TOKEN_RANGE; // same bit from every writer
    }
}

// one thread per (game, matrix): M = L * U, L unit-lower, U upper with diagonal +-1, off-diagonal entries
// -1/0/+1 with probabilities (p_nz/2, 1-p_nz, p_nz/2).  Draw for entry (r,c): byte (r*S+c)%16 of Philox block
// (r*S+c)/16 with ctr = (block, matrix f, 0x6D617473, d_lo), key as in the unimodular contract of the oracle.
// Everything stays in registers as packed bytes: the draws of a row become its L and U rows with SWAR compares, and
// row r of M is sum_{k<=r} L[r][k] * (row k of U) -- one IMAD per four entries (entries of M are at most S in size).
template <int S>
__global__ void __launch_bounds__(64)
    unimodular_kernel(unsigned long long seed, unsigned long long first, long long N, uint32_t thr_nz, int8_t *__restrict__ mats) {
    constexpr int NB = (S * S + 15) / 16, KW4 = (S + 3) / 4;
    // S not a multiple of 4: the S*S-byte matrices of the block's 64 threads are assembled in shared memory and leave
    // as coalesced words (64 * S * S is a multiple of 4)
    __shared__ __align__(16) uint8_t s_out[(S % 4) ? 64 * S * S : 16];
    const long long t0 = blockIdx.x * (long long)blockDim.x;
    const long long t = t0 + threadIdx.x;
    const bool live = t < N * 3;
    const long long n = live ? t / 3 : 0;
    const int f = (int)(t % 3);
    const unsigned long long d = first + (unsigned long long)n;
    const uint32_t k0 = (uint32_t)seed ^ ((uint32_t)(d >> 32) * 0x9E3779B9u), k1 = (uint32_t)(seed >> 32);
    uint32_t dw[4 * NB + 1];
#pragma unroll
    for (int b = 0; b < NB; b++) philox_block((uint32_t)b, (uint32_t)f, 0x6D617473u, (uint32_t)d, k0, k1, &dw[4 * b]);
    dw[4 * NB] = 0;
    const uint32_t cthr = (0x80u - (thr_nz > 0x80u ? 0x80u : thr_nz)) * ONES4; // (draw & 0x7F) + cthr sets bit 7 iff >= thr
    int32_t urow[S][KW4]; // rows of U in integer form (sum_b x_b 256^b)
    int8_t *out = (S % 4) ? reinterpret_cast<int8_t *>(s_out) + threadIdx.x * S * S : mats + (n * 3 + f) * S * S;
    if ((S % 4) == 0 && !live) return;
#pragma unroll
    for (int r = 0; r < S; r++) {
        uint32_t lrow[KW4];
        int32_t acc[KW4];
#pragma unroll
        for (int m = 0; m < KW4; m++) {
            // the draw bytes of entries (r, 4m .. 4m+3)
            const int o = r * S + 4 * m;
            uint32_t x = dw[o >> 2];
            if ((o & 3) != 0) x = __funnelshift_r(x, dw[(o >> 2) + 1], 8 * (o & 3));
            uint32_t colmask = 0, lowmask = 0, highmask = 0, diag = 0;
#pragma unroll
            for (int b = 0; b < 4; b++) {
                const int c = 4 * m + b;
                if (c < S) colmask |= 0xFFu << (8 * b);
                if (c < r) lowmask |= 0xFFu << (8 * b);
                if (c > r && c < S) highmask |= 0xFFu << (8 * b);
                if (c == r) diag |= 0xFFu << (8 * b);
            }
            const uint32_t notmag = ((x & 0x7F7F7F7Fu) + cthr) & H4;      // bit 7 set where the magnitude is 0
            const uint32_t magmask = (((notmag ^ H4) >> 7) * 0xFFu) & colmask;
            const uint32_t negmask = ((x & H4) >> 7) * 0xFFu;
            const uint32_t sgn1 = negmask | ONES4;                        // -1 or +1 in every byte
            const uint32_t val = magmask & sgn1;
            lrow[m] = (val & lowmask) | (ONES4 & diag);
            const uint32_t ub = (val & highmask) | (sgn1 & diag);
            urow[r][m] = (int32_t)((ub ^ H4) - H4);
            acc[m] = 0;
        }
#pragma unroll
        for (int k = 0; k <= r; k++) {
            const uint32_t w = lrow[k >> 2];
            const int l = (int)(int8_t)((w >> (8 * (k & 3))) & 0xFFu);
#pragma unroll
            for (int m = 0; m < KW4; m++) acc[m] += l * urow[k][m];
        }
        uint32_t words[KW4];
#pragma unroll
        for (int m = 0; m < KW4; m++) words[m] = ((uint32_t)acc[m] + H4) ^ H4;
        if constexpr (S % 4 == 0) {
#pragma unroll
            for (int m = 0; m < KW4; m++) reinterpret_cast<uint32_t *>(out + r * S)[m] = words[m];
        } else {
#pragma unroll
            for (int c = 0; c < S; c++) out[r * S + c] = (int8_t)(words[c >> 2] >> (8 * (c & 3)));
        }
    }
    if constexpr ((S % 4) != 0) {
        __syncthreads();
        const long long nlive = min((long long)blockDim.x, N * 3 - t0); // matrices of this block
        const long long bytes = nlive * S * S;
        int8_t *dst = mats + t0 * S * S;
        if ((((uintptr_t)dst) & 3) == 0) {
            for (long long w = threadIdx.x; w < bytes / 4; w += blockDim.x)
                reinterpret_cast<uint32_t *>(dst)[w] = reinterpret_cast<const uint32_t *>(s_out)[w];
            for (long long b = (bytes & ~3LL) + threadIdx.x; b < bytes; b += blockDim.x) dst[b] = (int8_t)s_out[b];
        } else {
            for (long long b = threadIdx.x; b < bytes; b += blockDim.x) dst[b] = (int8_t)s_out[b];
        }
    }
}

// ------------------------------------------------------------------ 4x4x4: one THREAD per game
// A 4x4x4 game is 64 bytes and its three matrices 48: the whole change of basis fits the registers of one thread, in int32
// ring arithmetic (the stored low bytes are those of the true T' for any int8 input): contract c with DP4A on the
// packed input words (Y[a][b][k'] = dp4a(T[a][b][.], C[k'][.])), then b and a with scalar matrix entries -- 64 DP4A + 512
// IMAD per game, no CTA barrier (the packed-lane kernel above needs three CTA barriers per 64 games and spends its time
// in them: 5.9 G games/s, 0.21 of HBM).  The 32 results of a warp are one contiguous block of the output slab: they go
// through a warp-private stage in shared memory (thread-major in, linear out) so that every store instruction writes 512
// contiguous bytes instead of 16-byte pieces of 32 different lines.
// |T'| <= 128 * nA * nB * nC (n = largest absolute row sum of a matrix).  Where that bound passes 2^31 - 1 an int32 result
// may have wrapped into the range it is tested against, so such a game's range test is redone here in 64 bit, one entry
// at a time from global memory (matrices whose row sums multiply to more than 2^24: never those of a game).
template <bool OUT16>
__device__ __noinline__ bool basis4_out_of_range_wide(const int8_t *__restrict__ game, const int8_t *__restrict__ m) {
    const long long lo = OUT16 ? -32768 : -64, hi = OUT16 ? 32767 : 63;
    bool bad = false;
#pragma unroll 1
    for (int e = 0; e < 64; e++) {
        const int i = e >> 4, j = (e >> 2) & 3, k = e & 3;
        long long v = 0;
#pragma unroll 1
        for (int abc = 0; abc < 64; abc++) {
            const int a = abc >> 4, b = (abc >> 2) & 3, c = abc & 3;
            v += (long long)(m[4 * i + a] * m[16 + 4 * j + b]) * (m[32 + 4 * k + c] * game[abc]);
        }
        bad |= v < lo || v > hi;
    }
    return bad;
}

template <bool OUT16>
__global__ void __launch_bounds__(128)
    basis4_thread_kernel(const int8_t *__restrict__ slab_in, const int8_t *__restrict__ mats, long long mat_stride,
                         void *__restrict__ slab_out, uint8_t *__restrict__ flags, long long N) {
    constexpr int IPG = OUT16 ? 8 : 4, PITCH = IPG * 16 + 16; // 16-byte items per game; stage pitch (conflict-free both ways)
    __shared__ __align__(16) uint8_t s_stage[4][32 * PITCH];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long nw0 = (long long)blockIdx.x * blockDim.x + warp * 32; // first game of the warp
    if (nw0 >= N) return;
    const long long n = min(nw0 + lane, N - 1); // spare lanes of the last warp repeat the last game
    const uint4 *mp = reinterpret_cast<const uint4 *>(mats + n * mat_stride);
    const uint4 mA = __ldg(mp), mB = __ldg(mp + 1), mC = __ldg(mp + 2); // row r of a matrix = word r
    const uint32_t rA[4] = {mA.x, mA.y, mA.z, mA.w}, rB[4] = {mB.x, mB.y, mB.z, mB.w}, rC[4] = {mC.x, mC.y, mC.z, mC.w};
    int cB[4][4]; // B[j][b]
#pragma unroll
    for (int j = 0; j < 4; j++)
#pragma unroll
        for (int b = 0; b < 4; b++) cB[j][b] = (int)(int8_t)(rB[j] >> (8 * b));
    int acc[4][16]; // T'[i][4 j + k]
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int e = 0; e < 16; e++) acc[i][e] = 0;
    const uint4 *tp = reinterpret_cast<const uint4 *>(slab_in + n * 64);
#pragma unroll
    for (int a = 0; a < 4; a++) {
        const uint4 t4 = __ldg(tp + a); // T[a][b][.] = word b
        const uint32_t tw[4] = {t4.x, t4.y, t4.z, t4.w};
        int z[16]; // Z[a][j][k] = sum_b B[j][b] Y[a][b][k]
#pragma unroll
        for (int e = 0; e < 16; e++) z[e] = 0;
#pragma unroll
        for (int b = 0; b < 4; b++) {
            int y[4];
#pragma unroll
            for (int k = 0; k < 4; k++) y[k] = __dp4a((int)tw[b], (int)rC[k], 0);
#pragma unroll
            for (int j = 0; j < 4; j++)
#pragma unroll
                for (int k = 0; k < 4; k++) z[4 * j + k] += cB[j][b] * y[k];
        }
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int aia = (int)(int8_t)(rA[i] >> (8 * a));
#pragma unroll
            for (int e = 0; e < 16; e++) acc[i][e] += aia * z[e];
        }
    }
    uint32_t bad = 0;
    if constexpr (OUT16) {
        uint4 *dst = reinterpret_cast<uint4 *>(s_stage[warp] + lane * PITCH);
#pragma unroll
        for (int i = 0; i < 4; i++) {
            uint32_t w[8];
#pragma unroll
            for (int p = 0; p < 8; p++) {
                const int lo = acc[i][2 * p], hi = acc[i][2 * p + 1];
                bad |= (uint32_t)(lo + 32768) | (uint32_t)(hi + 32768); // fits int16 <=> the biased value is below 2^16
                w[p] = ((uint32_t)lo & 0xFFFFu) | ((uint32_t)hi << 16);
            }
            dst[2 * i] = make_uint4(w[0], w[1], w[2], w[3]);
            dst[2 * i + 1] = make_uint4(w[4], w[5], w[6], w[7]);
        }
        bad >>= 16;
    } else {
        uint4 *dst = reinterpret_cast<uint4 *>(s_stage[warp] + lane * PITCH);
#pragma unroll
        for (int i = 0; i < 4; i++) {
            uint32_t w[4];
#pragma unroll
            for (int p = 0; p < 4; p++) {
                uint32_t word = 0;
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    const int v = acc[i][4 * p + q];
                    bad |= (uint32_t)(v + 64); // in [-64, 63] <=> the biased value is below 2^7
                    word |= ((uint32_t)v & 0xFFu) << (8 * q);
                }
                w[p] = word;
            }
            dst[i] = make_uint4(w[0], w[1], w[2], w[3]);
        }
        bad >>= 7;
    }
    if (flags && nw0 + lane < N) {
        uint32_t na = 0, nb = 0, nc = 0; // largest absolute row sums (|-128| counts 128: unsigned bytes of __vabs4)
#pragma unroll
        for (int r = 0; r < 4; r++) {
            na = max(na, __dp4a(__vabs4(rA[r]), 0x01010101u, 0u));
            nb = max(nb, __dp4a(__vabs4(rB[r]), 0x01010101u, 0u));
            nc = max(nc, __dp4a(__vabs4(rC[r]), 0x01010101u, 0u));
        }
        if (128ull * na * nb * nc > 0x7FFFFFFFull && basis4_out_of_range_wide<OUT16>(slab_in + n * 64, mats + n * mat_stride)) bad = 1;
        flags[n] = bad ? (uint8_t)TG_FLAG_RANGE : (uint8_t)0;
    }
    __syncwarp();
    const int total = (int)min(32LL, N - nw0) * IPG;
    uint4 *out = reinterpret_cast<uint4 *>(reinterpret_cast<uint8_t *>(slab_out) + nw0 * (IPG * 16));
    for (int x = lane; x < total; x += 32) out[x] = *reinterpret_cast<const uint4 *>(s_stage[warp] + (x / IPG) * PITCH + (x % IPG) * 16);
}

} // namespace tg

// int8 slab in; int8 slab out (out16 == 0) or int16 slab out
static int change_of_basis_impl(const int8_t *slab_in, const int8_t *mats, int per_game, void *slab_out, int out16, uint8_t *flags,
                                int64_t N, int S, void *stream) {
    if (!tg::basis_supported_S(S) || N < 0) return TG_E_ARG;
    if (N == 0) return TG_OK;
    if (!slab_in || !mats || !slab_out || (const void *)slab_in == (const void *)slab_out) return TG_E_ARG;
    if (((uintptr_t)slab_in | (uintptr_t)slab_out) & 15) return TG_E_ARG;
    if (N > 0x7FFFFFFFLL) return TG_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const long long ms = per_game ? 3LL * S * S : 0;
    // a fast kernel first (tensor cores for 9x9x9 and 16x16x16, packed integer lanes for 4x4x4); it marks the games whose
    // intermediates its arithmetic cannot hold exactly and the exact int32 kernel redoes exactly those (TG_FLAG_PATH_EXACT).
    // Without a flags array there is nowhere to leave the mark: exact kernel for all.
    const int exact_grid = (int)(N < 148 * 32 ? N : 148 * 32);
#define TG_BASIS_EXACT(SS, O16)                                                                                            \
    tg::basis_kernel<SS, O16><<<flags ? exact_grid : (int)N, tg::BasisCfg<SS>::NT, tg::BasisCfg<SS>::SMEM_BYTES, st>>>(    \
        slab_in, mats, ms, slab_out, flags, N, flags ? 1 : 0);
#define TG_BASIS_FAST(SS, O16)                                                                                             \
    {                                                                                                                      \
        using F = tg::BasisFast<SS, O16>;                                                                                  \
        auto fast = tg::basis_fast_kernel<SS, O16>;                                                                        \
        TG_CUDA(cudaFuncSetAttribute(fast, cudaFuncAttributeMaxDynamicSharedMemorySize, F::SMEM_BYTES));                   \
        fast<<<(unsigned)((N + F::GPC - 1) / F::GPC), F::NT, F::SMEM_BYTES, st>>>(slab_in, mats, ms, slab_out, flags, N);  \
    }
#ifdef TG_TUNING
    static const int variant = tg::tuning_env("TG_BASIS_VARIANT", 0); // 1: packed integer lanes instead of the tensor cores
#else
    constexpr int variant = 0;
#endif
    const bool mats_ok = (((uintptr_t)mats | (uintptr_t)ms) & 3) == 0;
    switch (S) {
    case 4:
        if (variant != 1 && ((((uintptr_t)mats | (uintptr_t)ms) & 15) == 0)) { // one thread per game, exact: nothing left to redo
            const unsigned grid = (unsigned)((N + 127) / 128);
            if (out16) tg::basis4_thread_kernel<true><<<grid, 128, 0, st>>>(slab_in, mats, ms, slab_out, flags, N);
            else tg::basis4_thread_kernel<false><<<grid, 128, 0, st>>>(slab_in, mats, ms, slab_out, flags, N);
            break;
        }
        if (flags) {
            if (out16) TG_BASIS_FAST(4, true) else TG_BASIS_FAST(4, false)
        }
        if (out16) { TG_BASIS_EXACT(4, true) } else { TG_BASIS_EXACT(4, false) }
        break;
    case 9:
        if (flags && variant != 1) {
            const int rc = tg::launch_basis_mma9(slab_in, mats, ms, slab_out, out16, flags, N, st);
            if (rc != TG_OK) return rc;
        }
#ifdef TG_TUNING
        else if (flags) { // the packed-lane kernel (3 x 10-bit lanes): A/B timing only
            if (out16) TG_BASIS_FAST(9, true) else TG_BASIS_FAST(9, false)
        }
#endif
        if (out16) { TG_BASIS_EXACT(9, true) } else { TG_BASIS_EXACT(9, false) }
        break;
    case 16:
        if (flags && variant != 1 && mats_ok) {
            const int rc = tg::launch_basis_mma16(slab_in, mats, ms, slab_out, out16, flags, N, st);
            if (rc != TG_OK) return rc;
        } else if (flags) {
#ifdef TG_TUNING
            if (out16) TG_BASIS_FAST(16, true) else TG_BASIS_FAST(16, false)
#else
            cudaMemsetAsync(flags, tg::BASIS_REDO, (size_t)N, st); // unaligned matrices: every game through the exact kernel
#endif
        }
        if (out16) { TG_BASIS_EXACT(16, true) } else { TG_BASIS_EXACT(16, false) }
        break;
    }
#undef TG_BASIS_EXACT
#undef TG_BASIS_FAST
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

extern "C" {

int tg_change_of_basis(const int8_t *slab_in, const int8_t *mats, int per_game, int8_t *slab_out, uint8_t *flags, int64_t N,
                       int S, void *stream) {
    return change_of_basis_impl(slab_in, mats, per_game, slab_out, 0, flags, N, S, stream);
}

int tg_change_of_basis_i16(const int8_t *slab_in, const int8_t *mats, int per_game, int16_t *slab16_out, uint8_t *flags, int64_t N,
                           int S, void *stream) {
    return change_of_basis_impl(slab_in, mats, per_game, slab16_out, 1, flags, N, S, stream);
}

int tg_change_of_basis_factors(const uint8_t *tape_in, int64_t in_step_stride, int shift_in, const int8_t *mats, int per_game,
                               uint8_t *tape_out, int64_t out_step_stride, int shift_out, uint8_t *flags, int64_t N, int R,
                               int S, void *stream) {
    if (!tg::basis_supported_S(S) || N < 0 || R < 1 || shift_in < 0 || shift_out < 1 || shift_out > 127) return TG_E_ARG;
    if (N == 0) return TG_OK;
    if (!tape_in || !mats || !tape_out || !flags) return TG_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const long long ms = per_game ? 3LL * S * S : 0;
    const long long blocks = (N + (256 / S) - 1) / (256 / S);
    const int grid = (int)(blocks < 148 * 16 ? blocks : 148 * 16);
    if (((uintptr_t)tape_in | (uintptr_t)in_step_stride) & 15) return TG_E_ARG;
    switch (S) {
    case 4: tg::basis_factors_kernel<4><<<grid, 256, 0, st>>>(tape_in, in_step_stride, shift_in, mats, ms, tape_out, out_step_stride, shift_out, flags, N, R); break;
    case 9: tg::basis_factors_kernel<9><<<grid, 256, 0, st>>>(tape_in, in_step_stride, shift_in, mats, ms, tape_out, out_step_stride, shift_out, flags, N, R); break;
    case 16: {
        const long long b16 = (N + 20) / 21;
        if ((((uintptr_t)tape_out | (uintptr_t)out_step_stride) & 3) == 0)
            tg::basis_factors16_kernel<<<(int)(b16 < 148 * 16 ? b16 : 148 * 16), 252, 0, st>>>(tape_in, in_step_stride, shift_in, mats, ms, tape_out, out_step_stride, shift_out, flags, N, R);
        else
            tg::basis_factors_kernel<16><<<grid, 256, 0, st>>>(tape_in, in_step_stride, shift_in, mats, ms, tape_out, out_step_stride, shift_out, flags, N, R);
    } break;
    }
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

int tg_sample_unimodular(uint64_t seed, uint64_t first, int64_t N, int S, double p_nonzero, int8_t *mats, void *stream) {
    if (!tg::basis_supported_S(S) || N < 0 || !(p_nonzero >= 0.0) || p_nonzero > 1.0) return TG_E_ARG;
    if (N == 0) return TG_OK;
    if (!mats) return TG_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const uint32_t thr = (uint32_t)(p_nonzero * 128.0);
    const int grid = (int)((N * 3 + 63) / 64);
    switch (S) {
    case 4: tg::unimodular_kernel<4><<<grid, 64, 0, st>>>(seed, first, N, thr, mats); break;
    case 9: tg::unimodular_kernel<9><<<grid, 64, 0, st>>>(seed, first, N, thr, mats); break;
    case 16: tg::unimodular_kernel<16><<<grid, 64, 0, st>>>(seed, first, N, thr, mats); break;
    }
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

} // extern "C"
