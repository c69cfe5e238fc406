// tg_basis_mma9.cu -- K5n: change of basis of 9x9x9 games on the tensor cores
// (called by tg_change_of_basis / tg_change_of_basis_i16 for S = 9; same contract as tg_basis.cu).
//
// ABSENT from the reference; spec as in tg_basis.cu:
//     T'[i][j][k] = sum_abc A[i][a] B[j][b] C[k][c] T[a][b][c]
//
// One WARP per game, three passes of mma.sync m16n8k16 (f16 operands, f32 accumulation), the 9x9 matrix always the A
// operand (zero-padded to 16x16), the tensor the B operand.  Everything is exact integer arithmetic: an f16 holds every
// integer up to 2048 and the f32 sums stay far below 2^24; the operands of passes 2 and 3 (Y and Z) are bounded a priori
// (max |T| times the largest absolute row sums of C and B, all three computed on the way in); only when that bound
// exceeds 2047 are Y and Z CHECKED as they are produced, and a game that then fails is left to the exact int32 kernel
// (BASIS_REDO) -- with SURVEY 8(d)'s matrices (off-diagonal density 0.3) max |Z| is ~170, so that practically never happens.
//   -. the 27 matrix rows become rows of halves (same conversion as 0.) in the not-yet-used Z bytes; one ldmatrix.x4 per
//      matrix yields its A fragment;
//   0. the int8 game becomes rows of halves in shared memory: row n' = 9a + b holds T[a][b][0..8] (byte -> half with one
//      PRMT per two entries: 0x6400 | (byte ^ 0x80) is the half 1024 + 128 + value, one HSUB2 removes the offset);
//   1. Y[k'][a][b] = sum_c C[k'][c] T[a][b][c]: per a one ldmatrix.x4 (rows b = 0..7 and b = 8 + seven zero rows) and
//      two MMAs (N tiles b = 0..7 and b = 8..15);
//   2. Z[j'][a][k'] = sum_b B[j'][b] Y[k'][a][b]: the accumulators of the two pass-1 MMAs ARE the B fragment of pass 2
//      (column <-> k', K slots <-> b), one cvt.rn.f16x2.f32 per two values; two MMAs per a (k' = 0..7 and k' = 8);
//   3. T'[i'][j'][k'] = sum_a A[i'][a] Z[j'][a][k']: the one transposition, through shared memory: Z is stored as halves
//      [a][n = 9 j' + k'] and read back with ldmatrix.x4.trans, eleven MMAs over the 81 (j', k') columns -- whose
//      accumulators land exactly in slab order (row i', entries n, n + 1), so the result leaves as aligned pairs into a
//      staging tile and from there with one TMA bulk store (768 bytes int8, 1536 bytes int16).
#include <cuda_fp16.h>

#include <type_traits>

#include "tg_common.cuh"

namespace tg {

namespace {

constexpr int WARPS = 4;             // games per CTA
constexpr int TS_PITCH = 48;         // bytes per row of halves (16 halves + pad: conflict-free ldmatrix rows)
constexpr int TS_BYTES = 82 * TS_PITCH; // 81 rows + one all-zero row = 3936
constexpr int ZS_PITCH = 208;        // bytes per row a of Z (104 halves >= 96; 52 words: conflict-free transposed reads)
constexpr int ZS_BYTES = 10 * ZS_PITCH; // rows a = 0..8 and one all-zero row (a = 9..15 all read it) = 2080
constexpr int MROWS = 28;            // the 27 matrix rows as halves + one all-zero row, staged in the (not yet used) Z bytes
constexpr int WARP_BYTES = TS_BYTES + ZS_BYTES; // 6016
static_assert(TS_BYTES >= 1536 && WARP_BYTES % 16 == 0, "the output stage overlays the T rows");
static_assert(MROWS * TS_PITCH <= 9 * ZS_PITCH, "the matrix rows must not reach the zero row of Z");

constexpr float MAGIC = 12582912.0f; // 1.5 * 2^23: float(MAGIC + n) has n in its low mantissa bits
constexpr uint32_t MAGIC_BITS = 0x4B400000u;

__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
}
__device__ __forceinline__ void mma_f16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// f16 accumulation (exact while every partial sum is an integer of magnitude <= 2048): the two result registers are the
// packed halves the next pass wants as its B fragment
__device__ __forceinline__ void mma_f16_h(uint32_t (&d)[2], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f16.f16.f16.f16 {%0,%1}, {%2,%3,%4,%5}, {%6,%7}, {%8,%8};"
                 : "=r"(d[0]), "=r"(d[1])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1), "r"(0u));
}
// D = A B + c with the same addend c in every accumulator slot (a loop-invariant register quad, no moves per tile)
__device__ __forceinline__ void mma_f16_bias(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1, const float (&c)[4]) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%11,%12,%13};"
                 : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1), "f"(c[0]), "f"(c[1]), "f"(c[2]), "f"(c[3]));
}
__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], uint32_t addr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t (&r)[4], uint32_t addr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(addr));
}
__device__ __forceinline__ uint32_t pack_f16(float lo, float hi) {
    const __half2 h = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<const uint32_t *>(&h);
}
__device__ __forceinline__ void track_abs_max(__half2 &m, uint32_t w) { m = __hmax2(m, __habs2(*reinterpret_cast<const __half2 *>(&w))); }

// nine int8 starting at byte (sh / 8) of the three words r0 r1 r2 -> ten halves (the tenth is 0) in five registers:
// 0x6400 | (byte ^ 0x80) is the half 1024 + 128 + value (one PRMT per two entries), one HSUB2 removes the offset
__device__ __forceinline__ void bytes9_to_halves(uint32_t r0, uint32_t r1, uint32_t r2, uint32_t sh, uint32_t (&h)[5]) {
    constexpr uint32_t KB = 0x00006480u; // bytes 0x80, 0x64 for PRMT: 0x64xx is the half 1024 + xx, 0x6480 the half 1152
    const __half2 ks = __halves2half2(__ushort_as_half((unsigned short)0x6480), __ushort_as_half((unsigned short)0x6480));
    const uint32_t x0 = __funnelshift_r(r0, r1, sh) ^ H4, x1 = __funnelshift_r(r1, r2, sh) ^ H4, x2 = (r2 >> sh) ^ H4;
    h[0] = prmt(x0, KB, 0x5150u), h[1] = prmt(x0, KB, 0x5352u), h[2] = prmt(x1, KB, 0x5150u), h[3] = prmt(x1, KB, 0x5352u);
    h[4] = prmt(x2, KB, 0x5450u);
#pragma unroll
    for (int e = 0; e < 5; e++) {
        const __half2 v = __hsub2(*reinterpret_cast<const __half2 *>(&h[e]), ks);
        h[e] = *reinterpret_cast<const uint32_t *>(&v);
    }
}

template <bool OUT16>
__global__ void __launch_bounds__(32 * WARPS)
    basis_mma9_kernel(const int8_t *__restrict__ slab_in, const int8_t *__restrict__ mats, long long mat_stride,
                      void *__restrict__ slab_out, uint8_t *__restrict__ flags, long long N) {
    extern __shared__ __align__(128) uint8_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    const long long n = (long long)blockIdx.x * WARPS + warp;
    if (n >= N) return;
    uint8_t *s_t = smem + (size_t)warp * WARP_BYTES; // T rows, later the output stage
    uint8_t *s_z = s_t + TS_BYTES;                    // first the matrix rows, then Z

    // ---- loads in flight first: row `lane` of the 27 matrix rows (9 bytes at any alignment: the three aligned words
    // around them) and the game's rows
    uint32_t mraw[3] = {0u, 0u, 0u}, msh = 0;
    if (lane < 27) {
        const int8_t *rp = mats + n * mat_stride + 9 * lane;
        const uint32_t o = (uint32_t)(reinterpret_cast<uintptr_t>(rp) & 3);
        const uint32_t *w = reinterpret_cast<const uint32_t *>(rp - o);
        mraw[0] = __ldg(w), mraw[1] = __ldg(w + 1);
        if (lane == 26 && (mat_stride == 0 || n == N - 1)) {
            // the last row of the last triple: its third word can reach up to 3 bytes past the triple, which may be the
            // end of the allocation; only the row's bytes of that word (0 .. o) are read
            const uint8_t *b = reinterpret_cast<const uint8_t *>(w + 2);
            mraw[2] = __ldg(b);
            for (uint32_t e = 1; e <= o; e++) mraw[2] |= (uint32_t)__ldg(b + e) << (8 * e);
        } else {
            mraw[2] = __ldg(w + 2);
        }
        msh = 8 * o;
    }
    const uint32_t *gw = reinterpret_cast<const uint32_t *>(slab_in + n * 768);
    uint32_t raw[3][3];
#pragma unroll
    for (int q = 0; q < 3; q++) {
        const int np = lane + 32 * q; // row n' = 9a + b
        if (np < 81) {
            const int off = np * 9 + 3 * (np / 9);
#pragma unroll
            for (int w = 0; w < 3; w++) raw[q][w] = __ldg(gw + (off >> 2) + w);
        } else {
            raw[q][0] = raw[q][1] = raw[q][2] = 0;
        }
    }
    // zero row of T, zero row of the matrices, zero row of Z for a = 9..15 (their A-operand columns are zero, but
    // 0 * NaN is not)
    if (lane < 3) reinterpret_cast<uint4 *>(s_t + 81 * TS_PITCH)[lane] = make_uint4(0, 0, 0, 0);
    if (lane >= 27 && lane < 30) reinterpret_cast<uint4 *>(s_z + 27 * TS_PITCH)[lane - 27] = make_uint4(0, 0, 0, 0);
    if (lane < ZS_PITCH / 16) reinterpret_cast<uint4 *>(s_z + 9 * ZS_PITCH)[lane] = make_uint4(0, 0, 0, 0);

    // ---- the matrices as rows of halves; their row sums bound Y and Z (below)
    int rowsum = 0;
    {
        uint32_t h[5];
        bytes9_to_halves(mraw[0], mraw[1], mraw[2], msh, h);
        if (lane < 27) {
            uint4 *row = reinterpret_cast<uint4 *>(s_z + lane * TS_PITCH);
            row[0] = make_uint4(h[0], h[1], h[2], h[3]);
            row[1] = make_uint4(h[4], 0, 0, 0);
            __half2 sm = __habs2(*reinterpret_cast<const __half2 *>(&h[0]));
#pragma unroll
            for (int e = 1; e < 5; e++) sm = __hadd2(sm, __habs2(*reinterpret_cast<const __half2 *>(&h[e])));
            rowsum = (int)(__low2float(sm) + __high2float(sm)); // <= 9 * 128: exact in f16
        }
    }
    // ---- 0. T[a][b][.] as rows of halves; the OR of |entry| (or |entry| - 1 for a negative one) bounds max |T|
    uint32_t tor = 0;
#pragma unroll
    for (int q = 0; q < 3; q++) {
        const int np = lane + 32 * q;
#pragma unroll
        for (int w = 0; w < 3; w++) tor |= raw[q][w] ^ prmt(raw[q][w], 0u, 0xBA98u); // sign-replicated bytes
        if (np < 81) {
            const int off = np * 9 + 3 * (np / 9);
            uint32_t h[5];
            bytes9_to_halves(raw[q][0], raw[q][1], raw[q][2], 8 * (off & 3), h);
            uint4 *row = reinterpret_cast<uint4 *>(s_t + np * TS_PITCH);
            row[0] = make_uint4(h[0], h[1], h[2], h[3]);
            row[1] = make_uint4(h[4], 0, 0, 0);
        }
    }
    // a-priori bounds: |Y| <= max|T| * max row sum of |C|, |Z| <= that * max row sum of |B|.  When both are <= 2047 (every
    // real game state: |T| is a few units) passes 1 and 2 need no run-time check of their operands.
    bool track, check3;
    {
        tor |= tor >> 16, tor |= tor >> 8;
        const int tb = (int)(__reduce_or_sync(0xFFFFFFFFu, tor) & 0xFFu) + 1;
        const int na = (int)__reduce_max_sync(0xFFFFFFFFu, lane < 9 ? rowsum : 0);
        const int nb = (int)__reduce_max_sync(0xFFFFFFFFu, (lane >= 9 && lane < 18) ? rowsum : 0);
        const int nc = (int)__reduce_max_sync(0xFFFFFFFFu, (lane >= 18 && lane < 27) ? rowsum : 0);
        track = !(tb * nc <= 2047 && tb * nc * nb <= 2047);
        // |T'| <= max row sum of |A| times the bound of Z: when that fits int16 the results need no range test either
        check3 = !OUT16 || track || tb * nc * nb * na > 32767;
    }
    __syncwarp();
    const uint32_t ts_base = smem_u32(s_t), zs_base = smem_u32(s_z);
    // ldmatrix row addresses of this lane: matrix = lane >> 3 (bit 0: rows 8..15, bit 1: halves 8..15), row = lane & 7
    const int lm_b = (lane & 7) + 8 * ((lane >> 3) & 1), lm_c = (lane >> 4) * 16;
    const bool lm_real = lm_b < 9;
    uint32_t fA[4], fB[4], fC[4]; // the m16n8k16 A fragments of the zero-padded 9x9 matrices
    ldmatrix_x4(fA, zs_base + (lm_real ? lm_b : 27) * TS_PITCH + lm_c);
    ldmatrix_x4(fB, zs_base + (lm_real ? 9 + lm_b : 27) * TS_PITCH + lm_c);
    ldmatrix_x4(fC, zs_base + (lm_real ? 18 + lm_b : 27) * TS_PITCH + lm_c);
    __syncwarp(); // the matrix rows are dead: Z takes over their bytes
    // columns n = 81..87 of Z are read by the last tile of pass 3: zero (n = 80 is written below, after the barrier)
    if (lane < 9) *reinterpret_cast<uint4 *>(s_z + lane * ZS_PITCH + 160) = make_uint4(0, 0, 0, 0);
    __syncwarp();

    // ---- 1 + 2, one a at a time
    __half2 ymax = __float2half2_rn(0.f), zmax = __float2half2_rn(0.f);
    // pass 1 reads the tensor with the other matrix order: bit 0 of the matrix index = halves 8..15, bit 1 = rows b = 8..15
    const int tl_b = (lane & 7) + 8 * (lane >> 4), tl_c = ((lane >> 3) & 1) * 16;
    const uint32_t tl_addr = ts_base + (tl_b < 9 ? tl_b : 81) * TS_PITCH + tl_c, tl_step = tl_b < 9 ? 9 * TS_PITCH : 0;
    uint16_t *zrow = reinterpret_cast<uint16_t *>(s_z);
    auto pass12 = [&](auto trk) { // two copies of the loop: predicated-off checks would still take issue slots
    constexpr bool TRACK = decltype(trk)::value;
#pragma unroll
    for (int a = 0; a < 9; a++) {
        uint32_t tb[4];
        ldmatrix_x4(tb, tl_addr + a * tl_step);
        uint32_t p0, p1, p2;
        if constexpr (TRACK) {
            float y0[4] = {0.f, 0.f, 0.f, 0.f}, y1[4] = {0.f, 0.f, 0.f, 0.f}; // rows k' = g | g+8 ; cols b = 2t, 2t+1 | 8+2t, 9+2t
            mma_f16(y0, fC, tb[0], tb[1]);
            mma_f16(y1, fC, tb[2], tb[3]);
            const uint32_t b00 = pack_f16(y0[0], y0[1]), b01 = pack_f16(y1[0], y1[1]); // k' = g
            const uint32_t b10 = pack_f16(y0[2], y0[3]), b11 = pack_f16(y1[2], y1[3]); // k' = g + 8
            track_abs_max(ymax, b00), track_abs_max(ymax, b01), track_abs_max(ymax, b10), track_abs_max(ymax, b11);
            float z0[4] = {0.f, 0.f, 0.f, 0.f}, z1[4] = {0.f, 0.f, 0.f, 0.f}; // rows j' = g | g+8 ; cols k' = 2t, 2t+1 | 8+2t, 9+2t
            mma_f16(z0, fB, b00, b01);
            mma_f16(z1, fB, b10, b11);
            p0 = pack_f16(z0[0], z0[1]), p1 = pack_f16(z0[2], z0[3]), p2 = pack_f16(z1[0], z1[2]);
            track_abs_max(zmax, p0), track_abs_max(zmax, p1), track_abs_max(zmax, p2);
        } else {
            // bounded a priori: f16 accumulators are exact, and they already are the packed operands of the next pass
            uint32_t y0[2], y1[2], z0[2], z1[2]; // [0]: row g, [1]: row g + 8; cols 2t, 2t+1 (y1 / z1: 8 + 2t, 9 + 2t)
            mma_f16_h(y0, fC, tb[0], tb[1]);
            mma_f16_h(y1, fC, tb[2], tb[3]);
            mma_f16_h(z0, fB, y0[0], y1[0]);
            mma_f16_h(z1, fB, y0[1], y1[1]);
            p0 = z0[0], p1 = z0[1], p2 = prmt(z1[0], z1[1], 0x5410u);
        }
        // Z as halves [a][n = 9 j' + k']
        uint16_t *zr = zrow + a * (ZS_PITCH / 2);
        zr[9 * g + 2 * t] = (uint16_t)p0, zr[9 * g + 2 * t + 1] = (uint16_t)(p0 >> 16); // j' = g, k' = 2t, 2t+1
        if (g == 0) *reinterpret_cast<uint32_t *>(zr + 72 + 2 * t) = p1;               // j' = 8
        if (t == 0) zr[9 * g + 8] = (uint16_t)p2;                                       // j' = g, k' = 8
        if (lane == 0) zr[80] = (uint16_t)(p2 >> 16);                                   // j' = 8, k' = 8
    }
    };
    if (track) pass12(std::true_type{}); else pass12(std::false_type{});
    if (track) {
        const float ym = fmaxf(__low2float(ymax), __high2float(ymax)), zm = fmaxf(__low2float(zmax), __high2float(zmax));
        // 2047 is the largest bound below which every integer is an f16 (a value that rounded is >= 2048 after rounding too)
        if (__any_sync(0xFFFFFFFFu, !(ym <= 2047.f && zm <= 2047.f))) {
            if (lane == 0) flags[n] = BASIS_REDO;
            return;
        }
    }
    __syncwarp(); // Z complete; the T rows are dead: their bytes become the output stage

    // ---- 3. eleven N tiles over n = 9 j' + k'; accumulator (row i', cols n, n+1) is slab entry i' * 84 + n.  The rows
    // i' = 9..15 of A and the columns n = 81..87 of Z are zero, so their accumulators hold exactly the bias: the range test
    // needs no masks, and entries 81..83 (the row padding) are stored as the zeros they are.
    uint32_t over = 0;
    const int zl_row = min((lane & 7) + 8 * ((lane >> 3) & 1), 9), zl_col = (lane >> 4) * 16; // ldmatrix.trans: rows a (9 = the zero row), 16 bytes of columns
    auto pass3 = [&](auto chk) {
    constexpr bool CHECK = decltype(chk)::value;
    // CHECK: int16 results are produced in offset binary so that "fits" is a test of the high half; without the test
    // (bounded a priori) the plain bias leaves the two's complement result in the low half
    constexpr float M0 = (OUT16 && CHECK) ? MAGIC + 32768.f : MAGIC;
    const float bias[4] = {M0, M0, M0, M0};
    uint32_t any1 = 0, all1 = 0xFFFFFFFFu;
#pragma unroll
    for (int tp = 0; tp < 6; tp++) {
        uint32_t zb[4];
        ldmatrix_x4_trans(zb, zs_base + zl_row * ZS_PITCH + tp * 32 + zl_col);
#pragma unroll
        for (int hh = 0; hh < 2; hh++) {
            const int tile = 2 * tp + hh;
            if (tile >= 11) break;
            float d[4];
            mma_f16_bias(d, fA, zb[2 * hh], zb[2 * hh + 1], bias);
            const int nn = 8 * tile + 2 * t; // entries nn, nn + 1 of row i' = g (d[0], d[1]) and i' = g + 8 (d[2], d[3])
            const bool st = tile != 10 || t < 2; // the last tile: entries 80..83 only (84.. is the next row)
            const uint32_t u0 = __float_as_uint(d[0]), u1 = __float_as_uint(d[1]), u2 = __float_as_uint(d[2]), u3 = __float_as_uint(d[3]);
            if constexpr (OUT16) {
                uint32_t wA = prmt(u0, u1, 0x5410u), wB = prmt(u2, u3, 0x5410u);
                if constexpr (CHECK) {
                    // low half = result in offset binary; it fits int16 iff the high half is still 0x4B40: OR and AND of all words
                    any1 |= u0 | u1, any1 |= u2 | u3;
                    all1 &= u0 & u1, all1 &= u2 & u3;
                    wA ^= 0x80008000u, wB ^= 0x80008000u;
                }
                if (st) {
                    reinterpret_cast<uint32_t *>(s_t)[(g * 84 + nn) >> 1] = wA;
                    if (g == 0) reinterpret_cast<uint32_t *>(s_t)[(8 * 84 + nn) >> 1] = wB;
                }
            } else {
                // in [-64, 63]  <=>  bits - (MAGIC_BITS - 64) < 128
                over |= ((u0 - (MAGIC_BITS - 64u)) | (u1 - (MAGIC_BITS - 64u))) & ~127u;
                over |= ((u2 - (MAGIC_BITS - 64u)) | (u3 - (MAGIC_BITS - 64u))) & ~127u;
                if (st) {
                    reinterpret_cast<uint16_t *>(s_t)[(g * 84 + nn) >> 1] = (uint16_t)prmt(u0, u1, 0x4040u);
                    if (g == 0) reinterpret_cast<uint16_t *>(s_t)[(8 * 84 + nn) >> 1] = (uint16_t)prmt(u2, u3, 0x4040u);
                }
            }
        }
    }
    if constexpr (OUT16 && CHECK) over = ((any1 >> 16) ^ 0x4B40u) | ((all1 >> 16) ^ 0x4B40u);
    };
    if (check3) pass3(std::true_type{}); else pass3(std::false_type{});
    // game padding (entries 756..767) is zero
    if (lane < (OUT16 ? 6 : 3)) reinterpret_cast<uint32_t *>(s_t)[(OUT16 ? 378 : 189) + lane] = 0u;
    const bool bad = __any_sync(0xFFFFFFFFu, over != 0);
    fence_proxy_async();
    __syncwarp();
    if (lane == 0) {
        flags[n] = bad ? (uint8_t)TG_FLAG_RANGE : (uint8_t)0;
        constexpr uint32_t OB = OUT16 ? 1536u : 768u;
        bulk_s2g(reinterpret_cast<uint8_t *>(slab_out) + n * OB, s_t, OB);
        bulk_commit();
        bulk_wait_read<0>();
    }
}

} // namespace

int launch_basis_mma9(const int8_t *slab_in, const int8_t *mats, long long mat_stride, void *slab_out, int out16, uint8_t *flags,
                      long long N, cudaStream_t st) {
    constexpr int SMEM = WARPS * WARP_BYTES;
    const unsigned grid = (unsigned)((N + WARPS - 1) / WARPS);
    if (out16) {
        auto kern = basis_mma9_kernel<true>;
        TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
        kern<<<grid, 32 * WARPS, SMEM, st>>>(slab_in, mats, mat_stride, slab_out, flags, N);
    } else {
        auto kern = basis_mma9_kernel<false>;
        TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
        kern<<<grid, 32 * WARPS, SMEM, st>>>(slab_in, mats, mat_stride, slab_out, flags, N);
    }
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

} // namespace tg
