// tg_aux.cu -- K4 demo_sample (training-sample batcher), K6 slice_rank (int8 and int16 slabs), K7 state_key.
#include <mutex>
#include <type_traits>

#include "tg_step.cuh"

namespace tg {

// ------------------------------------------------------------------ K4
// SyntheticDemoDataset.__getitem__ (datasets.py:77-122) for a batch of sample
// indices, straight from the in-HBM demo store (no torch.load, no Python
// replay).  idx = demo * R + action.  Emits, per sample,
//   state  float32 [dim_t][S][S][S]: slot 0 = target - sum_{j>a} rank1(tok_j),
//          slots 1.. = rank1 of actions min(a+dim_t-1,R-1) .. a+1, zero padded
//   scalar float32 = R - a, reward float32 = -(a+1), action int64 [3S] = tok_a.
// rank1 uses coefficient = token - replay_shift; the reference hard-codes 1
// there (SURVEY Q1), callers wanting the true residual pass the demo's shift.
// One thread per (sample, word column); per-entry int32 accumulators, so any
// magnitude the float32 reference can hold exactly is exact here too.
template <int S, typename TB>
__device__ __forceinline__ void vw_bytes(const TB *tok, const Lane<S> &L, int shift, int vw[4]) {
    const int vA = (int)tok[L.off_vA] - shift, vB = (int)tok[L.off_vB] - shift;
#pragma unroll
    for (int b = 0; b < 4; b++) {
        const bool inA = (L.maskA >> (8 * b)) & 1u, inB = (L.maskB >> (8 * b)) & 1u;
        const int w = (int)tok[L.off_w[b]] - shift;
        vw[b] = inA ? vA * w : (inB ? vB * w : 0);
    }
}

// sign-extended byte B of a word (one PRMT with a sign-replicating selector)
template <int B>
__device__ __forceinline__ int sext_byte(uint32_t w) {
    constexpr uint32_t sel = (uint32_t)B | ((uint32_t)(B | 8) << 4) | ((uint32_t)(B | 8) << 8) | ((uint32_t)(B | 8) << 12);
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(w), "r"(0u), "r"(sel));
    return (int)d;
}

// sample index -> (demo, action); indices below 2^32 (every realistic store) take a 32-bit division
__device__ __forceinline__ void split_index(long long id, int R, long long &demo, int &a) {
    if ((unsigned long long)id < 0x100000000ULL) {
        const uint32_t d = (uint32_t)id / (uint32_t)R;
        demo = (long long)d;
        a = (int)((uint32_t)id - d * (uint32_t)R);
    } else {
        demo = id / R;
        a = (int)(id - demo * R);
    }
}

// PACK16: the head is accumulated two entries per 32-bit word (16-bit lanes in integer form, one IMAD per two
// entries, half the registers -> more samples in flight); the host takes this path when R * cmax^3 + 128 fits int16.
// STAGE: the CTA first copies the action records a .. R-1 of all its samples into shared memory, every load in flight at
// once (the step-major tape puts each record of a demo in a different DRAM page; read one after the other inside the
// replay loop they serialise into R - a round trips per sample, which is what bounded this kernel).
template <int S, bool PACK16, bool STAGE>
__global__ void __launch_bounds__(128, PACK16 ? (S == 16 ? 6 : (S == 25 ? 3 : 8)) : 1)
    demo_sample_kernel(const uint8_t *__restrict__ tape, long long tape_step_stride,
                                   const int8_t *__restrict__ slab, long long N, int R, int dim_t, int replay_shift,
                                   const long long *__restrict__ idx, long long nb, float *__restrict__ states,
                                   float *__restrict__ scalars, long long *__restrict__ actions,
                                   float *__restrict__ rewards) {
    using G = Geo<S>;
    // COEF (the production variant): the staged records after the sample's own action hold int8 coefficients; exact under the
    // same contract PACK16 already needs (tokens <= 8, 0 <= replay_shift <= 8)
    constexpr bool COEF = PACK16 && STAGE;
    extern __shared__ __align__(16) uint8_t s_tok[]; // STAGE: [samples of the CTA][R][TP]
    const long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long b = t / G::WR;
    const long long b0 = (blockIdx.x * (long long)blockDim.x) / G::WR; // first sample this CTA touches
    // this thread's own sample first: its index and the words of the target it owns are in flight while the CTA stages the
    // action records (otherwise a third dependent DRAM round trip after the barrier)
    Lane<S> L;
    L.init((int)(t % G::WR));
    long long demo = -1;
    int a = 0;
    if (b < nb) split_index(idx[b], R, demo, a);
    const bool live = b < nb && demo >= 0 && demo < N;
    uint32_t head[S];
    if (live) {
        const int8_t *tg = slab + demo * G::GP + 4 * L.c;
#pragma unroll
        for (int i = 0; i < S; i++) head[i] = __ldg(reinterpret_cast<const uint32_t *>(tg + i * G::RP));
    }
    if constexpr (STAGE) {
        constexpr int SLOTS = (128 + G::WR - 1) / G::WR + 1;
        const int nslots = (int)min((long long)SLOTS, nb - b0);
        for (int item = threadIdx.x; item < nslots * R; item += 128) {
            const int sl = item / R, j = item - sl * R;
            long long demo2;
            int a2;
            split_index(idx[b0 + sl], R, demo2, a2);
            if (demo2 >= 0 && demo2 < N && j >= a2) {
                const uint4 *src = reinterpret_cast<const uint4 *>(tape + (size_t)j * tape_step_stride + demo2 * G::TP);
                uint4 *dst = reinterpret_cast<uint4 *>(s_tok + ((size_t)sl * R + j) * G::TP);
                if (COEF && j > a2) {
                    // records that are only ever replayed are staged as int8 coefficients (token - replay_shift, no borrow
                    // between bytes: token | 0x80 > shift), so the replay loop needs no subtraction per byte
                    const uint32_t sh4 = (uint32_t)replay_shift * ONES4;
#pragma unroll
                    for (int w = 0; w < G::TP / 16; w++) {
                        const uint4 x = __ldg(src + w);
                        dst[w] = make_uint4(((x.x | H4) - sh4) ^ H4, ((x.y | H4) - sh4) ^ H4, ((x.z | H4) - sh4) ^ H4, ((x.w | H4) - sh4) ^ H4);
                    }
                } else {
#pragma unroll
                    for (int w = 0; w < G::TP / 16; w++) dst[w] = __ldg(src + w);
                }
            }
        }
        __syncthreads();
    }
    if (!live) return;
    const uint8_t *tk = STAGE ? s_tok + (size_t)(b - b0) * R * G::TP : tape + demo * G::TP;
    if constexpr (STAGE) tape_step_stride = G::TP;
    // head
    float *st = states + b * (long long)dim_t * G::S3;
    const int nv = min(4, G::S2 - 4 * L.c); // entries of this word column inside a row (the last column of 9x9x9 holds one)
    if constexpr (PACK16) {
        int acc[S][2];
#pragma unroll
        for (int i = 0; i < S; i++) {
            const uint32_t t = head[i];
            acc[i][0] = (int)(int8_t)(t & 0xFFu) + ((int)(int8_t)((t >> 8) & 0xFFu)) * 65536;
            acc[i][1] = (int)(int8_t)((t >> 16) & 0xFFu) + ((int)(int8_t)(t >> 24)) * 65536;
        }
        if constexpr (COEF) {
            // entries outside the row (last word column of 9x9x9) pick up a v of their own; they are never stored and a low
            // 16-bit lane does not depend on the lane above it
            const bool inA0 = !G::STRADDLE || (L.maskA & 0x1u), inA1 = !G::STRADDLE || (L.maskA & 0x100u),
                       inA2 = !G::STRADDLE || (L.maskA & 0x10000u), inA3 = !G::STRADDLE || (L.maskA & 0x1000000u);
            const int8_t *rec = reinterpret_cast<const int8_t *>(tk) + (size_t)(a + 1) * G::TP;
#pragma unroll 2
            for (int j = a + 1; j < R; j++, rec += G::TP) {
                const int nvA = -(int)rec[L.off_vA], nvB = G::STRADDLE ? -(int)rec[L.off_vB] : nvA;
                const int w0 = rec[L.off_w[0]], w1 = rec[L.off_w[1]], w2 = rec[L.off_w[2]], w3 = rec[L.off_w[3]];
                const int np0 = (inA0 ? nvA : nvB) * w0 + ((inA1 ? nvA : nvB) * w1) * 65536;
                const int np1 = (inA2 ? nvA : nvB) * w2 + ((inA3 ? nvA : nvB) * w3) * 65536;
                uint32_t uq[UW<S>];
                if constexpr (S <= 4) {
                    uq[0] = *reinterpret_cast<const uint32_t *>(rec);
                } else {
                    load_u<S>(reinterpret_cast<const uint8_t *>(rec), uq);
                }
#pragma unroll
                for (int i = 0; i < S; i++) {
                    int u;
                    switch (i & 3) {
                    case 0: u = sext_byte<0>(uq[i >> 2]); break;
                    case 1: u = sext_byte<1>(uq[i >> 2]); break;
                    case 2: u = sext_byte<2>(uq[i >> 2]); break;
                    default: u = sext_byte<3>(uq[i >> 2]); break;
                    }
                    acc[i][0] += u * np0;
                    acc[i][1] += u * np1;
                }
            }
        } else {
            for (int j = a + 1; j < R; j++) {
                const uint8_t *tok = tk + (size_t)j * tape_step_stride;
                int vw[4];
                vw_bytes<S, uint8_t>(tok, L, replay_shift, vw);
                const int p0 = vw[0] + vw[1] * 65536, p1 = vw[2] + vw[3] * 65536;
#pragma unroll
                for (int i = 0; i < S; i++) {
                    const int u = (int)tok[i] - replay_shift;
                    acc[i][0] -= u * p0;
                    acc[i][1] -= u * p1;
                }
            }
        }
#pragma unroll
        for (int i = 0; i < S; i++) {
            float f[4];
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const int x = acc[i][q >> 1];
                const int lo = (int)(short)(x & 0xFFFF);
                f[q] = (float)((q & 1) ? (x - lo) >> 16 : lo);
            }
            store_run<S>(st + i * G::S2 + 4 * L.c, nv, f[0], f[1], f[2], f[3]);
        }
    } else {
        int acc[S][4];
#pragma unroll
        for (int i = 0; i < S; i++)
#pragma unroll
            for (int q = 0; q < 4; q++) acc[i][q] = (int)(int8_t)((head[i] >> (8 * q)) & 0xFFu);
        for (int j = a + 1; j < R; j++) {
            const uint8_t *tok = tk + (size_t)j * tape_step_stride;
            int vw[4];
            vw_bytes<S, uint8_t>(tok, L, replay_shift, vw);
#pragma unroll
            for (int i = 0; i < S; i++) {
                const int u = (int)tok[i] - replay_shift;
#pragma unroll
                for (int q = 0; q < 4; q++) acc[i][q] -= u * vw[q];
            }
        }
#pragma unroll
        for (int i = 0; i < S; i++)
            store_run<S>(st + i * G::S2 + 4 * L.c, nv, (float)acc[i][0], (float)acc[i][1], (float)acc[i][2], (float)acc[i][3]);
    }
    // history slots: rank-1 tensors of the next actions, latest first
    const int hi = min(a + dim_t, R);
    for (int s = 1; s < dim_t; s++) {
        const int j = hi - s;
        float *ss = st + (long long)s * G::S3;
        if (j >= a + 1) {
            using TB = typename std::conditional<COEF, int8_t, uint8_t>::type; // COEF: the record already holds coefficients
            const int hshift = COEF ? 0 : replay_shift;
            const TB *tok = reinterpret_cast<const TB *>(tk + (size_t)j * tape_step_stride);
            int vw[4];
            vw_bytes<S, TB>(tok, L, hshift, vw);
#pragma unroll
            for (int i = 0; i < S; i++) {
                const int u = (int)tok[i] - hshift;
                store_run<S>(ss + i * G::S2 + 4 * L.c, nv, (float)(u * vw[0]), (float)(u * vw[1]), (float)(u * vw[2]), (float)(u * vw[3]));
            }
        } else {
#pragma unroll
            for (int i = 0; i < S; i++) store_run<S>(ss + i * G::S2 + 4 * L.c, nv, 0.f, 0.f, 0.f, 0.f);
        }
    }
    if (L.c == 0) {
        scalars[b] = (float)(R - a);
        rewards[b] = -(float)(a + 1);
    }
    const uint8_t *ta = tk + (size_t)a * tape_step_stride;
    for (int q = L.c; q < 3 * S; q += G::WR) actions[b * 3 * S + q] = (long long)ta[q];
}

// ------------------------------------------------------------------ K4, demo-major store
// The same samples from the DEMO-MAJOR store: action records uint8 [N][R][TP] (the records a .. R-1 a sample needs are one
// contiguous run of HBM) and targets as an int8 slab [N][GP] or an int16 slab [N][GP] (entry (i,j,k) at element
// i*RP + j*S + k, two bytes each).  Every byte a CTA reads or writes moves by TMA:
//   in:  per sample one bulk copy of its records a .. R-1 and one of its target, completion on one mbarrier;
//   out: the CTA builds the float32 states of its SPC samples in shared memory as the exact image of their (contiguous)
//        region of the states array, which leaves with ONE bulk store (a cooperative scalar copy when the region is not
//        16-byte aligned / sized: odd tails, caller buffers at odd offsets).
// In between, thread (sample, word column c) replays the later actions on packed 16-bit lanes exactly as above.  The rows
// of 9x9x9 (81 floats) are not 16-byte aligned in that image, so a thread stores its four floats of a row one by one; to
// keep those stores free of bank conflicts, a thread holds its four entries ROTATED by (c >> 3) & 3 -- position q of
// thread c is entry (q + (c >> 3)) & 3 of its word column, a per-thread constant baked into the offsets it reads its w
// coefficients and target bytes from -- so that lanes c, c + 8, c + 16 (same bank for the same entry) store different
// entries in the same instruction.
template <int S>
struct SampleCfg {
    static_assert(S == 9 || S == 16, "4x4x4 and 25x25x25 samples have kernels of their own");
    using G = Geo<S>;
    static constexpr int SPC = S == 9 ? 4 : 2;                        // samples per CTA: SPC * dim_t * S^3 * 4 bytes is a multiple of 16
    static constexpr int NT = ((SPC * G::WR + 31) / 32) * 32;         // 96 / 128
    static __host__ __device__ constexpr long long smem_bytes(int R, int dim_t, bool tgt16) {
        return (((long long)SPC * dim_t * G::S3 * 4 + 15) & ~15LL) + (long long)SPC * R * G::TP + (long long)SPC * G::GP * (tgt16 ? 2 : 1) +
               ((SPC * 4 + 15) & ~15) + 16;
    }
};

// sign-extended 16-bit entry e (0..3) of the pair of words (w0 = entries 0,1; w1 = entries 2,3): one PRMT, selector in a register
__device__ __forceinline__ int sext_half_sel(uint32_t w0, uint32_t w1, uint32_t sel) {
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(w0), "r"(w1), "r"(sel));
    return (int)d;
}

template <int S, bool TGT16, bool PACK16>
__global__ void __launch_bounds__(SampleCfg<S>::NT)
    demo_sample_dm_kernel(const uint8_t *__restrict__ tape_dm, const uint8_t *__restrict__ targets, long long N, int R, int dim_t,
                          int replay_shift, const long long *__restrict__ idx, long long nb, float *__restrict__ states,
                          float *__restrict__ scalars, long long *__restrict__ actions, float *__restrict__ rewards) {
    using G = Geo<S>;
    using C = SampleCfg<S>;
    constexpr int SPC = C::SPC, NT = C::NT, GPB = G::GP * (TGT16 ? 2 : 1);
    extern __shared__ __align__(128) uint8_t smem[];
    float *s_tile = reinterpret_cast<float *>(smem);                                   // [SPC][dim_t][S^3]
    uint8_t *s_rec = smem + (((size_t)SPC * dim_t * G::S3 * 4 + 15) & ~(size_t)15);   // [SPC][R][TP]
    uint8_t *s_tgt = s_rec + (size_t)SPC * R * G::TP;                                  // [SPC][GPB]
    int *s_a = reinterpret_cast<int *>(s_tgt + (size_t)SPC * GPB);                     // [SPC] action index, -1 = bad sample
    uint64_t *s_bar = reinterpret_cast<uint64_t *>(reinterpret_cast<uint8_t *>(s_a) + ((SPC * 4 + 15) & ~15));
    const int tid = threadIdx.x;
    const long long b0 = (long long)blockIdx.x * SPC;
    const int ns = (int)min((long long)SPC, nb - b0);
    if (tid == 0) {
        mbar_init(s_bar, (uint32_t)ns);
        mbar_fence_init();
    }
    __syncthreads();
    if (tid < ns) {
        const long long id = idx[b0 + tid];
        long long demo = -1;
        int a = 0;
        if (id >= 0) split_index(id, R, demo, a);
        const bool ok = demo >= 0 && demo < N;
        s_a[tid] = ok ? a : -1;
        if (ok) {
            const uint32_t rb = (uint32_t)(R - a) * G::TP;
            mbar_expect_tx(s_bar, rb + (uint32_t)GPB);
            bulk_g2s(s_rec + ((size_t)tid * R + a) * G::TP, tape_dm + ((size_t)demo * R + a) * G::TP, rb, s_bar);
            bulk_g2s(s_tgt + (size_t)tid * GPB, targets + (size_t)demo * GPB, (uint32_t)GPB, s_bar);
        } else {
            asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(s_bar)) : "memory");
        }
    }
    __syncthreads(); // s_a
    mbar_wait(s_bar, 0);
    // the records that are only replayed (j > a) become int8 coefficients in place (token - replay_shift; no borrow between
    // bytes: token | 0x80 > shift), so the replay loop has no subtraction per byte
    {
        const uint32_t sh4 = (uint32_t)replay_shift * ONES4;
        for (int sl = 0; sl < ns; sl++) {
            const int a = s_a[sl];
            if (a < 0) continue;
            uint32_t *rw = reinterpret_cast<uint32_t *>(s_rec + ((size_t)sl * R + a + 1) * G::TP);
            for (int w = tid; w < (R - a - 1) * (G::TP / 4); w += NT) rw[w] = ((rw[w] | H4) - sh4) ^ H4;
        }
    }
    __syncthreads();

    const int sl = tid / G::WR;
    const bool worker = tid < SPC * G::WR && sl < ns;
    if (worker) {
        Lane<S> L;
        L.init(tid % G::WR);
        const int a = s_a[sl];
        const long long b = b0 + sl;
        float *st = s_tile + (size_t)sl * dim_t * G::S3;
        const int nv = min(4, G::S2 - 4 * L.c); // entries of this word column inside a row
        // position q of this thread is entry ord(q) = (q + rot) & 3 of its word column (rot = 0 unless the rows are unaligned)
        const int rot = (G::S2 % 4 != 0) ? ((L.c >> 3) & 3) : 0;
        int offw[4], wpos[4];
        bool inA[4], valid[4];
        uint32_t tsel[4];
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int e = (q + rot) & 3;
            offw[q] = L.off_w[0], inA[q] = true;
#pragma unroll
            for (int x = 0; x < 4; x++)
                if (x == e) offw[q] = L.off_w[x], inA[q] = !G::STRADDLE || ((L.maskA >> (8 * x)) & 1u);
            valid[q] = e < nv;
            wpos[q] = 4 * L.c + e;
            // target entry e as a sign-extended int: int8 slab -> byte e of the word; int16 slab -> half e of the word pair
            tsel[q] = TGT16 ? ((uint32_t)(2 * e) | ((uint32_t)(2 * e + 1) << 4) | ((uint32_t)(8 | (2 * e + 1)) << 8) | ((uint32_t)(8 | (2 * e + 1)) << 12))
                            : ((uint32_t)e | ((uint32_t)(8 | e) << 4) | ((uint32_t)(8 | e) << 8) | ((uint32_t)(8 | e) << 12));
        }
        auto put4 = [&](float *row, float f0, float f1, float f2, float f3) {
            if constexpr (G::S2 % 4 == 0) {
                *reinterpret_cast<float4 *>(row + 4 * L.c) = make_float4(f0, f1, f2, f3);
            } else {
                if (valid[0]) row[wpos[0]] = f0;
                if (valid[1]) row[wpos[1]] = f1;
                if (valid[2]) row[wpos[2]] = f2;
                if (valid[3]) row[wpos[3]] = f3;
            }
        };
        if (a < 0) {
            for (int s = 0; s < dim_t; s++)
#pragma unroll
                for (int i = 0; i < S; i++) put4(st + (size_t)s * G::S3 + i * G::S2, 0.f, 0.f, 0.f, 0.f);
        } else {
            const int8_t *rec0 = reinterpret_cast<const int8_t *>(s_rec + (size_t)sl * R * G::TP);
            const uint8_t *tg = s_tgt + (size_t)sl * GPB;
            // ---- head = target - sum of the later actions
            int acc[S][PACK16 ? 2 : 4];
#pragma unroll
            for (int i = 0; i < S; i++) {
                uint32_t w0, w1 = 0;
                if constexpr (TGT16) {
                    const uint2 p = *reinterpret_cast<const uint2 *>(tg + (size_t)(i * G::RP + 4 * L.c) * 2);
                    w0 = p.x, w1 = p.y;
                } else {
                    w0 = *reinterpret_cast<const uint32_t *>(tg + i * G::RP + 4 * L.c);
                }
                const int e0 = sext_half_sel(w0, w1, tsel[0]), e1 = sext_half_sel(w0, w1, tsel[1]), e2 = sext_half_sel(w0, w1, tsel[2]),
                          e3 = sext_half_sel(w0, w1, tsel[3]);
                if constexpr (PACK16) {
                    acc[i][0] = e0 + e1 * 65536, acc[i][1] = e2 + e3 * 65536;
                } else {
                    acc[i][0] = e0, acc[i][1] = e1, acc[i][2] = e2, acc[i][3] = e3;
                }
            }
            const int8_t *rec = rec0 + (size_t)(a + 1) * G::TP;
#pragma unroll 2
            for (int j = a + 1; j < R; j++, rec += G::TP) {
                const int nvA = -(int)rec[L.off_vA], nvB = G::STRADDLE ? -(int)rec[L.off_vB] : nvA;
                const int p0 = (inA[0] ? nvA : nvB) * (int)rec[offw[0]], p1 = (inA[1] ? nvA : nvB) * (int)rec[offw[1]],
                          p2 = (inA[2] ? nvA : nvB) * (int)rec[offw[2]], p3 = (inA[3] ? nvA : nvB) * (int)rec[offw[3]];
                uint32_t uq[4];
                const uint4 q4 = *reinterpret_cast<const uint4 *>(rec);
                uq[0] = q4.x, uq[1] = q4.y, uq[2] = q4.z, uq[3] = q4.w;
                const int np0 = p0 + p1 * 65536, np1 = p2 + p3 * 65536;
#pragma unroll
                for (int i = 0; i < S; i++) {
                    int u;
                    switch (i & 3) {
                    case 0: u = sext_byte<0>(uq[i >> 2]); break;
                    case 1: u = sext_byte<1>(uq[i >> 2]); break;
                    case 2: u = sext_byte<2>(uq[i >> 2]); break;
                    default: u = sext_byte<3>(uq[i >> 2]); break;
                    }
                    if constexpr (PACK16) {
                        acc[i][0] += u * np0, acc[i][1] += u * np1;
                    } else {
                        acc[i][0] += u * p0, acc[i][1] += u * p1, acc[i][2] += u * p2, acc[i][3] += u * p3;
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < S; i++) {
                float f[4];
                if constexpr (PACK16) {
#pragma unroll
                    for (int h = 0; h < 2; h++) {
                        const int x = acc[i][h];
                        const int lo = (int)(short)(x & 0xFFFF);
                        f[2 * h] = (float)lo, f[2 * h + 1] = (float)((x - lo) >> 16);
                    }
                } else {
#pragma unroll
                    for (int q = 0; q < 4; q++) f[q] = (float)acc[i][q];
                }
                put4(st + i * G::S2, f[0], f[1], f[2], f[3]);
            }
            // ---- history slots: rank-1 tensors of the next actions, latest first
            const int hi = min(a + dim_t, R);
            for (int s = 1; s < dim_t; s++) {
                const int j = hi - s;
                float *ss = st + (size_t)s * G::S3;
                if (j >= a + 1) {
                    const int8_t *hr = rec0 + (size_t)j * G::TP;
                    const int vA = (int)hr[L.off_vA], vB = G::STRADDLE ? (int)hr[L.off_vB] : vA;
                    const float pf0 = (float)((inA[0] ? vA : vB) * (int)hr[offw[0]]), pf1 = (float)((inA[1] ? vA : vB) * (int)hr[offw[1]]),
                                pf2 = (float)((inA[2] ? vA : vB) * (int)hr[offw[2]]), pf3 = (float)((inA[3] ? vA : vB) * (int)hr[offw[3]]);
#pragma unroll
                    for (int i = 0; i < S; i++) {
                        const float uf = (float)(int)hr[i];
                        put4(ss + i * G::S2, uf * pf0, uf * pf1, uf * pf2, uf * pf3);
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < S; i++) put4(ss + i * G::S2, 0.f, 0.f, 0.f, 0.f);
                }
            }
            if (L.c == 0) {
                scalars[b] = (float)(R - a);
                rewards[b] = -(float)(a + 1);
            }
            const uint8_t *ta = s_rec + ((size_t)sl * R + a) * G::TP; // the sample's own action: raw tokens
            for (int q = L.c; q < 3 * S; q += G::WR) actions[b * 3 * S + q] = (long long)ta[q];
        }
    }
    fence_proxy_async();
    __syncthreads();
    float *dst = states + b0 * (long long)dim_t * G::S3;
    const size_t bytes = (size_t)ns * dim_t * G::S3 * 4;
    if ((bytes & 15) == 0 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
        if (tid == 0) {
            bulk_s2g(dst, s_tile, (uint32_t)bytes);
            bulk_commit();
            bulk_wait_read<0>();
        }
    } else {
        for (size_t e = tid; e < bytes / 4; e += NT) dst[e] = s_tile[e];
    }
}

// ------------------------------------------------------------------ K4 at 25x25x25, demo-major store
// One 25x25x25 state slot is 62.5 KB of float32, so the shared-memory image of whole samples that demo_sample_dm_kernel
// builds does not fit from dim_t = 4 on.  Here a CTA serves one sample: its records a .. R-1 (one contiguous run of the
// demo-major store) arrive with one bulk copy, thread c (one of the 157 word columns) keeps the four entries
// (i, 4c .. 4c+3) of every row of the head in registers -- exact int32 entries, or two 16-bit lanes per register under the
// same bound as above -- and every state slot leaves straight from the registers with the widest stores each address
// allows (store_run), so states may start at any float.
template <bool TGT16, bool PACK16>
__global__ void __launch_bounds__(160, PACK16 ? 3 : 1)
    demo_sample_dm25_kernel(const uint8_t *__restrict__ tape_dm, const uint8_t *__restrict__ targets, long long N, int R, int dim_t,
                            int replay_shift, const long long *__restrict__ idx, float *__restrict__ states,
                            float *__restrict__ scalars, long long *__restrict__ actions, float *__restrict__ rewards) {
    constexpr int S = 25;
    using G = Geo<S>;
    extern __shared__ __align__(16) uint8_t s_rec[]; // [R][TP]: record a raw, records a+1 .. R-1 as int8 coefficients
    __shared__ uint64_t s_bar;
    const int tid = threadIdx.x;
    const long long b = blockIdx.x;
    long long demo = -1;
    int a = 0;
    const long long id = idx[b];
    if (id >= 0) split_index(id, R, demo, a);
    const bool worker = tid < G::WR;
    Lane<S> L;
    L.init(worker ? tid : 0);
    const int nv = min(4, G::S2 - 4 * L.c);
    float *st = states + b * (long long)dim_t * G::S3;
    if (demo < 0 || demo >= N) { // bad index: zero states, nothing else written
        if (worker)
            for (int s = 0; s < dim_t; s++)
#pragma unroll
                for (int i = 0; i < S; i++) store_run<S>(st + (size_t)s * G::S3 + i * G::S2 + 4 * L.c, nv, 0.f, 0.f, 0.f, 0.f);
        return;
    }
    if (tid == 0) {
        mbar_init(&s_bar, 1);
        mbar_fence_init();
    }
    __syncthreads();
    if (tid == 0) {
        const uint32_t rb = (uint32_t)(R - a) * G::TP;
        mbar_expect_tx(&s_bar, rb);
        bulk_g2s(s_rec + (size_t)a * G::TP, tape_dm + ((size_t)demo * R + a) * G::TP, rb, &s_bar);
    }
    // the target words of this word column are in flight while the records land
    int acc[S][PACK16 ? 2 : 4];
    if (worker) {
#pragma unroll
        for (int i = 0; i < S; i++) {
            int e[4];
            if constexpr (TGT16) {
                const uint2 p = __ldg(reinterpret_cast<const uint2 *>(targets + ((size_t)demo * G::GP + i * G::RP + 4 * L.c) * 2));
                e[0] = (int)(short)(p.x & 0xFFFFu), e[1] = (int)p.x >> 16, e[2] = (int)(short)(p.y & 0xFFFFu), e[3] = (int)p.y >> 16;
            } else {
                const uint32_t w = __ldg(reinterpret_cast<const uint32_t *>(targets + (size_t)demo * G::GP + i * G::RP + 4 * L.c));
                e[0] = sext_byte<0>(w), e[1] = sext_byte<1>(w), e[2] = sext_byte<2>(w), e[3] = sext_byte<3>(w);
            }
            if constexpr (PACK16) {
                acc[i][0] = e[0] + e[1] * 65536, acc[i][1] = e[2] + e[3] * 65536;
            } else {
                acc[i][0] = e[0], acc[i][1] = e[1], acc[i][2] = e[2], acc[i][3] = e[3];
            }
        }
    }
    mbar_wait(&s_bar, 0);
    {   // records that are only replayed become int8 coefficients in place (no borrow between bytes: token | 0x80 > shift)
        const uint32_t sh4 = (uint32_t)replay_shift * ONES4;
        uint32_t *rw = reinterpret_cast<uint32_t *>(s_rec + (size_t)(a + 1) * G::TP);
        for (int w = tid; w < (R - a - 1) * (G::TP / 4); w += 160) rw[w] = ((rw[w] | H4) - sh4) ^ H4;
    }
    __syncthreads();
    if (!worker) return;
    // entries outside the row (last word column) take v_B; they are never stored, and a 16-bit lane never reads the one above it
    const bool inA[4] = {(L.maskA & 0x1u) != 0, (L.maskA & 0x100u) != 0, (L.maskA & 0x10000u) != 0, (L.maskA & 0x1000000u) != 0};
    const int8_t *rec0 = reinterpret_cast<const int8_t *>(s_rec);
#pragma unroll 2
    for (int j = a + 1; j < R; j++) {
        const int8_t *rec = rec0 + (size_t)j * G::TP;
        const int nvA = -(int)rec[L.off_vA], nvB = -(int)rec[L.off_vB];
        int p[4];
#pragma unroll
        for (int q = 0; q < 4; q++) p[q] = (inA[q] ? nvA : nvB) * (int)rec[L.off_w[q]];
        uint32_t uq[UW<S>];
        load_u<S>(reinterpret_cast<const uint8_t *>(rec), uq);
        const int np0 = p[0] + p[1] * 65536, np1 = p[2] + p[3] * 65536;
#pragma unroll
        for (int i = 0; i < S; i++) {
            int u;
            switch (i & 3) {
            case 0: u = sext_byte<0>(uq[i >> 2]); break;
            case 1: u = sext_byte<1>(uq[i >> 2]); break;
            case 2: u = sext_byte<2>(uq[i >> 2]); break;
            default: u = sext_byte<3>(uq[i >> 2]); break;
            }
            if constexpr (PACK16) {
                acc[i][0] += u * np0, acc[i][1] += u * np1;
            } else {
                acc[i][0] += u * p[0], acc[i][1] += u * p[1], acc[i][2] += u * p[2], acc[i][3] += u * p[3];
            }
        }
    }
#pragma unroll
    for (int i = 0; i < S; i++) {
        float f[4];
        if constexpr (PACK16) {
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const int x = acc[i][h];
                const int lo = (int)(short)(x & 0xFFFF);
                f[2 * h] = (float)lo, f[2 * h + 1] = (float)((x - lo) >> 16);
            }
        } else {
#pragma unroll
            for (int q = 0; q < 4; q++) f[q] = (float)acc[i][q];
        }
        store_run<S>(st + i * G::S2 + 4 * L.c, nv, f[0], f[1], f[2], f[3]);
    }
    // history slots: rank-1 tensors of the next actions, latest first
    const int hi = min(a + dim_t, R);
    for (int s = 1; s < dim_t; s++) {
        const int j = hi - s;
        float *ss = st + (size_t)s * G::S3;
        if (j >= a + 1) {
            const int8_t *hr = rec0 + (size_t)j * G::TP;
            const int vA = (int)hr[L.off_vA], vB = (int)hr[L.off_vB];
            float pf[4];
#pragma unroll
            for (int q = 0; q < 4; q++) pf[q] = (float)((inA[q] ? vA : vB) * (int)hr[L.off_w[q]]);
#pragma unroll
            for (int i = 0; i < S; i++) {
                const float uf = (float)(int)hr[i];
                store_run<S>(ss + i * G::S2 + 4 * L.c, nv, uf * pf[0], uf * pf[1], uf * pf[2], uf * pf[3]);
            }
        } else {
#pragma unroll
            for (int i = 0; i < S; i++) store_run<S>(ss + i * G::S2 + 4 * L.c, nv, 0.f, 0.f, 0.f, 0.f);
        }
    }
    if (tid == 0) {
        scalars[b] = (float)(R - a);
        rewards[b] = -(float)(a + 1);
    }
    const uint8_t *ta = s_rec + (size_t)a * G::TP; // the sample's own action: raw tokens
    for (int q = tid; q < 3 * S; q += G::WR) actions[b * 3 * S + q] = (long long)ta[q];
}

// ------------------------------------------------------------------ K4r: 9x9x9, one thread per (sample, row i)
// The word-column kernel above spends ~1270 warp-instructions per 9x9x9 sample: every one of a sample's 21 threads
// extracts all nine u coefficients of every replayed action and walks all of them.  Here a thread owns ROW i of its sample
// (81 entries as 45 packed pairs of 16-bit lanes): per replayed action it needs ONE u coefficient -- and skips the action
// altogether when that coefficient is zero (70 % of them with the reference's distributions; every lane walks its own list
// of non-zero actions) -- forms c_j = u_i v_j once and adds c_j * pack(w) to its nine runs: 45 IMADs for 81 entries.  A WARP
// is self-contained (three samples, no CTA barrier): it converts the later records of its samples into replay form (w as
// five 16-bit pairs, u and v as int8 coefficients) in shared memory, and builds one state slot at a time in a warp-private
// tile that is the image of the slot's 729 floats in HBM -- placed at the same offset modulo 16 bytes, so the aligned body
// leaves with one TMA bulk store per (sample, slot) and at most three floats at either end with plain stores.  A row of 81
// floats is 81 consecutive words of the tile and lanes are 81 words apart: conflict-free for the lanes of one sample.
namespace rows9 {
constexpr int S = 9, S2 = 81, S3 = 729, TP = 32, RP = 84, GP = 768;
constexpr int WARPS = 4, SPW = 3;            // warps per CTA; samples per warp (27 of 32 lanes own a row)
constexpr int RECB = 48;                     // replay record: 5 words pack16(w) | 5 words coefficient bytes (u 0..8, v 9..17) | pad
constexpr int PIECE = 736;                   // floats per sample in the warp tile (729 + alignment phase, multiple of 4 and of 32)
__host__ __device__ constexpr int warp_bytes(int R) { return ((SPW * R * RECB + 15) & ~15) + SPW * PIECE * 4; }

template <int B>
__device__ __forceinline__ int sx(uint32_t w) { return sext_byte<B>(w); }

template <bool TGT16, bool PACK16>
__global__ void __launch_bounds__(32 * WARPS, 4)
    demo_sample_rows9_kernel(const uint8_t *__restrict__ tape_dm, const uint8_t *__restrict__ targets, long long N, int R, int dim_t,
                             int replay_shift, const long long *__restrict__ idx, long long nb, float *__restrict__ states,
                             float *__restrict__ scalars, long long *__restrict__ actions, float *__restrict__ rewards,
                             unsigned long long *__restrict__ ticket) {
    static_assert(PACK16, "the row kernel keeps 16-bit lanes; the host routes larger bounds to the column kernel");
    extern __shared__ __align__(128) uint8_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint8_t *s_rec = smem + (size_t)warp * warp_bytes(R);
    float *s_tile = reinterpret_cast<float *>(s_rec + ((SPW * R * RECB + 15) & ~15));
    // a warp starts with triple number (its own index) and then takes tickets from a global counter (a triple replays 0 .. R-1
    // actions per sample, so equal COUNTS of triples per warp leave the last wave of a launch a fifth full): the index of
    // the NEXT triple is read while this one is processed, and its records and target rows are pulled into L2 before the
    // slots of this one are built, so that the two dependent DRAM round trips at the head of a triple (index -> records /
    // targets) are hidden behind the previous one
    const long long nwarps = (long long)gridDim.x * WARPS, ntrip = (nb + SPW - 1) / SPW;
    long long trip = (long long)blockIdx.x * WARPS + warp;
    if (trip >= ntrip) return;
    auto decode = [&](long long id, long long &dm, int &aa) {
        dm = -1, aa = -1;
        if (id >= 0) {
            split_index(id, R, dm, aa);
            if (dm >= N) dm = -1, aa = -1;
        }
    };
    long long my_demo = -1;
    int my_a = -1;
    if (lane < (int)min((long long)SPW, nb - trip * SPW)) decode(idx[trip * SPW + lane], my_demo, my_a);
    for (;;) {
    const long long b0 = trip * SPW;
    const int ns = (int)min((long long)SPW, nb - b0);
    unsigned long long tk = 0;
    if (lane == 0) tk = atomicAdd(ticket, 1ULL);
    const long long ntr = nwarps + (long long)__shfl_sync(0xFFFFFFFFu, tk, 0);
    long long nid = -1;
    if (ntr < ntrip && lane < (int)min((long long)SPW, nb - ntr * SPW)) nid = idx[ntr * SPW + lane];
    // ---- the warp's samples: lane q < ns holds sample q; everybody gets (demo, a) of every sample by shuffle
    long long demo_q[SPW];
    int a_q[SPW];
#pragma unroll
    for (int q = 0; q < SPW; q++) {
        demo_q[q] = __shfl_sync(0xFFFFFFFFu, my_demo, q);
        a_q[q] = __shfl_sync(0xFFFFFFFFu, my_a, q);
    }
    const int q = lane / S, i = lane - q * S; // this lane's sample and row (lanes 27..31: q == 3, helpers only)
    const bool owner = q < ns;
    long long demo = -1;
    int a = -1;
#pragma unroll
    for (int x = 0; x < SPW; x++)
        if (x == q) demo = demo_q[x], a = a_q[x];
    const bool live = owner && a >= 0;
    // ---- this lane's target row in flight: 84 bytes (int8) / 162 bytes (int16) at a 4-byte aligned address; and its three
    // tokens of the sample's own action (raw tokens: the actions output)
    constexpr int TW = TGT16 ? 41 : 21;
    uint32_t tw[TW];
    uint32_t own[3] = {0, 0, 0};
    if (live) {
        const uint8_t *ta = tape_dm + ((size_t)demo * R + a) * TP;
#pragma unroll
        for (int x = 0; x < 3; x++) own[x] = __ldg(ta + i * 3 + x);
        const uint32_t *tp = reinterpret_cast<const uint32_t *>(targets + ((size_t)demo * GP + i * RP) * (TGT16 ? 2 : 1));
#pragma unroll
        for (int w = 0; w < TW; w++) tw[w] = __ldg(tp + w);
    }
    // ---- the records j > a of the three samples -> replay form in shared memory, one record per lane and round
    {
        const uint32_t sh4 = (uint32_t)replay_shift * ONES4;
        int n0 = a_q[0] >= 0 ? R - 1 - a_q[0] : 0, n1 = a_q[1] >= 0 ? R - 1 - a_q[1] : 0, n2 = a_q[2] >= 0 ? R - 1 - a_q[2] : 0;
        for (int e = lane; e < n0 + n1 + n2; e += 32) {
            const int x = (e >= n0) + (e >= n0 + n1);
            const int j = (x == 0 ? a_q[0] + 1 + e : (x == 1 ? a_q[1] + 1 + e - n0 : a_q[2] + 1 + e - n0 - n1));
            const long long d = x == 0 ? demo_q[0] : (x == 1 ? demo_q[1] : demo_q[2]);
            const uint4 *src = reinterpret_cast<const uint4 *>(tape_dm + ((size_t)d * R + j) * TP);
            const uint4 r0 = __ldg(src), r1 = __ldg(src + 1);
            const uint32_t c0 = ((r0.x | H4) - sh4) ^ H4, c1 = ((r0.y | H4) - sh4) ^ H4, c2 = ((r0.z | H4) - sh4) ^ H4,
                           c3 = ((r0.w | H4) - sh4) ^ H4, c4 = ((r1.x | H4) - sh4) ^ H4, c5 = ((r1.y | H4) - sh4) ^ H4,
                           c6 = ((r1.z | H4) - sh4) ^ H4;
            // w coefficients are bytes 18..26: c4.2, c4.3, c5.0..3, c6.0..2
            const int p0 = sx<2>(c4) + sx<3>(c4) * 65536, p1 = sx<0>(c5) + sx<1>(c5) * 65536, p2 = sx<2>(c5) + sx<3>(c5) * 65536,
                      p3 = sx<0>(c6) + sx<1>(c6) * 65536, p4 = sx<2>(c6);
            uint4 *dst = reinterpret_cast<uint4 *>(s_rec + ((size_t)x * R + j) * RECB);
            dst[0] = make_uint4((uint32_t)p0, (uint32_t)p1, (uint32_t)p2, (uint32_t)p3);
            dst[1] = make_uint4((uint32_t)p4, c0, c1, c2);
            dst[2] = make_uint4(c3, c4, 0u, 0u);
        }
    }
    __syncwarp();
    const uint8_t *rbase = s_rec + (size_t)(owner ? q : 0) * R * RECB;
    // ---- head: target row as packed pairs, minus the later actions whose u_i is not zero
    int acc[S][5];
    if (live) {
#pragma unroll
        for (int j = 0; j < S; j++)
#pragma unroll
            for (int p = 0; p < 5; p++) {
                const int e0 = 9 * j + 2 * p; // entries e0, e0 + 1 of the row (the fifth pair of a run holds one entry)
                if constexpr (TGT16) {
                    uint32_t pr;
                    if ((e0 & 1) == 0)
                        pr = tw[e0 >> 1];
                    else
                        pr = __byte_perm(tw[e0 >> 1], tw[(e0 >> 1) + 1 < TW ? (e0 >> 1) + 1 : e0 >> 1], 0x5432);
                    // two's complement halves -> lo + 65536 * hi (a negative low half borrows from the high one); the fifth
                    // pair of a run holds a single entry
                    acc[j][p] = p < 4 ? (int)(pr - ((pr & 0x8000u) << 1)) : (int)(short)(pr & 0xFFFFu);
                } else {
                    auto ent = [&](int e) -> int {
                        switch (e & 3) {
                        case 0: return sx<0>(tw[e >> 2]);
                        case 1: return sx<1>(tw[e >> 2]);
                        case 2: return sx<2>(tw[e >> 2]);
                        default: return sx<3>(tw[e >> 2]);
                        }
                    };
                    acc[j][p] = p < 4 ? ent(e0) + ent(e0 + 1) * 65536 : ent(e0);
                }
            }
        // bit x of mask: action a + 1 + x has u_i != 0
        uint32_t mask = 0;
        for (int j = a + 1, x = 0; j < R; j++, x++)
            if (reinterpret_cast<const int8_t *>(rbase + (size_t)j * RECB)[20 + i] != 0) mask |= 1u << x;
        if (R - 1 - a > 32) mask = 0xFFFFFFFFu; // longer lists: plain walk below
        auto apply = [&](int j) {
            const uint8_t *rec = rbase + (size_t)j * RECB;
            const uint4 w03 = *reinterpret_cast<const uint4 *>(rec), w47 = *reinterpret_cast<const uint4 *>(rec + 16);
            const uint2 w89 = *reinterpret_cast<const uint2 *>(rec + 32);
            const int nu = -(int)reinterpret_cast<const int8_t *>(rec)[20 + i];
            // v coefficients: record bytes 29..37 = w47.w bytes 1..3, w89.x bytes 0..3, w89.y bytes 0..1
            const int c[S] = {nu * sx<1>(w47.w), nu * sx<2>(w47.w), nu * sx<3>(w47.w), nu * sx<0>(w89.x), nu * sx<1>(w89.x),
                              nu * sx<2>(w89.x), nu * sx<3>(w89.x), nu * sx<0>(w89.y), nu * sx<1>(w89.y)};
            const int pw[5] = {(int)w03.x, (int)w03.y, (int)w03.z, (int)w03.w, (int)w47.x};
#pragma unroll
            for (int j2 = 0; j2 < S; j2++)
#pragma unroll
                for (int p = 0; p < 5; p++) acc[j2][p] += c[j2] * pw[p];
        };
        if (R - 1 - a <= 32) {
            while (mask) {
                const int x = __ffs((int)mask) - 1;
                mask &= mask - 1;
                apply(a + 1 + x);
            }
        } else {
            for (int j = a + 1; j < R; j++) apply(j);
        }
    }
    // ---- the next triple: decode its indices (read at the top) and pull its records and target rows into L2
    long long nx_demo;
    int nx_a;
    decode(nid, nx_demo, nx_a);
    {
        const long long pd = __shfl_sync(0xFFFFFFFFu, nx_demo, q < SPW ? q : 0);
        const int pa = __shfl_sync(0xFFFFFFFFu, nx_a, q < SPW ? q : 0);
        if (q < SPW && pa >= 0) {
            const uint8_t *trow = targets + ((size_t)pd * GP + i * RP) * (TGT16 ? 2 : 1);
            asm volatile("prefetch.global.L2 [%0];" ::"l"(trow));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(trow + (TGT16 ? 161 : 83)));
            if (i * 128 < (R - pa) * TP) asm volatile("prefetch.global.L2 [%0];" ::"l"(tape_dm + ((size_t)pd * R + pa) * TP + i * 128));
        }
    }
    // ---- slots, one at a time through the warp tile
    const long long b = b0 + (owner ? q : 0);
    const int hi = min(a + dim_t, R);
    for (int s = 0; s < dim_t; s++) {
        float *gdst = states + (b * dim_t + s) * (long long)S3;
        const int ph = (int)((reinterpret_cast<uintptr_t>(gdst) >> 2) & 3); // the piece sits at the same offset modulo 16 bytes
        float *row = s_tile + q * PIECE + ph + i * S2;
        if (owner) {
            if (live && s == 0) {
#pragma unroll
                for (int j = 0; j < S; j++)
#pragma unroll
                    for (int p = 0; p < 5; p++) {
                        const int x = acc[j][p];
                        if (p < 4) {
                            const int lo = (int)(short)(x & 0xFFFF);
                            row[9 * j + 2 * p] = (float)lo;
                            row[9 * j + 2 * p + 1] = (float)((x - lo) >> 16);
                        } else {
                            row[9 * j + 8] = (float)x;
                        }
                    }
            } else if (live && hi - s >= a + 1) {
                const uint8_t *rec = rbase + (size_t)(hi - s) * RECB;
                const uint4 w03 = *reinterpret_cast<const uint4 *>(rec), w47 = *reinterpret_cast<const uint4 *>(rec + 16);
                const uint2 w89 = *reinterpret_cast<const uint2 *>(rec + 32);
                const int u = (int)reinterpret_cast<const int8_t *>(rec)[20 + i];
                const float cf[S] = {(float)(u * sx<1>(w47.w)), (float)(u * sx<2>(w47.w)), (float)(u * sx<3>(w47.w)),
                                     (float)(u * sx<0>(w89.x)), (float)(u * sx<1>(w89.x)), (float)(u * sx<2>(w89.x)),
                                     (float)(u * sx<3>(w89.x)), (float)(u * sx<0>(w89.y)), (float)(u * sx<1>(w89.y))};
                // w back from the pairs: lo + 65536 * hi
                float wf[S];
#pragma unroll
                for (int p = 0; p < 4; p++) {
                    const int x = p == 0 ? (int)w03.x : (p == 1 ? (int)w03.y : (p == 2 ? (int)w03.z : (int)w03.w));
                    const int lo = (int)(short)(x & 0xFFFF);
                    wf[2 * p] = (float)lo, wf[2 * p + 1] = (float)((x - lo) >> 16);
                }
                wf[8] = (float)(int)w47.x;
#pragma unroll
                for (int j = 0; j < S; j++)
#pragma unroll
                    for (int k = 0; k < S; k++) row[9 * j + k] = cf[j] * wf[k];
            } else {
#pragma unroll
                for (int e = 0; e < S2; e++) row[e] = 0.f;
            }
        }
        fence_proxy_async();
        __syncwarp();
        // copy-out: lane 9 x leads sample x: aligned body by TMA, up to three floats at either end by lanes 9x+1 .. 9x+6
        if (owner) {
            const int hc = (4 - ph) & 3, nbody = (S3 - hc) & ~3, tail = S3 - hc - nbody;
            const float *piece = s_tile + q * PIECE + ph;
            if (i == 0) {
                bulk_s2g(gdst + hc, piece + hc, (uint32_t)nbody * 4u);
                bulk_commit();
            } else if (i <= 3) {
                if (i - 1 < hc) gdst[i - 1] = piece[i - 1];
            } else if (i <= 6) {
                if (i - 4 < tail) gdst[hc + nbody + i - 4] = piece[hc + nbody + i - 4];
            }
            if (i == 0) bulk_wait_read<0>();
        }
        __syncwarp(); // the tile may be rewritten
    }
    if (live) {
        if (i == 0) {
            scalars[b] = (float)(R - a);
            rewards[b] = -(float)(a + 1);
        }
#pragma unroll
        for (int x = 0; x < 3; x++) actions[b * 27 + i * 3 + x] = (long long)own[x];
    }
    if (ntr >= ntrip) break;
    trip = ntr, my_demo = nx_demo, my_a = nx_a;
    __syncwarp(); // the records of this triple are dead: the next conversion may overwrite them
    } // triples
}
} // namespace rows9

// ------------------------------------------------------------------ K4 at 4x4x4: one thread per (sample, row i)
// A 4x4x4 sample is tiny (64-byte target, <= R 16-byte records, dim_t * 256 bytes out): the word-column kernel above spends
// 165 warp-instructions per sample in staging loops and CTA barriers (0.15-0.28 of HBM).  Here four threads own the four
// rows of a sample entirely in registers -- 16 int32 entries, exact for any target bound, no shared memory, no barrier: the
// target row is one 16-byte load, every record one 16-byte load (the four threads of a sample read the same one), a
// replayed action whose u_i is zero is skipped, and a state row leaves as four 16-byte stores; the four threads of a
// sample write 256 contiguous bytes per slot.
namespace rows4 {
template <bool TGT16>
__global__ void __launch_bounds__(128)
    demo_sample_rows4_kernel(const uint8_t *__restrict__ tape_dm, const uint8_t *__restrict__ targets, long long N, int R, int dim_t,
                             int replay_shift, const long long *__restrict__ idx, long long nb, float *__restrict__ states,
                             float *__restrict__ scalars, long long *__restrict__ actions, float *__restrict__ rewards) {
    const long long gt = (long long)blockIdx.x * 128 + threadIdx.x;
    const long long b = gt >> 2;
    const int i = (int)(gt & 3);
    if (b >= nb) return;
    const long long id = idx[b];
    long long demo = -1;
    int a = 0;
    if (id >= 0) split_index(id, R, demo, a);
    float *st = states + b * (long long)dim_t * 64 + i * 16; // row i of slot 0
    const bool aligned = (reinterpret_cast<uintptr_t>(states) & 15) == 0; // then every row of every sample is 16-byte aligned
    auto put_row = [&](float *row, const float (&f)[16]) {
        if (aligned) {
#pragma unroll
            for (int j = 0; j < 4; j++) st_f32x4(row + 4 * j, f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
        } else {
#pragma unroll
            for (int j = 0; j < 4; j++) store_run<4>(row + 4 * j, 4, f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
        }
    };
    const float zeros[16] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (demo < 0 || demo >= N) { // bad index: zero states, nothing else written (as the column kernel)
        for (int s = 0; s < dim_t; s++) put_row(st + (size_t)s * 64, zeros);
        return;
    }
    // ---- head = target - sum of the later actions
    int acc[16];
    if constexpr (TGT16) {
        const uint4 *tp = reinterpret_cast<const uint4 *>(reinterpret_cast<const int16_t *>(targets) + demo * 64 + i * 16);
        const uint4 t0 = __ldg(tp), t1 = __ldg(tp + 1);
        const uint32_t tw[8] = {t0.x, t0.y, t0.z, t0.w, t1.x, t1.y, t1.z, t1.w};
#pragma unroll
        for (int e = 0; e < 8; e++) acc[2 * e] = (int)(short)(tw[e] & 0xFFFFu), acc[2 * e + 1] = (int)tw[e] >> 16;
    } else {
        const uint4 t0 = __ldg(reinterpret_cast<const uint4 *>(targets + demo * 64 + i * 16));
        const uint32_t tw[4] = {t0.x, t0.y, t0.z, t0.w};
#pragma unroll
        for (int e = 0; e < 16; e++) acc[e] = (int)(int8_t)(tw[e >> 2] >> (8 * (e & 3)));
    }
    const uint4 *rec = reinterpret_cast<const uint4 *>(tape_dm + (size_t)demo * R * 16); // record j: x = u, y = v, z = w tokens
    const int ush = 8 * i;
    const uint32_t sh4 = (uint32_t)replay_shift * ONES4;
    auto replay = [&](const uint4 &q) { // acc -= u_i * v (x) w of one record
        // tokens -> int8 coefficients, four at a time (no borrow between bytes: token | 0x80 > shift), then one sign-
        // extending PRMT per coefficient
        const uint32_t cv = ((q.y | H4) - sh4) ^ H4, cw = ((q.z | H4) - sh4) ^ H4;
        const int nui = replay_shift - (int)((q.x >> ush) & 0xFFu);
        const int w[4] = {sext_byte<0>(cw), sext_byte<1>(cw), sext_byte<2>(cw), sext_byte<3>(cw)};
        const int v[4] = {sext_byte<0>(cv), sext_byte<1>(cv), sext_byte<2>(cv), sext_byte<3>(cv)};
#pragma unroll
        for (int jj = 0; jj < 4; jj++) {
            const int c = nui * v[jj];
#pragma unroll
            for (int k = 0; k < 4; k++) acc[4 * jj + k] += c * w[k];
        }
    };
    constexpr int RMAX = 8;
    uint4 qa; // the sample's own action
    if (R <= RMAX) {
        // every record of the demo in flight at once (the loads do not wait for each other, nor for the target row)
        uint4 q[RMAX];
#pragma unroll
        for (int j = 0; j < RMAX; j++) q[j] = (j < R && j >= a) ? __ldg(rec + j) : make_uint4(0, 0, 0, 0);
        qa = q[0];
#pragma unroll
        for (int j = 1; j < RMAX; j++) {
            if (j == a) qa = q[j];
            if (j > a && j < R) replay(q[j]);
        }
    } else {
        qa = __ldg(rec + a);
#pragma unroll 2
        for (int j = a + 1; j < R; j++) replay(__ldg(rec + j));
    }
    {
        float f[16];
#pragma unroll
        for (int e = 0; e < 16; e++) f[e] = (float)acc[e];
        put_row(st, f);
    }
    // ---- history slots: rank-1 tensors of the next actions, latest first
    const int hi = min(a + dim_t, R);
    for (int s = 1; s < dim_t; s++) {
        const int j = hi - s;
        float *row = st + (size_t)s * 64;
        if (j >= a + 1) {
            const uint4 q = __ldg(rec + j);
            const int ui = (int)((q.x >> ush) & 0xFFu) - replay_shift;
            float f[16];
#pragma unroll
            for (int jj = 0; jj < 4; jj++) {
                const int c = ui * ((int)((q.y >> (8 * jj)) & 0xFFu) - replay_shift);
#pragma unroll
                for (int k = 0; k < 4; k++) f[4 * jj + k] = (float)(c * ((int)((q.z >> (8 * k)) & 0xFFu) - replay_shift));
            }
            put_row(row, f);
        } else {
            put_row(row, zeros);
        }
    }
    if (i == 0) {
        scalars[b] = (float)(R - a);
        rewards[b] = -(float)(a + 1);
    }
    // the sample's own action: raw tokens; thread i writes tokens 3i .. 3i+2
#pragma unroll
    for (int x = 0; x < 3; x++) {
        const int qi = 3 * i + x;
        const uint32_t word = qi < 4 ? qa.x : (qi < 8 ? qa.y : qa.z);
        actions[b * 12 + qi] = (long long)((word >> (8 * (qi & 3))) & 0xFFu);
    }
}
} // namespace rows4

// step-major tape [R][N][TP] -> demo-major records [N][R][TP], 16 bytes per thread
__global__ void tape_to_demo_major_kernel(const uint4 *__restrict__ src, long long src_step_stride16, uint4 *__restrict__ dst,
                                          long long N, int R, int tp16) {
    const long long total = N * R * tp16;
    for (long long x = blockIdx.x * (long long)blockDim.x + threadIdx.x; x < total; x += (long long)gridDim.x * blockDim.x) {
        const int w = (int)(x % tp16);
        const long long nr = x / tp16;
        const int r = (int)(nr % R);
        const long long n = nr / R;
        dst[x] = __ldg(src + (size_t)r * src_step_stride16 + n * tp16 + w);
    }
}

// ------------------------------------------------------------------ K6
// get_rank (utils.py:134-140): sum over the S slices T[i,:,:] of the matrix rank.  The reference takes a float32 SVD;
// here the rank over Q is computed exactly: fraction-free elimination (row <- row*piv - row[c]*pivrow) over GF(p), one
// matrix per group of S lanes, lane = matrix row.  rank_p <= rank_Q.  With r the largest rank_p over primes p_1 .. p_k,
// rank_Q > r needs a non-zero (r+1) x (r+1) minor divisible by every p_j, i.e. one of size >= p_1 ... p_k > 2^(30 k)
// (primes 2^31 - c).  By Hadamard a minor is at most the product of the norms of its rows; a lane bounds its row's
// |row|^2 by 2^e (e = ceil(log2 |row|^2): <= 19 for int8, <= 35 for int16), so once the r+1 largest e of the slice sum
// to at most 60 k -- or r is the slice's count of non-zero rows -- r = rank_Q.  Until then the slice is eliminated again
// mod the next prime: one prime for the few-unit entries of most game states, up to eight for int8 extremes and
// fifteen (a product above 2^900 against r+1 largest e summing to at most 875) for int16 extremes at 25x25x25.
__constant__ uint32_t c_rank_c[15] = {1, 19, 61, 69, 85, 99, 105, 151, 159, 171, 225, 249, 295, 325, 379}; // p = 2^31 - c, all prime
template <typename T>
constexpr int RANK_PRIMES = sizeof(T) == 1 ? 8 : 15;

template <int S, typename T>
__device__ __forceinline__ int rank_mod_p(const T *__restrict__ src, bool live, int lane, uint32_t gmask, uint32_t P, uint32_t C) {
    uint32_t row[S];
#pragma unroll
    for (int c = 0; c < S; c++) {
        const int v = live ? src[c] : 0;
        row[c] = v >= 0 ? (uint32_t)v : P - (uint32_t)(-v);
    }
    bool used = !live;
    int rank = 0;
#pragma unroll
    for (int c = 0; c < S; c++) {
        const uint32_t cand = __ballot_sync(0xFFFFFFFFu, !used && row[c] != 0) & gmask;
        const bool has = cand != 0; // uniform within the group; all 32 lanes keep executing the same shuffles
        const int pl = has ? __ffs(cand) - 1 : lane;
        const uint32_t pv = __shfl_sync(0xFFFFFFFFu, row[c], pl);
        const uint32_t mine = row[c];
        const bool elim = has && !used && lane != pl && mine != 0;
        // columns <= c of the rows still in play are zero from here on: only k > c needs the update
        //   row[k] <- row[k] * pv - mine * pk  =  row[k] * pv + (P - mine) * pk   (mod P), one reduction for both products
        const uint32_t nmine = P - mine;
#pragma unroll
        for (int k = c + 1; k < S; k++) {
            const uint32_t pk = __shfl_sync(0xFFFFFFFFu, row[k], pl);
            if (elim) {
                // 2^31 = C (mod P): fold the bits above 31 twice, then one conditional subtraction (C < 2^9)
                const unsigned long long z = (unsigned long long)row[k] * pv + (unsigned long long)nmine * pk; // < 2^63
                unsigned long long r = (z & 0x7FFFFFFFull) + (z >> 31) * C;                                    // < 2^41
                uint32_t q = (uint32_t)(r & 0x7FFFFFFFull) + (uint32_t)(r >> 31) * C;                          // < P + 2^19
                row[k] = q >= P ? q - P : q;
            }
        }
        if (has && lane == pl) used = true;
        rank += has ? 1 : 0;
    }
    return rank;
}

template <int S, typename T>
__global__ void slice_rank_kernel(const T *__restrict__ slab, int32_t *__restrict__ ranks, long long B) {
    using G = Geo<S>;
    constexpr int LG = S;       // lanes per matrix: 4 / 9 / 16 (the shuffles address absolute lanes, so any group size works)
    constexpr int MPW = 32 / LG; // matrices per warp: 8 / 3 (lanes 27..31 idle; two per warp with groups of 16 was 1.5x slower) / 2
    const int lane = threadIdx.x & 31;
    const int sub = lane / LG, r = lane % LG;
    const long long warp = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    const long long mat = warp * MPW + sub; // matrix index = game * S + slice
    const long long game = mat / S;
    const int slice = (int)(mat - game * S);
    const bool live = sub < MPW && game < B && r < S;
    const T *src = slab + (live ? game * G::GP + slice * G::RP + r * S : 0);
    const uint32_t gmask = sub < MPW ? (((1u << LG) - 1u) << (sub * LG)) : 0u;
    int rank = rank_mod_p<S>(src, live, lane, gmask, 0x7FFFFFFFu, 1u);
    using N2 = std::conditional_t<sizeof(T) == 1, uint32_t, unsigned long long>;
    N2 n2 = 0; // |row|^2 <= 25 * 128^2 < 2^19 (int8), 25 * 2^30 < 2^35 (int16)
#pragma unroll
    for (int c = 0; c < S; c++) {
        const int v = live ? src[c] : 0;
        n2 += (N2)(v * v);
    }
    int e = 0; // |row|^2 <= 2^e
    if constexpr (sizeof(N2) == 4) e = n2 <= 1 ? 0 : 32 - __clz(n2 - 1);
    else e = n2 <= 1 ? 0 : 64 - __clzll((long long)(n2 - 1));
    const int emax = (int)__reduce_max_sync(0xFFFFFFFFu, (unsigned)e);
    const int nzrows = __popc(__ballot_sync(0xFFFFFFFFu, n2 != 0) & gmask);
    // sum of the m largest e of the group (sum over t of min(m, #{e >= t})): an m x m minor is at most 2^(that / 2)
    auto top_e = [&](int m) {
        int E = 0;
        for (int t = 1; t <= emax; t++) E += min(m, __popc(__ballot_sync(0xFFFFFFFFu, e >= t) & gmask));
        return E;
    };
    // rank_Q > r (the largest rank_p so far) needs a non-zero (r+1) x (r+1) minor that every prime so far divides: none
    // exists once the product of the primes (> 2^(30 j)) exceeds the minor's Hadamard bound, or once r = nzrows
    bool fin = rank == nzrows;
    if (!__all_sync(0xFFFFFFFFu, fin)) {
        const int E = top_e(rank + 1);
        fin = fin || E <= 60;
    }
#pragma unroll 1
    for (int j = 1; j < RANK_PRIMES<T> && !__all_sync(0xFFFFFFFFu, fin); j++) { // every lane runs the shuffles
        const int rj = rank_mod_p<S>(src, live, lane, gmask, 0x80000000u - c_rank_c[j], c_rank_c[j]);
        if (!fin) rank = max(rank, rj);
        const int E = top_e(rank + 1);
        fin = fin || rank == nzrows || E <= 60 * (j + 1);
    }
    // every lane of a group counted the same pivots; add the slices of a game
    if (live && r == 0) atomicAdd(&ranks[game], rank);
}

// ------------------------------------------------------------------ K7
// tg_state_key: the 64-bit state key of tg_common.cuh (key_const).
// key(T) = sum T[i][j][k] * A_i * B_j * C_k (mod 2^64).  One thread per word column of a game: its four entries of row i
// as unsigned offset-binary bytes (entry + 128) times the compile-time A_i go into four 64-bit accumulators (one wide
// and one 32-bit multiply-add per entry; the offset's share -128 sum_i A_i is their start value), which then meet the
// column's four B_j C_k (registers).  The WR partial sums of a game meet in shared memory -- no atomics, no table.
template <int S>
__global__ void __launch_bounds__(256) state_key_kernel(const int8_t *__restrict__ slab, unsigned long long *__restrict__ keys,
                                                        long long B) {
    using G = Geo<S>;
    constexpr int TG = 256 / G::WR; // games per pass of the CTA
    __shared__ unsigned long long s_ph[256];
    const int tid = threadIdx.x;
    const int gl = tid / G::WR, c = tid % G::WR;
    unsigned long long kb[4];
#pragma unroll
    for (int q = 0; q < 4; q++) {
        const int jk = 4 * c + q;
        kb[q] = jk < G::S2 ? key_const(0x2000, jk / S) * key_const(0x3000, jk % S) : 0ull;
    }
    unsigned long long a0 = 0;
#pragma unroll
    for (int i = 0; i < S; i++) a0 -= 128ull * key_const(0x1000, i);
    uint32_t w[S];
    auto fetch = [&](long long g0) { // this thread's word column of its game of the pass starting at g0 (zero state beyond B)
        const long long g = g0 + gl;
        if (gl < TG && g < B) {
            const uint32_t *col = reinterpret_cast<const uint32_t *>(slab + g * G::GP) + c;
#pragma unroll
            for (int i = 0; i < S; i++) w[i] = __ldg(col + i * G::WR) ^ 0x80808080u;
        } else {
#pragma unroll
            for (int i = 0; i < S; i++) w[i] = 0x80808080u;
        }
    };
    fetch((long long)blockIdx.x * TG);
    for (long long g0 = (long long)blockIdx.x * TG; g0 < B; g0 += (long long)gridDim.x * TG) {
        unsigned long long acc[4] = {a0, a0, a0, a0};
#pragma unroll
        for (int i = 0; i < S; i++) {
#pragma unroll
            for (int q = 0; q < 4; q++) acc[q] += (unsigned long long)((w[i] >> (8 * q)) & 0xFFu) * key_const(0x1000, i);
        }
        const unsigned long long h = acc[0] * kb[0] + acc[1] * kb[1] + acc[2] * kb[2] + acc[3] * kb[3];
        fetch(g0 + (long long)gridDim.x * TG); // the next pass's loads fly over this pass's reduction
        s_ph[tid] = h;
        __syncthreads();
        if constexpr (G::WR <= 32) {
            if (tid < TG && g0 + tid < B) {
                unsigned long long k = 0;
#pragma unroll
                for (int x = 0; x < G::WR; x++) k += s_ph[tid * G::WR + x];
                keys[g0 + tid] = k;
            }
        } else if constexpr (G::WR > 64) { // S = 25: one game per pass (157 partial sums), reduced by warp 0
            static_assert(TG == 1, "one game per pass");
            if (tid < 32 && g0 < B) {
                unsigned long long k = 0;
                for (int x = tid; x < G::WR; x += 32) k += s_ph[x];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) k += __shfl_xor_sync(0xFFFFFFFFu, k, o);
                if (tid == 0) keys[g0] = k;
            }
        } else { // S = 16: 64 partial sums per game, one warp per game
            static_assert(G::WR <= 32 || (G::WR == 64 && TG <= 8), "warp-per-game reduction");
            const int wp = tid >> 5, ln = tid & 31;
            if (wp < TG && g0 + wp < B) {
                unsigned long long k = s_ph[wp * 64 + ln] + s_ph[wp * 64 + 32 + ln];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) k += __shfl_xor_sync(0xFFFFFFFFu, k, o);
                if (ln == 0) keys[g0 + wp] = k;
            }
        }
        __syncthreads();
    }
}

template <int S, bool P16, bool STG>
static int launch_demo_sample_variant(unsigned grid, size_t smem, const uint8_t *tape, long long tape_step_stride, const int8_t *slab,
                                      long long N, int R, int dim_t, int replay_shift, const long long *idx, long long nb,
                                      float *states, float *scalars, long long *actions, float *rewards, cudaStream_t st) {
    auto kern = demo_sample_kernel<S, P16, STG>;
    if (STG) TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, 128, STG ? smem : 0, st>>>(tape, tape_step_stride, slab, N, R, dim_t, replay_shift, idx, nb, states, scalars,
                                            actions, rewards);
    return TG_OK;
}

template <int S>
static int launch_demo_sample(const uint8_t *tape, long long tape_step_stride, const int8_t *slab, long long N, int R, int dim_t,
                              int replay_shift, const long long *idx, long long nb, float *states, float *scalars,
                              long long *actions, float *rewards, bool pack16, cudaStream_t st) {
    using G = Geo<S>;
    const unsigned grid = (unsigned)((nb * G::WR + 127) / 128);
    // staging needs 16-byte aligned records and room for the records of every sample a CTA touches
    const long long smem = ((128 + G::WR - 1) / G::WR + 1) * (long long)R * G::TP;
    const bool stage = (((uintptr_t)tape | (uintptr_t)tape_step_stride) & 15) == 0 && smem <= 64 * 1024;
#define TG_ARGS grid, (size_t)smem, tape, tape_step_stride, slab, N, R, dim_t, replay_shift, idx, nb, states, scalars, actions, rewards, st
    if (pack16) return stage ? launch_demo_sample_variant<S, true, true>(TG_ARGS) : launch_demo_sample_variant<S, true, false>(TG_ARGS);
    return stage ? launch_demo_sample_variant<S, false, true>(TG_ARGS) : launch_demo_sample_variant<S, false, false>(TG_ARGS);
#undef TG_ARGS
}

template <int S, bool T16, bool P16>
static int launch_demo_sample_dm_variant(const uint8_t *tape_dm, const uint8_t *targets, long long N, int R, int dim_t, int replay_shift,
                                         const long long *idx, long long nb, float *states, float *scalars, long long *actions,
                                         float *rewards, cudaStream_t st) {
    using C = SampleCfg<S>;
    const long long smem = C::smem_bytes(R, dim_t, T16);
    if (smem > 227 * 1024) return TG_E_ARG;
    const unsigned grid = (unsigned)((nb + C::SPC - 1) / C::SPC);
    auto kern = demo_sample_dm_kernel<S, T16, P16>;
    TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, C::NT, (size_t)smem, st>>>(tape_dm, targets, N, R, dim_t, replay_shift, idx, nb, states, scalars, actions, rewards);
    return TG_OK;
}

template <int S>
static int launch_demo_sample_dm(const uint8_t *tape_dm, const uint8_t *targets, bool t16, bool p16, long long N, int R, int dim_t,
                                 int replay_shift, const long long *idx, long long nb, float *states, float *scalars,
                                 long long *actions, float *rewards, cudaStream_t st) {
#define TG_ARGS tape_dm, targets, N, R, dim_t, replay_shift, idx, nb, states, scalars, actions, rewards, st
    if (t16) return p16 ? launch_demo_sample_dm_variant<S, true, true>(TG_ARGS) : launch_demo_sample_dm_variant<S, true, false>(TG_ARGS);
    return p16 ? launch_demo_sample_dm_variant<S, false, true>(TG_ARGS) : launch_demo_sample_dm_variant<S, false, false>(TG_ARGS);
#undef TG_ARGS
}

} // namespace tg

namespace tg {
// Work counters of the persistent batcher: static device memory (the library allocates nothing), one slot per launch, handed
// out round robin per device.  A slot is zeroed on the launch's stream right before the kernel; its event (recorded after
// the kernel) keeps a later launch that comes round to the same slot from zeroing it while the earlier one still runs.
constexpr int TICKET_SLOTS = 64, TICKET_MAXDEV = 64;
__device__ unsigned long long g_tickets[TICKET_SLOTS];
static cudaEvent_t g_ticket_done[TICKET_MAXDEV][TICKET_SLOTS];
static unsigned g_ticket_next[TICKET_MAXDEV];
static std::mutex g_ticket_mu;
static int ticket_acquire(cudaStream_t st, unsigned long long **ticket, cudaEvent_t *done) {
    int dev = 0;
    TG_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= TICKET_MAXDEV) return TG_E_ARG;
    unsigned long long *base = nullptr;
    TG_CUDA(cudaGetSymbolAddress(reinterpret_cast<void **>(&base), g_tickets));
    std::lock_guard<std::mutex> lock(g_ticket_mu);
    const int slot = (int)(g_ticket_next[dev]++ % TICKET_SLOTS);
    cudaEvent_t &ev = g_ticket_done[dev][slot];
    if (!ev) TG_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    else TG_CUDA(cudaStreamWaitEvent(st, ev, 0));
    TG_CUDA(cudaMemsetAsync(base + slot, 0, sizeof(unsigned long long), st));
    *ticket = base + slot, *done = ev;
    return TG_OK;
}
} // namespace tg

extern "C" {

int tg_demo_sample(const uint8_t *tape, int64_t tape_step_stride, const int8_t *slab, int64_t N, int R, int S, int dim_t,
                   int replay_shift, const int64_t *idx, int64_t nb, float *states, float *scalars, int64_t *actions,
                   float *rewards, void *stream) {
    const int rc = tg::check_demo_sample(S, N, R, dim_t, 0, nb, false, replay_shift, tape, slab, idx, states, scalars, actions, rewards);
    if (rc != tg::LAUNCH) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    // tokens are <= 2 * 4 (tape contract), so |coefficient| <= cmax; the 16-bit packed head is exact while
    // 127 + R * cmax^3 fits an int16 lane
    const long long cmax = replay_shift > 8 - replay_shift ? replay_shift : 8 - replay_shift;
    const bool pack16 = replay_shift >= 0 && replay_shift <= 8 && 127 + (long long)R * cmax * cmax * cmax <= 32767;
    return tg::with_S(S, [&](auto s) {
        constexpr int kS = decltype(s)::value;
        const int rc = tg::launch_demo_sample<kS>(tape, tape_step_stride, slab, N, R, dim_t, replay_shift, (const long long *)idx, nb,
                                                  states, scalars, (long long *)actions, rewards, pack16, st);
        if (rc != TG_OK) return rc;
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    });
}

int tg_demo_sample_dm(const uint8_t *tape_dm, const void *targets, int targets_i16, int target_bound, int64_t N, int R, int S,
                      int dim_t, int replay_shift, const int64_t *idx, int64_t nb, float *states, float *scalars, int64_t *actions,
                      float *rewards, void *stream) {
    const int rc = tg::check_demo_sample(S, N, R, dim_t, target_bound, nb, true, replay_shift, tape_dm, targets, idx, states, scalars,
                                         actions, rewards);
    if (rc != tg::LAUNCH) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    // tokens are <= 8 (tape contract), so |coefficient| <= cmax; the 16-bit packed head is exact while
    // target_bound + R * cmax^3 fits an int16 lane
    const long long cmax = replay_shift > 8 - replay_shift ? replay_shift : 8 - replay_shift;
    const bool pack16 = (long long)target_bound + (long long)R * cmax * cmax * cmax <= 32767;
    return tg::with_S(S, [&](auto s) {
        constexpr int kS = decltype(s)::value;
        if constexpr (kS == 4) { // one thread per (sample, row), exact int32 (any target bound)
            auto kern = targets_i16 ? tg::rows4::demo_sample_rows4_kernel<true> : tg::rows4::demo_sample_rows4_kernel<false>;
            kern<<<(unsigned)((nb * 4 + 127) / 128), 128, 0, st>>>(tape_dm, (const uint8_t *)targets, N, R, dim_t, replay_shift,
                                                                   (const long long *)idx, nb, states, scalars, (long long *)actions, rewards);
        } else if constexpr (kS == 25) { // one CTA per sample, states straight from the registers
            const long long smem = (long long)R * tg::Geo<25>::TP;
            if (smem > 227 * 1024 || nb > 0x7FFFFFFFLL) return TG_E_ARG;
            auto kern = targets_i16 ? (pack16 ? tg::demo_sample_dm25_kernel<true, true> : tg::demo_sample_dm25_kernel<true, false>)
                                    : (pack16 ? tg::demo_sample_dm25_kernel<false, true> : tg::demo_sample_dm25_kernel<false, false>);
            TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            kern<<<(unsigned)nb, 160, (size_t)smem, st>>>(tape_dm, (const uint8_t *)targets, N, R, dim_t, replay_shift, (const long long *)idx,
                                                         states, scalars, (long long *)actions, rewards);
        } else if (kS == 9 && pack16 && (long long)tg::rows9::WARPS * tg::rows9::warp_bytes(R) <= 200 * 1024) {
            // 9x9x9: one thread per (sample, row), three samples per warp
            const int smem = tg::rows9::WARPS * tg::rows9::warp_bytes(R);
            const long long per_cta = (long long)tg::rows9::WARPS * tg::rows9::SPW;
            const long long want = (nb + per_cta - 1) / per_cta;
            const unsigned grid = (unsigned)(want < 148 * 4 ? want : 148 * 4); // persistent warps: four CTAs per SM
            unsigned long long *ticket = nullptr;
            cudaEvent_t done = nullptr;
            if (const int trc = tg::ticket_acquire(st, &ticket, &done); trc != TG_OK) return trc;
            auto kern = targets_i16 ? tg::rows9::demo_sample_rows9_kernel<true, true> : tg::rows9::demo_sample_rows9_kernel<false, true>;
            TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
            kern<<<grid, 32 * tg::rows9::WARPS, smem, st>>>(tape_dm, (const uint8_t *)targets, N, R, dim_t, replay_shift, (const long long *)idx,
                                                            nb, states, scalars, (long long *)actions, rewards, ticket);
            TG_CUDA(cudaGetLastError());
            TG_CUDA(cudaEventRecord(done, st));
            return TG_OK;
        } else {
            const int lrc = tg::launch_demo_sample_dm<kS>(tape_dm, (const uint8_t *)targets, targets_i16 != 0, pack16, N, R, dim_t,
                                                          replay_shift, (const long long *)idx, nb, states, scalars, (long long *)actions,
                                                          rewards, st);
            if (lrc != TG_OK) return lrc;
        }
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    });
}

int tg_tape_to_demo_major(const uint8_t *tape, int64_t tape_step_stride, uint8_t *tape_dm, int64_t N, int R, int S, void *stream) {
    if (const int rc = tg::check_tape_to_demo_major(S, N, R, tape, tape_step_stride, tape_dm); rc != tg::LAUNCH) return rc;
    const int tp16 = ((3 * S + 15) & ~15) / 16;
    const long long total = N * R * tp16;
    const long long blocks = (total + 255) / 256;
    tg::tape_to_demo_major_kernel<<<(unsigned)(blocks < 148 * 32 ? blocks : 148 * 32), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const uint4 *>(tape), tape_step_stride / 16, reinterpret_cast<uint4 *>(tape_dm), N, R, tp16);
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

int tg_slice_rank(const int8_t *slab, int32_t *ranks, int64_t B, int S, void *stream) {
    if (const int rc = tg::check_pair(S, B, slab, 16, ranks, 1); rc != tg::LAUNCH) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    TG_CUDA(cudaMemsetAsync(ranks, 0, (size_t)B * 4, st));
    return tg::with_S(S, [&](auto s) {
        constexpr int kS = decltype(s)::value;
        const long long warps = (B * kS + (32 / kS) - 1) / (32 / kS);
        tg::slice_rank_kernel<kS><<<(unsigned)((warps * 32 + 127) / 128), 128, 0, st>>>(slab, ranks, B);
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    });
}

int tg_slice_rank_i16(const int16_t *slab16, int32_t *ranks, int64_t B, int S, void *stream) {
    if (const int rc = tg::check_pair(S, B, slab16, 16, ranks, 1); rc != tg::LAUNCH) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    TG_CUDA(cudaMemsetAsync(ranks, 0, (size_t)B * 4, st));
    return tg::with_S(S, [&](auto s) {
        constexpr int kS = decltype(s)::value;
        const long long warps = (B * kS + (32 / kS) - 1) / (32 / kS);
        tg::slice_rank_kernel<kS><<<(unsigned)((warps * 32 + 127) / 128), 128, 0, st>>>(slab16, ranks, B);
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    });
}

int tg_state_key(const int8_t *slab, uint64_t *keys, int64_t B, int S, void *stream) {
    if (const int rc = tg::check_pair(S, B, slab, 16, keys, 1); rc != tg::LAUNCH) return rc;
    return tg::with_S(S, [&](auto s) {
        constexpr int kS = decltype(s)::value;
        const long long tiles = (B + (256 / tg::Geo<kS>::WR) - 1) / (256 / tg::Geo<kS>::WR);
        tg::state_key_kernel<kS><<<(unsigned)(tiles < 148 * 16 ? tiles : 148 * 16), 256, 0, (cudaStream_t)stream>>>(
            slab, (unsigned long long *)keys, B);
        TG_CUDA(cudaGetLastError());
        return TG_OK;
    });
}

} // extern "C"
