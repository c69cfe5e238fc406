// tg_demo_tc.cu -- K3t: the target tensor of a 16x16x16 action list on the 5th-generation tensor cores
// (tcgen05.mma kind::i8, accumulators in TMEM): the experimental entry point tg_demo_accumulate_tc (S = 16, R <= 64).
// tg_demo_accumulate / tg_demo_gen_philox use the mma.sync f16 kernel of tg_demo_mma.cu instead, which is 1.5x faster
// than this one (profiles/README.md).
//
// Reference restated: target = sum_r u_r (x) v_r (x) w_r (utils.py:40-53 uvw_to_demo, utils.py:232,
// datasets.py:141).  As a GEMM per demo:
//     T[(i,j)][k] = sum_r  KR[r][(i,j)] * W[r][k],      KR[r][(i,j)] = u_r[i] * v_r[j]      (Khatri-Rao rows)
// with M = (i,j) = 256 (two 128-row MMAs, no padding), N = k = 16, K = r padded to 32 or 64.  Row (i,j) of the
// result is the 16 contiguous bytes i*256 + j*16 of the slab, so TMEM lane m of the accumulator IS slab row m.
// Both operands are "MN-major" in shared memory (canonical no-swizzle layout: 8 K-rows x 16 bytes per core matrix),
// which is exactly how the data is produced: one action r gives sixteen 16-byte rows of KR (u_i * pack(v), one
// packed IMAD per four entries) and one 16-byte row of W (its w coefficients) -- no transposition anywhere.
// (An M = i formulation pads 16 rows to 64 and needs 256 TMEM columns per demo; it was measured slower.)
//
// STATUS: experimental.  Bit-exact against the packed-IMAD path for every R <= 64, but only 1.3x faster (0.23 ms vs
// 0.30 ms for 65536 demos, R = 49): with MN-major no-swizzle int8 operands each tcgen05.mma costs ~350 cycles whatever its
// size, so the four MMAs of a demo pace the CTA at ~1450 cycles per demo (profiles/README.md).  This entry point stays for
// tests and profiling.
//
// Warp-specialised CTA, rings of mbarriers (no CTA-wide barrier in the loop):
//   producers (8 warps): thread (r, quarter) turns action r of the demo (tape rows prefetched from HBM one demo
//      ahead) into operand rows of a free operand stage;
//   MMA warp: per demo 2 x K/32 tcgen05.mma (128 x 16 x 32, int8 -> int32 in TMEM, 32 columns per demo);
//   consumers (8 warps): tcgen05.ld 16 columns of their 32 lanes, saturate to int8, range-test, one 16-byte store
//      per lane: a warp writes 512 contiguous bytes of the slab.

#include "tg_common.cuh"

namespace tg {

namespace tc {

#ifdef TG_TC_DEBUG
__device__ unsigned long long g_dbg[16];
#define DBG_T0 long long _t0 = clock64();
#define DBG_ADD(i) dbg_acc[i] += clock64() - _t0;
#else
#define DBG_T0
#define DBG_ADD(i)
#endif

constexpr int S = 16;
constexpr int NT = 256;                 // producer threads (8 warps); as many consumers
constexpr int NT_ALL = 2 * NT + 32;     // producers + consumers + the MMA warp
constexpr int A_BYTES = 8 * 128;        // W operand: 8 K-groups of 8 rows x 16 bytes (k = 0..15)
constexpr int B_BYTES = 8 * 16 * 128;   // KR operand: 8 K-groups x 16 chunks (i) x (8 rows x 16 bytes (j))
constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
#ifndef TG_TC_DEPTH
#define TG_TC_DEPTH 2
#endif
constexpr int DEPTH = TG_TC_DEPTH;      // demos the tensor core runs ahead of the epilogue
constexpr int OPST = DEPTH + 1;         // operand stages
constexpr int TMST = 4;                 // accumulator stages of 32 TMEM columns
constexpr int ACC_COLS = 32;            // two 128 x 16 accumulators per demo
constexpr int CTAS_BY_THREADS = 2; // 544 threads x ~50 registers: two CTAs per SM
constexpr int CTAS_BY_SMEM = 227 * 1024 / (OPST * (8 * 128 + 8 * 16 * 128) + 1024);
constexpr int CTAS_PER_SM = CTAS_BY_SMEM < CTAS_BY_THREADS ? CTAS_BY_SMEM : CTAS_BY_THREADS;
constexpr int SMEM_BYTES = OPST * STAGE_BYTES + 128;
constexpr int TMEM_COLS = ACC_COLS * TMST;

__device__ __forceinline__ uint64_t smem_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    // UMMA shared-memory descriptor, no swizzle: start address, leading (K-group) and stride (MN-chunk) byte offsets in
    // 16-byte units, descriptor version 1 (sm_100)
    return (uint64_t)((addr >> 4) & 0x3FFFu) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}
// kind::i8 instruction descriptor: D = s32, A = B = signed int8, both MN-major, M = 128, N = 16
constexpr uint32_t IDESC = (2u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((16u >> 3) << 17) | ((128u >> 4) << 24);

__device__ __forceinline__ void mma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(IDESC), "r"(accumulate), "r"(0u)
        : "memory");
}
// the same with a disable-output-lane mask (one word per 32 TMEM lanes, bit set = lane not written)
__device__ __forceinline__ void mma_i8_q(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate, uint32_t m0,
                                         uint32_t m1, uint32_t m2, uint32_t m3) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(IDESC), "r"(accumulate), "r"(m0), "r"(m1), "r"(m2), "r"(m3)
        : "memory");
}
__device__ __forceinline__ void mma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// one lane of a converged warp (the compiler knows the result is warp-uniform single-lane: no per-lane loops around
// the uniform-datapath tensor instructions)
__device__ __forceinline__ bool elect_one() {
    uint32_t p;
    asm volatile("{\n.reg .pred P;\nelect.sync _|P, 0xffffffff;\nselp.b32 %0, 1, 0, P;\n}" : "=r"(p));
    return p != 0;
}
__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// two s32 -> saturated s8 pair in the low half, c's low half moved to the high half
__device__ __forceinline__ uint32_t pack_sat(int a, int b, uint32_t c) {
    uint32_t d;
    asm("cvt.pack.sat.s8.s32.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(b), "r"(a), "r"(c));
    return d;
}

struct Action { // the token words of one action that a (r, quarter) thread needs
    uint4 v, w;
    uint32_t u;
};

__device__ __forceinline__ Action load_action(const uint8_t *rec, int quarter) {
    Action a;
    a.v = *reinterpret_cast<const uint4 *>(rec + 16);
    a.u = *reinterpret_cast<const uint32_t *>(rec + 4 * quarter);
    a.w = quarter == 0 ? *reinterpret_cast<const uint4 *>(rec + 32) : make_uint4(0, 0, 0, 0);
    return a;
}

// action r -> four of the sixteen 16-byte rows of KR (i = 4*quarter .. +3: u_i * pack(v)) and, for quarter 0, the
// 16-byte row of W (the w coefficients)
__device__ __forceinline__ void expand_action(const Action &a, int r, int quarter, uint32_t sh4, int shift, uint8_t *s_w,
                                              uint8_t *s_kr) {
    const uint32_t vt[4] = {a.v.x, a.v.y, a.v.z, a.v.w};
    int32_t vp[4]; // pack(v) in integer form: sum_b (v_b - shift) 256^b
#pragma unroll
    for (int m = 0; m < 4; m++) vp[m] = (int32_t)(vt[m] - sh4);
    uint8_t *krow = s_kr + (r >> 3) * 2048 + (4 * quarter) * 128 + (r & 7) * 16;
#pragma unroll
    for (int ii = 0; ii < 4; ii++) {
        const int ui = (int)((a.u >> (8 * ii)) & 0xFFu) - shift;
        uint4 o;
        o.x = ((uint32_t)(ui * vp[0]) + H4) ^ H4; // integer form -> two's complement bytes
        o.y = ((uint32_t)(ui * vp[1]) + H4) ^ H4;
        o.z = ((uint32_t)(ui * vp[2]) + H4) ^ H4;
        o.w = ((uint32_t)(ui * vp[3]) + H4) ^ H4;
        *reinterpret_cast<uint4 *>(krow + ii * 128) = o;
    }
    if (quarter == 0) {
        uint4 o;
        o.x = ((a.w.x | H4) - sh4) ^ H4;
        o.y = ((a.w.y | H4) - sh4) ^ H4;
        o.z = ((a.w.z | H4) - sh4) ^ H4;
        o.w = ((a.w.w | H4) - sh4) ^ H4;
        *reinterpret_cast<uint4 *>(s_w + (r >> 3) * 128 + (r & 7) * 16) = o;
    }
}

// mbarrier operations on precomputed 32-bit shared addresses (keeps the address arithmetic out of the loop)
__device__ __forceinline__ void mbar_arrive_a(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait_a(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(bar),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void mma_commit_a(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// Warp roles: warps 0..7 producers (expand), warps 8..15 consumers (epilogue), warp 16 issues the MMAs.  Rings of
// mbarriers, no CTA-wide barrier in the loop.  For demo `it` of the CTA (operand stage op = it % OPST, accumulator
// stage tm = it % TMST):
//   producers: wait opfree[op] (MMAs of demo it-OPST done)     -> expand -> proxy fence -> arrive ready[op]
//   MMA warp : wait ready[op], wait tmfree[tm] (epilogue it-TMST) -> NQ x K/32 MMAs -> commit full[tm], opfree[op]
//   consumers: wait full[tm] -> tcgen05.ld -> arrive tmfree[tm]  -> saturate, range test, store to HBM
// Producers never store to global memory, so their proxy fence (a CTA-scope memory barrier under the hood) waits only
// for their own shared-memory writes.
__global__ void __launch_bounds__(NT_ALL) demo_tc_kernel(const uint8_t *__restrict__ tape, long long tape_step_stride,
                                                         long long N, int R, int shift, int8_t *__restrict__ slab,
                                                         uint8_t *__restrict__ flags) {
    using G = Geo<S>;
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t *s_op = smem; // OPST operand stages, each A (1 KB) then B (16 KB)
    uint64_t *s_full = reinterpret_cast<uint64_t *>(smem + OPST * STAGE_BYTES); // [TMST] accumulator stage written
    uint64_t *s_tmfree = s_full + TMST;                                          // [TMST] accumulator stage read
    uint64_t *s_ready = s_tmfree + TMST;                                         // [OPST] operand stage written
    uint64_t *s_opfree = s_ready + OPST;                                         // [OPST] operand stage consumed
    uint32_t *s_tmem = reinterpret_cast<uint32_t *>(s_opfree + OPST);

#ifdef TG_TC_DEBUG
    long long dbg_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#endif
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)), "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 0) {
        for (int i = 0; i < TMST; i++) mbar_init(&s_full[i], 1), mbar_init(&s_tmfree[i], NT / 32);
        for (int i = 0; i < OPST; i++) mbar_init(&s_ready[i], NT / 32), mbar_init(&s_opfree[i], 1);
        mbar_fence_init();
    }
    // rows r >= R of the W operands stay zero for the whole kernel: they cancel whatever the KR rows r >= R hold
    for (int st = 0; st < OPST; st++)
        for (int w = tid; w < A_BYTES / 4; w += NT_ALL) reinterpret_cast<uint32_t *>(s_op + st * STAGE_BYTES)[w] = 0;
    fence_proxy_async();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem = *s_tmem;
    const uint32_t a_full = smem_u32(s_full), a_tmfree = smem_u32(s_tmfree), a_ready = smem_u32(s_ready),
                   a_opfree = smem_u32(s_opfree), a_op = smem_u32(s_op);
    const int ksteps = (R + 31) >> 5;
    const long long step = gridDim.x, d0 = blockIdx.x;
    const int niter = d0 < N ? (int)((N - d0 + step - 1) / step) : 0;

    if (warp == 2 * (NT / 32)) {
        // ---------------- MMA warp: T[(i,j)][k] for i < 8 into columns tm*32 .. +15, for i >= 8 into the next 16
        for (int it = 0; it < niter; it++) {
            const int op = it % OPST, tm = it & (TMST - 1);
            { DBG_T0 mbar_wait_a(a_ready + 8 * op, (uint32_t)(it / OPST) & 1u); DBG_ADD(0) }
            { DBG_T0 if (it >= TMST) mbar_wait_a(a_tmfree + 8 * tm, (uint32_t)(it / TMST - 1) & 1u); DBG_ADD(1) }
            fence_after_sync();
            DBG_T0
            if (elect_one()) {
                const uint32_t base = a_op + op * STAGE_BYTES;
                const uint64_t wdesc = smem_desc(base, 128, 0);                 // B operand: W, one 16-column chunk
                const uint64_t krdesc = smem_desc(base + A_BYTES, 2048, 128);   // A operand: KR, chunk i at + i*128
#pragma unroll
                for (int half = 0; half < 2; half++)
                    for (int ks = 0; ks < ksteps; ks++) // 32 actions = 4 K-groups per instruction
                        mma_i8_q(tmem + tm * ACC_COLS + 16 * half, krdesc + (uint64_t)((ks * 4 * 2048 + half * 8 * 128) >> 4),
                                 wdesc + (uint64_t)((ks * 4 * 128) >> 4), ks > 0, 0u, 0u, 0u, 0u);
                mma_commit_a(a_full + 8 * tm);
                mma_commit_a(a_opfree + 8 * op);
            }
            __syncwarp();
            DBG_ADD(2)
        }
    } else if (warp < NT / 32) {
        // ---------------- producers.  expand task: action r = tid % 64, j quarter = tid / 64
        const uint32_t sh4 = (uint32_t)shift * ONES4;
        const int r = tid & 63, quarter = tid >> 6;
        const bool expander = r < R;
        const long long rec_step = step * G::TP;
        const uint8_t *rec = tape + (size_t)(expander ? r : 0) * tape_step_stride + d0 * G::TP; // next tape row to load
        Action cur, nxt;
        if (expander && niter > 0) nxt = load_action(rec, quarter);
        rec += rec_step;
        for (int it = 0; it < niter; it++) {
            const int op = it % OPST;
            cur = nxt;
            if (expander && it + 1 < niter) nxt = load_action(rec, quarter); // consumed one iteration later
            rec += rec_step;
            { DBG_T0 if (it >= OPST) mbar_wait_a(a_opfree + 8 * op, (uint32_t)(it / OPST - 1) & 1u); DBG_ADD(3) }
            uint8_t *st = s_op + op * STAGE_BYTES;
            { DBG_T0
            if (expander) expand_action(cur, r, quarter, sh4, shift, st, st + A_BYTES);
            DBG_ADD(4) }
            { DBG_T0
            fence_proxy_async(); // generic-proxy writes -> visible to the tensor core (async proxy)
            __syncwarp();
            DBG_ADD(5) }
            if (lane == 0) mbar_arrive_a(a_ready + 8 * op);
        }
    } else {
        // ---------------- consumers: warp w reads its 32 lanes (slab rows 32 (w & 3) + lane of half w >> 2)
        const int w = warp - NT / 32;
        const int row = 128 * (w >> 2) + 32 * (w & 3) + lane; // (i, j) = (row / 16, row % 16)
        int8_t *out = slab + d0 * G::GP + row * 16;
        uint8_t *fl = flags ? flags + d0 : nullptr;
        for (int it = 0; it < niter; it++, out += step * G::GP, fl += fl ? step : 0) {
            const int tm = it & (TMST - 1);
            { DBG_T0 mbar_wait_a(a_full + 8 * tm, (uint32_t)(it / TMST) & 1u); DBG_ADD(6) }
            fence_after_sync();
            DBG_T0
            uint32_t v[16];
            const uint32_t taddr = tmem + ((uint32_t)(32 * (w & 3)) << 16) + (uint32_t)(tm * ACC_COLS + 16 * (w >> 2));
            asm volatile(
                "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
                : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
                  "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                : "r"(taddr));
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            DBG_ADD(7)
            fence_before_sync(); // the loads are done: hand the accumulator stage back
            __syncwarp();
            if (lane == 0) mbar_arrive_a(a_tmfree + 8 * tm);
            uint32_t words[4], bad = 0;
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const uint32_t hi = pack_sat((int)v[4 * q + 2], (int)v[4 * q + 3], 0u);
                const uint32_t t = pack_sat((int)v[4 * q], (int)v[4 * q + 1], hi);
                bad |= (t ^ (t << 1)) & H4;
                words[q] = t;
            }
            *reinterpret_cast<uint4 *>(out) = make_uint4(words[0], words[1], words[2], words[3]);
            if (bad && fl) *fl = (uint8_t)TG_FLAG_RANGE; // every writer stores the same byte over the zeroed array
        }
    }
#ifdef TG_TC_DEBUG
    if (lane == 0)
        for (int i = 0; i < 8; i++)
            if (dbg_acc[i]) atomicAdd(&g_dbg[i], (unsigned long long)dbg_acc[i]);
#endif
    fence_before_sync();
    __syncthreads();
    if (warp == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(TMEM_COLS) : "memory");
}

} // namespace tc

// slab[n] = sum_r rank1(tape[r][n]) for S = 16, R <= 64 on the tensor cores
int launch_demo_tc(const uint8_t *tape, long long stride, long long N, int R, int shift, int8_t *slab, uint8_t *flags,
                   cudaStream_t st) {
    if (R < 1 || R > 64) return TG_E_ARG;
    auto kern = tc::demo_tc_kernel;
    TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::SMEM_BYTES));
    int per_sm = tc::CTAS_PER_SM; // limited by threads and shared memory
#ifdef TG_TUNING
    if (tuning_env("TG_TC_CTAS", 0) > 0) per_sm = tuning_env("TG_TC_CTAS", 0);
#endif
    const long long grid = N < 148 * per_sm ? N : 148 * per_sm;
    // the kernel only ever SETS flag bytes
    if (flags) TG_CUDA(cudaMemsetAsync(flags, 0, (size_t)N, st));
    kern<<<(int)grid, tc::NT_ALL, tc::SMEM_BYTES, st>>>(tape, stride, N, R, shift, slab, flags);
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

} // namespace tg

#ifdef TG_TC_DEBUG
extern "C" int tg_debug_tc(unsigned long long *out, int reset) {
    if (reset) { unsigned long long z[16] = {0}; cudaMemcpyToSymbol(tg::tc::g_dbg, z, sizeof(z)); return 0; }
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out, tg::tc::g_dbg, 16 * 8);
    return 0;
}
#endif

extern "C" int tg_demo_accumulate_tc(const uint8_t *tape, int64_t tape_step_stride, int64_t N, int R, int S, int shift,
                                     int8_t *slab, uint8_t *flags, void *stream) {
    if (R > 64) return TG_E_ARG; // the MMA's K dimension is the demo's R terms, padded to 32 or 64
    if (const int rc = tg::check_accumulate(S == 16, N, R, shift, 1, 4, tape, tape_step_stride, slab); rc != tg::LAUNCH) return rc;
    return tg::launch_demo_tc(tape, tape_step_stride, N, R, shift, slab, flags, (cudaStream_t)stream);
}
