// tg_common.cuh -- shared device helpers for the TensorGame kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "../../include/tensorgame.h"

namespace tg {

// ---------------------------------------------------------------- geometry
// Device slab: int8 [B][GP]; entry (i,j,k) at i*RP + j*S + k.  One 32-bit word
// holds four consecutive (j,k) entries of one i-row, so the rank-1 update of a
// word is  u_i * pack(v_j w_k)  -- one IMAD per word (see tg_step.cuh).
template <int S>
struct Geo {
    static constexpr int S2 = S * S;
    static constexpr int S3 = S2 * S;
    static constexpr int RP = (S2 + 3) & ~3;       // row pitch (bytes)
    static constexpr int WR = RP / 4;              // 32-bit words per row
    static constexpr int GP = (S * RP + 15) & ~15; // game pitch (bytes)
    static constexpr int TP = (3 * S + 15) & ~15;  // token pitch (bytes)
    static constexpr bool STRADDLE = (S % 4) != 0; // a word can span two j
};

// the game path (layout, conversions, step, expansion, rollout, keys, ranks, demos, samples, host buffers)
__host__ __device__ constexpr bool supported_S(int S) { return S == 4 || S == 9 || S == 16 || S == 25; }
// change of basis (tg_change_of_basis*, tg_sample_unimodular): kernels specialised per size, not built for 25x25x25
__host__ __device__ constexpr bool basis_supported_S(int S) { return S == 4 || S == 9 || S == 16; }

extern int g_last_cuda_error;

// Kernel variants for tuning sweeps exist only in the -DTG_TUNING build (libtensorgame_b200_tuning.so, selected with
// TG_TUNING=1 by mat_mul_b200/_lib.py): there an environment variable picks the variant; the production library compiles
// the measured-best path alone and reads no environment.
#ifdef TG_TUNING
}
#include <cstdlib>
namespace tg {
inline int tuning_env(const char *name, int dflt) {
    const char *e = getenv(name);
    return e ? atoi(e) : dflt;
}
#endif

inline int cuda_fail(cudaError_t e) {
    g_last_cuda_error = (int)e;
    return TG_E_CUDA;
}
#define TG_CUDA(call)                                  \
    do {                                               \
        cudaError_t _e = (call);                       \
        if (_e != cudaSuccess) return tg::cuda_fail(_e); \
    } while (0)

// multiprocessors of the current device (148 if the runtime cannot tell), cached per device
int sm_count();

// f(std::integral_constant<int, S>{}) for a game-path size, TG_E_ARG for any other S.  In f: constexpr int kS =
// decltype(s)::value.  For the switches whose cases make the same call with only S changing; the switches that pick a
// measured configuration per size stay written out.
template <class F>
int with_S(int S, F &&f) {
    switch (S) {
    case 4: return f(std::integral_constant<int, 4>{});
    case 9: return f(std::integral_constant<int, 9>{});
    case 16: return f(std::integral_constant<int, 16>{});
    case 25: return f(std::integral_constant<int, 25>{});
    }
    return TG_E_ARG;
}

// ---------------------------------------------------------------- argument rules of the game path
// One function per shape of entry point, shared by the int8, int16 and bit-slab twins.  In order: the scalars (TG_E_ARG),
// an empty batch (TG_OK, before any pointer is looked at), null pointers (TG_E_ARG), alignment (TG_E_ARG).  LAUNCH means
// the arguments hold and there is work; the entry point goes on to launch.  It never leaves the library.
constexpr int LAUNCH = 1;

inline bool misaligned(const void *p, uintptr_t align) { return ((uintptr_t)p & (align - 1)) != 0; }

// tg_step*: slab_in, slab_out and tape 16-byte aligned
inline int check_step(int S, long long B, int shift, const void *in, const void *tape, const void *out, const void *flags,
                      const void *nnz) {
    if (!supported_S(S) || B < 0 || shift < 1 || shift > 4) return TG_E_ARG;
    if (B == 0) return TG_OK;
    if (!in || !tape || !out || !flags || !nnz) return TG_E_ARG;
    if (misaligned(in, 16) || misaligned(out, 16) || misaligned(tape, 16)) return TG_E_ARG;
    return LAUNCH;
}

// tg_expand_children*: tg_step's rules with k >= 1 children per parent (keys may be NULL)
inline int check_expand(int S, long long B, int k, int shift, const void *parents, const void *tape, const void *children,
                        const void *flags, const void *nnz) {
    if (k < 1) return TG_E_ARG;
    return check_step(S, B, shift, parents, tape, children, flags, nnz);
}

// tg_rollout* (freeze: steps required) and tg_replay*: the tape only when K > 0; slabs, tape and step stride 16-byte aligned
inline int check_rollout(int S, long long B, int K, int shift, const void *in, const void *tape, long long stride, const void *out,
                         const void *flags, const void *nnz, const void *steps, bool freeze) {
    if (!supported_S(S) || B < 0 || K < 0 || shift < 1 || shift > 4) return TG_E_ARG;
    if (B == 0) return TG_OK;
    if (!in || !out || !flags || !nnz || (freeze && !steps) || (K > 0 && !tape)) return TG_E_ARG;
    if (misaligned(in, 16) || misaligned(out, 16) || misaligned(tape, 16) || (stride & 15)) return TG_E_ARG;
    return LAUNCH;
}

// one source and one destination buffer per game (keys, ranks and the conversions), each aligned to its own boundary:
// slabs and tapes 16, float32 values 4, int64 tokens 8, keys and ranks 1 (not checked)
inline int check_pair(int S, long long B, const void *src, uintptr_t src_align, const void *dst, uintptr_t dst_align) {
    if (!supported_S(S) || B < 0) return TG_E_ARG;
    if (B == 0) return TG_OK;
    if (!src || !dst) return TG_E_ARG;
    if (misaligned(src, src_align) || misaligned(dst, dst_align)) return TG_E_ARG;
    return LAUNCH;
}

// tg_change_of_basis_gf2: bit slabs 16-byte aligned, the uint32 matrix rows 4-byte aligned
inline int check_basis_gf2(int S, long long N, const void *in, const void *mats, const void *out) {
    if (!supported_S(S) || N < 0) return TG_E_ARG;
    if (N == 0) return TG_OK;
    if (!in || !mats || !out) return TG_E_ARG;
    if (misaligned(in, 16) || misaligned(out, 16) || misaligned(mats, 4)) return TG_E_ARG;
    return LAUNCH;
}

// tg_change_of_basis_factors_gf2: both shifts in [1, 4], R >= 1; tapes and step strides 16-byte aligned, matrices 4
inline int check_basis_factors_gf2(int S, long long N, int R, int shift_in, int shift_out, const void *tape_in, long long in_stride,
                                   const void *mats, const void *tape_out, long long out_stride) {
    if (!supported_S(S) || N < 0 || R < 1 || shift_in < 1 || shift_in > 4 || shift_out < 1 || shift_out > 4) return TG_E_ARG;
    if (N == 0) return TG_OK;
    if (!tape_in || !mats || !tape_out) return TG_E_ARG;
    if (misaligned(tape_in, 16) || misaligned(tape_out, 16) || (in_stride & 15) || (out_stride & 15) || misaligned(mats, 4)) return TG_E_ARG;
    return LAUNCH;
}

// tg_sample_invertible_gf2: p_nonzero in [0, 1] (NaN refused), matrices 4-byte aligned
inline int check_sample_gf2(int S, long long N, double p_nonzero, const void *mats) {
    if (!supported_S(S) || N < 0 || !(p_nonzero >= 0.0 && p_nonzero <= 1.0)) return TG_E_ARG;
    if (N == 0) return TG_OK;
    if (!mats) return TG_E_ARG;
    if (misaligned(mats, 4)) return TG_E_ARG;
    return LAUNCH;
}

// tg_demo_sample_gf2: the rules of tg_demo_sample_dm in its order -- the scalars, an empty batch, null pointers, tape_dm
// and the targets 16-byte aligned, then replay_shift in [0, 8]; states may start at any float
inline int check_demo_sample_gf2(int S, long long N, int R, int dim_t, int replay_shift, long long nb, const void *tape_dm,
                                 const void *targets, const void *idx, const void *states, const void *scalars, const void *actions,
                                 const void *rewards) {
    if (!supported_S(S) || N < 0 || R < 1 || dim_t < 1 || nb < 0) return TG_E_ARG;
    if (nb == 0) return TG_OK;
    if (!tape_dm || !targets || !idx || !states || !scalars || !actions || !rewards) return TG_E_ARG;
    if (misaligned(tape_dm, 16) || misaligned(targets, 16)) return TG_E_ARG;
    if (replay_shift < 0 || replay_shift > 8) return TG_E_ARG;
    return LAUNCH;
}

// change of basis: set by a fast kernel on the games it leaves to the exact int32 kernel, which clears it
constexpr uint8_t BASIS_REDO = 0x80;
// tg_basis_mma.cu: 16x16x16 games, one warp per game on mma.sync int8 + f16; tg_basis_mma9.cu: 9x9x9 games on mma.sync f16.
// slab_out is an int8 slab (out16 == 0) or an int16 slab.
int launch_basis_mma16(const int8_t *slab_in, const int8_t *mats, long long mat_stride, void *slab_out, int out16, uint8_t *flags,
                       long long N, cudaStream_t st);
int launch_basis_mma9(const int8_t *slab_in, const int8_t *mats, long long mat_stride, void *slab_out, int out16, uint8_t *flags,
                      long long N, cudaStream_t st);

// tg_rollout9.cu: tg_rollout / tg_replay at 9x9x9 and 16x16x16, one thread per row of a game
int launch_rollout_rows(const int8_t *slab_in, const uint8_t *tape, long long stride, int K, int8_t *slab_out, uint8_t *flags,
                        int32_t *nnz, int32_t *steps, long long B, int S, int shift, int freeze, cudaStream_t st);
// tg_demo_mma.cu: sum of the R rank-1 terms of 16x16x16 action lists, one warp per demo on mma.sync f16 (R <= 64)
bool demo_acc16_mma_applies(int R);
int launch_demo_acc16_mma(const uint8_t *tape, long long tape_step_stride, long long N, int R, int shift, int8_t *slab,
                          uint8_t *flags, int or_flags, cudaStream_t st);

// Philox4x32-10 (oracle/tg_oracle.c orc_philox4x32_10): the block of counter (c0, c1, c2, c3) under key (k0, k1)
__device__ __forceinline__ void philox_block(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1,
                                             uint32_t out[4]) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ k0, c1 = lo1, c2 = hi0 ^ c3 ^ k1, c3 = lo0;
        k0 += 0x9E3779B9u, k1 += 0xBB67AE85u;
    }
    out[0] = c0, out[1] = c1, out[2] = c2, out[3] = c3;
}

// 64-bit state key replacing the string key of utils.py:164-169 (dict key of the MCTS tree, act.py:37...210): a linear
// hash, key(T) = sum T[i][j][k] * A_i * B_j * C_k (mod 2^64), the trilinear form of the state at three fixed odd 64-bit
// vectors, A_i = key_const(0x1000, i), B_j = key_const(0x2000, j), C_k = key_const(0x3000, k), distinct per mode
// so that transposed states differ.  The int8, int16 and bit-slab kernels use the same constants, so a state has the
// same key in every format that holds it.  The product structure is what lets the leaf expansion get a child's key
// from its action's 3 S tokens alone.
__device__ __forceinline__ unsigned long long splitmix64(unsigned long long z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__device__ __forceinline__ unsigned long long key_const(unsigned base, int i) { return splitmix64((unsigned long long)(base + i)) | 1ull; }

// ---------------------------------------------------------------- PTX: mbarrier + bulk async copy (TMA 1-D)
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// global -> shared, completion counted on the mbarrier (UBLKCP in SASS)
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// shared -> global, tracked by bulk async-groups
__device__ __forceinline__ void bulk_s2g(void *dst_gmem, const void *src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait() {
    asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
// generic-proxy smem writes -> visible to the async proxy (bulk store source)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---------------------------------------------------------------- SWAR helpers on 4 packed int8
constexpr uint32_t H4 = 0x80808080u;
constexpr uint32_t ONES4 = 0x01010101u;

// bit 7 of each byte set iff that byte is non-zero
__device__ __forceinline__ uint32_t nonzero_mask(uint32_t x) { return (((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x) & H4; }

// sum of the four unsigned bytes of x
__device__ __forceinline__ uint32_t byte_sum(uint32_t x) { return __dp4a(x, ONES4, 0u); }

// vector accesses as PTX, so that the access width is exactly the one the alignment test in front of it allows (the
// compiler re-vectorised the plain C++ stores of the misaligned branch into an 8-byte store at p + 2)
__device__ __forceinline__ void st_f32x4(float *p, float a, float b, float c, float d) {
    asm volatile("st.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(__cvta_generic_to_global(p)), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ void st_f32x2(float *p, float a, float b) {
    asm volatile("st.global.v2.f32 [%0], {%1, %2};" ::"l"(__cvta_generic_to_global(p)), "f"(a), "f"(b) : "memory");
}
__device__ __forceinline__ void st_f32(float *p, float a) {
    asm volatile("st.global.f32 [%0], %1;" ::"l"(__cvta_generic_to_global(p)), "f"(a) : "memory");
}
__device__ __forceinline__ void ld_f32x4(const float *p, float f[4]) {
    asm volatile("ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(f[0]), "=f"(f[1]), "=f"(f[2]), "=f"(f[3]) : "l"(__cvta_generic_to_global(p)));
}
__device__ __forceinline__ void ld_f32x2(const float *p, float &a, float &b) {
    asm volatile("ld.global.nc.v2.f32 {%0, %1}, [%2];" : "=f"(a), "=f"(b) : "l"(__cvta_generic_to_global(p)));
}
__device__ __forceinline__ float ld_f32(const float *p) {
    float a;
    asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(a) : "l"(__cvta_generic_to_global(p)));
    return a;
}

// four consecutive float32 entries of one output row (entries 4c .. 4c+3, the first nv of them inside the row) leave with
// the widest stores the address allows: one 16-byte store when S^2 is a multiple of four (4x4x4, 16x16x16: every run of a
// 16-byte aligned batch is aligned), at 9x9x9 (rows of 81 floats: the alignment of a run alternates with the row) two
// 8-byte stores, or 4 + 8 + 4 bytes around the aligned pair in the middle.  p points to global memory.
template <int S>
__device__ __forceinline__ void store_run(float *p, int nv, float a, float b, float c, float d) {
    const uint32_t lo = (uint32_t)reinterpret_cast<uintptr_t>(p);
    if constexpr (Geo<S>::S2 % 4 == 0) {
        if ((lo & 15u) == 0) {
            st_f32x4(p, a, b, c, d);
            return;
        }
    }
    if (nv == 4) {
        if ((lo & 7u) == 0) {
            st_f32x2(p, a, b);
            st_f32x2(p + 2, c, d);
        } else {
            st_f32(p, a);
            st_f32x2(p + 1, b, c);
            st_f32(p + 3, d);
        }
    } else {
        if (nv > 0) st_f32(p, a);
        if (nv > 1) st_f32(p + 1, b);
        if (nv > 2) st_f32(p + 2, c);
    }
}

// counterpart of store_run: four consecutive float32 entries of a row (the first nv of them exist) with the widest loads
// the address allows
template <int S>
__device__ __forceinline__ void load_run(const float *p, int nv, float f[4]) {
    const uint32_t lo = (uint32_t)reinterpret_cast<uintptr_t>(p);
    f[0] = f[1] = f[2] = f[3] = 0.f;
    if constexpr (Geo<S>::S2 % 4 == 0) {
        if ((lo & 15u) == 0) {
            ld_f32x4(p, f);
            return;
        }
    }
    if (nv == 4) {
        if ((lo & 7u) == 0) {
            ld_f32x2(p, f[0], f[1]);
            ld_f32x2(p + 2, f[2], f[3]);
        } else {
            f[0] = ld_f32(p);
            ld_f32x2(p + 1, f[1], f[2]);
            f[3] = ld_f32(p + 3);
        }
    } else {
        if (nv > 0) f[0] = ld_f32(p);
        if (nv > 1) f[1] = ld_f32(p + 1);
        if (nv > 2) f[2] = ld_f32(p + 2);
    }
}

} // namespace tg
