// tg_host.cu -- host-buffer entry points: the end-to-end path a caller with
// data in host memory takes (H2D copy -> kernel -> D2H copy).  Chunks flow through three dedicated streams -- every H2D
// copy on one, every kernel on another, every D2H copy on a third -- chained by events per staging buffer, so that the
// two copy engines stream back to back: a chunk's upload never queues behind another chunk's download (with one stream
// per buffer it did: at 8 ranks per host the path reached half of the raw pinned-copy rate).
//
// Every entry point, for int8, int16 and bit slabs, runs the one chunk loop of host_chunks: the formats differ only in
// the bytes per game of a slab and in the device call that processes a chunk.
#include <new>
#include <type_traits>

#include "tg_common.cuh"

struct tg_host_ctx {
    int device;
    int S;
    int64_t chunk;
    static constexpr int NBUF = 4;
    cudaStream_t s_in, s_k, s_out;
    cudaEvent_t ev_in[NBUF], ev_k[NBUF], ev_out[NBUF];
    int8_t *slab[NBUF];     // slab staging of one chunk in any format: GP * chunk bytes, grown to 2 GP * chunk for int16
    int64_t slab_bytes[NBUF];
    uint8_t *tape[NBUF];
    uint8_t *flags[NBUF];
    int32_t *nnz[NBUF];
    int32_t *steps[NBUF];
    uint8_t *tape_k[NBUF]; // multi-step tape staging [K][chunk][TP], grown on demand
    int64_t tape_k_bytes[NBUF];
};

// device staging kept in the context, grown when a call needs more (after the device has finished with the old buffer)
template <class T>
static int ensure_staging(T *&buf, int64_t &have, int64_t bytes) {
    if (have >= bytes) return TG_OK;
    TG_CUDA(cudaDeviceSynchronize());
    cudaFree(buf);
    buf = nullptr, have = 0;
    TG_CUDA(cudaMalloc(&buf, (size_t)bytes));
    have = bytes;
    return TG_OK;
}

// every staging buffer: slabs of `slab_bytes` per game and K-step tapes of `tape_rows` records per game (0: none)
static int ensure_chunk_staging(tg_host_ctx *c, int64_t slab_bytes, int64_t tape_rows, int tp) {
    for (int i = 0; i < tg_host_ctx::NBUF; i++) {
        int rc = ensure_staging(c->slab[i], c->slab_bytes[i], slab_bytes * c->chunk);
        if (rc == TG_OK && tape_rows > 0) rc = ensure_staging(c->tape_k[i], c->tape_k_bytes[i], tape_rows * c->chunk * tp);
        if (rc != TG_OK) return rc;
    }
    return TG_OK;
}

// bytes per game of a host slab: GP for int8, 2 GP for int16, GB for a bit slab
template <class T>
static int64_t game_bytes(int S) {
    int rp, gp, tp;
    tg_layout(S, &rp, &gp, &tp);
    if constexpr (std::is_same_v<T, uint32_t>) {
        int rw, gb;
        tg_layout_gf2(S, &rw, &gb);
        return gb;
    }
    return (int64_t)gp * (int64_t)sizeof(T);
}

// What one host call moves per game.  Host buffers need only their element type's alignment: every copy is a byte copy
// between them and the aligned staging.  Chunk q reads and writes games [b0, b0 + n) of every buffer and nothing else,
// so in place (slab_out == slab_in) holds.
struct HostIO {
    int64_t slab_bytes;    // per game, game_bytes<T>
    const void *slab_in;   // uploaded per chunk; null when the device call writes the slab (demos)
    void *slab_out;        // downloaded per chunk
    const uint8_t *tape;   // uploaded: a step's records [B][TP] (tape_rows == 0) or a step-major [K][B][TP] tape (K rows)
    uint8_t *tape_out;     // downloaded: a step-major [R][N][TP] tape (R rows)
    int tape_rows;
    uint8_t *flags;
    int32_t *nnz, *steps;  // downloaded when not null
};

// Enqueues every chunk: upload on s_in, run(i, b0, n) on s_k with staging buffer i = q % NBUF, download on s_out.  The
// first stream to touch buffer i waits for the buffer's last download.
template <class Run>
static int enqueue_chunks(tg_host_ctx *c, const HostIO &io, int64_t B, int tp, Run &run) {
    const int64_t sb = io.slab_bytes;
    const uint8_t *slab_in = (const uint8_t *)io.slab_in;
    uint8_t *slab_out = (uint8_t *)io.slab_out;
    int q = 0;
    for (int64_t b0 = 0; b0 < B; b0 += c->chunk, q++) {
        const int i = q % tg_host_ctx::NBUF;
        const int64_t n = (B - b0 < c->chunk) ? B - b0 : c->chunk;
        if (q >= tg_host_ctx::NBUF) TG_CUDA(cudaStreamWaitEvent(slab_in ? c->s_in : c->s_k, c->ev_out[i], 0));
        if (slab_in) {
            TG_CUDA(cudaMemcpyAsync(c->slab[i], slab_in + b0 * sb, (size_t)(n * sb), cudaMemcpyHostToDevice, c->s_in));
            if (io.tape && io.tape_rows == 0)
                TG_CUDA(cudaMemcpyAsync(c->tape[i], io.tape + b0 * tp, (size_t)n * tp, cudaMemcpyHostToDevice, c->s_in));
            // the chunk's columns of the step-major host tape [K][B][TP] -> a dense [K][n][TP] staging tape
            else if (io.tape)
                TG_CUDA(cudaMemcpy2DAsync(c->tape_k[i], (size_t)n * tp, io.tape + b0 * tp, (size_t)B * tp, (size_t)n * tp,
                                          (size_t)io.tape_rows, cudaMemcpyHostToDevice, c->s_in));
            TG_CUDA(cudaEventRecord(c->ev_in[i], c->s_in));
            TG_CUDA(cudaStreamWaitEvent(c->s_k, c->ev_in[i], 0));
        }
        const int rc = run(i, b0, n);
        if (rc != TG_OK) return rc;
        TG_CUDA(cudaEventRecord(c->ev_k[i], c->s_k));
        TG_CUDA(cudaStreamWaitEvent(c->s_out, c->ev_k[i], 0));
        // dense [R][n][TP] staging tape -> the chunk's columns of the step-major host tape [R][N][TP]
        if (io.tape_out)
            TG_CUDA(cudaMemcpy2DAsync(io.tape_out + b0 * tp, (size_t)B * tp, c->tape_k[i], (size_t)n * tp, (size_t)n * tp,
                                      (size_t)io.tape_rows, cudaMemcpyDeviceToHost, c->s_out));
        TG_CUDA(cudaMemcpyAsync(slab_out + b0 * sb, c->slab[i], (size_t)(n * sb), cudaMemcpyDeviceToHost, c->s_out));
        TG_CUDA(cudaMemcpyAsync(io.flags + b0, c->flags[i], (size_t)n, cudaMemcpyDeviceToHost, c->s_out));
        if (io.nnz) TG_CUDA(cudaMemcpyAsync(io.nnz + b0, c->nnz[i], (size_t)n * 4, cudaMemcpyDeviceToHost, c->s_out));
        if (io.steps) TG_CUDA(cudaMemcpyAsync(io.steps + b0, c->steps[i], (size_t)n * 4, cudaMemcpyDeviceToHost, c->s_out));
        TG_CUDA(cudaEventRecord(c->ev_out[i], c->s_out));
    }
    return TG_OK;
}

// The chunk loop of every host entry point; returns when the results are in host memory.  A call that fails part way
// waits for what it had enqueued, so no copy from or to the caller's buffers is in flight after it returns.
template <class Run>
static int host_chunks(tg_host_ctx *c, const HostIO &io, int64_t B, Run &&run) {
    int rp, gp, tp;
    tg_layout(c->S, &rp, &gp, &tp);
    const int rc = enqueue_chunks(c, io, B, tp, run);
    if (rc != TG_OK) {
        cudaStreamSynchronize(c->s_in);
        cudaStreamSynchronize(c->s_k);
        cudaStreamSynchronize(c->s_out);
        return rc;
    }
    TG_CUDA(cudaStreamSynchronize(c->s_out));
    return TG_OK;
}

// the device calls behind the host entry points, one signature per shape for the three slab formats
template <class T>
using StepFn = int (*)(const T *, const uint8_t *, T *, uint8_t *, int32_t *, int64_t, int, int, void *);
template <class T>
using RolloutFn = int (*)(const T *, const uint8_t *, int64_t, int, T *, uint8_t *, int32_t *, int32_t *, int64_t, int, int, void *);
template <class T>
using DemoFn = int (*)(uint64_t, uint64_t, int64_t, int, int, int, const int8_t *, const double *, int, int, uint8_t *, int64_t, T *,
                       uint8_t *, void *);

// Argument rules of the host entry points, in order: a null context, B < 0 or K < 0 (TG_E_ARG); B == 0 (TG_OK); a null
// host pointer (TG_E_ARG); then the device call's own checks, all before the first copy.  The device call is first made
// on an empty chunk: an empty batch returns TG_OK after the scalar checks (shift, K, R, ...) and launches nothing, and the
// staging buffers pass its pointer checks.  The demo generators check their alphabet after that; there the first chunk's
// device call comes before any copy.
template <class T>
static int step_host(StepFn<T> step, tg_host_ctx *c, const T *slab_in, const uint8_t *tape, T *slab_out, uint8_t *flags,
                     int32_t *nnz, int64_t B, int shift) {
    if (!c || B < 0) return TG_E_ARG;
    if (B == 0) return TG_OK;
    if (!slab_in || !tape || !slab_out || !flags || !nnz) return TG_E_ARG;
    TG_CUDA(cudaSetDevice(c->device));
    if (const int rc = step((T *)c->slab[0], c->tape[0], (T *)c->slab[0], c->flags[0], c->nnz[0], 0, c->S, shift, c->s_k); rc != TG_OK)
        return rc;
    const int64_t sb = game_bytes<T>(c->S);
    if (const int rc = ensure_chunk_staging(c, sb, 0, 0); rc != TG_OK) return rc;
    const HostIO io = {sb, slab_in, slab_out, tape, nullptr, 0, flags, nnz, nullptr};
    return host_chunks(c, io, B, [&](int i, int64_t, int64_t n) {
        T *s = (T *)c->slab[i];
        return step(s, c->tape[i], s, c->flags[i], c->nnz[i], n, c->S, shift, c->s_k);
    });
}

template <class T>
static int rollout_host(RolloutFn<T> rollout, tg_host_ctx *c, const T *slab_in, const uint8_t *tape, int K, T *slab_out,
                        uint8_t *flags, int32_t *nnz, int32_t *steps, int64_t B, int shift) {
    if (!c || B < 0 || K < 0) return TG_E_ARG;
    if (B == 0) return TG_OK;
    if (!slab_in || (K > 0 && !tape) || !slab_out || !flags || !nnz || !steps) return TG_E_ARG;
    int rp, gp, tp;
    tg_layout(c->S, &rp, &gp, &tp);
    TG_CUDA(cudaSetDevice(c->device));
    if (const int rc = rollout((T *)c->slab[0], c->tape_k[0], 0, K, (T *)c->slab[0], c->flags[0], c->nnz[0], c->steps[0], 0, c->S,
                               shift, c->s_k);
        rc != TG_OK)
        return rc;
    const int64_t sb = game_bytes<T>(c->S);
    if (const int rc = ensure_chunk_staging(c, sb, K > 0 ? K : 1, tp); rc != TG_OK) return rc;
    const HostIO io = {sb, slab_in, slab_out, K > 0 ? tape : nullptr, nullptr, K, flags, nnz, steps};
    return host_chunks(c, io, B, [&](int i, int64_t, int64_t n) {
        T *s = (T *)c->slab[i];
        return rollout(s, c->tape_k[i], n * tp, K, s, c->flags[i], c->nnz[i], c->steps[i], n, c->S, shift, c->s_k);
    });
}

// demos are keyed by their global index first_demo + n0 + n, so the chunking does not show in the output
template <class T>
static int demo_host(DemoFn<T> gen, tg_host_ctx *c, uint64_t seed, uint64_t first_demo, int64_t N, int R, int shift,
                     const int8_t *values, const double *probs, int n_values, int max_tries, uint8_t *tape, T *slab, uint8_t *flags) {
    if (!c || N < 0 || R < 1) return TG_E_ARG;
    if (N == 0) return TG_OK;
    if (!tape || !slab || !flags) return TG_E_ARG;
    int rp, gp, tp;
    tg_layout(c->S, &rp, &gp, &tp);
    TG_CUDA(cudaSetDevice(c->device));
    if (const int rc = gen(seed, first_demo, 0, R, c->S, shift, values, probs, n_values, max_tries, c->tape_k[0], 0, (T *)c->slab[0],
                           c->flags[0], c->s_k);
        rc != TG_OK)
        return rc;
    const int64_t sb = game_bytes<T>(c->S);
    if (const int rc = ensure_chunk_staging(c, sb, R, tp); rc != TG_OK) return rc;
    const HostIO io = {sb, nullptr, slab, nullptr, tape, R, flags, nullptr, nullptr};
    return host_chunks(c, io, N, [&](int i, int64_t n0, int64_t n) {
        return gen(seed, first_demo + (uint64_t)n0, n, R, c->S, shift, values, probs, n_values, max_tries, c->tape_k[i], n * tp,
                   (T *)c->slab[i], c->flags[i], c->s_k);
    });
}

extern "C" {

int tg_host_ctx_create(tg_host_ctx **out, int device, int S, int64_t max_chunk) {
    if (!out || !tg::supported_S(S) || max_chunk <= 0) return TG_E_ARG;
    int rp, gp, tp;
    tg_layout(S, &rp, &gp, &tp);
    TG_CUDA(cudaSetDevice(device));
    tg_host_ctx *c = new (std::nothrow) tg_host_ctx();
    if (!c) return TG_E_ARG;
    c->device = device, c->S = S, c->chunk = max_chunk;
    c->s_in = c->s_k = c->s_out = nullptr;
    for (int i = 0; i < tg_host_ctx::NBUF; i++) {
        c->ev_in[i] = c->ev_k[i] = c->ev_out[i] = nullptr;
        c->slab[i] = nullptr, c->slab_bytes[i] = 0, c->tape[i] = nullptr, c->flags[i] = nullptr, c->nnz[i] = nullptr;
        c->steps[i] = nullptr, c->tape_k[i] = nullptr, c->tape_k_bytes[i] = 0;
    }
    cudaError_t e = cudaStreamCreateWithFlags(&c->s_in, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->s_k, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->s_out, cudaStreamNonBlocking);
    for (int i = 0; i < tg_host_ctx::NBUF && e == cudaSuccess; i++) {
        e = cudaEventCreateWithFlags(&c->ev_in[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_k[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_out[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaMalloc(&c->slab[i], (size_t)max_chunk * gp);
        if (e == cudaSuccess) c->slab_bytes[i] = max_chunk * gp;
        if (e == cudaSuccess) e = cudaMalloc(&c->tape[i], (size_t)max_chunk * tp);
        if (e == cudaSuccess) e = cudaMalloc(&c->flags[i], (size_t)max_chunk);
        if (e == cudaSuccess) e = cudaMalloc(&c->nnz[i], (size_t)max_chunk * 4);
        if (e == cudaSuccess) e = cudaMalloc(&c->steps[i], (size_t)max_chunk * 4);
    }
    if (e != cudaSuccess) {
        tg_host_ctx_destroy(c);
        return tg::cuda_fail(e);
    }
    *out = c;
    return TG_OK;
}

int tg_host_ctx_destroy(tg_host_ctx *c) {
    if (!c) return TG_OK;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    for (int i = 0; i < tg_host_ctx::NBUF; i++) {
        cudaFree(c->slab[i]);
        cudaFree(c->tape[i]);
        cudaFree(c->flags[i]);
        cudaFree(c->nnz[i]);
        cudaFree(c->steps[i]);
        cudaFree(c->tape_k[i]);
        if (c->ev_in[i]) cudaEventDestroy(c->ev_in[i]);
        if (c->ev_k[i]) cudaEventDestroy(c->ev_k[i]);
        if (c->ev_out[i]) cudaEventDestroy(c->ev_out[i]);
    }
    if (c->s_in) cudaStreamDestroy(c->s_in);
    if (c->s_k) cudaStreamDestroy(c->s_k);
    if (c->s_out) cudaStreamDestroy(c->s_out);
    delete c;
    return TG_OK;
}

int tg_step_host(tg_host_ctx *c, const int8_t *slab_in, const uint8_t *tape, int8_t *slab_out, uint8_t *flags,
                 int32_t *nnz, int64_t B, int shift) {
    return step_host<int8_t>(tg_step, c, slab_in, tape, slab_out, flags, nnz, B, shift);
}

int tg_step_host_i16(tg_host_ctx *c, const int16_t *slab_in, const uint8_t *tape, int16_t *slab_out, uint8_t *flags,
                     int32_t *nnz, int64_t B, int shift) {
    return step_host<int16_t>(tg_step_i16, c, slab_in, tape, slab_out, flags, nnz, B, shift);
}

int tg_step_host_gf2(tg_host_ctx *c, const uint32_t *bits_in, const uint8_t *tape, uint32_t *bits_out, uint8_t *flags,
                     int32_t *nnz, int64_t B, int shift) {
    return step_host<uint32_t>(tg_step_gf2, c, bits_in, tape, bits_out, flags, nnz, B, shift);
}

int tg_rollout_host(tg_host_ctx *c, const int8_t *slab_in, const uint8_t *tape, int K, int8_t *slab_out, uint8_t *flags,
                    int32_t *nnz, int32_t *steps, int64_t B, int shift) {
    return rollout_host<int8_t>(tg_rollout, c, slab_in, tape, K, slab_out, flags, nnz, steps, B, shift);
}

int tg_rollout_host_i16(tg_host_ctx *c, const int16_t *slab_in, const uint8_t *tape, int K, int16_t *slab_out, uint8_t *flags,
                        int32_t *nnz, int32_t *steps, int64_t B, int shift) {
    return rollout_host<int16_t>(tg_rollout_i16, c, slab_in, tape, K, slab_out, flags, nnz, steps, B, shift);
}

int tg_rollout_host_gf2(tg_host_ctx *c, const uint32_t *bits_in, const uint8_t *tape, int K, uint32_t *bits_out, uint8_t *flags,
                        int32_t *nnz, int32_t *steps, int64_t B, int shift) {
    return rollout_host<uint32_t>(tg_rollout_gf2, c, bits_in, tape, K, bits_out, flags, nnz, steps, B, shift);
}

int tg_demo_gen_host(tg_host_ctx *c, uint64_t seed, uint64_t first_demo, int64_t N, int R, int shift, const int8_t *values,
                     const double *probs, int n_values, int max_tries, uint8_t *tape, int8_t *slab, uint8_t *flags) {
    return demo_host<int8_t>(tg_demo_gen_philox, c, seed, first_demo, N, R, shift, values, probs, n_values, max_tries, tape, slab, flags);
}

int tg_demo_gen_host_gf2(tg_host_ctx *c, uint64_t seed, uint64_t first_demo, int64_t N, int R, int shift, const int8_t *values,
                         const double *probs, int n_values, int max_tries, uint8_t *tape, uint32_t *bits, uint8_t *flags) {
    return demo_host<uint32_t>(tg_demo_gen_gf2, c, seed, first_demo, N, R, shift, values, probs, n_values, max_tries, tape, bits, flags);
}

} // extern "C"
