/*
 * tensorgame.h -- C ABI of libtensorgame_b200.so (sm_100a).
 *
 * Drop-in boundary for the data-parallel hot path of kurtosis/mat_mul's
 * TensorGame environment.  The reference has no FFI: its boundary is the
 * Python surface of utils.py / datasets.py / act.py.  Each entry point below
 * names the reference code it replaces (file:line in /root/reference); the
 * Python mirrors in mat_mul_b200/{utils,datasets,act}.py bind them with
 * ctypes (see INTEGRATION.md for the stub a maintainer would add).
 *
 * Conventions
 *   - plain pointers and sizes only; no torch types.
 *   - unless the name ends in _host, every pointer is a CUDA DEVICE pointer
 *     owned by the caller; calls are asynchronous on `stream` (a cudaStream_t
 *     passed as void*), never allocate and never synchronise -- with one
 *     exception: tg_demo_gen_philox and tg_demo_gen_gf2 keep the device form
 *     of up to eight alias-table sets per device in static device memory,
 *     one cache for both (uploaded on `stream` the first time a distribution
 *     is used; launches on other streams wait for that upload by event; the
 *     mod-2 tables of an alphabet whose only even value is 0 are the integer
 *     ones and share their slot); a NINTH distinct set evicts one after a
 *     cudaDeviceSynchronize.  tg_demo_sample_dm (9x9x9)
 *     zeroes a per-launch work counter in static device memory on `stream`.
 *   - *_host entry points take HOST pointers (pinned for full speed), move the
 *     data themselves through a caller-created tg_host_ctx and return after
 *     the results are in host memory.
 *   - return value: 0 on success, a negative TG_E_* code otherwise; nothing
 *     throws.  There is no CPU fallback: without a CUDA device every compute
 *     entry point returns TG_E_CUDA.
 *   - argument rules of the game path (tg_step, tg_expand_children,
 *     tg_rollout, tg_replay, tg_state_key, tg_slice_rank and the conversions,
 *     for every slab format), checked in this order: a bad scalar (S, B < 0,
 *     shift outside [1, 4], k < 1, K < 0) returns TG_E_ARG; an empty batch
 *     (B == 0) returns TG_OK before any pointer is looked at; a null pointer
 *     the call needs returns TG_E_ARG; a misaligned buffer returns TG_E_ARG.
 *     Slabs of every format, tapes and tape_step_stride are 16-byte aligned,
 *     float32 arrays 4-byte and int64 token arrays 8-byte aligned; flags, nnz,
 *     steps, keys and ranks are naturally aligned arrays (not checked).
 *
 * Sizes: S = dim_3d in {4, 9, 16, 25} on the game path (layout, conversions,
 * K1-K4, K6-K8, parity mode, host buffers, the int16 and mod-2 game paths, and the change of basis mod 2).  The
 * change of basis over Z (K5) stays {4, 9, 16} and tg_demo_accumulate_tc 16; at 25 tg_demo_gen_philox keeps
 * contract v1 for every alphabet (tg_demo_alias_tables returns TG_E_ARG).
 *
 * Device formats (see DESIGN.md "Data layout")
 *   slab   int8  [B][GP]   residual tensors, entry (i,j,k) at i*RP + j*S + k,
 *                          RP = roundup4(S*S), GP = roundup16(S*RP); padding
 *                          bytes are zero.  (S=4: 16/64, S=9: 84/768,
 *                          S=16: 256/4096, S=25: 628/15712.)  Values must stay in [-64, 63]
 *                          for the next step to be guaranteed (TG_FLAG_RANGE).
 *   tape   uint8 [B][TP]   action tokens cat(u,v,w)+shift in bytes [0,3S),
 *                          TP = roundup16(3S) (16/32/48/80), padding zero.
 *                          Token bound: every token is <= 2*shift (|coefficient|
 *                          <= shift <= 4) for the shift handed to the same call;
 *                          tg_step, tg_rollout, tg_replay and tg_expand_children
 *                          test it and raise TG_FLAG_RANGE for a game whose
 *                          record breaks it (its result is then unspecified).
 *                          A caller with another token convention re-bases:
 *                          coefficient c = token - s is passed as token c + 4
 *                          with shift 4.
 *   flags  uint8 [B]       TG_FLAG_* bits per game.
 *   nnz    int32 [B]       count of non-zero residual entries (rank upper
 *                          bound, training.py:259-266).
 */
#ifndef TENSORGAME_H
#define TENSORGAME_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TG_VERSION 205

#define TG_OK 0
#define TG_E_ARG (-1)     /* bad argument (unsupported S, null pointer, misaligned buffer) */
#define TG_E_CUDA (-2)    /* CUDA runtime error; tg_last_cuda_error() has the code */
#define TG_E_RANGE (-3)   /* value does not fit the device format */

#define TG_FLAG_TERMINAL 1u /* new head all zero: utils.py:181-188 on the head (act.py:177) */
#define TG_FLAG_NULL 2u     /* rank-1 update all zero: utils.py:191-194 */
#define TG_FLAG_RANGE 4u    /* a residual entry left the guaranteed zone ([-64, 63] int8, [-16384, 16383] int16) or a token exceeded 2*shift */
#define TG_FLAG_EXHAUSTED 8u /* demo generation: a term hit max_tries and was forced to a unit triple */
#define TG_FLAG_TOKEN_RANGE 16u /* change of basis: a transformed factor entry left [-shift_out, shift_out] */
#define TG_FLAG_PATH_PLANES 32u /* change of basis, informational: 16x16x16 game computed on int8 byte planes (not f16) */
#define TG_FLAG_PATH_EXACT 64u  /* change of basis, informational: game computed by the exact int32 kernel (no fast path held it) */

int tg_version(void);
int tg_last_cuda_error(void);
const char *tg_error_string(int code);

/* geometry of the device formats for a given S; returns TG_E_ARG for unsupported S */
int tg_layout(int S, int *row_pitch, int *game_pitch, int *token_pitch);

/* ---- boundary conversions (reference dtypes <-> device formats) ---------- */
/* float32 residuals, game b at src + b*src_stride (elements), dense (S,S,S)
 * -> slab.  range_flag (device int32, may be NULL) is OR-ed with 1 if a value
 * is non-integral or outside [-128,127].  Replaces the float32 state tensors
 * of utils.py:99-111 / datasets.py:94-114 at the boundary. */
int tg_pack_f32(const float *src, int64_t src_stride, int8_t *slab, int64_t B, int S, int32_t *range_flag, void *stream);
/* slab -> float32 dense (S,S,S) at dst + b*dst_stride: the state the model
 * consumes (model.py:101-103).  The slab is 16-byte aligned like every slab;
 * dst may start at any float (rows leave with the widest stores each address
 * allows). */
int tg_expand_f32(const int8_t *slab, float *dst, int64_t dst_stride, int64_t B, int S, void *stream);
/* int64 tokens (B,3S) (reference action format, utils.py:56-66) <-> tape */
/* the same two conversions for int16 slabs (range: integers in [-32768, 32767]) */
int tg_pack_f32_i16(const float *src, int64_t src_stride, int16_t *slab16, int64_t B, int S, int32_t *range_flag, void *stream);
int tg_expand_f32_i16(const int16_t *slab16, float *dst, int64_t dst_stride, int64_t B, int S, void *stream);
int tg_pack_actions_i64(const int64_t *actions, uint8_t *tape, int64_t B, int S, int32_t *range_flag, void *stream);
int tg_unpack_actions_i64(const uint8_t *tape, int64_t *actions, int64_t B, int S, void *stream);

/* ---- K1: batched transition --------------------------------------------- */
/* slab_out[b] = slab_in[b] - u(x)v(x)w of tape[b] with coefficient = token -
 * shift; flags/nnz per game.  In place (slab_out == slab_in) is allowed.
 * Replaces act.py:266-275 (get_child_states), training.py:253-267
 * (_take_action arithmetic), utils.py:181-188 (tensor_factorized on the head),
 * utils.py:191-194 (remove_null_actions), utils.py:69-96.  shift in [1,4]. */
int tg_step(const int8_t *slab_in, const uint8_t *tape, int8_t *slab_out, uint8_t *flags, int32_t *nnz,
            int64_t B, int S, int shift, void *stream);

/* ---- K8: batched leaf expansion ------------------------------------------ */
/* children[b][c] = parents[b] - u(x)v(x)w of tape[b][c] for c < k (tape uint8 [B][k][TP], children int8
 * [B][k][GP], flags / nnz / keys [B][k]); each parent is read once.  flags as in tg_step (TERMINAL = the child's
 * head is all zero, NULL = the action changed nothing, RANGE), keys = tg_state_key of the child (may be NULL).
 * Replaces, for B states at once, act.py:266-275 (get_child_states) together with the per-child
 * remove_null_actions (utils.py:191-194), tensor_factorized (utils.py:181-188, act.py:177) and state key
 * (utils.py:164-169, act.py:185-195) that extend_tree applies to the children. */
int tg_expand_children(const int8_t *parents, const uint8_t *tape, int k, int8_t *children, uint8_t *flags, int32_t *nnz,
                       uint64_t *keys, int64_t B, int S, int shift, void *stream);

/* ---- K2: fused K-step rollout --------------------------------------------- */
/* Applies tape[0..K-1] (step-major uint8 [K][B_total][TP], byte stride
 * tape_step_stride between steps) to every game, freezing a game once its
 * head is all zero (the break at act.py:49); steps[b] = actions applied, so
 * the game's return is -steps[b] (act.py:60-62) before the terminal -get_rank
 * term.  flags: TG_FLAG_TERMINAL | TG_FLAG_RANGE; nnz of the final head.
 * Replaces datasets.py:144-153 (_take_actions) and the loop at
 * training.py:336-342.  In place (slab_out == slab_in) is allowed. */
int tg_rollout(const int8_t *slab_in, const uint8_t *tape, int64_t tape_step_stride, int K, int8_t *slab_out,
               uint8_t *flags, int32_t *nnz, int32_t *steps, int64_t B, int S, int shift, void *stream);

/* Same fused kernel WITHOUT the freeze: all K actions are applied even if the
 * residual passes through zero -- SyntheticDemoDataset._take_actions
 * (datasets.py:144-153) literally. */
int tg_replay(const int8_t *slab_in, const uint8_t *tape, int64_t tape_step_stride, int K, int8_t *slab_out, uint8_t *flags,
              int32_t *nnz, int64_t B, int S, int shift, void *stream);

/* ---- K3: synthetic demonstrations ----------------------------------------- */
/* Multi-step tapes are step-major: uint8 [R][N_total][TP]; `tape_step_stride`
 * is the byte distance between consecutive steps (N_total*TP), so a rank can
 * write its shard of demos straight into a larger tape.
 *
 * Throughput mode (device RNG; contracts in DESIGN.md, restated by the oracle):
 * demo d = first_demo + n draws its R factor triples from Philox4x32-10 keyed
 * by seed.  `values` / `probs` are HOST arrays, n_values <= 8, values in
 * [-shift, shift].
 *  v2 (n_values <= 5 and P(0) <= 0.999) "group alias": an accepted triple of the
 *   reference's rejection loop is three independent factors, each conditioned on
 *   being non-zero; that conditional distribution is sampled directly, three
 *   entries at a time, from alias tables of 128 buckets (tg_demo_alias_tables)
 *   with one 16-bit draw per group, counter (d_lo, d_hi, term, block).  No tries:
 *   max_tries does not apply and TG_FLAG_EXHAUSTED is never raised.
 *  v1 (other alphabets): counter (d_lo, d_hi, term | try << 16, block), 15-bit
 *   draws against floor(cdf * 2^15); a triple is rejected iff u, v or w is all
 *   zero (utils.py:229), at most max_tries <= 65535 tries per term
 *   (TG_FLAG_EXHAUSTED).
 * Writes tokens (values + shift) to the tape, the summed
 * target tensors to slab [N][GP] and TG_FLAG_RANGE/EXHAUSTED to flags (may be
 * NULL).  Replaces utils.py:203-233 and datasets.py:124-142 (different RNG
 * stream than torch: see tg_demo_from_ustream for same-seed parity). */
int tg_demo_gen_philox(uint64_t seed, uint64_t first_demo, int64_t N, int R, int S, int shift, const int8_t *values,
                       const double *probs, int n_values, int max_tries, uint8_t *tape, int64_t tape_step_stride,
                       int8_t *slab, uint8_t *flags, void *stream);
/* HOST function: the alias tables of contract v2 as uint16 [8][128] -- [0] the plain distribution of a group of three
 * entries, [1] of a single entry, [2 + g] the tilted table of group g; bucket = 9-bit threshold | alias outcome << 9.
 * TG_E_ARG where v2 does not apply (also at S = 25: nine groups per factor, the tables hold six). */
int tg_demo_alias_tables(const int8_t *values, const double *probs, int n_values, int S, uint16_t *tables_host);
/* slab[n] = sum_r rank1(tape[r][n]) -- the target tensor of a given action
 * list (utils.py:40-53 uvw_to_demo, utils.py:232, datasets.py:141). */
int tg_demo_accumulate(const uint8_t *tape, int64_t tape_step_stride, int64_t N, int R, int S, int shift, int8_t *slab,
                       uint8_t *flags, void *stream);
/* the same sum into an int16 slab [N][GP] of int16 (exact for every tape and any shift in [0,127]: int32 arithmetic per
 * entry while R * max(shift, 255 - shift)^3 fits int32, 64-bit beyond; TG_FLAG_RANGE = an entry does not fit int16).  The reference accumulates targets in float32
 * without limit (utils.py:218-232); this is where targets beyond the int8 slab's zone go. */
int tg_demo_accumulate_i16(const uint8_t *tape, int64_t tape_step_stride, int64_t N, int R, int S, int shift, int16_t *slab16,
                           uint8_t *flags, void *stream);
/* For S = 16 and R <= 64 tg_demo_accumulate and tg_demo_gen_philox sum the targets on the tensor cores
 * (mma.sync f16, exact integer arithmetic; csrc/tg_demo_mma.cu) -- same results.
 * tg_demo_accumulate_tc: the same sum with tcgen05.mma kind::i8 (int32 accumulators in TMEM), an experimental entry
 * point kept for tests and profiling: S = 16 and R <= 64 only (TG_E_ARG otherwise); entries beyond int8 are stored
 * saturated (and flagged) instead of wrapped. */
int tg_demo_accumulate_tc(const uint8_t *tape, int64_t tape_step_stride, int64_t N, int R, int S, int shift, int8_t *slab,
                          uint8_t *flags, void *stream);

/* Parity mode: same-seed demos as the reference.  tg_mt19937_fill_f64 is a
 * HOST function reproducing torch's CPU uniform stream (MT19937, 53-bit
 * doubles; torch.manual_seed(seed); torch.rand(dtype=float64)), optionally
 * continuing from a generator state (the 624 words and position stored in
 * torch.get_rng_state()).  tg_demo_from_ustream consumes a DEVICE copy of
 * that stream exactly as the reference's rejection loop does (utils.py:
 * 222-232; Categorical == multinomial, float32 CDF) and emits the first N
 * demos: result[0] = demos completed (<= N), result[1] = doubles consumed by
 * them.  workspace: tg_demo_from_ustream_workspace(n_u, S) bytes, 16-aligned. */
int tg_mt19937_fill_f64(uint32_t seed, int64_t skip, int64_t n, double *out_host);
int tg_mt19937_fill_f64_state(const uint32_t *state624, int pos, int64_t skip, int64_t n, double *out_host);
int64_t tg_demo_from_ustream_workspace(int64_t n_u, int S);
int tg_demo_from_ustream(const double *u, int64_t n_u, const int8_t *values, const float *probs, int n_values, int R, int S,
                         int shift, int64_t N, uint8_t *tape, int64_t tape_step_stride, int8_t *slab, uint8_t *flags,
                         int64_t *result, void *workspace, int64_t workspace_bytes, void *stream);

/* ---- K4: training-sample batcher ------------------------------------------ */
/* SyntheticDemoDataset.__getitem__ (datasets.py:77-122) for nb sample indices
 * idx[b] = demo * R + action, read from the in-HBM demo store (step-major tape
 * + target slab): states float32 [nb][dim_t][S][S][S], scalars [nb] = R - a,
 * actions int64 [nb][3S], rewards [nb] = -(a+1).  replay_shift is the shift
 * action_to_tensor applies while replaying (the reference hard-codes 1,
 * utils.py:88-96); pass the demos' own shift for the true residual. */
int tg_demo_sample(const uint8_t *tape, int64_t tape_step_stride, const int8_t *slab, int64_t N, int R, int S, int dim_t,
                   int replay_shift, const int64_t *idx, int64_t nb, float *states, float *scalars, int64_t *actions,
                   float *rewards, void *stream);

/* The same samples from a DEMO-MAJOR store: action records uint8 [N][R][TP] (tg_tape_to_demo_major of a step-major tape;
 * the records a .. R-1 a sample needs are one contiguous run) and targets as an int8 slab (targets_i16 == 0) or an int16
 * slab [N][GP] of int16 (targets_i16 != 0; entry (i,j,k) at element i*RP + j*S + k -- the format targets beyond int8
 * are kept in, tg_demo_accumulate_i16).  target_bound >= max |target entry| (127 for an int8 slab) selects the packed
 * 16-bit arithmetic when target_bound + R * cmax^3 fits an int16.  Inputs and outputs move by TMA bulk copies; states may
 * start at any float (16-byte aligned batches leave with one bulk store per CTA).  Samples whose index is out of range
 * get all-zero states (scalars / actions / rewards untouched). */
int tg_demo_sample_dm(const uint8_t *tape_dm, const void *targets, int targets_i16, int target_bound, int64_t N, int R, int S,
                      int dim_t, int replay_shift, const int64_t *idx, int64_t nb, float *states, float *scalars, int64_t *actions,
                      float *rewards, void *stream);
/* step-major tape uint8 [R][N][TP] (byte stride tape_step_stride between steps) -> demo-major records uint8 [N][R][TP] */
int tg_tape_to_demo_major(const uint8_t *tape, int64_t tape_step_stride, uint8_t *tape_dm, int64_t N, int R, int S, void *stream);

/* ---- K6: rank reward ------------------------------------------------------ */
/* ranks[b] = sum_i rank(T_b[i,:,:]) -- get_rank (utils.py:134-140), the
 * terminal reward -get_rank of act.py:59,214.  Exact rank over Q for every
 * int8 slab (over GF(2^31-1), and over further 31-bit primes where a slice's
 * Hadamard bound exceeds the first) instead of the reference's float32 SVD. */
int tg_slice_rank(const int8_t *slab, int32_t *ranks, int64_t B, int S, void *stream);

/* ---- K7: state keys ------------------------------------------------------- */
/* 64-bit key per head tensor, replacing the string keys of utils.py:164-169
 * used by the MCTS tree (act.py:37,93,146,171,189,192,210): equal states <=>
 * equal keys (up to a ~2^-60 collision); the all-zero state has key 0.
 * key(T) = sum_{i,j,k} T[i][j][k] * A_i * B_j * C_k  (mod 2^64) with A_i = splitmix64(0x1000 + i) | 1,
 * B_j = splitmix64(0x2000 + j) | 1, C_k = splitmix64(0x3000 + k) | 1 -- the trilinear form of the state at three fixed
 * odd vectors: linear in T, and the key of a rank-1 action u (x) v (x) w is (sum u_i A_i)(sum v_j B_j)(sum w_k C_k),
 * which is how tg_expand_children keys a child without a pass over it.  (TG_VERSION 200 changed the constants.) */
int tg_state_key(const int8_t *slab, uint64_t *keys, int64_t B, int S, void *stream);

/* ---- int16 game path: K1, K8, K2, K7, K6 on int16 slabs (S in {4, 9, 16, 25}) ----------------------------------- */
/* The int16 twins of tg_step, tg_expand_children, tg_rollout, tg_replay, tg_state_key and tg_slice_rank, for residuals
 * the int8 slab cannot hold (tg_change_of_basis_i16 outputs, tg_demo_accumulate_i16 targets, start tensors with large
 * entries).  Same arguments, checks and outputs as the int8 twin, with int16 slabs [B][GP] of int16: entry (i,j,k) at
 * element i*RP + j*S + k, padding elements zero, 16-byte aligned.
 *   - Tokens: the same token bound (every token <= 2*shift, shift in [1,4], so |u v w| <= 64 per step); a record that
 *     breaks it raises TG_FLAG_RANGE (the game's result is then unspecified).
 *   - Zone: entries are guaranteed while they stay in [-16384, 16383] (the top two bits of a 16-bit lane are equal).
 *     A step whose result leaves the zone raises TG_FLAG_RANGE and is still exact; the next one is not guaranteed.
 *     tg_rollout_i16 / tg_replay_i16 test the zone after every applied step: RANGE = the start state or the state after
 *     an applied step had an entry outside the zone, or an applied step's record broke the token bound.
 *   - TG_FLAG_TERMINAL, TG_FLAG_NULL, nnz and steps mean what they mean on int8.
 *   - tg_state_key_i16 is tg_state_key's trilinear form over the int16 values: a state whose values fit int8 has the
 *     same key in both formats, so int8 and int16 nodes share one MCTS tree.  tg_expand_children_i16 keys its children
 *     by the same parent-minus-action rule as tg_expand_children.
 *   - tg_slice_rank_i16: exact rank over Q for every int16 slab (no zone), with up to fifteen 31-bit primes.
 * tg_expand_children_i16 holds a CTA's k records in shared memory and returns TG_E_ARG when they do not fit
 * (k above about 1200 at 25x25x25, more at the smaller sizes). */
int tg_step_i16(const int16_t *slab_in, const uint8_t *tape, int16_t *slab_out, uint8_t *flags, int32_t *nnz, int64_t B, int S,
                int shift, void *stream);
int tg_expand_children_i16(const int16_t *parents, const uint8_t *tape, int k, int16_t *children, uint8_t *flags, int32_t *nnz,
                           uint64_t *keys, int64_t B, int S, int shift, void *stream);
int tg_rollout_i16(const int16_t *slab_in, const uint8_t *tape, int64_t tape_step_stride, int K, int16_t *slab_out, uint8_t *flags,
                   int32_t *nnz, int32_t *steps, int64_t B, int S, int shift, void *stream);
int tg_replay_i16(const int16_t *slab_in, const uint8_t *tape, int64_t tape_step_stride, int K, int16_t *slab_out, uint8_t *flags,
                  int32_t *nnz, int64_t B, int S, int shift, void *stream);
int tg_state_key_i16(const int16_t *slab16, uint64_t *keys, int64_t B, int S, void *stream);
int tg_slice_rank_i16(const int16_t *slab16, int32_t *ranks, int64_t B, int S, void *stream);

/* ---- mod-2 game path: K1, K8, K2, K7, K6 on bit slabs (S in {4, 9, 16, 25}) ------------------------------------- */
/* The game over Z_2 (the AlphaTensor paper's "modular" arithmetic): T' = T xor (u (x) v (x) w mod 2).
 *   bit slab  uint32 [B][GB/4]  row i of a game is the S^2 bits (j,k) in RW = ceil(S^2/32) little-endian words: entry
 *                          (i,j,k) is bit (j*S+k) % 32 of word i*RW + (j*S+k)/32; padding bits and words are zero; games
 *                          are 16-byte aligned at GB = roundup16(4*S*RW) bytes (S=4: 1/16, S=9: 3/112, S=16: 8/512,
 *                          S=25: 20/2000 words per row / bytes per game).  In torch an int32 tensor [B][GB/4].
 *   Tapes are unchanged: token t stands for the coefficient t - shift (shift in [1,4], checked as on int8), whose residue
 *   is (t - shift) & 1.  Every byte is a valid token, so TG_FLAG_RANGE is never raised.
 *   Each entry point takes its int8 twin's arguments, checks and aliasing rules (in place allowed for step, rollout and
 *   replay), with bit slabs for slabs:
 *   - tg_step_gf2: TERMINAL = T' all zero; NULL = the term vanishes mod 2 (u, v or w has only even coefficients; then
 *     T' = T); nnz = popcount of T'.
 *   - tg_expand_children_gf2: k children per parent as tg_expand_children, keys optional.
 *   - tg_rollout_gf2 / tg_replay_gf2: tg_rollout / tg_replay (freeze at solved, steps, tape step stride); flags TERMINAL.
 *   - tg_state_key_gf2: tg_state_key of the 0/1 unpacking (the trilinear form over the values 0 and 1), so a mod-2 state
 *     and the int8 slab of its 0/1 values share a key.  tg_expand_children_gf2 keys its children the same way, from the
 *     child itself (parent-minus-action does not hold under xor).
 *   - tg_slice_rank_gf2: sum_i rank over GF(2) of T[i,:,:], the slices of tg_slice_rank.
 * Conversions: tg_pack_gf2 (int8 slab) and tg_pack_gf2_i16 (int16 slab) keep the low bit of each two's-complement entry
 * (-1 -> 1); tg_unpack_gf2 writes the int8 slab of 0/1 values (to float32 through tg_expand_f32).  tg_demo_accumulate
 * and tg_demo_gen_philox store the low byte of each entry and tg_demo_accumulate_i16 its int16 value, so packing their
 * targets gives the mod-2 sum of the tape, RANGE-flagged targets included (tg_demo_accumulate_tc saturates instead: its
 * targets keep their parity only where they fit int8). */
int tg_layout_gf2(int S, int *row_words, int *game_bytes);
int tg_pack_gf2(const int8_t *slab, uint32_t *bits, int64_t B, int S, void *stream);
int tg_pack_gf2_i16(const int16_t *slab16, uint32_t *bits, int64_t B, int S, void *stream);
int tg_unpack_gf2(const uint32_t *bits, int8_t *slab, int64_t B, int S, void *stream);
int tg_step_gf2(const uint32_t *bits_in, const uint8_t *tape, uint32_t *bits_out, uint8_t *flags, int32_t *nnz, int64_t B, int S,
                int shift, void *stream);
int tg_expand_children_gf2(const uint32_t *parents, const uint8_t *tape, int k, uint32_t *children, uint8_t *flags, int32_t *nnz,
                           uint64_t *keys, int64_t B, int S, int shift, void *stream);
int tg_rollout_gf2(const uint32_t *bits_in, const uint8_t *tape, int64_t tape_step_stride, int K, uint32_t *bits_out, uint8_t *flags,
                   int32_t *nnz, int32_t *steps, int64_t B, int S, int shift, void *stream);
int tg_replay_gf2(const uint32_t *bits_in, const uint8_t *tape, int64_t tape_step_stride, int K, uint32_t *bits_out, uint8_t *flags,
                  int32_t *nnz, int64_t B, int S, int shift, void *stream);
int tg_state_key_gf2(const uint32_t *bits, uint64_t *keys, int64_t B, int S, void *stream);
int tg_slice_rank_gf2(const uint32_t *bits, int32_t *ranks, int64_t B, int S, void *stream);

/* ---- change of basis mod 2: K5 over GF(2) on bit slabs (S in {4, 9, 16, 25}) -------------------------------------- */
/* The AlphaTensor augmentation of the game over Z_2: T'[i][j][k] = sum_abc A[i][a] B[j][b] C[k][c] T[a][b][c] mod 2 with
 * (A, B, C) invertible over GF(2), and the factors u' = A u, v' = B v, w' = C w of the same basis, so that a transformed
 * tape still sums to the transformed tensor.
 *   mats  uint32 [N or 1][3][S]  a triple (A, B, C) mod 2: word r of matrix f is row r, bit c is M[r][c] mod 2; bits S to
 *                          31 are ignored.  4-byte aligned; per_game != 0: one triple per game, otherwise one shared triple.
 *                          In torch an int32 tensor (N, 3, S).
 * Over GF(2) no entry and no token can leave its format, so none of the three takes a flags array.  Argument rules as on
 * the game path: a bad scalar (S, N < 0, R < 1, shift_in or shift_out outside [1, 4], p_nonzero outside [0, 1] or NaN)
 * returns TG_E_ARG; N == 0 returns TG_OK; a null pointer returns TG_E_ARG; bit slabs, tapes and step strides must be
 * 16-byte aligned and mats 4-byte aligned (TG_E_ARG). */
/* T' = T x1 A x2 B x3 C over GF(2); in place allowed; padding bits and words of the output zero */
int tg_change_of_basis_gf2(const uint32_t *bits_in, const uint32_t *mats, int per_game, uint32_t *bits_out, int64_t N, int S,
                           void *stream);
/* u' = A u, v' = B v, w' = C w over GF(2) for every record of a step-major tape uint8 [R][N][TP]: the residue of token t
 * is (t - shift_in) & 1, the output token is residue' + shift_out, padding bytes zero; in place allowed */
int tg_change_of_basis_factors_gf2(const uint8_t *tape_in, int64_t in_step_stride, int shift_in, const uint32_t *mats,
                                   int per_game, uint8_t *tape_out, int64_t out_step_stride, int shift_out, int64_t N, int R,
                                   int S, void *stream);
/* (A, B, C) per game, each L*U mod 2 and so invertible over GF(2) -> uint32 [N][3][S].  The draws of
 * tg_sample_unimodular (Philox ctr = (block, f, 0x6D617473, d_lo), the demo-stream key of (seed, d = first + n)): L[r][c]
 * = 1 below the diagonal and U[r][c] = 1 above it where the low 7 bits of the draw byte are below floor(128 p_nonzero),
 * both diagonals 1.  At S <= 16 the result is tg_sample_unimodular of the same arguments mod 2; at 25 the same recipe
 * reads 40 Philox blocks per matrix. */
int tg_sample_invertible_gf2(uint64_t seed, uint64_t first, int64_t N, int S, double p_nonzero, uint32_t *mats, void *stream);

/* ---- mod-2 training samples: K4 and the float32 conversion on bit slabs (S in {4, 9, 16, 25}) ---------------------- */
/* SyntheticDemoDataset.__getitem__ (datasets.py:77-122) modulo 2, from a demo-major store with bit-slab targets: the
 * arguments of tg_demo_sample_dm without targets_i16 and target_bound, the targets a bit slab [N][GB/4].  The records are
 * tg_demo_sample_dm's uint8 [N][R][TP]; token t has residue (t - replay_shift) & 1, replay_shift in [0, 8].  With
 * idx[b] = d*R + a and term(r) = (u mod 2) (x) (v mod 2) (x) (w mod 2) of record r of demo d:
 *   - slot 0 of states[b] = target_d xor term(a+1) xor ... xor term(R-1) (the target as given, so a target transformed
 *     by tg_change_of_basis_gf2 works too);
 *   - slot t, 1 <= t < dim_t, = term(hi - t) with hi = min(a + dim_t, R), zero where hi - t <= a;
 *   - entries 0.0f or 1.0f, dense (dim_t, S, S, S) per sample; states may start at any float;
 *   - scalars = R - a, actions = the record's 3S tokens as int64, rewards = -(a+1), as tg_demo_sample_dm writes them;
 *   - an index outside [0, N*R) gets all-zero states, its other outputs untouched.
 * Checks in tg_demo_sample_dm's order: a bad scalar (S, N < 0, R < 1, dim_t < 1, nb < 0) returns TG_E_ARG; nb == 0
 * returns TG_OK; a null pointer returns TG_E_ARG; tape_dm and the targets must be 16-byte aligned (TG_E_ARG); then
 * replay_shift outside [0, 8] returns TG_E_ARG.  Records are read from the store as they are replayed, so R has no upper
 * bound. */
int tg_demo_sample_gf2(const uint8_t *tape_dm, const uint32_t *targets_bits, int64_t N, int R, int S, int dim_t,
                       int replay_shift, const int64_t *idx, int64_t nb, float *states, float *scalars, int64_t *actions,
                       float *rewards, void *stream);
/* bit slab -> float32 dense (S,S,S) of 0.0f / 1.0f at dst + b*dst_stride: the state the model consumes;
 * tg_expand_f32(tg_unpack_gf2(bits)) in one pass.  The game path's argument rules (bits 16-byte aligned, dst 4-byte);
 * dst may start at any float, and floats outside each game's S^3 are not written. */
int tg_expand_f32_gf2(const uint32_t *bits, float *dst, int64_t dst_stride, int64_t B, int S, void *stream);

/* ---- mod-2 synthetic demonstrations: K3 with bit-slab targets (S in {4, 9, 16, 25}) -------------------------------- */
/* tg_demo_gen_philox modulo 2: the same arguments, with a bit slab [N][GB/4] (16-byte aligned) for the int8 slab.  Each
 * factor is an i.i.d. factor of the alphabet conditioned on having at least one ODD entry -- the reference's rejection
 * rule (utils.py:222-232) with "zero" read as "zero mod 2" -- so every term of a demo is a non-null action of the mod-2
 * game.  (tg_demo_gen_philox conditions on non-zero over Z: with an even value besides 0, such as 2 in {-2..2}, some of
 * its terms vanish mod 2.)  Demo d = first_demo + n is keyed by its global index, as there.
 *  v2 mod 2 (n_values <= 5, S <= 16, P(value even) <= 0.999): contract v2 with its groups, counters, 16-bit draws,
 *   128-bucket tables and Vose order; in the tilted table of group g EVERY outcome whose entries are all even is weighed
 *   by 1 - P(every later entry even), and "all groups so far even" selects the tilted tables.  max_tries does not apply.
 *  v1 mod 2 (other alphabets, and every alphabet at 25): contract v1's counters and draws; a try is rejected iff u, v or
 *   w has no odd entry; after max_tries tries the term is u = v = w = x e_0 with x the LAST ODD value of the alphabet,
 *   and the demo gets TG_FLAG_EXHAUSTED.
 * Writes the tape (tokens = value + shift, step-major [R][N][TP], padding zero, tape_step_stride as there), the bit
 * target = the xor of the R terms mod 2 (padding bits and words zero) and flags (may be NULL): TG_FLAG_EXHAUSTED or 0;
 * TG_FLAG_RANGE is never raised.  Checks in tg_demo_gen_philox's order: a bad scalar (S, N < 0, R outside [1, 65535],
 * shift outside [1, 4], n_values outside [1, 8], max_tries outside [1, 65535]) returns TG_E_ARG; N == 0 returns TG_OK;
 * a null values, probs, tape or bits returns TG_E_ARG; a misaligned tape, step stride or bit slab returns TG_E_ARG;
 * then a negative or NaN probability, a zero sum, a value outside [-shift, shift] or an alphabet with no odd value
 * returns TG_E_ARG.
 * Where 0 is the only even value (listed once) and, under v1, the last value is odd, the tables and the accept rule are
 * the integer ones: the tape is tg_demo_gen_philox's byte for byte, the bits are tg_pack_gf2 of its targets and the
 * EXHAUSTED flags are the same -- a mod-2 run and an integer run with one seed see the same demos. */
int tg_demo_gen_gf2(uint64_t seed, uint64_t first_demo, int64_t N, int R, int S, int shift, const int8_t *values,
                    const double *probs, int n_values, int max_tries, uint8_t *tape, int64_t tape_step_stride,
                    uint32_t *bits, uint8_t *flags, void *stream);
/* HOST function: the tables of v2 mod 2 in tg_demo_alias_tables' layout (uint16 [8][128]); TG_E_ARG where v2 mod 2 does
 * not apply (also at S = 25). */
int tg_demo_alias_tables_gf2(const int8_t *values, const double *probs, int n_values, int S, uint16_t *tables_host);

/* ---- K5: change-of-basis augmentation (S in {4, 9, 16}; TG_E_ARG at 25) ------ */
/* ABSENT from the reference; specified from the AlphaTensor paper (Methods,
 * "Change of basis"): T'[i][j][k] = sum_abc A[i][a] B[j][b] C[k][c] T[a][b][c].
 * mats: int8 [N or 1][3][S][S] = (A, B, C) row-major, one triple per game
 * (per_game != 0) or one shared triple.  slab_out must differ from slab_in.
 * flags (may be NULL): TG_FLAG_RANGE if an entry of T' left [-64,63] (the
 * int8 slab's guaranteed zone; the test is on the exact value, which for int8
 * input and int8 matrices can reach 2^40; the stored byte is its low byte). */
int tg_change_of_basis(const int8_t *slab_in, const int8_t *mats, int per_game, int8_t *slab_out, uint8_t *flags, int64_t N,
                       int S, void *stream);
/* The same contraction with the result as an int16 slab [N][GP] of int16 (entry (i,j,k) at element i*RP + j*S + k) --
 * SURVEY 8(d)'s format "int8 in, int16 out": unimodular matrices with off-diagonal density 0.3 take 16x16x16 residuals to
 * |T'| ~ 1000.  TG_FLAG_RANGE here means an entry does not fit int16.  The informational bits TG_FLAG_PATH_* say which
 * kernel computed each game (both entry points). */
int tg_change_of_basis_i16(const int8_t *slab_in, const int8_t *mats, int per_game, int16_t *slab16_out, uint8_t *flags, int64_t N,
                           int S, void *stream);
/* factors follow: u' = A u, v' = B v, w' = C w for every step of a step-major
 * tape; token' = coef' + shift_out.  ORs TG_FLAG_TOKEN_RANGE into flags[n] if a
 * transformed entry leaves [-shift_out, shift_out] (flags must be initialised). */
int tg_change_of_basis_factors(const uint8_t *tape_in, int64_t in_step_stride, int shift_in, const int8_t *mats, int per_game,
                               uint8_t *tape_out, int64_t out_step_stride, int shift_out, uint8_t *flags, int64_t N, int R,
                               int S, void *stream);
/* random unimodular triples M = L*U (L unit lower, U upper with +-1 diagonal,
 * off-diagonal entries -1/0/+1, P(non-zero) = p_nonzero quantised to 1/128),
 * Philox-keyed by (seed, first + n) like the demo stream -> int8 [N][3][S][S]. */
int tg_sample_unimodular(uint64_t seed, uint64_t first, int64_t N, int S, double p_nonzero, int8_t *mats, void *stream);

/* ---- host-buffer path (end-to-end through PCIe) -------------------------- */
typedef struct tg_host_ctx tg_host_ctx;
/* creates three streams, events and four device staging buffers for chunks of up to max_chunk games */
int tg_host_ctx_create(tg_host_ctx **ctx, int device, int S, int64_t max_chunk);
int tg_host_ctx_destroy(tg_host_ctx *ctx);
/* same contract as tg_step with HOST slabs/tapes/flags/nnz; chunks flow
 * through dedicated H2D / kernel / D2H streams chained by events per staging
 * buffer (both copy engines stream back to back); returns when done. */
int tg_step_host(tg_host_ctx *ctx, const int8_t *slab_in, const uint8_t *tape, int8_t *slab_out, uint8_t *flags,
                 int32_t *nnz, int64_t B, int shift);
/* tg_rollout with HOST buffers: the slab crosses PCIe once per K steps instead of once per step -- the case where the
 * caller holds the whole action list (SyntheticDemoDataset._take_actions, datasets.py:144-153).  tape is the dense
 * step-major host tape uint8 [K][B][TP]. */
int tg_rollout_host(tg_host_ctx *ctx, const int8_t *slab_in, const uint8_t *tape, int K, int8_t *slab_out, uint8_t *flags,
                    int32_t *nnz, int32_t *steps, int64_t B, int shift);
/* tg_demo_gen_philox into HOST buffers (dense step-major tape uint8 [R][N][TP], slab [N][GP], flags [N]): chunks are
 * generated on the device and copied out over three streams; the end-to-end form of utils.py:203-233 /
 * datasets.py:124-142 for a caller that wants the demonstrations in host memory. */
int tg_demo_gen_host(tg_host_ctx *ctx, uint64_t seed, uint64_t first_demo, int64_t N, int R, int shift, const int8_t *values,
                     const double *probs, int n_values, int max_tries, uint8_t *tape, int8_t *slab, uint8_t *flags);

#ifdef TG_TUNING
/* Sweep build only (-DTG_TUNING, libtensorgame_b200_tuning.so): CTAs launched per SM (0 = default) and kernel
 * variant of tg_step; the production library does not export them. */
int tg_tune_step_ctas_per_sm(int n);
int tg_tune_step_variant(int v);
#endif

#ifdef __cplusplus
}
#endif
#endif /* TENSORGAME_H */
