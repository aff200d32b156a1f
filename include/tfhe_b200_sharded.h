/*
 * tfhe_b200_sharded.h -- C ABI of the sharded program executor of libtfhe_b200.so: any program recorded with tfhe_b200_program_build,
 * run across the ranks of a tfhe_b200_exchange (one process per GPU, or every rank of one GPU in one call).  Same conventions as
 * tfhe_b200.h: int return, 0 = success, the message of a failure in tfhe_b200_last_error.
 */
#ifndef TFHE_B200_SHARDED_H
#define TFHE_B200_SHARDED_H
#include "tfhe_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ---- multi-GPU: any recorded program across the ranks of an exchange -----------------------------------------------------------------
 * A level of w PBS jobs with w > min_shard_width (and world > 1) is split: rank r keyswitches and bootstraps jobs [lo_r, hi_r) only
 * (contiguous, balanced, the first w % world ranks take one more; shares may be empty), its PBS writes them into its exchange send area,
 * and one scatter kernel per split level pulls every rank's share over peer memory into every rank's arena.  Every other level and every
 * linear instruction runs in full on every rank, with no communication.  The plan depends only on (program, world, min_shard_width).
 *   shard_plan: out = {split levels, largest share in rows (the exchange needs max_rows >= it), rows each rank receives}
 *   level_share: out = {lo, hi, split} of `rank` in level `level` ([0, width) and split = 0 for a replicated level)
 *   run_sharded: one rank per GPU (one process each, or attach_local across GPUs); every rank passes all inputs and receives all outputs
 *     (device buffers, enqueued on cuda_stream, NULL = the context's stream, without synchronising).  Every rank must run the same
 *     program with the same min_shard_width.
 *   run_sharded_group: all `world` ranks on ONE GPU in one call on one stream; rank r brings its own context, program object and exchange.
 * The send area of the exchange is double-buffered: 2 x max_rows x (k*N+1) x 8 bytes per rank.  program_last_ms covers the whole run,
 * exchanges included. */
int tfhe_b200_program_shard_plan(const tfhe_b200_program *prog, uint32_t world, uint64_t min_shard_width, uint64_t out[3]);
int tfhe_b200_program_level_share(const tfhe_b200_program *prog, uint32_t level, uint32_t rank, uint32_t world, uint64_t min_shard_width,
                                  uint64_t out[3]);
int tfhe_b200_program_run_sharded(tfhe_b200_ctx *ctx, tfhe_b200_program *prog, tfhe_b200_exchange *ex, const uint64_t *d_inputs,
                                  uint64_t *d_outputs, uint64_t min_shard_width, void *cuda_stream);
int tfhe_b200_program_run_sharded_group(tfhe_b200_ctx *const *ctxs, tfhe_b200_program *const *progs, tfhe_b200_exchange *const *exs,
                                        uint32_t world, const uint64_t *const *d_inputs, uint64_t *const *d_outputs, uint64_t min_shard_width,
                                        void *cuda_stream);

#ifdef __cplusplus
}
#endif
#endif
