/*
 * tfhe_b200_many_lut.h -- C ABI of the many-LUT PBS of libtfhe_b200.so: several functions of one input from one keyswitch and one
 * blind rotation.  Same conventions as tfhe_b200.h: int return, 0 = success, the message of a failure in tfhe_b200_last_error.
 */
#ifndef TFHE_B200_MANY_LUT_H
#define TFHE_B200_MANY_LUT_H
#include "tfhe_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* These entries are declared here rather than in tfhe_b200.h so that the C-linkage checks of that header stay as they are; this header
 * includes it.
 *
 * Many-LUT PBS: several functions of one input from one keyswitch and one blind rotation (tfhe-rs ServerKey::generate_many_lookup_table
 * and apply_many_lookup_table, shortint/server_key/mod.rs).  With total = msg_mod * carry_mod, box = N / total, F functions and
 * chunk = total / F (integer division), accumulator l holds f_f(x) * Delta in box f * chunk + x for x < chunk, 0 in the boxes from
 * F * chunk on, then the same half-box rotation (and negation of the first half box) as generate_lookup_table.  Function f is extracted
 * at monomial f * chunk * box.  The input's degree must be below chunk; every output has the noise of one PBS.
 *
 * upload_many_luts     n_luts accumulators of (k + 1) * N words and their function counts fn_count[l] in 2 ... total.  Replaces the
 *                      uploaded lookup tables: until tfhe_b200_upload_luts is called again, the single-function batch entries
 *                      (pbs_batch, ks_pbs_batch, pbs_ks_batch, their _device and _partial forms) refuse to run.
 * pbs_many_batch       apply_many_lookup_table on small-key inputs; ks_pbs_many_batch keyswitches big-key inputs first (as
 *                      ks_pbs_batch).  Output: batch x S rows of k * N + 1 words, S = the largest fn_count of the table; function f of
 *                      ciphertext i is row i * S + f.  With one function count F for every table, S = F and this is row i * F + f.
 *                      Tables of different F may be mixed in one batch; the rows of ciphertext i past its own table's F are zero in
 *                      the host entries and left untouched by the _device entries.  lut_idx as for pbs_batch.
 * _partial             test hook as tfhe_b200_pbs_batch_partial. */
int tfhe_b200_upload_many_luts(tfhe_b200_ctx *ctx, const uint64_t *accs, uint32_t n_luts, const uint32_t *fn_count);
int tfhe_b200_pbs_many_batch(tfhe_b200_ctx *ctx, const uint64_t *lwe_small, const uint32_t *lut_idx, uint64_t *lwe_big_rows,
                             size_t batch);
int tfhe_b200_pbs_many_batch_partial(tfhe_b200_ctx *ctx, const uint64_t *lwe_small, const uint32_t *lut_idx, uint64_t *lwe_big_rows,
                                     size_t batch, uint32_t n_iters);
int tfhe_b200_ks_pbs_many_batch(tfhe_b200_ctx *ctx, const uint64_t *lwe_big_in, const uint32_t *lut_idx, uint64_t *lwe_big_rows,
                                size_t batch);
int tfhe_b200_pbs_many_batch_device(tfhe_b200_ctx *ctx, const uint64_t *d_lwe_small, const uint32_t *d_lut_idx,
                                    uint64_t *d_lwe_big_rows, size_t batch, void *cuda_stream);
int tfhe_b200_ks_pbs_many_batch_device(tfhe_b200_ctx *ctx, const uint64_t *d_lwe_big_in, const uint32_t *d_lut_idx,
                                       uint64_t *d_lwe_big_rows, size_t batch, void *cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* TFHE_B200_MANY_LUT_H */
