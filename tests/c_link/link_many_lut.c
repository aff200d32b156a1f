/* Plain-C consumer of include/tfhe_b200_many_lut.h: the many-LUT header is self-sufficient C and every entry point it declares resolves in
 * libtfhe_b200.so.  Runs without a GPU: it takes the address of each entry point and checks the argument refusals that need no context. */
#include <stdio.h>
#include "tfhe_b200_many_lut.h"

typedef void (*any_fn)(void);
#define ADDR(f) do { any_fn p = (any_fn)(f); if (!p) { printf("missing %s\n", #f); return 2; } n_syms++; } while (0)

int main(void) {
    int n_syms = 0;
    ADDR(tfhe_b200_upload_many_luts); ADDR(tfhe_b200_pbs_many_batch); ADDR(tfhe_b200_pbs_many_batch_partial);
    ADDR(tfhe_b200_ks_pbs_many_batch); ADDR(tfhe_b200_pbs_many_batch_device); ADDR(tfhe_b200_ks_pbs_many_batch_device);
    uint32_t fn[1] = {2};
    if (tfhe_b200_upload_many_luts(NULL, NULL, 1, fn) == 0) return 3;          /* null context and table: refused with a message */
    printf("upload_many_luts(NULL): %s\n", tfhe_b200_last_error());
    if (tfhe_b200_pbs_many_batch(NULL, NULL, NULL, NULL, 1) == 0) return 4;
    printf("ok: %d symbols resolved\n", n_syms);
    return 0;
}
