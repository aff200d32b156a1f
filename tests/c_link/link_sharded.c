/* Plain-C consumer of include/tfhe_b200_sharded.h: the header of the sharded program executor is self-sufficient C and every entry point
 * it declares resolves in libtfhe_b200.so.  Runs without a GPU: it takes the address of the entry points that need one and computes the
 * shard plan of a recorded program, which is pure host arithmetic. */
#include <stdio.h>
#include "tfhe_b200_sharded.h"

typedef void (*any_fn)(void);
#define ADDR(f) do { any_fn p = (any_fn)(f); if (!p) { printf("missing %s\n", #f); return 2; } n_syms++; } while (0)

int main(void) {
    int n_syms = 0;
    ADDR(tfhe_b200_program_shard_plan); ADDR(tfhe_b200_program_level_share); ADDR(tfhe_b200_program_run_sharded);
    ADDR(tfhe_b200_program_run_sharded_group);

    /* PARAM_MESSAGE_2_CARRY_2_KS_PBS; string_eq(8, 8) has levels [32, 3, 1] */
    tfhe_b200_params p = {742, 1, 2048, 23, 1, 3, 5, 0, 4, 4};
    tfhe_b200_program *prog = NULL;
    uint64_t args[2] = {8, 8};
    if (tfhe_b200_program_build(&p, "string_eq", args, 2, NULL, &prog) != 0 || !prog) { printf("program_build: %s\n", tfhe_b200_last_error()); return 3; }
    uint64_t plan[3], share[3];
    if (tfhe_b200_program_shard_plan(prog, 3, 2, plan) != 0) return 4;
    printf("string_eq(8, 8) at world 3, min_shard_width 2: %llu split levels, largest share %llu, %llu rows received\n",
           (unsigned long long)plan[0], (unsigned long long)plan[1], (unsigned long long)plan[2]);
    if (plan[0] != 2 || plan[1] != 11 || plan[2] != 35) return 5;
    if (tfhe_b200_program_level_share(prog, 0, 2, 3, 2, share) != 0 || share[0] != 22 || share[1] != 32 || share[2] != 1) return 6;
    if (tfhe_b200_program_level_share(prog, 2, 1, 3, 2, share) != 0 || share[0] != 0 || share[1] != 1 || share[2] != 0) return 7;
    if (tfhe_b200_program_level_share(prog, 3, 0, 3, 2, share) == 0) return 8;      /* no such level: refused with a message */
    tfhe_b200_program_destroy(prog);
    printf("ok: %d symbols resolved\n", n_syms);
    return 0;
}
