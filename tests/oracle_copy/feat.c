/* Test helper: branching for the C oracle of oracle/features_oracle.c, compiled into a helper library of its own by
 * tests/test_checkpoint.py.  The oracle's source is included unchanged, so the structs below have its exact layout and
 * the function works on handles the oracle library created.  Env dst[i] takes the whole state of env src[i] (all
 * sources are read before any destination is written: the sets may overlap) and keeps its own env_id, i.e. continues
 * on its own random stream; seed, configuration and the static tables are the same for every env of a batch. */
#include "../../oracle/features_oracle.c"

int feat_oracle_copy_envs(void* h, const int32_t* src, const int32_t* dst, int count)
{
    fbatch* b = (fbatch*)h;
    fenv* tmp = (fenv*)malloc((size_t)(count > 0 ? count : 1) * sizeof(fenv));
    if (!tmp) return -1;
    for (int i = 0; i < count; i++) tmp[i] = b->envs[src[i]];
    for (int i = 0; i < count; i++) {
        fenv* d = &b->envs[dst[i]];
        const uint32_t id = d->env_id;
        *d = tmp[i];
        d->env_id = id;
    }
    free(tmp);
    return 0;
}
