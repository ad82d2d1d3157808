/* Plain-C client of the data-parallel PPO entry points of libb200env.so: they resolve, b2e_config keeps its size with
 * env_base in place of the reserved word, and the argument checks that need no GPU report as documented.  Built and run
 * by tests/test_ppo_dist_host.py. */
#include <dlfcn.h>
#include <stdio.h>
#include <string.h>

#include "b200env.h"
#include "b200policy.h"

#define RESOLVE(name)                                        \
    do {                                                     \
        if (!dlsym(lib, #name)) {                            \
            fprintf(stderr, "missing symbol %s\n", #name);   \
            return 2;                                        \
        }                                                    \
    } while (0)

int main(int argc, char **argv) {
    void *lib;
    size_t (*partial_size)(b2p_handle);
    int (*adv_combine)(const double *, int, int64_t, double *, void *);
    int (*adv_moments)(const b2p_ppo_batch *, uint64_t, int64_t, double *, void *, void *);
    int (*combine)(b2p_handle, const double *, int, int64_t, float, float, float, float *, double *, void *);
    int (*env_create)(const b2e_config *, b2e_handle *);
    const char *(*policy_error)(b2p_handle);
    const char *(*env_error)(b2e_handle);
    double host[8];
    b2e_config cfg;
    b2e_handle env = NULL;
    if (argc < 2) return 64;
    lib = dlopen(argv[1], RTLD_NOW);
    if (!lib) { fprintf(stderr, "%s\n", dlerror()); return 1; }
    RESOLVE(b2p_set_row_base); RESOLVE(b2p_ppo_partial_size); RESOLVE(b2p_ppo_grad_partial); RESOLVE(b2p_ppo_combine);
    RESOLVE(b2p_ppo_adv_moments); RESOLVE(b2p_ppo_adv_combine);
    if (sizeof(b2e_config) != 4 * 20 + 4 * B2E_MAX_LAYERS + 8) return 3;
    *(void **)&partial_size = dlsym(lib, "b2p_ppo_partial_size");
    *(void **)&adv_combine = dlsym(lib, "b2p_ppo_adv_combine");
    *(void **)&adv_moments = dlsym(lib, "b2p_ppo_adv_moments");
    *(void **)&combine = dlsym(lib, "b2p_ppo_combine");
    *(void **)&env_create = dlsym(lib, "b2e_create");
    *(void **)&policy_error = dlsym(lib, "b2p_last_error");
    *(void **)&env_error = dlsym(lib, "b2e_last_error");
    /* argument errors are reported before any CUDA call */
    if (partial_size(NULL) != 0) return 4;
    if (combine(NULL, host, 1, 1, 0.f, 0.f, 0.f, NULL, NULL, NULL) == 0) return 5;
    if (adv_combine(host, 0, 1, host, NULL) == 0 || !strstr(policy_error(NULL), "ranks must be")) return 6;
    if (adv_combine(NULL, 1, 1, host, NULL) == 0 || !strstr(policy_error(NULL), "null")) return 7;
    if (adv_moments(NULL, 1, 1, host, host, NULL) == 0 || !strstr(policy_error(NULL), "b2p_ppo_adv_moments")) return 8;
    memset(&cfg, 0, sizeof(cfg));
    cfg.struct_size = (int32_t)sizeof(cfg);
    cfg.env_kind = B2E_ENV_MULTIOPTLRS; cfg.problem_kind = B2E_PROBLEM_FUNC;
    cfg.history_version = 3; cfg.observation_version = 3;
    cfg.num_envs = 4; cfg.max_history = 5; cfg.max_batches = 10;
    cfg.env_base = -1;
    if (env_create(&cfg, &env) == 0 || !strstr(env_error(NULL), "env_base")) return 9;
    cfg.env_base = 0x7FFFFFFF - 3;
    if (env_create(&cfg, &env) == 0 || !strstr(env_error(NULL), "env_base")) return 10;
    printf("c dist abi ok\n");
    return 0;
}
