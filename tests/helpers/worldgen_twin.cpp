// Host-compiled twin of csrc/d2d_worldgen.cuh for the CPU test-suite (tests/test_worldgen_host.py).
// Build: g++ -O2 -ffp-contract=off -shared -fPIC (no FMA contraction: same arithmetic as nvcc -fmad=false).
#include <vector>
#include "../../gym_drone2d_activeperception_b200/csrc/d2d_worldgen.cuh"

extern "C" {
long wt_sizeof_source(void) { return (long)sizeof(d2d_world_source); }

// The worlds of seeds[0..n) into env-major arrays laid out as world.generate_worlds returns them (gt as 50 row bitmasks).
// Returns 0, a positive count of seeds given up (their fail[] entry is 1), or -1 with the reason in *why.
long wt_generate(const d2d_world_source *src, const double *targets, int n_targets, double scale, int num_agents, int rvo,
                 int noisy, const uint32_t *seeds, long n, double *apos, double *apref, double *arad, double *trad,
                 uint64_t *gt_rows, double *pose, uint32_t *rng_key, double *avel, double *obs, int *nobs, int *fail,
                 const char **why) {
    std::vector<unsigned char> buf(sizeof(WgTables));
    WgTables *T = (WgTables *)buf.data();
    *why = wg_build_tables(T, src, (const double(*)[2])targets, n_targets, scale, num_agents, rvo, noisy);
    if (*why) return -1;
    const long N = num_agents;
    long failed = 0;
    for (long i = 0; i < n; i++) {
        fail[i] = wg_generate_host(*T, seeds[i], apos + i * N * 2, apref + i * N * 2, arad + i * N, trad + i * N, gt_rows + i * 50,
                                   pose + i * 3, rng_key + (noisy ? i * 624 : 0), avel + (rvo ? i * N * 2 : 0),
                                   obs + (rvo ? i * 48 : 0), nobs + (rvo ? i : 0)) != 0;
        failed += fail[i];
    }
    return failed;
}
}
