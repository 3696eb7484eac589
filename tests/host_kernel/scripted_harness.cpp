// scripted_harness.cpp -- TEST INFRASTRUCTURE. The harness of harness.cpp plus the scripted player
// of inv_scripted_actions (load_board + scripted_action of csrc/inversus_kernels.cuh), compiled for
// the host through host_shim.h. See tests/test_scripted_host.py.
#include "harness.cpp"

extern "C" {

// The scripted player of inv_scripted_actions for `seat` on env 0..n-1 (same decode, same device
// function); out[i] = its action id.
int hk_scripted_actions(const uint32_t *planes, int64_t n, int seat, int difficulty, uint64_t seed,
                        uint32_t env_id_base, int8_t *out)
{
    Params p;
    memset(&p, 0, sizeof(p));
    p.seed_lo = (uint32_t)seed;
    p.seed_hi = (uint32_t)(seed >> 32);
    for (int64_t i = 0; i < n; ++i) {
        Env s;
        load_board(s, reinterpret_cast<const uint4 *>(planes), n, i);
        out[i] = (int8_t)scripted_action(s, p, env_id_base + (uint32_t)i, seat, difficulty);
    }
    return 0;
}

} // extern "C"
