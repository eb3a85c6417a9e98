// Host emulation of the 3-robot throughput rollout WITH the shared robot-robot sphere leaves -- DEBUGGING AID FOR THE
// CPU TEST SUITE ONLY (see mrf_emul.cpp, which emulates the full leaf set).  Walks a CTA tile thread by thread: Phase A
// for every thread, barrier, stage 1 (pair_leaves_eval) for every pair lane, barrier, fabric_action with the leaf slots
// for every thread -- the order of the kernel's barriers.  Instantiated for FP64, it checks the pair algebra against
// the oracle; for FP32, it follows the kernel's arithmetic.
#include <vector>

#include "../../multi-robot-fabrics_b200/csrc/mrf_devcfg.h"

using namespace mrf;

template <typename T>
static int rollout_pair(const MrfConfig* mc, const double* rec, int N, double* avg, double* qN, double* qdN, long long B) {
    DevCfg<T> cfg;
    fill_devcfg(*mc, cfg);
    if (cfg.n_robots != 3 || !cfg.uniform_obst) return -1;
    constexpr int R = 3, NT = kTile * R;
    // the leaf slots follow the parameter blocks, as in the kernel's shared memory
    std::vector<T> kin((size_t)kKinRows<T> * NT), prm((size_t)(P_N + kPairRows) * NT), q((size_t)NT * 7),
        qd((size_t)NT * 7), acc(NT), pnum(NT);
    std::vector<Chain<T>> ch(NT);
    std::vector<char> pon(NT, 0);
    T* const pls = prm.data() + P_N * NT;
    const bool pair_cfg = kPairLeaves && pair_leaves_cfg(cfg);
    const T vref = cfg.static_or_dyn ? T(1) : T(0), aref = cfg.static_or_dyn ? cfg.sref : T(0);
    for (long long t0 = 0; t0 < B; t0 += kTile) {
        for (int tid = 0; tid < NT; ++tid) {
            const int lane = tid % kTile, r = tid / kTile;
            const long long b = t0 + lane, bb = b < B ? b : B - 1;
            auto ld = [&](int f) { return (T)rec[(bb * R + r) * MRF_REC + f]; };
            for (int i = 0; i < 7; ++i) {
                q[tid * 7 + i] = ld(MRF_Q + i);
                qd[tid * 7 + i] = ld(MRF_QD + i);
            }
            load_params<T>(ld, prm.data(), NT, tid);
            acc[tid] = 0;
        }
        for (int tid = 0; tid < NT; ++tid) pon[tid] = pair_cfg && pair_leaves_lane(prm.data(), NT, tid % kTile);
        for (int k = 0; k < N; ++k) {
            for (int tid = 0; tid < NT; ++tid) {
                for (int i = 0; i < 7; ++i) q[tid * 7 + i] += cfg.dt * qd[tid * 7 + i];
                chain_forward(cfg, tid / kTile, &q[tid * 7], &qd[tid * 7], ch[tid], kin.data(), NT, tid);
            }
            for (int tid = 0; tid < NT; ++tid)
                if (pon[tid]) pnum[tid] = pair_leaves_eval(cfg, tid / kTile, kin.data(), prm.data(), pls, NT, tid, tid % kTile);
            for (int tid = 0; tid < NT; ++tid) {
                const int lane = tid % kTile, r = tid / kTile;
                const long long b = t0 + lane;
                SmemSrcUniform<T, R> src{kin.data(), lane, r, vref, aref, cfg.r_obst};
                PairLeaves<T> pl{T(0), pon[tid] != 0};
                if (pl.on) pl.num = pnum[tid] + pls[2 * kPairSlots * NT + (r == 0 ? 2 : r - 1) * kTile + lane];
                T act[7];
                fabric_action(cfg, r, &q[tid * 7], &qd[tid * 7], ch[tid], kin.data(), prm.data(), NT, tid, src, act,
                              (T*)nullptr, &pl);
                for (int i = 0; i < 7; ++i) {
                    qd[tid * 7 + i] = act[i];
                    acc[tid] += act[i] * act[i];
                    if (b < B) {
                        if (qN) qN[(((b * R + r) * N) + k) * 7 + i] = q[tid * 7 + i];
                        if (qdN) qdN[(((b * R + r) * N) + k) * 7 + i] = act[i];
                    }
                }
            }
        }
        for (int tid = 0; tid < NT; ++tid) {
            const long long b = t0 + tid % kTile;
            if (avg && b < B) avg[b * R + tid / kTile] = acc[tid] / (T(N) * T(7));
        }
    }
    return 0;
}

extern "C" {
int emul_pair_rollout_f64(const MrfConfig* c, const double* rec, int N, double* avg, double* qN, double* qdN, long long B) { return rollout_pair<double>(c, rec, N, avg, qN, qdN, B); }
int emul_pair_rollout_f32(const MrfConfig* c, const double* rec, int N, double* avg, double* qN, double* qdN, long long B) { return rollout_pair<float>(c, rec, N, avg, qN, qdN, B); }
}
