// mrf_b200.cu -- __global__ kernels and the C-ABI (include/mrf_b200.h) of the B200-native
// multi-robot-fabrics hot path.  Build: see __graft_entry__.build()
//   nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -shared ...
//
// Kernels
//   rollout_kernel<T>   coupled joint-space Rollout Fabrics (RF / RF-CV), persistent over the horizon.
//                       CTA = R warps x 32 lanes; warp r = robot r, lane = scenario of the CTA's 32-scenario
//                       tile.  Every step each thread re-computes its own chain (Phase A), publishes its five
//                       moving link points through shared memory, and evaluates its fabric action against the
//                       other robots' points (Phase B).  Reference: ForwardFabricsPlanner
//                       multi_robot_fabrics/fabrics_planner/forward_planner_Jointspace.py:118-296,298-423.
//   action_kernel<T>    one fabric action per (scenario, robot) against caller-supplied obstacle spheres.
//                       Reference: planner.compute_action, examples/example_pandas_Jointspace.py:417-445.
//   cart_kernel<T>      decoupled rollout with constant-velocity obstacles.  Reference: FabricsRollouts
//                       multi_robot_fabrics/fabrics_planner/forward_planner_Cartesian.py:347-489.
//   kinematics_kernel   fk / J qdot / Jdot qdot of the 8 collision links (utils.py:16-54).
//   deadlock_kernel     deadlockprevention.deadlock_checking (others_planner/deadlock_prevention.py:50-118).
//   transpose kernels   AoS <-> SoA staging for the host-pointer entries.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "../../include/mrf_b200.h"
#include "mrf_device.cuh"
#include "mrf_devcfg.h"
#include "mrf_coop.cuh"

namespace mrf {

// ------------------------------------------------------------------------------------------------
// deadlock heuristic, one thread per scenario (deadlock_prevention.py:50-118)
// ------------------------------------------------------------------------------------------------
struct DlCfg {
    // goal element (robot i, component k, scenario b) at goals[i * g_sr + k * g_sc + b]; weight at weights[i * w_sr + b]
    long long g_sr, g_sc, w_sr;
    int est_robot; // >= 0: goals of this robot are first overwritten by goal_est (RF-CV), -1: off
    int R, time_wait, time_gate;
    double avg_vel_constant, dist_constant, w_follower, w_leader, goal_scale, dist_endeff, backoff;
};

// Euclidean norm exactly as numpy computes it for a 3-vector (np.linalg.norm -> sqrt(x.dot(x)), OpenBLAS ddot: an
// FMA-chained accumulation; checked against numpy on 200 000 random vectors) -- explicit rounding intrinsics so the
// compiler can neither fuse nor un-fuse anything; the follower goal then matches the reference bit for bit.
__device__ __forceinline__ double np_norm3(double x, double y, double z) {
    return __dsqrt_rn(__fma_rn(z, z, __fma_rn(y, y, __dmul_rn(x, x))));
}

// Optional FP64 overrides for scenarios the FP32 rollout could not decide safely (see guard_select_one): slot[b] >= 0
// selects column slot[b] of the compact FP64 results avg [R][cap], x_ee [R][3][cap], goal_est [3][cap].
struct DlOverride {
    const int* slot;
    const double* avg;
    const double* x_ee;
    const double* goal_est;
    long long cap;
    unsigned* counters; // the list counter is reset once its consumers are done
};

// One scenario of the heuristic.  os >= 0: this scenario was re-rolled in FP64, its rollout outputs are column os of the
// compact arrays of `ov`.
template <typename T>
__device__ __forceinline__ void deadlock_one(const DlCfg& c, long long b, long long B, int os, const DlOverride& ov,
                                             const T* __restrict__ x_ee, T* __restrict__ goals, T* __restrict__ weights,
                                             const T* __restrict__ avg_vel, const T* __restrict__ avg_sum_in,
                                             const int* __restrict__ sm_state, const int* __restrict__ time_step,
                                             int* __restrict__ tdo, int* __restrict__ st_int, T* __restrict__ st_goal,
                                             int* __restrict__ flag, const T* __restrict__ goal_est, T* __restrict__ result) {
    const int R = c.R;
    if (c.est_robot >= 0 && goal_est != nullptr) // goal_pandas[1] = estimate (example_pandas_Jointspace.py:346-348)
        for (int k = 0; k < 3; ++k)
            goals[c.est_robot * c.g_sr + k * c.g_sc + b] = os >= 0 ? (T)ov.goal_est[k * ov.cap + os] : goal_est[(long long)k * B + b];
    // the reference does this arithmetic in float64 whatever the planner precision
    double x[MRF_MAX_ROBOTS][3], g[MRF_MAX_ROBOTS][3], dist_goal[MRF_MAX_ROBOTS];
    int st[MRF_MAX_ROBOTS];
    double avg_sum = 0.0;
    for (int i = 0; i < R; ++i) {
        for (int k = 0; k < 3; ++k) {
            x[i][k] = os >= 0 ? ov.x_ee[((long long)i * 3 + k) * ov.cap + os] : (double)x_ee[((long long)i * 3 + k) * B + b];
            g[i][k] = (os >= 0 && i == c.est_robot && goal_est != nullptr) ? ov.goal_est[k * ov.cap + os]
                                                                           : (double)goals[i * c.g_sr + k * c.g_sc + b];
        }
        dist_goal[i] = np_norm3(__dsub_rn(x[i][0], g[i][0]), __dsub_rn(x[i][1], g[i][1]), __dsub_rn(x[i][2], g[i][2]));
        st[i] = sm_state[(long long)i * B + b];
        if (avg_vel) {
            const double a = os >= 0 ? ov.avg[(long long)i * ov.cap + os] : (double)avg_vel[(long long)i * B + b];
            avg_sum += a;
            if (result) result[(long long)i * B + b] = (T)a;
        }
    }
    // vel_avg_tot = sum(vel_avg)/nr_robots (example_pandas_Jointspace.py:375), or the caller's scalar
    avg_sum = avg_vel ? avg_sum / (double)R : (double)avg_sum_in[b];
    const int ts = time_step[b];
    int t_out = tdo[b];
    int i_leader = st_int[0 * B + b], i_follower = st_int[1 * B + b];
    int dead0 = st_int[2 * B + b], dead1 = st_int[3 * B + b];
    bool deadlock = false;
    double min_dist = 100.0; // deadlock_distance initial value / deadlock_min_dist (:57,74)
    for (int a = 0; a < R; ++a)
        for (int bq = a + 1; bq < R; ++bq) { // itertools.combinations order (:29-30)
            double dsum = __dadd_rn(dist_goal[a], dist_goal[bq]);
            bool check_state = (st[a] == 0 || st[a] == 1) && (st[bq] == 0 || st[bq] == 1);
            double de = np_norm3(__dsub_rn(x[a][0], x[bq][0]), __dsub_rn(x[a][1], x[bq][1]), __dsub_rn(x[a][2], x[bq][2]));
            if (avg_sum < c.avg_vel_constant && dsum > c.dist_constant && ts > c.time_gate && check_state &&
                de < c.dist_endeff) {
                deadlock = true;
                // after each hit the reference rescans all pairs for the minimum recorded distance with a
                // strict '<' (:74-80): the first pair reaching the minimum wins
                if (de < min_dist) {
                    min_dist = de;
                    dead0 = a;
                    dead1 = bq;
                }
            }
        }
    int fl = 0;
    double g0[3] = {(double)st_goal[0 * B + b], (double)st_goal[1 * B + b], (double)st_goal[2 * B + b]};
    bool apply = false;
    if (deadlock && ts > c.time_gate) {
        fl = 1;
        if (dist_goal[dead0] > dist_goal[dead1]) {
            i_leader = dead1;
            i_follower = dead0;
        } else {
            i_leader = dead0;
            i_follower = dead1;
        }
        double d[3], dg[3];
        for (int k = 0; k < 3; ++k) {
            d[k] = __dsub_rn(x[i_leader][k], x[i_follower][k]);
            dg[k] = __dmul_rn(d[k], c.goal_scale);
        }
        const double nrm = np_norm3(dg[0], dg[1], dg[2]);
        const double sc = __ddiv_rn(c.backoff, nrm);       // 0.3 / norm, then elementwise * and - as numpy does
        for (int k = 0; k < 3; ++k)
            g0[k] = nrm > 0.05 ? __dsub_rn(x[i_follower][k], __dmul_rn(sc, dg[k]))
                               : __dsub_rn(x[i_follower][k], __dmul_rn(d[k], c.goal_scale));
        if (g0[2] < 0.0) g0[2] = 0.1;
        apply = true;
        t_out = 0;
    } else if (st[dead0] == 2 || st[dead1] == 2) {
        t_out = 400;
    } else if (t_out < c.time_wait) {
        apply = true;
        t_out = t_out + 1;
    }
    if (apply) {
        weights[i_leader * c.w_sr + b] = (T)c.w_leader;
        weights[i_follower * c.w_sr + b] = (T)c.w_follower;
        for (int k = 0; k < 3; ++k) goals[i_follower * c.g_sr + k * c.g_sc + b] = (T)g0[k];
    }
    tdo[b] = t_out;
    st_int[0 * B + b] = i_leader;
    st_int[1 * B + b] = i_follower;
    st_int[2 * B + b] = dead0;
    st_int[3 * B + b] = dead1;
    for (int k = 0; k < 3; ++k) st_goal[k * B + b] = (T)g0[k];
    if (flag) flag[b] = fl;
    if (result) result[(long long)R * B + b] = (T)fl; // what a sweep gathers per scenario: avg_vel[R] and the flag
}

template <typename T>
__global__ void deadlock_kernel(DlCfg c, const T* __restrict__ x_ee, T* __restrict__ goals, T* __restrict__ weights,
                                const T* __restrict__ avg_vel, const T* __restrict__ avg_sum_in,
                                const int* __restrict__ sm_state,
                                const int* __restrict__ time_step, int* __restrict__ tdo, int* __restrict__ st_int,
                                T* __restrict__ st_goal, int* __restrict__ flag, const T* __restrict__ goal_est,
                                long long B, DlOverride ov, T* __restrict__ result) {
    // grid-stride over the scenarios: a few fat CTAs instead of B / 128 thin ones -- next to a sweep whose rollout kernels
    // fill every SM's register file, each CTA of a small kernel delays one rollout CTA slot at a wave boundary
    if (ov.counters != nullptr && blockIdx.x == 0 && threadIdx.x == 0) ov.counters[0] = 0; // list consumed (same stream order)
    for (long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += (long long)gridDim.x * blockDim.x)
        deadlock_one<T>(c, b, B, ov.slot != nullptr ? ov.slot[b] : -1, ov, x_ee, goals, weights, avg_vel, avg_sum_in, sm_state,
                        time_step, tdo, st_int, st_goal, flag, goal_est, result);
}

// ------------------------------------------------------------------------------------------------
// "deadlock flags identical" for the FP32 path.  The heuristic compares rollout outputs with thresholds
// (deadlock_prevention.py:61-66: vel_avg_tot < 0.16, ee distance < 0.35) and with each other (:76,85: closest pair,
// leader = closer to its goal); an FP32 rollout answers those tests like the reference's float64 one unless a value sits
// within the FP32 error of the threshold.  guard_select_one lists exactly those scenarios -- a narrow band for
// ordinary scenarios, a wide one for numerically stiff ones (risk = max over the horizon of the summed leaf metric:
// near contact the explicit dt = 0.01 integration amplifies rounding) and anything non-finite; they are re-rolled by the
// FP64 kernel from the same records and the deadlock kernel reads the FP64 values for them (DlOverride).
// ------------------------------------------------------------------------------------------------
struct GuardCfg {
    int R, est_robot;
    double c_avg, c_dist, band_dist;
    double band[3], rel[3], edge[2]; // |vel_avg_tot - c_avg| <= band[t] + rel[t] vel_avg_tot, tier t = (risk >= edge[0]) + (risk >= edge[1])
    unsigned cap;
};
// counters: [0] listed this call (may exceed cap), [1] not used, [2] cumulative re-rolled, [3] cumulative overflow
// One scenario of the selection; returns its slot in the list (-1: not listed, or the list is full).
template <typename T>
__device__ __forceinline__ int guard_select_one(const GuardCfg& c, long long b, long long B, const T* __restrict__ avg_vel,
                                                const T* __restrict__ x_ee, const T* __restrict__ rec,
                                                const T* __restrict__ goal_est, const T* __restrict__ risk,
                                                const int* __restrict__ sm_state, const int* __restrict__ time_step,
                                                int time_gate, double dist_constant, unsigned* __restrict__ counters,
                                                int* __restrict__ list) {
    const int R = c.R;
    const long long RB = (long long)R * B;
    double s = 0.0, rk = 0.0, x[MRF_MAX_ROBOTS][3], dg[MRF_MAX_ROBOTS];
    int st[MRF_MAX_ROBOTS];
    for (int i = 0; i < R; ++i) {
        s += (double)avg_vel[(long long)i * B + b];
        if (risk) rk = fmax(rk, (double)risk[(long long)i * B + b]);
        st[i] = sm_state[(long long)i * B + b];
        double d2 = 0.0;
        for (int k = 0; k < 3; ++k) {
            x[i][k] = (double)x_ee[((long long)i * 3 + k) * B + b];
            const double g = (i == c.est_robot && goal_est != nullptr) ? (double)goal_est[(long long)k * B + b]
                                                                       : (double)rec[(MRF_G0 + k) * RB + (long long)i * B + b];
            d2 += (x[i][k] - g) * (x[i][k] - g);
        }
        dg[i] = sqrt(d2);
    }
    s /= (double)R;
    // Only a scenario with a candidate pair -- both robots in state 0 / 1, hands closer than the distance threshold (plus
    // the band), goal distances above the constant, time gate open (deadlock_prevention.py:61-66) -- can raise the flag at
    // all; for every other scenario the velocity test is never consulted and nothing needs FP64.
    bool cand = false, knife = false;
    double de[MRF_MAX_ROBOTS * (MRF_MAX_ROBOTS - 1) / 2];
    int np = 0;
    if (time_step[b] > time_gate) {
        for (int a = 0; a < R; ++a)
            for (int q = a + 1; q < R; ++q) {
                if (!((st[a] == 0 || st[a] == 1) && (st[q] == 0 || st[q] == 1))) continue;
                const double d = sqrt((x[a][0] - x[q][0]) * (x[a][0] - x[q][0]) + (x[a][1] - x[q][1]) * (x[a][1] - x[q][1]) +
                                      (x[a][2] - x[q][2]) * (x[a][2] - x[q][2]));
                if (!(d >= c.c_dist + c.band_dist) && !(dg[a] + dg[q] <= dist_constant - c.band_dist)) { // NaN counts as candidate
                    cand = true;
                    knife = knife || fabs(d - c.c_dist) <= c.band_dist;                           // :64 distance test
                    knife = knife || fabs(dg[a] + dg[q] - dist_constant) <= c.band_dist;          // :61 goal-distance test
                    knife = knife || fabs(dg[a] - dg[q]) <= c.band_dist;                          // :85 leader choice
                    for (int e = 0; e < np; ++e) knife = knife || fabs(de[e] - d) <= c.band_dist; // :76 closest pair
                    de[np++] = d;
                }
            }
    }
    bool guard = false;
    if (cand) {
        const double da = fabs(s - c.c_avg);
        const int tier = (rk >= c.edge[0] ? 1 : 0) + (rk >= c.edge[1] ? 1 : 0);
        const double band = c.band[tier] + c.rel[tier] * fabs(s);
        guard = !(da == da) || !(rk == rk) || isinf(s) || isinf(rk);   // non-finite FP32 rollout
        guard = guard || da <= band;                                   // velocity knife edge, widened by stiffness tier
        guard = guard || (knife && s < c.c_avg + band);                // geometric knife edges matter if the velocity test can pass
    }
    int slot = -1;
    if (guard) {
        const unsigned t = atomicAdd(&counters[0], 1u);
        if (t < c.cap) {
            slot = (int)t;
            list[t] = (int)b;
        }
    }
    return slot;
}

// Arguments of the heuristic as the post step of a sweep hands them to the kernels (FP32 arrays; see deadlock_one)
struct DlPost {
    int enabled;
    DlCfg c;
    long long B;
    const float* x_ee;
    float* goals;
    float* weights;
    const float* avg_vel;
    const int* sm_state;
    const int* time_step;
    int* tdo;
    int* st_int;
    float* st_goal;
    int* flag;
    const float* goal_est;
    float* result;
    DlOverride ov;
    unsigned* done; // CTAs of the re-roll kernel that have finished: the last one resets the list counter
};

// First kernel of the post step: list the scenarios the FP32 rollout could not decide safely -- and run the heuristic right
// away for all the others.  The listed ones get theirs from the FP64 re-roll kernel (rollout_kernel<double, ..., STRIDE>),
// each CTA for the scenarios it has just re-rolled: two launches per step instead of three next to the rollouts.
template <typename T>
__global__ void __launch_bounds__(256, 4)
    guard_deadlock_kernel(GuardCfg g, const T* __restrict__ rec, const T* __restrict__ risk, int time_gate,
                          double dist_constant, int* __restrict__ slot_of, unsigned* __restrict__ counters,
                          int* __restrict__ list, DlPost d) {
    const long long B = d.B;
    for (long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += (long long)gridDim.x * blockDim.x) {
        const int slot = guard_select_one<T>(g, b, B, (const T*)d.avg_vel, (const T*)d.x_ee, rec, (const T*)d.goal_est, risk,
                                             d.sm_state, d.time_step, time_gate, dist_constant, counters, list);
        slot_of[b] = slot;
        if (slot < 0)
            deadlock_one<T>(d.c, b, B, -1, d.ov, (const T*)d.x_ee, (T*)d.goals, (T*)d.weights, (const T*)d.avg_vel, nullptr,
                            d.sm_state, d.time_step, d.tdo, d.st_int, (T*)d.st_goal, d.flag, (const T*)d.goal_est, (T*)d.result);
    }
}

// ------------------------------------------------------------------------------------------------
// coupled joint-space rollout
// ------------------------------------------------------------------------------------------------
#ifndef MRF_ROLLOUT_MINBLOCKS
#define MRF_ROLLOUT_MINBLOCKS 4
#endif
#ifndef MRF_ROLLOUT_MINBLOCKS_F64
#define MRF_ROLLOUT_MINBLOCKS_F64 1
#endif
#ifdef MRF_EXP_NOBAR // timing experiment only (racy): what the two per-step CTA barriers cost
#define MRF_STEP_SYNC() __syncwarp()
#else
#define MRF_STEP_SYNC() __syncthreads()
#endif
// Host-record mode (AOS): `rec` holds the caller's own records rec[B][R][44] (the reference's argument order), normally
// in PAGE-LOCKED HOST memory that the kernel reads over PCIe.  A tile's records are one contiguous block, fetched with
// coalesced 16-byte loads into the (not yet used) point table; results go back in the matching layout (avg[B][R],
// x_ee[B][R][3], goal[B][3]).  No staging copy, no transpose kernel: the CTA scheduler overlaps the host reads of later
// tiles with the horizons of earlier ones.  Tiles are handed out by an atomic ticket and admitted to the bus in ticket
// order, `window` tiles at a time (sync[0] = tickets, sync[1] = tiles loaded): without that every CTA of a wave would
// share the bus, all would start -- and later finish -- together, and each wave would stall for its whole transfer.
// the rarely used arguments of rollout_kernel
template <typename T> struct RollExtra {
    // STRIDE (FP64 re-roll of the guard band): count, list, and the FP32 records the listed scenarios are read from --
    // element (field f, robot r, scenario b) at src[f * sf + r * sr + b * sb] (SoA device tensor or the caller's AoS host
    // records); fields >= src_nvar come from src_tail [R][MRF_REC] (compact host records)
    unsigned* n_live;
    const float* src;
    const int* list;
    long long sf, sr, sb;
    int src_nvar;
    const float* src_tail;
    // static spheres of the rollout planners (generic kernel): stat [n_static][4][R][B]
    int n_static;
    const T* stat;
    // host-record mode feeding the device post step: results in the SoA layout of the device entries (not the caller's
    // record order), and the record fields read from the host copied to rec_out [n_var][R][B] on the device (SoA) -- the
    // post step (goal rows for the heuristic, whole records of the re-rolled scenarios) then never touches the bus
    int out_soa;
    T* rec_out;
    // STRIDE as the second kernel of a sweep's post step: every CTA runs the deadlock heuristic for the scenarios it has
    // just re-rolled (dl.enabled), and the last CTA to finish resets the list counter
    DlPost dl;
};

template <typename T, int R, bool UNIFORM, bool AOS, bool STRIDE = false>
__global__ void __launch_bounds__(kTile* R, (R == 3 && sizeof(T) == 4) ? MRF_ROLLOUT_MINBLOCKS : MRF_ROLLOUT_MINBLOCKS_F64)
    rollout_kernel(const __grid_constant__ DevCfg<T> cfg, const T* __restrict__ rec, int N, T* __restrict__ avg_vel,
                   T* __restrict__ x_ee, T* __restrict__ goal_est, T* __restrict__ qN, T* __restrict__ qdN, long long B,
                   unsigned* __restrict__ sync, unsigned window, int n_var, const T* __restrict__ rec_tail,
                   T* __restrict__ risk, const __grid_constant__ RollExtra<T> ex) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    unsigned* const n_live = ex.n_live;
    const int n_static = ex.n_static;
    const bool rec_order_out = AOS && !ex.out_soa; // results in the caller's record order (AoS) or in the device SoA layout
    // STRIDE (FP64 re-roll of the guard band): the scenarios are the first min(*n_live, B) entries of `list` -- produced
    // on the device by guard_deadlock_kernel -- read from the FP32 records rec_f32 [44][R][B_src] (exact promotion); results
    // go to compact arrays of stride B.  The grid is a handful of CTAs that stride over the tiles, so only a few
    // (register-heavy) CTAs have to find room next to the FP32 sweep.  Ordinary launches: one CTA per tile, no loop.
    const long long Bn = STRIDE ? ((long long)*n_live < B ? (long long)*n_live : B) : B;
    if (STRIDE && blockIdx.x == 0 && threadIdx.x == 0) { // guard statistics: [1] listed by this call, [2] re-rolled, [3] overflow
        n_live[1] = n_live[0];
        n_live[2] += (unsigned)Bn;
        n_live[3] += n_live[0] - (unsigned)Bn;
    }
    constexpr int NT = kTile * R; // compile-time so every shared-memory offset is an immediate
    unsigned tile_first = blockIdx.x;
    const bool fused_post = STRIDE && ex.dl.enabled != 0;
    bool has_work = !(STRIDE && (long long)tile_first * kTile >= Bn);
    if (!has_work && !fused_post) return;
  while (has_work) {
    const int tid = threadIdx.x, lane = tid & (kTile - 1), r = tid / kTile;
    // (a double-buffered point table with one barrier per step was measured 2 % slower: more shared memory per CTA
    //  and non-immediate offsets; the barrier stall is load imbalance between the robots' warps, not barrier count)
    T* kin = reinterpret_cast<T*>(smem_raw);
    T* prm = kin + kKinRows<T> * NT;
    unsigned tile = tile_first;
    if (AOS) {
        unsigned* tk = reinterpret_cast<unsigned*>(prm);
        if (tid == 0) {
            const unsigned t = atomicAdd(&sync[0], 1u);
            while (*reinterpret_cast<volatile unsigned*>(&sync[1]) + window <= t) __nanosleep(100);
            *tk = t;
        }
        __syncthreads();
        tile = *tk;
    }
    const long long b = (long long)tile * kTile + lane;
    const bool live = b < Bn;
    const long long bb = live ? b : Bn - 1; // idle lanes shadow the last scenario so barriers stay uniform
    const T* ld_base = rec + (long long)r * B + bb;
    long long ld_stride = (long long)R * B;
    const T* tail = rec_tail; // shared trailing fields (device memory, [R][MRF_REC]) when the records are compact
    if (AOS) {
        // each host record holds the first n_var fields (n_var = MRF_REC: whole records; n_var = MRF_G1 = 18: q, qdot,
        // x_goal_0, weight_goal_0 -- what changes from scenario to scenario; the rest comes from rec_tail)
        const long long first = (long long)tile * kTile;
        const int nb = (int)(B - first < kTile ? B - first : kTile);
        const int nvals = nb * R * n_var;
        const int nvec = nvals * (int)sizeof(T) / 16; // a full tile is a whole number of 16-byte words; a ragged one may not be
        const T* srcT = rec + first * R * n_var;
        const int4* src = reinterpret_cast<const int4*>(srcT);
        int4* dst = reinterpret_cast<int4*>(kin);
        for (int i = tid; i < nvec; i += NT) dst[i] = src[i];
        for (int i = nvec * (16 / (int)sizeof(T)) + tid; i < nvals; i += NT) kin[i] = srcT[i];
        __syncthreads();
        if (tid == 0) atomicAdd(&sync[1], 1u);
        ld_base = kin + ((live ? lane : nb - 1) * R + r) * n_var;
        ld_stride = 1;
        tail += r * MRF_REC;
    }
    const long long b_src = STRIDE ? (long long)ex.list[bb] : 0;
    auto ld = [&](int f) {
        if (STRIDE)
            return f < ex.src_nvar ? (T)ex.src[f * ex.sf + r * ex.sr + b_src * ex.sb] : (T)ex.src_tail[r * MRF_REC + f];
        return AOS ? (f < n_var ? ld_base[f] : tail[f]) : rec[((long long)f * R + r) * B + bb];
    };
    (void)ld_stride;

    T q[kDof], qd[kDof];
#pragma unroll
    for (int i = 0; i < kDof; ++i) {
        q[i] = ld(MRF_Q + i);
        qd[i] = ld(MRF_QD + i);
    }
    load_params<T>(ld, prm, NT, tid);
    // static spheres of this robot's rollout planner (generic kernel only): stat [n_static][4][R][B] = x, y, z, radius
    T* st_sph = prm + P_N * NT;
    if (!UNIFORM && !AOS && n_static > 0) {
        for (int i = 0; i < 4 * n_static; ++i) st_sph[i * NT + tid] = ex.stat[((long long)i * R + r) * B + bb];
    }
    if (AOS && ex.rec_out != nullptr && live) { // device SoA copy of the host record fields for the post step
        for (int f = 0; f < n_var; ++f) ex.rec_out[((long long)f * R + r) * B + b] = ld_base[f];
    }
    Chain<T> ch;
    const T vref = cfg.static_or_dyn ? T(1) : T(0), aref = cfg.static_or_dyn ? cfg.sref : T(0);
    // shared robot-robot leaves (mrf_device.cuh, pair_leaves_eval): decided per scenario from its parameter blocks
    constexpr bool kPair = kPairPath<T, R, UNIFORM>;
    const bool pair_cfg = kPair && pair_leaves_cfg(cfg); // uniform over the grid: the extra barrier is not divergent
    bool pair_on = false;
    T* const pls = prm + P_N * NT;
    if (pair_cfg) {
        __syncthreads(); // every robot's parameter block is in shared memory
        pair_on = pair_leaves_lane(prm, NT, lane);
    }
    T acc = T(0);
    prm[P_RISK * NT + tid] = T(0); // running maximum of the stiffness indicator (shared memory: no register held)
    // k = -1: FK at the measured state only (end-effector position, RF-CV goal estimate); k >= 0: horizon steps.
    // One loop body keeps a single copy of chain_forward in the instruction stream.
    const bool want_pre = x_ee != nullptr || goal_est != nullptr || cfg.estimate_goal != 0;
    for (int k = want_pre ? -1 : 0; k < N; ++k) {
        // Phase A (forward_planner_Jointspace.py:191-209): step with the stale velocity, then FK
        if (k >= 0) {
#pragma unroll
            for (int i = 0; i < kDof; ++i) q[i] += cfg.dt * qd[i];
        }
        MRF_STEP_SYNC(); // readers of the previous step are done
        chain_forward(cfg, r, q, qd, ch, kin, NT, tid);
        if (k < 0) {
            // end-effector FK at the measured state (example_pandas_Jointspace.py:236-238,328-329) and the RF-CV
            // constant-velocity goal estimate of one robot (:346-348)
            V3<T> p8 = kin_load(kin, NT, tid, 4, 0);
            if (x_ee != nullptr && live) {
                T* o = rec_order_out ? x_ee + (b * R + r) * 3 : x_ee + (long long)r * 3 * B + b;
                const long long st = rec_order_out ? 1 : B;
                o[0] = p8.x;
                o[st] = p8.y;
                o[2 * st] = p8.z;
            }
            if (r == cfg.estimate_robot) {
                V3<T> g = mk(prm[(P_G0 + 0) * NT + tid], prm[(P_G0 + 1) * NT + tid], prm[(P_G0 + 2) * NT + tid]);
                if (cfg.estimate_goal) {
                    V3<T> l1 = mk(cfg.link1[r][0], cfg.link1[r][1], cfg.link1[r][2]);
                    // mode 1: first COLUMN of the hand Jacobian (the reference's "v_ee"); mode 2: J qdot
                    V3<T> v = cfg.estimate_goal == 1 ? cross(ch.z[0], p8 - l1) : kin_load(kin, NT, tid, 4, 3);
                    g = p8 + v * cfg.est_h;
                    prm[(P_G0 + 0) * NT + tid] = g.x;
                    prm[(P_G0 + 1) * NT + tid] = g.y;
                    prm[(P_G0 + 2) * NT + tid] = g.z;
                }
                if (goal_est != nullptr && live) {
                    T* o = rec_order_out ? goal_est + b * 3 : goal_est + b;
                    const long long st = rec_order_out ? 1 : B;
                    o[0] = g.x;
                    o[st] = g.y;
                    o[2 * st] = g.z;
                }
            }
            continue;
        }
        MRF_STEP_SYNC(); // every robot of the tile has published
        // Phase B (:211-249): action against the other robots' published spheres
        T act[kDof], stiff;
        if (UNIFORM) {
            SmemSrcUniform<T, R> src{kin, lane, r, vref, aref, cfg.r_obst};
            PairLeaves<T> pl{T(0), pair_on};
            if (pair_cfg) {
                if (pair_on) pl.num = pair_leaves_eval(cfg, r, kin, prm, pls, NT, tid, lane);
                __syncthreads(); // every robot's leaf slots are written
                if (pair_on) pl.num += pls[2 * kPairSlots * NT + (r == 0 ? 2 : r - 1) * kTile + lane];
            }
            fabric_action(cfg, r, q, qd, ch, kin, prm, NT, tid, src, act, &stiff, kPair ? &pl : nullptr);
        } else {
            SmemSrc<T> src{cfg, kin, NT, lane, r, vref, aref, st_sph, AOS ? 0 : n_static, tid};
            fabric_action(cfg, r, q, qd, ch, kin, prm, NT, tid, src, act, &stiff);
        }
        prm[P_RISK * NT + tid] = Mth<T>::max(prm[P_RISK * NT + tid], stiff);
#pragma unroll
        for (int i = 0; i < kDof; ++i) {
            qd[i] = act[i];
            acc += act[i] * act[i];
        }
        if (qN != nullptr && live) {
#pragma unroll
            for (int i = 0; i < kDof; ++i) qN[(((long long)r * N + k) * kDof + i) * B + b] = q[i];
        }
        if (qdN != nullptr && live) {
#pragma unroll
            for (int i = 0; i < kDof; ++i) qdN[(((long long)r * N + k) * kDof + i) * B + b] = qd[i];
        }
    }
    // compute_velocity_average (:102-116): mean SQUARE joint velocity over the horizon
    if (avg_vel != nullptr && live) avg_vel[rec_order_out ? b * R + r : (long long)r * B + b] = acc / (T(N) * T(kDof));
    // stiffness indicator (maximum over the horizon of fabric_action's sum of leaf metrics), see mrf_rfcv_post_dev_f32
    if (risk != nullptr && live) risk[rec_order_out ? b * R + r : (long long)r * B + b] = prm[P_RISK * NT + tid];
    if (STRIDE) {
        __syncthreads(); // the next tile of this CTA overwrites the tables; this tile's results are visible to the CTA
        if (fused_post && tid < kTile && live) // one thread per re-rolled scenario: its robots' FP64 results are column b
            deadlock_one<float>(ex.dl.c, (long long)ex.list[b], ex.dl.B, (int)b, ex.dl.ov, ex.dl.x_ee, ex.dl.goals, ex.dl.weights,
                                ex.dl.avg_vel, nullptr, ex.dl.sm_state, ex.dl.time_step, ex.dl.tdo, ex.dl.st_int, ex.dl.st_goal,
                                ex.dl.flag, ex.dl.goal_est, ex.dl.result);
        tile_first += gridDim.x;
    }
    has_work = STRIDE && (long long)tile_first * kTile < Bn;
  }
    if (fused_post) { // every CTA has read the list counter at entry: the last one out resets it for the next post step
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();
            if (atomicAdd(ex.dl.done, 1u) == gridDim.x - 1) {
                *ex.dl.done = 0;
                n_live[0] = 0;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// single action / decoupled rollout: thread = (robot, scenario), obstacles from global memory
// ------------------------------------------------------------------------------------------------
constexpr int kActThreads = 128;

#ifndef MRF_ACTION_MINBLOCKS
#define MRF_ACTION_MINBLOCKS 1
#endif
template <typename T, bool CART>
__global__ void __launch_bounds__(kActThreads, sizeof(T) == 4 ? MRF_ACTION_MINBLOCKS : 1)
    action_kernel(const __grid_constant__ DevCfg<T> cfg, int robot_first, int n_rob, const T* __restrict__ rec, int S,
                  const T* __restrict__ obst, int N, T* __restrict__ out, T* __restrict__ qN, T* __restrict__ qdN,
                  long long B, const int32_t* __restrict__ sm_state) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int NT = blockDim.x, tid = threadIdx.x;
    T* kin = reinterpret_cast<T*>(smem_raw);
    T* prm = kin + kKinRows<T> * NT;
    const long long total = (long long)n_rob * B;
    long long idx = (long long)blockIdx.x * NT + tid;
    const bool live = idx < total;
    if (!live) idx = total - 1;
    const int rl = (int)(idx / B);
    const long long b = idx - (long long)rl * B;
    const int r = robot_first + rl;
    const long long stride = total;
    auto ld = [&](int f) { return rec[(long long)f * stride + idx]; };
    T q[kDof], qd[kDof];
#pragma unroll
    for (int i = 0; i < kDof; ++i) {
        q[i] = ld(MRF_Q + i);
        qd[i] = ld(MRF_QD + i);
    }
    load_params<T>(ld, prm, NT, tid);
    Chain<T> ch;
    GlobalSrc<T, CART> src{obst, stride, idx, S, T(0), T(1), T(1), prm + P_N * NT, NT, tid};
    // state-machine code 2 ("from pregrasp to the block"): the reference switches to the planner built without collision
    // links (example_pandas_Jointspace.py:440)
    src.grasp = sm_state != nullptr && sm_state[idx] == 2;
    if (!CART) {
        T act[kDof];
        chain_forward(cfg, r, q, qd, ch, kin, NT, tid);
        fabric_action(cfg, r, q, qd, ch, kin, prm, NT, tid, src, act);
        if (live) {
#pragma unroll
            for (int i = 0; i < kDof; ++i) out[(long long)i * stride + idx] = act[i];
        }
    } else {
        // forward_planner_Cartesian.py:421-458: evaluate, then step robot and obstacles.  Outputs per robot of the call:
        // avg_vel [n_rob][B], qN / qdN [n_rob][N][7][B] (n_rob = 1: the single-robot layouts [B], [N][7][B])
        T acc = T(0);
        const long long tb = (long long)rl * N * kDof * B + b; // column of this thread in qN / qdN
        for (int k = 0; k < N; ++k) {
            T act[kDof];
            src.tk = T(k) * cfg.dt;
            chain_forward(cfg, r, q, qd, ch, kin, NT, tid);
            fabric_action(cfg, r, q, qd, ch, kin, prm, NT, tid, src, act);
#pragma unroll
            for (int i = 0; i < kDof; ++i) {
                if (cfg.mode == 1) { // 'vel': the action is the new velocity (system_step, forward_planner_Cartesian.py:85-87)
                    qd[i] = act[i];
                    q[i] += cfg.dt * act[i];
                } else {             // 'acc': the action is qdd (:81-84)
                    q[i] += cfg.dt * qd[i] + T(0.5) * cfg.dt * cfg.dt * act[i];
                    qd[i] += cfg.dt * act[i];
                }
                acc += qd[i] * qd[i];
            }
            if (live) {
#pragma unroll
                for (int i = 0; i < kDof; ++i) {
                    if (qN != nullptr) qN[((long long)k * kDof + i) * B + tb] = q[i];
                    if (qdN != nullptr) qdN[((long long)k * kDof + i) * B + tb] = qd[i];
                }
            }
        }
        if (out != nullptr && live) out[src.off] = acc / (T(N) * T(kDof)); // src.off == idx = rl * B + b
    }
}

// fk / J qdot / jdot_ref_sign * Jdot qdot of the 8 collision links
template <typename T>
__global__ void __launch_bounds__(kActThreads)
    kinematics_kernel(const __grid_constant__ DevCfg<T> cfg, const T* __restrict__ qin, const T* __restrict__ qdin,
                      T* __restrict__ x, T* __restrict__ v, T* __restrict__ a, long long B) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int NT = blockDim.x, tid = threadIdx.x, R = cfg.n_robots;
    T* kin = reinterpret_cast<T*>(smem_raw);
    const long long total = (long long)R * B;
    long long idx = (long long)blockIdx.x * NT + tid;
    const bool live = idx < total;
    if (!live) idx = total - 1;
    const int r = (int)(idx / B);
    T q[kDof], qd[kDof];
#pragma unroll
    for (int i = 0; i < kDof; ++i) {
        q[i] = qin[(long long)i * total + idx];
        qd[i] = qdin[(long long)i * total + idx];
    }
    Chain<T> ch;
    chain_forward(cfg, r, q, qd, ch, kin, NT, tid);
    if (!live) return;
    const int emap[8] = {-1, -1, 0, 1, 2, 2, 3, 4};
#pragma unroll
    for (int l = 0; l < 8; ++l) {
        V3<T> xx, vv, aa;
        if (emap[l] < 0) {
            xx = mk(cfg.link1[r][0], cfg.link1[r][1], cfg.link1[r][2]);
            vv = mk(T(0), T(0), T(0));
            aa = vv;
        } else {
            xx = kin_load(kin, NT, tid, emap[l], 0);
            vv = kin_load(kin, NT, tid, emap[l], 3);
            aa = kin_load(kin, NT, tid, emap[l], 6) * cfg.sref;
        }
        if (x) { x[((long long)l * 3 + 0) * total + idx] = xx.x; x[((long long)l * 3 + 1) * total + idx] = xx.y; x[((long long)l * 3 + 2) * total + idx] = xx.z; }
        if (v) { v[((long long)l * 3 + 0) * total + idx] = vv.x; v[((long long)l * 3 + 1) * total + idx] = vv.y; v[((long long)l * 3 + 2) * total + idx] = vv.z; }
        if (a) { a[((long long)l * 3 + 0) * total + idx] = aa.x; a[((long long)l * 3 + 1) * total + idx] = aa.y; a[((long long)l * 3 + 2) * total + idx] = aa.z; }
    }
}

// ------------------------------------------------------------------------------------------------
// Staging layout of the host-pointer entries: host [B][A][F] (array of records) <-> device [F][A][B] (the kernels'
// structure of arrays).  The host side is a [B][A*F] matrix with column j = a*F + f, the device side holds that column
// in row f*A + a; tiled through shared memory so that both sides coalesce.  A = 1 is the plain transpose.
// ------------------------------------------------------------------------------------------------
template <typename T, bool TO_DEVICE>
__global__ void layout_kernel(const T* __restrict__ in, T* __restrict__ out, long long B, int A, int F) {
    __shared__ T tile[32][33];
    const int AF = A * F;
    const long long b0 = (long long)blockIdx.x * 32;
    const int j0 = blockIdx.y * 32;
    auto row = [&](int j) { return (long long)(j % F) * A + j / F; }; // device row of host column j
    if (TO_DEVICE) {
        for (int i = threadIdx.y; i < 32; i += blockDim.y) { // rows = b, cols = j (contiguous on the host side)
            long long b = b0 + i;
            int j = j0 + threadIdx.x;
            if (b < B && j < AF) tile[i][threadIdx.x] = in[b * AF + j];
        }
        __syncthreads();
        for (int i = threadIdx.y; i < 32; i += blockDim.y) {
            int j = j0 + i;
            long long b = b0 + threadIdx.x;
            if (b < B && j < AF) out[row(j) * B + b] = tile[threadIdx.x][i];
        }
    } else {
        for (int i = threadIdx.y; i < 32; i += blockDim.y) { // rows = j, cols = b (contiguous on the device side)
            int j = j0 + i;
            long long b = b0 + threadIdx.x;
            if (b < B && j < AF) tile[i][threadIdx.x] = in[row(j) * B + b];
        }
        __syncthreads();
        for (int i = threadIdx.y; i < 32; i += blockDim.y) {
            long long b = b0 + i;
            int j = j0 + threadIdx.x;
            if (b < B && j < AF) out[b * AF + j] = tile[threadIdx.x][i];
        }
    }
}

// ------------------------------------------------------------------------------------------------
// obstacle staging for the executed action: collision spheres of every robot with per-link offsets
// (n_obst_per_link spheres per link, offsets in the link frame as placed by
// examples/simulation_environments/create_simulation_manipulators.py:188-245 and evaluated symbolically by
// multi_robot_fabrics/utils/utils.py:87-119), assembled per ego robot like
// examples/example_pandas_Jointspace.py:400-412 / multi_robot_fabrics/utils/utils_apply_fk.py:3-33.
// thread = (robot j, scenario b): computes robot j's 8n spheres and scatters them into the obstacle lists of every
// other robot i (block j' = index of j among i's others, ascending).
// ------------------------------------------------------------------------------------------------
template <typename T> struct SphereOffsets {
    int n;
    T t[MRF_NLINKS][MRF_MAX_SPHERES_PER_LINK][3];
};

template <typename T>
__global__ void __launch_bounds__(kActThreads)
    obstacles_kernel(const __grid_constant__ DevCfg<T> cfg, const __grid_constant__ SphereOffsets<T> off, int vel_mode,
                     const T* __restrict__ qin, const T* __restrict__ qdin, T* __restrict__ obst, T* __restrict__ sx,
                     T* __restrict__ sv, long long B) {
    const int R = cfg.n_robots, n = off.n;
    const long long total = (long long)R * B;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int j = (int)(idx / B);
    const long long b = idx - (long long)j * B;
    T q[kDof], qd[kDof];
#pragma unroll
    for (int i = 0; i < kDof; ++i) {
        q[i] = qin[(long long)i * total + idx];
        qd[i] = qdin[(long long)i * total + idx];
    }
    const int S = MRF_NLINKS * n * (R - 1);
    const T vsc = cfg.static_or_dyn ? T(1) : T(0); // STATIC_OR_DYN_FABRICS == 0: zero velocities (:337-338)
    auto emit = [&](int link, const Frame<T>& f) {
        for (int s = 0; s < n; ++s) {
            const T* t = off.t[link][s];
            V3<T> rt = f.a * t[0] + f.b * t[1] + f.n * t[2];
            V3<T> xs = f.p + rt;
            V3<T> vs = vel_mode ? f.v + cross(f.w, rt) : f.v; // 1: J_sphere qdot; 0: link-origin velocity replicated
            vs = vs * vsc;
            const int k = link * n + s;
            if (sx) { sx[((long long)k * 3 + 0) * total + idx] = xs.x; sx[((long long)k * 3 + 1) * total + idx] = xs.y; sx[((long long)k * 3 + 2) * total + idx] = xs.z; }
            if (sv) { sv[((long long)k * 3 + 0) * total + idx] = vs.x; sv[((long long)k * 3 + 1) * total + idx] = vs.y; sv[((long long)k * 3 + 2) * total + idx] = vs.z; }
            if (obst) {
                for (int i = 0; i < R; ++i) {
                    if (i == j) continue;
                    const int o = (j - (j > i ? 1 : 0)) * MRF_NLINKS * n + k;
                    T* p = obst + ((long long)o * MRF_OBST * R + i) * B + b;
                    const long long st = (long long)R * B;
                    p[0 * st] = xs.x; p[1 * st] = xs.y; p[2 * st] = xs.z;
                    p[3 * st] = vs.x; p[4 * st] = vs.y; p[5 * st] = vs.z;
                    p[6 * st] = T(0); p[7 * st] = T(0); p[8 * st] = T(0); // accelerations are not communicated (:411)
                    p[9 * st] = (T)cfg.r_link[j][link];
                }
            }
        }
    };
    (void)S;
    Frame<T> f;
    const T* Rm = cfg.R0[j];
    f.a = mk(Rm[0], Rm[3], Rm[6]);
    f.b = mk(Rm[1], Rm[4], Rm[7]);
    f.n = mk(Rm[2], Rm[5], Rm[8]);
    f.p = mk(cfg.link1[j][0], cfg.link1[j][1], cfg.link1[j][2]);
    f.w = mk(T(0), T(0), T(0));
    f.al = f.w; f.v = f.w; f.ac = f.w;
    (void)fr_joint<T, 0>(f, q[0], qd[0]);  emit(0, f);
    (void)fr_joint<T, -1>(f, q[1], qd[1]); emit(1, f);
    fr_advance(f, f.b * T(-0.316));
    (void)fr_joint<T, 1>(f, q[2], qd[2]);  emit(2, f);
    fr_advance(f, f.a * T(0.0825));
    (void)fr_joint<T, 1>(f, q[3], qd[3]);  emit(3, f);
    fr_advance(f, f.a * T(-0.0825) + f.b * T(0.384));
    (void)fr_joint<T, -1>(f, q[4], qd[4]); emit(4, f);
    (void)fr_joint<T, 1>(f, q[5], qd[5]);  emit(5, f);
    fr_advance(f, f.a * T(0.088));
    (void)fr_joint<T, 1>(f, q[6], qd[6]);  emit(6, f);
    fr_advance(f, f.n * T(0.107));
    emit(7, f);
}

// ------------------------------------------------------------------------------------------------
// point-mass planner (BASELINE config C1): examples/example_pointmasses_static.py:102-129,
// examples/example_pointmasses_dynamic.py:102-131.  3 dof (x, y, theta); collision link base_link at (x, y, 0.05)
// (pointRobot1.urdf:91-113); collision_geometry "-2/x xdot^2", collision_finsler "1/x^2 (1 - heaviside(xdot)) xdot^2";
// one 2-D attractor; no limits; mode 'acc'.  thread = scenario (one robot each).
//   rec [10][B]: q[3], qdot[3], x_goal_0[2], weight_goal_0, radius_body_base_link
//   stat [Ss][4][B]: x[3], radius          dyn [Sd][7][B]: x[2], xdot[2], xddot[2], radius
// ------------------------------------------------------------------------------------------------
// point_action: the planner for one robot with ego state (qx, qy, theta), (vx, vy, vth), goal (gx, gy), weight wg.
// `each(leaf)` enumerates the obstacle spheres in order, calling leaf(dx, dy, dz, wx, wy, ax, ay, rho) with the offset
// ego - obstacle, the relative velocity, the obstacle's acceleration and rho = radius_obst + radius_body.  Writes the
// action (a0, a1, a2).  Shared by point_action_kernel (obstacles from global memory) and point_episode_kernel (scene
// spheres from shared memory, other robots from neighbouring lanes).
template <typename T, typename Each>
__device__ __forceinline__ void point_action(T eps, T sigma, T s2, T qx, T qy, T vx, T vy, T vth, T gx, T gy, T wg, Each each,
                                             T& a0, T& a1, T& a2) {
    T m00 = T(0.2), m01 = T(0), m11 = T(0.2), f0 = T(0), f1 = T(0), num = T(0);
    each([&](T dx, T dy, T dz, T wx, T wy, T ax, T ay, T rho) {
        const T n2 = dx * dx + dy * dy + dz * dz;
        const T in1 = Mth<T>::rsqrt(n2), n = n2 * in1;
        const T t = n - rho, nr = n * rho, u = Mth<T>::rcp(nr * t);
        const T gs = u * t, ix = (u * nr) * rho;         // 1/(n rho), 1/x
        const T dw = dx * wx + dy * wy, ww = wx * wx + wy * wy;
        const T xd = dw * gs;
        const T kappa = (ww - dw * dw * (in1 * in1)) * gs;
        const T s = xd < T(0) ? T(1) : (xd > T(0) ? T(0) : T(0.5)); // 1 - heaviside(xdot)
        const T Ml = T(2) * s * ix * ix;
        const T fel = T(-2) * s * xd * xd * ix * ix * ix;
        const T fl = Ml * (T(-2) * ix * xd * xd);
        const T acc_o = (dx * ax + dy * ay) * gs;
        const T fq = fl + Ml * (sigma * kappa - acc_o), feq = fel + Ml * (kappa - acc_o);
        const T g0 = dx * gs, g1 = dy * gs;
        f0 += g0 * fq; f1 += g1 * fq;
        m00 += Ml * g0 * g0; m01 += Ml * g0 * g1; m11 += Ml * g1 * g1;
        num += (g0 * vx + g1 * vy) * (fq - feq);
    });
    const T xg0 = qx - gx, xg1 = qy - gy;
    const T ng = Mth<T>::sqrt(xg0 * xg0 + xg1 * xg1);
    T dpsi, mm;
    attractor_scalars(ng, wg, dpsi, mm);
    const T ff0 = f0 + mm * dpsi * xg0 * Mth<T>::rcp(ng), ff1 = f1 + mm * dpsi * xg1 * Mth<T>::rcp(ng);
    auto solve2 = [&](T a00, T a01, T a11, T b0, T b1, T& h0, T& h1) {
        a00 += eps; a11 += eps;
        const T idet = Mth<T>::rcp(a00 * a11 - a01 * a01);
        h0 = (a11 * b0 - a01 * b1) * idet;
        h1 = (a00 * b1 - a01 * b0) * idet;
    };
    T hg0, hg1, hf0, hf1;
    solve2(m00, m01, m11, f0, f1, hg0, hg1);
    solve2(m00 + mm, m01, m11 + mm, ff0, ff1, hf0, hf1);
    const T qMq = m00 * vx * vx + T(2) * m01 * vx * vy + m11 * vy * vy + T(0.2) * vth * vth;
    const T qq = vx * vx + vy * vy + vth * vth;
    const T a_geom = -num * Mth<T>::rcp(eps + qMq);
    const T iden = Mth<T>::rcp(eps + s2 * qq);
    const T a_ex0 = -s2 * (vx * hg0 + vy * hg1) * iden, a_exf = -s2 * (vx * hf0 + vy * hf1) * iden;
    const T eta = T(0.5) * (Mth<T>::tanh(T(-0.45) * qq - T(0.5)) + T(1));
    const T a_ex = eta * a_ex0 + (T(1) - eta) * a_exf;
    const T beta = T(0.5) * (Mth<T>::tanh(T(-0.5) * (ng - T(0.02))) + T(1)) * T(6.5) + T(0.01) +
                   Mth<T>::max(T(0), a_geom - a_ex);
    const T damp = a_ex + beta;
    a0 = -hf0 - damp * vx;
    a1 = -hf1 - damp * vy;
    a2 = -damp * vth;
}

template <typename T>
__global__ void __launch_bounds__(kActThreads)
    point_action_kernel(T eps, T sigma, T s2, const T* __restrict__ rec, int Ss, const T* __restrict__ stat, int Sd,
                        const T* __restrict__ dyn, T* __restrict__ action, long long B) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    auto ld = [&](int f) { return rec[(long long)f * B + b]; };
    const T qx = ld(0), qy = ld(1), vx = ld(3), vy = ld(4), vth = ld(5);
    const T gx = ld(6), gy = ld(7), wg = ld(8), rb = ld(9);
    auto each = [&](auto&& leaf) {
        for (int o = 0; o < Ss + Sd; ++o) {
            T dx, dy, dz, wx, wy, ax = T(0), ay = T(0), rho;
            if (o < Ss) {
                const T* p = stat + (long long)o * 4 * B + b;
                dx = qx - p[0]; dy = qy - p[B]; dz = T(0.05) - p[2 * B];
                wx = vx; wy = vy;
                rho = p[3 * B] + rb;
            } else {
                const T* p = dyn + (long long)(o - Ss) * 7 * B + b;
                dx = qx - p[0]; dy = qy - p[B]; dz = T(0);
                wx = vx - p[2 * B]; wy = vy - p[3 * B];
                ax = p[4 * B]; ay = p[5 * B];
                rho = p[6 * B] + rb;
            }
            leaf(dx, dy, dz, wx, wy, ax, ay, rho);
        }
    };
    T a0, a1, a2;
    point_action<T>(eps, sigma, s2, qx, qy, vx, vy, vth, gx, gy, wg, each, a0, a1, a2);
    action[b] = a0;
    action[B + b] = a1;
    action[2 * B + b] = a2;
}

// ------------------------------------------------------------------------------------------------
// closed-loop point-mass episodes (examples/example_pointmasses_static.py, _dynamic.py), many control steps per launch.
// thread = (scenario, robot): the R robots of a scenario sit in W consecutive lanes (W = R rounded up to a power of two,
// lanes R..W-1 idle) and read each other's state by __shfl_sync(..., W).  q, qdot and the running metrics stay in
// registers for the whole launch; the scenario's scene spheres are staged once in shared memory.  Per step, every
// robot i of every scenario at once, all robots reading the state at the start of the step:
//   metrics of the measured state: reached (every robot within eps_goal of its goal in x-y; done_at = first such step),
//     x-y robot-robot clearance |p_i - p_j| - (r_i + r_j), scene clearance |(x, y, 0.05) - c_o| - (r_o + r_i)
//   obstacles: the scene spheres, then the other robots ascending -- DYN = false: a static sphere at q_j = (x, y, theta)
//     of radius r_j (the reference's static example passes the whole joint vector, so theta lands in the sphere's z;
//     theta is only ever damped); DYN = true: a 2-D sphere at q_j[0:2] moving with qdot_j[0:2], no acceleration
//   action: point_action (the planner of mrf_point_action_dev)
//   environment: a non-finite action becomes 0 for the step and the step is counted; qdot += dt a, q += dt qdot
//     (semi-implicit Euler, every product and sum rounded on its own: no FMA contraction)
// The one barrier (scene staging) comes before any per-lane branch, so a scenario's bits never depend on its neighbours.
// ------------------------------------------------------------------------------------------------
constexpr int kPointThreads = 128;

template <typename T> __device__ __forceinline__ T mul_rn(T a, T b);
template <> __device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
template <> __device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
template <typename T> __device__ __forceinline__ T add_rn(T a, T b);
template <> __device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
template <> __device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }

template <typename T, bool DYN>
__global__ void __launch_bounds__(kPointThreads)
    point_episode_kernel(T eps, T sigma, T s2, T dt, T eps_goal, int R, int W, int n_scene, int n_steps,
                         T* __restrict__ state, const T* __restrict__ goal, const T* __restrict__ weight,
                         const T* __restrict__ radius, const T* __restrict__ scene, int32_t* __restrict__ time_step,
                         int32_t* __restrict__ done_at, int32_t* __restrict__ nonfinite, T* __restrict__ min_rr,
                         T* __restrict__ min_sc, T* __restrict__ traj, long long B) {
    extern __shared__ __align__(16) unsigned char point_smem[];
    T* sc = reinterpret_cast<T*>(point_smem);        // [spb][n_scene][4]
    const int spb = blockDim.x / W, g = threadIdx.x / W, i = threadIdx.x % W;
    const long long b0 = (long long)blockIdx.x * spb, b = b0 + g;
    const int nf = n_scene * 4;
    for (int k = threadIdx.x; k < spb * nf; k += blockDim.x) { // scenario fastest: coalesced reads
        const int s = k % spb, f = k / spb;
        sc[s * nf + f] = b0 + s < B ? scene[(long long)f * B + b0 + s] : T(0);
    }
    __syncthreads();
    const bool live = b < B && i < R;
    const long long RB = (long long)R * B, idx = (long long)i * B + b;
    T qx = T(0), qy = T(0), qt = T(0), vx = T(0), vy = T(0), vt = T(0), gx = T(0), gy = T(0), wg = T(0), rb = T(0);
    if (live) {
        qx = state[idx]; qy = state[RB + idx]; qt = state[2 * RB + idx];
        vx = state[3 * RB + idx]; vy = state[4 * RB + idx]; vt = state[5 * RB + idx];
        gx = goal[((long long)i * 2) * B + b]; gy = goal[((long long)i * 2 + 1) * B + b];
        wg = weight[idx]; rb = radius[idx];
    }
    int t0 = 0, done = -1, nbad = 0;
    if (b < B) { t0 = time_step[b]; done = done_at[b]; nbad = nonfinite[b]; }
    const T inf = T(INFINITY);
    T mrr = inf, msc = inf;                          // this robot's running minima; reduced over the group at the end
    const unsigned gmask = ((1u << R) - 1u) << ((threadIdx.x & 31) & ~(W - 1));
    const T* my_sc = sc + g * nf;
    for (int k = 0; k < n_steps; ++k) {
        const T ex = qx - gx, ey = qy - gy;
        const unsigned near = __ballot_sync(0xffffffffu, Mth<T>::sqrt(ex * ex + ey * ey) < eps_goal);
        if ((near & gmask) == gmask && done < 0) done = t0 + k;
        auto each = [&](auto&& leaf) {
            for (int o = 0; o < n_scene; ++o) {
                const T* p = my_sc + o * 4;
                const T dx = qx - p[0], dy = qy - p[1], dz = T(0.05) - p[2], rho = p[3] + rb;
                const T c = Mth<T>::sqrt(dx * dx + dy * dy + dz * dz) - rho;
                msc = c < msc ? c : msc;
                leaf(dx, dy, dz, vx, vy, T(0), T(0), rho);
            }
            for (int j = 0; j < R; ++j) { // every lane shuffles (uniform trip count); the leaf skips robot i itself
                const T xj = __shfl_sync(0xffffffffu, qx, j, W), yj = __shfl_sync(0xffffffffu, qy, j, W);
                const T rj = __shfl_sync(0xffffffffu, rb, j, W);
                const T uj = __shfl_sync(0xffffffffu, DYN ? vx : qt, j, W); // DYN: x-velocity of robot j, else its theta
                const T wj = DYN ? __shfl_sync(0xffffffffu, vy, j, W) : T(0);
                if (j == i) continue;
                const T dx = qx - xj, dy = qy - yj, rho = rj + rb;
                const T c = Mth<T>::sqrt(dx * dx + dy * dy) - rho;
                mrr = c < mrr ? c : mrr;
                if (DYN) leaf(dx, dy, T(0), vx - uj, vy - wj, T(0), T(0), rho);
                else leaf(dx, dy, T(0.05) - uj, vx, vy, T(0), T(0), rho);
            }
        };
        T a0, a1, a2;
        point_action<T>(eps, sigma, s2, qx, qy, vx, vy, vt, gx, gy, wg, each, a0, a1, a2);
        const bool bad = !(a0 - a0 == T(0) && a1 - a1 == T(0) && a2 - a2 == T(0));
        if (bad) { a0 = T(0); a1 = T(0); a2 = T(0); }
        if (__ballot_sync(0xffffffffu, bad) & gmask) ++nbad;
        vx = add_rn(vx, mul_rn(dt, a0)); vy = add_rn(vy, mul_rn(dt, a1)); vt = add_rn(vt, mul_rn(dt, a2));
        qx = add_rn(qx, mul_rn(dt, vx)); qy = add_rn(qy, mul_rn(dt, vy)); qt = add_rn(qt, mul_rn(dt, vt));
        if (traj != nullptr && live) {
            T* p = traj + (long long)k * 3 * RB + idx;
            p[0] = qx; p[RB] = qy; p[2 * RB] = qt;
        }
    }
    if (!live) { mrr = inf; msc = inf; }
    for (int off = W / 2; off > 0; off >>= 1) { // min is exact: the order of the reduction does not matter
        const T orr = __shfl_xor_sync(0xffffffffu, mrr, off, W), osc = __shfl_xor_sync(0xffffffffu, msc, off, W);
        mrr = orr < mrr ? orr : mrr;
        msc = osc < msc ? osc : msc;
    }
    if (live) {
        state[idx] = qx; state[RB + idx] = qy; state[2 * RB + idx] = qt;
        state[3 * RB + idx] = vx; state[4 * RB + idx] = vy; state[5 * RB + idx] = vt;
    }
    if (b < B && i == 0) {
        time_step[b] = t0 + n_steps;
        done_at[b] = done;
        nonfinite[b] = nbad;
        if (mrr < min_rr[b]) min_rr[b] = mrr;
        if (msc < min_sc[b]) min_sc[b] = msc;
    }
}

// ------------------------------------------------------------------------------------------------
// pick-and-place state machine, one thread per (robot, scenario):
// StateMachine.get_state_machine_panda + get_gripper_action_panda
// (multi_robot_fabrics/others_planner/state_machine.py:70-84,133-214).  Distances are float64 with numpy's rounding
// (np_norm3) so the threshold tests agree with the reference bit for bit.
//   x_ee, goal_block, start_goal, goal (in/out), above (in/out)  [R][3][B];  q_grip, grip_action [R][2][B]
//   weight [R][B] (in/out);  st [6][R][B] in/out: state, nr_success, nr_failed, time_gripping, gripper_closed, stop_time
// ------------------------------------------------------------------------------------------------
struct FsmCfg {
    int R;
    int nr_blocks[MRF_MAX_ROBOTS];
};
template <typename T>
__global__ void fsm_kernel(FsmCfg c, const T* __restrict__ x_ee, const T* __restrict__ q_grip,
                           const T* __restrict__ goal_block, const T* __restrict__ start_goal, T* __restrict__ goal,
                           T* __restrict__ above, T* __restrict__ weight, int* __restrict__ st, T* __restrict__ grip_action,
                           long long B) {
    const long long total = (long long)c.R * B;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int r = (int)(idx / B);
    const long long b = idx - (long long)r * B;
    auto v3 = [&](const T* p, int k) { return (double)p[((long long)r * 3 + k) * B + b]; };
    const double x[3] = {v3(x_ee, 0), v3(x_ee, 1), v3(x_ee, 2)};
    const double gb[3] = {v3(goal_block, 0), v3(goal_block, 1), v3(goal_block, 2)};
    const double sg[3] = {v3(start_goal, 0), v3(start_goal, 1), v3(start_goal, 2)};
    double g[3] = {v3(goal, 0), v3(goal, 1), v3(goal, 2)};
    double ab[3] = {v3(above, 0), v3(above, 1), v3(above, 2)};
    const double qg0 = (double)q_grip[((long long)r * 2 + 0) * B + b], qg1 = (double)q_grip[((long long)r * 2 + 1) * B + b];
    int state = st[0 * total + idx], n_ok = st[1 * total + idx], n_fail = st[2 * total + idx], t_grip = st[3 * total + idx];
    int closed = st[4 * total + idx], stop = st[5 * total + idx];
    double w = (double)weight[idx];
    const double pre[3] = {gb[0], gb[1], __dadd_rn(gb[2], 0.1)};                                   // :134-135
    auto norm2 = [](double a, double bb) { return __dsqrt_rn(__fma_rn(bb, bb, __dmul_rn(a, a))); };
    const double d_start = np_norm3(__dsub_rn(x[0], sg[0]), __dsub_rn(x[1], sg[1]), __dsub_rn(x[2], sg[2]));
    const double d_pre = norm2(__dsub_rn(x[0], pre[0]), __dsub_rn(x[1], pre[1]));
    const double d_block = np_norm3(__dsub_rn(x[0], gb[0]), __dsub_rn(x[1], gb[1]), __dsub_rn(x[2], gb[2]));
    const double d_open = norm2(__dsub_rn(qg0, 0.04), __dsub_rn(qg1, 0.04));
    if (n_ok > c.nr_blocks[r] - 1) {                                                               // :141-142
        state = 10;
    } else if (gb[2] < 0.6) {                                                                      // :143-147
        n_ok += 1; n_fail += 1; state = 0;
    }
    const int s = state;
    if (s == 0) {                                                                                  // :150-155
        g[0] = sg[0]; g[1] = sg[1]; g[2] = sg[2]; closed = 0;
        if (d_start < 0.05) state = 1;
    } else if (s == 1) {                                                                           // :158-162
        g[0] = pre[0]; g[1] = pre[1]; g[2] = pre[2];
        if (d_pre < 0.013) state = 2;
    } else if (s == 2) {                                                                           // :164-170
        g[0] = gb[0]; g[1] = gb[1]; g[2] = gb[2];
        if (d_block < 0.013) { closed = 1; w = 0.0; state = 3; }
    } else if (s == 3) {                                                                           // :172-181
        g[0] = gb[0]; g[1] = gb[1]; g[2] = gb[2];
        ab[0] = gb[0]; ab[1] = gb[1]; ab[2] = __dadd_rn(gb[2], 0.15);
        t_grip += 1;
        if ((double)t_grip > 0.3 / 0.01) { t_grip = 0; g[0] = sg[0]; g[1] = sg[1]; g[2] = sg[2]; w = 2.0; state = 12; }
    } else if (s == 12) {                                                                          // :183-186
        g[0] = ab[0]; g[1] = ab[1]; g[2] = ab[2];
        if (norm2(__dsub_rn(x[0], g[0]), __dsub_rn(x[1], g[1])) < 0.04) state = 4;
    } else if (s == 4) {                                                                           // :188-194
        g[0] = sg[0]; g[1] = sg[1]; g[2] = sg[2];
        if (d_start < 0.15) { state = 5; closed = 0; }
    } else if (s == 5) {                                                                           // :196-200
        if (d_open < 0.005) { state = 0; n_ok += 1; g[0] = sg[0]; g[1] = sg[1]; g[2] = sg[2]; }
    } else if (s == 10) {                                                                          // :202-206
        stop = 1;
    }
    // gripper action (:70-84)
    double a0 = 0.0, a1 = 0.0;
    if (closed) { a0 = -0.05; a1 = -0.05; }
    else if (d_open > 0.005) { a0 = qg0 > 0.04 ? -0.4 : 0.4; a1 = qg1 > 0.04 ? -0.4 : 0.4; }
    for (int k = 0; k < 3; ++k) {
        goal[((long long)r * 3 + k) * B + b] = (T)g[k];
        above[((long long)r * 3 + k) * B + b] = (T)ab[k];
    }
    weight[idx] = (T)w;
    st[0 * total + idx] = state; st[1 * total + idx] = n_ok; st[2 * total + idx] = n_fail; st[3 * total + idx] = t_grip;
    st[4 * total + idx] = closed; st[5 * total + idx] = stop;
    if (grip_action) {
        grip_action[((long long)r * 2 + 0) * B + b] = (T)a0;
        grip_action[((long long)r * 2 + 1) * B + b] = (T)a1;
    }
}

// ------------------------------------------------------------------------------------------------
// FMA peak micro-benchmark: the roofline denominator for the compute-bound rollout (MEASURED_PEAKS.json
// holds HBM and bf16 tensor peaks only).  8 independent FMA chains per thread.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) fma2_peak_kernel(float* out, int iters, float b, float c) {
    float a0 = threadIdx.x * 1e-3f;
    float2 p0 = make_float2(a0, a0 + 1), p1 = make_float2(a0 + 2, a0 + 3), p2 = make_float2(a0 + 4, a0 + 5),
           p3 = make_float2(a0 + 6, a0 + 7);
    const float2 bb = make_float2(b, b), cc = make_float2(c, c);
#pragma unroll 4
    for (int i = 0; i < iters; ++i) {
        p0 = __ffma2_rn(p0, bb, cc); p1 = __ffma2_rn(p1, bb, cc); p2 = __ffma2_rn(p2, bb, cc); p3 = __ffma2_rn(p3, bb, cc);
    }
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = ((p0.x + p0.y) + (p1.x + p1.y)) + ((p2.x + p2.y) + (p3.x + p3.y));
}

template <typename T> __global__ void __launch_bounds__(256) fma_peak_kernel(T* out, int iters, T b, T c) {
    T a0 = T(threadIdx.x) * T(1e-3), a1 = a0 + T(1), a2 = a0 + T(2), a3 = a0 + T(3);
    T a4 = a0 + T(4), a5 = a0 + T(5), a6 = a0 + T(6), a7 = a0 + T(7);
#pragma unroll 4
    for (int i = 0; i < iters; ++i) {
        a0 = a0 * b + c; a1 = a1 * b + c; a2 = a2 * b + c; a3 = a3 * b + c;
        a4 = a4 * b + c; a5 = a5 * b + c; a6 = a6 * b + c; a7 = a7 * b + c;
    }
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
}

} // namespace mrf

// =================================================================================================
// C-ABI
// =================================================================================================
using namespace mrf;

static thread_local std::string g_err;
static int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}
#define MRF_CUDA(call)                                                                             \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(MRF_ECUDA, std::string(#call) + ": " + cudaGetErrorString(e_));            \
    } while (0)

struct MrfHandle_ {
    MrfConfig cfg;
    int device;
    DevCfg<float> c32;
    DevCfg<double> c64;
    cudaStream_t stream, s_copy, s_chunk[8];
    cudaEvent_t ev0, ev1, ev_up[8], ev_free, ev_chunk[8];
    // device scratch of the synchronous host entries (scratch_reset / scratch_take): blocks, the last one being filled
    std::vector<void*> scratch;
    size_t scratch_cap, scratch_off, scratch_used; // size and fill of the last block, bytes taken by the current call
    long long launches;
    double last_ms;
    long long coop_max_batch; // batches up to this size use the cooperative low-latency rollout kernel
    int zero_copy;            // page-locked host records are read by the kernel directly (MRF_ZERO_COPY=0 disables)
    int zc_window;            // tiles admitted to the bus at a time in that mode
    unsigned* d_sync;         // its ticket / loaded counters: one pair per in-flight launch (slot 0 = synchronous entry)
    void* d_tail[2];          // shared trailing record fields of compact submissions, one per pipeline slot
    int zc_slot;              // next slot of the submit/wait pipeline
    int zc_pending[2];        // submissions in flight per pipeline slot
    int zc_oldest;
    // FP64 re-roll of guard-band scenarios (mrf_rfcv_post_dev_f32)
    double guard_band[3], guard_rel[3], guard_edge[2], guard_band_dist;
    long long guard_cap;      // 0 = max(256, B / 16)
    void* rf_buf[4];          // per pipeline slot: device buffers of mrf_rfcv_host_submit (its own four-deep pipeline)
    size_t rf_bytes[4];
    void* d_tail_rf[4];
    cudaEvent_t ev_rf[4], ev_rf_roll[4]; // batch complete / its rollout kernel complete
    cudaStream_t s_rf_post[4];           // high-priority streams of the post steps
    int rf_roll_valid[4];
    int rf_head, rf_count;
    void* guard_buf[MRF_GUARD_SLOTS];   // per scratch slot: list, slot_of, compact FP64 records and results
    size_t guard_bytes[MRF_GUARD_SLOTS];
};

extern "C" int mrf_version(void) { return 100; }
extern "C" const char* mrf_last_error(void) { return g_err.c_str(); }

extern "C" int mrf_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

extern "C" int mrf_config_default(MrfConfig* c, int n_robots) {
    if (!c || n_robots < 1 || n_robots > MRF_MAX_ROBOTS) return fail(MRF_EINVAL, "mrf_config_default: bad arguments");
    memset(c, 0, sizeof(*c));
    c->struct_size = (int32_t)sizeof(MrfConfig);
    c->n_robots = n_robots;
    c->mode = 1;                // fabrics_mode "vel", parameters_manipulators.py:12
    c->static_or_dyn = 1;       // panda_config.yaml:4
    c->has_collision_links = 1;
    c->estimate_goal = 0;
    c->estimate_robot = 1;      // example_pandas_Jointspace.py:347-348
    c->estimate_horizon = 20 * 0.01;
    c->dt = 0.01;
    c->eps = 1e-6;
    c->jdot_sign = -1.0;
    c->jdot_ref_sign = -1.0;    // utils.py:28
    c->exec_scale = 1.0;
    static const double pos[4][3] = {{0.0, 0.0, 0.65}, {1.0, 0.0, 0.65}, {0.7, 0.6, 0.65}, {0.0, 0.0, 0.65}};
    for (int r = 0; r < MRF_MAX_ROBOTS; ++r) { // parameters_manipulators.py:83-110,138-150
        const double yaw = (r == 1 || r == 2) ? M_PI : 0.0; // set_planner_panda: i_robot in {1, 2} (parameters_manipulators.py:138-150)
        double* T = c->mount[r];
        T[0] = cos(yaw); T[1] = -sin(yaw); T[4] = sin(yaw); T[5] = cos(yaw); T[10] = 1.0; T[15] = 1.0;
        T[3] = pos[r][0]; T[7] = pos[r][1]; T[11] = pos[r][2];
        for (int l = 0; l < MRF_NLINKS; ++l) c->r_robots[r][l] = 0.08; // parameters_manipulators.py:23
        c->collision_link_mask[r] = 0xFF;                              // collision_links_nrs = [1..8], :25
    }
    static const double lim[7][2] = {{-2.8973, 2.8973}, {-1.7628, 1.7628}, {-2.8973, 2.8973}, {-3.0718, -0.0698},
                                     {-2.8973, 2.8973}, {-0.0175, 3.7525}, {-2.8973, 2.8973}};
    memcpy(c->limits, lim, sizeof(lim));
    c->dl_avg_vel_constant = 0.16;  // deadlock_prevention.py:20-27
    c->dl_dist_constant = 0.0;
    c->dl_goal_weight_follower = 2.0;
    c->dl_goal_weight_leader = 3.0;
    c->dl_nr_goal_scale = 2.0;
    c->dl_dist_endeff = 0.35;       // :64
    c->dl_backoff = 0.3;            // :96
    c->dl_time_wait = 300;
    c->dl_time_gate = 10;           // :66,83
    return MRF_OK;
}

static int create_resources(MrfHandle_* h) {
    for (int i = 0; i < 2; ++i) MRF_CUDA(cudaMalloc(&h->d_tail[i], sizeof(double) * MRF_MAX_ROBOTS * MRF_REC));
    // [0..13] ticket pairs (slot 0 synchronous entry, 1..2 rollout submit pipeline, 3..6 RF-CV submit pipeline), [16..] guard counters
    // [0, 16): ticket / loaded pairs of the in-place host launches; then 4 guard counters per scratch slot; then one
    // finished-CTA counter per scratch slot (fused post step)
    MRF_CUDA(cudaMalloc(&h->d_sync, (16 + 5 * MRF_GUARD_SLOTS) * sizeof(unsigned)));
    MRF_CUDA(cudaMemset(h->d_sync, 0, (16 + 5 * MRF_GUARD_SLOTS) * sizeof(unsigned)));
    int prio_lo = 0, prio_hi = 0;
    MRF_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    for (int i = 0; i < 4; ++i) {
        MRF_CUDA(cudaMalloc(&h->d_tail_rf[i], sizeof(float) * MRF_MAX_ROBOTS * MRF_REC));
        MRF_CUDA(cudaEventCreateWithFlags(&h->ev_rf[i], cudaEventDisableTiming));
        MRF_CUDA(cudaEventCreateWithFlags(&h->ev_rf_roll[i], cudaEventDisableTiming));
        MRF_CUDA(cudaStreamCreateWithPriority(&h->s_rf_post[i], cudaStreamNonBlocking, prio_hi));
    }
    MRF_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    MRF_CUDA(cudaStreamCreateWithFlags(&h->s_copy, cudaStreamNonBlocking));
    MRF_CUDA(cudaEventCreate(&h->ev0));
    MRF_CUDA(cudaEventCreate(&h->ev1));
    for (int i = 0; i < 8; ++i) MRF_CUDA(cudaEventCreateWithFlags(&h->ev_up[i], cudaEventDisableTiming));
    MRF_CUDA(cudaEventCreateWithFlags(&h->ev_free, cudaEventDisableTiming));
    for (int i = 0; i < 8; ++i) {
        MRF_CUDA(cudaStreamCreateWithFlags(&h->s_chunk[i], cudaStreamNonBlocking));
        MRF_CUDA(cudaEventCreateWithFlags(&h->ev_chunk[i], cudaEventDisableTiming));
    }
    return MRF_OK;
}

extern "C" int mrf_destroy(mrf_handle_t h);

extern "C" int mrf_create(const MrfConfig* cfg, int device, mrf_handle_t* out) {
    if (!cfg || !out) return fail(MRF_EINVAL, "mrf_create: null argument");
    if (cfg->struct_size != (int32_t)sizeof(MrfConfig)) return fail(MRF_EINVAL, "mrf_create: MrfConfig size mismatch");
    if (cfg->n_robots < 1 || cfg->n_robots > MRF_MAX_ROBOTS) return fail(MRF_EINVAL, "mrf_create: n_robots out of range");
    if (cfg->mode != 0 && cfg->mode != 1) return fail(MRF_EINVAL, "mrf_create: mode must be 0 (acc) or 1 (vel)");
    if (cfg->estimate_goal && (cfg->estimate_robot < 0 || cfg->estimate_robot >= cfg->n_robots))
        return fail(MRF_EINVAL, "mrf_create: estimate_robot out of range");
    int n = 0;
    cudaError_t ce = cudaGetDeviceCount(&n);
    if (ce != cudaSuccess || n == 0) {
        cudaGetLastError();
        return fail(MRF_ENODEV, std::string("mrf_create: no CUDA device (this library has no CPU fallback): ") +
                                    (ce != cudaSuccess ? cudaGetErrorString(ce) : "device count is 0"));
    }
    if (device < 0 || device >= n) return fail(MRF_EINVAL, "mrf_create: bad device index");
    MRF_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    MRF_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail(MRF_EUNSUPPORTED, "mrf_create: built for sm_100a (B200) only");
    MrfHandle_* h = new (std::nothrow) MrfHandle_();
    if (!h) return fail(MRF_ENOMEM, "mrf_create: out of memory");
    h->cfg = *cfg;
    h->device = device;
    h->coop_max_batch = 512;
    if (const char* e = getenv("MRF_COOP_MAX_BATCH")) h->coop_max_batch = atoll(e);
    h->zero_copy = 1;
    if (const char* e = getenv("MRF_ZERO_COPY")) h->zero_copy = atoi(e);
    h->zc_window = 32;
    if (const char* e = getenv("MRF_ZC_WINDOW")) h->zc_window = atoi(e) > 0 ? atoi(e) : 32;
    h->d_sync = nullptr;
    h->zc_slot = 0;
    h->zc_pending[0] = h->zc_pending[1] = 0;
    h->zc_oldest = 0;
    h->d_tail[0] = h->d_tail[1] = nullptr;
    // defaults calibrated on B200 (tools/guard_probe.py, profiles/r2_guard_calibration.md)
    // FP32 error of vel_avg_tot against FP64 over 4 x 65536 random scenarios, by stiffness tier: risk < 40: max 7e-6;
    // 40..200: max 9.3e-4; >= 200: max 3.1e-4 while the rollout stays calm (vel_avg_tot < 1), and up to 15 % of
    // vel_avg_tot when it blows up in both precisions (explicit Euler near contact, vel_avg_tot 2..160).  A flag can only
    // flip if |vel_avg_tot - 0.16| <= that error, hence an absolute plus a relative band per tier (margins: 3x, 4x, 13x / 2.7x).
    h->guard_band[0] = 2e-5;
    h->guard_band[1] = 4e-3;
    h->guard_band[2] = 4e-3;
    h->guard_rel[0] = 0.0;
    h->guard_rel[1] = 0.02;
    h->guard_rel[2] = 0.4;
    h->guard_edge[0] = 40.0;
    h->guard_edge[1] = 200.0;
    h->guard_band_dist = 1e-5;
    h->guard_cap = 0;
    for (int i = 0; i < MRF_GUARD_SLOTS; ++i) {
        h->guard_buf[i] = nullptr;
        h->guard_bytes[i] = 0;
    }
    fill_devcfg(*cfg, h->c32);
    fill_devcfg(*cfg, h->c64);
    // every failure below releases what was created so far (the handle is value-initialised: null streams / events /
    // buffers are skipped by mrf_destroy)
    int rc = create_resources(h);
    if (rc != MRF_OK) {
        const std::string msg = g_err;
        mrf_destroy(h);
        return fail(rc, msg);
    }
    *out = h;
    return MRF_OK;
}

extern "C" int mrf_destroy(mrf_handle_t h) {
    if (!h) return MRF_OK;
    cudaSetDevice(h->device);
    for (void* p : h->scratch) cudaFree(p);
    if (h->d_sync) cudaFree(h->d_sync);
    for (int i = 0; i < 4; ++i) {
        if (h->rf_buf[i]) cudaFree(h->rf_buf[i]);
        if (h->d_tail_rf[i]) cudaFree(h->d_tail_rf[i]);
        if (h->ev_rf[i]) cudaEventDestroy(h->ev_rf[i]);
        if (h->ev_rf_roll[i]) cudaEventDestroy(h->ev_rf_roll[i]);
        if (h->s_rf_post[i]) cudaStreamDestroy(h->s_rf_post[i]);
    }
    for (int i = 0; i < MRF_GUARD_SLOTS; ++i)
        if (h->guard_buf[i]) cudaFree(h->guard_buf[i]);
    for (int i = 0; i < 2; ++i)
        if (h->d_tail[i]) cudaFree(h->d_tail[i]);
    // a partially created handle (mrf_create failure path) holds null streams / events: skip them
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    for (int i = 0; i < 8; ++i)
        if (h->ev_up[i]) cudaEventDestroy(h->ev_up[i]);
    if (h->ev_free) cudaEventDestroy(h->ev_free);
    for (int i = 0; i < 8; ++i) {
        if (h->ev_chunk[i]) cudaEventDestroy(h->ev_chunk[i]);
        if (h->s_chunk[i]) cudaStreamDestroy(h->s_chunk[i]);
    }
    if (h->stream) cudaStreamDestroy(h->stream);
    if (h->s_copy) cudaStreamDestroy(h->s_copy);
    (void)cudaGetLastError();
    delete h;
    return MRF_OK;
}

extern "C" int mrf_set_coop_max_batch(mrf_handle_t h, int64_t max_batch) {
    if (!h || max_batch < 0) return fail(MRF_EINVAL, "mrf_set_coop_max_batch: bad argument");
    h->coop_max_batch = max_batch;
    return MRF_OK;
}
extern "C" int64_t mrf_launch_count(mrf_handle_t h) { return h ? h->launches : 0; }
extern "C" double mrf_last_kernel_ms(mrf_handle_t h) { return h ? h->last_ms : 0.0; }

template <typename T> static const DevCfg<T>& devcfg(mrf_handle_t h);
template <> const DevCfg<float>& devcfg<float>(mrf_handle_t h) { return h->c32; }
template <> const DevCfg<double>& devcfg<double>(mrf_handle_t h) { return h->c64; }

template <typename K> static int set_smem(K kernel, size_t bytes) {
    if (bytes > 48 * 1024) MRF_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    return MRF_OK;
}
// Kernels that run NEXT TO the rollout kernels on the same SMs (the post step of a sweep: guard select, FP64 re-roll,
// deadlock heuristic) ask for the same L1 / shared-memory split as the rollouts: an SM changes its carve-out only when it
// is empty, so a kernel preferring another split has to wait for -- and idles -- whole SMs.
template <typename K> static void same_carveout(K kernel) {
#ifndef MRF_NO_CARVEOUT
    cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
#endif
}

// ---------------------------------- device-pointer entries --------------------------------------
template <typename T>
static int rollout_dev(mrf_handle_t h, const T* rec, int N, T* avg_vel, T* x_ee, T* goal_est, T* qN, T* qdN, int64_t B,
                       void* stream, bool aos = false, int sync_slot = 0, int n_var = MRF_REC, const T* rec_tail = nullptr,
                       T* risk = nullptr, RollExtra<T> ex = RollExtra<T>{}) {
    unsigned* const n_live = ex.n_live;
    const int n_static = ex.n_static;
    const T* const stat = ex.stat;
    if (!h || (!rec && !n_live)) return fail(MRF_EINVAL, "mrf_rollout: null argument");
    if (B <= 0 || N <= 0) return fail(MRF_EINVAL, "mrf_rollout: B and N must be positive");
    // mode 'acc' (MrfConfig.mode = 0) is the reference's own recurrence for that mode: it integrates a zero acceleration and
    // stores the planner output in q_dot (forward_planner_Jointspace.py:195,202,233) -- the same loop with action = qdd
    MRF_CUDA(cudaSetDevice(h->device));
    const int R = h->cfg.n_robots, NT = kTile * R;
    if (aos && (qN || qdN)) return fail(MRF_EINVAL, "mrf_rollout: record-order input has no trajectory output");
    if (n_static < 0 || n_static > MRF_MAX_STATIC || (n_static > 0 && (!stat || aos || n_live)))
        return fail(MRF_EINVAL, "mrf_rollout: bad static-obstacle arguments");
    if (!aos && R >= 2 && B <= h->coop_max_batch && !risk && !n_live && n_static == 0) {
        // few scenarios: latency matters, not throughput -> one CTA per scenario, one warp per robot (mrf_coop.cuh)
        switch (R) {
            case 2: rollout_coop_kernel<T, 2><<<(unsigned)B, 64, 0, (cudaStream_t)stream>>>(devcfg<T>(h), rec, N, avg_vel, x_ee, goal_est, qN, qdN, (long long)B); break;
            case 3: rollout_coop_kernel<T, 3><<<(unsigned)B, 96, 0, (cudaStream_t)stream>>>(devcfg<T>(h), rec, N, avg_vel, x_ee, goal_est, qN, qdN, (long long)B); break;
            case 4: rollout_coop_kernel<T, 4><<<(unsigned)B, 128, 0, (cudaStream_t)stream>>>(devcfg<T>(h), rec, N, avg_vel, x_ee, goal_est, qN, qdN, (long long)B); break;
            default: return fail(MRF_EINVAL, "mrf_rollout: n_robots out of range");
        }
        MRF_CUDA(cudaGetLastError());
        h->launches += 1;
        return MRF_OK;
    }
    const size_t smem = sizeof(T) * (size_t)(kKinRows<T> + P_N + 4 * n_static) * NT;
    long long grid = (B + kTile - 1) / kTile;
    if (n_live != nullptr && grid > 16) grid = 16; // device-side count: a few CTAs stride over the tiles (see the kernel)
    int rc = MRF_OK;
#define MRF_LAUNCH_ROLLOUT_K(RR, UU, AA, SS)                                                                         \
    {                                                                                                                \
        const size_t smem_k = smem + (kPairPath<T, RR, UU> ? sizeof(T) * (size_t)kPairRows * NT : 0);               \
        rc = set_smem(rollout_kernel<T, RR, UU, AA, SS>, smem_k);                                                    \
        same_carveout(rollout_kernel<T, RR, UU, AA, SS>);                                                            \
        if (rc) return rc;                                                                                           \
        rollout_kernel<T, RR, UU, AA, SS><<<(unsigned)grid, NT, smem_k, (cudaStream_t)stream>>>(                     \
            devcfg<T>(h), rec, N, avg_vel, x_ee, goal_est, qN, qdN, (long long)B, h->d_sync + 2 * sync_slot,        \
            (unsigned)h->zc_window, n_var, rec_tail, risk, ex);                                                      \
    }
#define MRF_LAUNCH_ROLLOUT(RR)                                                                                       \
    case RR:                                                                                                         \
        if (devcfg<T>(h).uniform_obst && n_static == 0) {                                                            \
            if (aos) MRF_LAUNCH_ROLLOUT_K(RR, true, true, false)                                                     \
            else if (stride) MRF_LAUNCH_ROLLOUT_STRIDE(RR, true)                                                     \
            else MRF_LAUNCH_ROLLOUT_K(RR, true, false, false)                                                        \
        } else {                                                                                                     \
            if (aos) MRF_LAUNCH_ROLLOUT_K(RR, false, true, false)                                                    \
            else if (stride) MRF_LAUNCH_ROLLOUT_STRIDE(RR, false)                                                    \
            else MRF_LAUNCH_ROLLOUT_K(RR, false, false, false)                                                       \
        }                                                                                                            \
        break;
    // the strided variant exists for FP64 only (the guard re-roll)
#define MRF_LAUNCH_ROLLOUT_STRIDE(RR, UU)                                                                            \
    {                                                                                                                \
        if constexpr (sizeof(T) == 8) MRF_LAUNCH_ROLLOUT_K(RR, UU, false, true)                                      \
        else return fail(MRF_EINVAL, "mrf_rollout: device-side count is FP64 only");                                 \
    }
    const bool stride = n_live != nullptr;
    if (aos) MRF_CUDA(cudaMemsetAsync(h->d_sync + 2 * sync_slot, 0, 2 * sizeof(unsigned), (cudaStream_t)stream));
    switch (R) {
        MRF_LAUNCH_ROLLOUT(1)
        MRF_LAUNCH_ROLLOUT(2)
        MRF_LAUNCH_ROLLOUT(3)
        MRF_LAUNCH_ROLLOUT(4)
        default: return fail(MRF_EINVAL, "mrf_rollout: n_robots out of range");
    }
#undef MRF_LAUNCH_ROLLOUT_STRIDE
#undef MRF_LAUNCH_ROLLOUT_K
#undef MRF_LAUNCH_ROLLOUT
    MRF_CUDA(cudaGetLastError());
    h->launches += 1;
    return MRF_OK;
}

template <typename T, bool CART>
static int action_dev(mrf_handle_t h, int robot_first, int n_rob, const T* rec, int S, const T* obst, int N, T* out,
                      T* qN, T* qdN, int64_t B, void* stream, const int32_t* sm_state = nullptr) {
    if (!h || !rec || (S > 0 && !obst)) return fail(MRF_EINVAL, "mrf_action: null argument");
    if (B <= 0 || S < 0 || n_rob < 1 || robot_first < 0 || robot_first + n_rob > h->cfg.n_robots)
        return fail(MRF_EINVAL, "mrf_action: bad sizes");
    if (CART && N <= 0) return fail(MRF_EINVAL, "mrf_rollout_cart: needs N > 0");
    MRF_CUDA(cudaSetDevice(h->device));
    // FP64: the per-thread tables (point table + axes + parameters + sphere ring: 142 doubles) bound the occupancy through
    // shared memory -- 128-thread CTAs fit once per SM (4 warps, one per scheduler: the FP64 pipe idles on every dependent
    // DFMA), one-warp CTAs six times (6 warps).  Measured (65 536 scenarios, Cartesian rollout S = 32 / 64): 6.09 / 30.9 ms
    // at 128 threads, 4.77 / 23.8 at 64, 4.63 / 23.0 at 32.
    static const int env_thr = getenv("MRF_ACTION_THREADS_F64") ? atoi(getenv("MRF_ACTION_THREADS_F64")) : 32;
    const int threads = sizeof(T) == 8 ? env_thr : kActThreads;
    const size_t smem = sizeof(T) * (size_t)(kKinRows<T> + P_N + kObstRing * MRF_OBST) * threads;
    int rc = set_smem(action_kernel<T, CART>, smem);
    if (rc) return rc;
    const long long total = (long long)n_rob * B;
    const long long grid = (total + threads - 1) / threads;
    action_kernel<T, CART><<<(unsigned)grid, threads, smem, (cudaStream_t)stream>>>(
        devcfg<T>(h), robot_first, n_rob, rec, S, obst, N, out, qN, qdN, (long long)B, sm_state);
    MRF_CUDA(cudaGetLastError());
    h->launches += 1;
    return MRF_OK;
}

template <typename T>
static int kinematics_dev(mrf_handle_t h, const T* q, const T* qd, T* x, T* v, T* a, int64_t B, void* stream) {
    if (!h || !q || !qd) return fail(MRF_EINVAL, "mrf_kinematics: null argument");
    if (B <= 0) return fail(MRF_EINVAL, "mrf_kinematics: B must be positive");
    MRF_CUDA(cudaSetDevice(h->device));
    const size_t smem = sizeof(T) * (size_t)kKinRows<T> * kActThreads;
    int rc = set_smem(kinematics_kernel<T>, smem);
    if (rc) return rc;
    const long long total = (long long)h->cfg.n_robots * B;
    kinematics_kernel<T><<<(unsigned)((total + kActThreads - 1) / kActThreads), kActThreads, smem, (cudaStream_t)stream>>>(
        devcfg<T>(h), q, qd, x, v, a, (long long)B);
    MRF_CUDA(cudaGetLastError());
    h->launches += 1;
    return MRF_OK;
}

template <typename T>
static int deadlock_dev(mrf_handle_t h, const T* x_ee, T* goals, T* weights, const T* avg_vel, const T* avg_sum,
                        const int32_t* sm_state, const int32_t* time_step, int32_t* tdo, int32_t* st_int, T* st_goal,
                        int32_t* flag, int64_t B, void* stream, bool rec_layout = false, const T* goal_est = nullptr,
                        DlOverride ov = DlOverride{nullptr, nullptr, nullptr, nullptr, 0, nullptr}, T* result = nullptr) {
    if (!h || !x_ee || !goals || !weights || !sm_state || !time_step || !tdo || !st_int || !st_goal)
        return fail(MRF_EINVAL, "mrf_deadlock: null argument");
    if (h->cfg.n_robots < 2)
        return fail(MRF_EINVAL, "mrf_deadlock: the heuristic is defined on robot pairs, n_robots must be >= 2 "
                                "(deadlock_prevention.py:29-30)");
    if (result && !avg_vel) return fail(MRF_EINVAL, "mrf_deadlock: the result tensor needs per-robot avg_vel");
    if ((avg_vel == nullptr) == (avg_sum == nullptr))
        return fail(MRF_EINVAL, "mrf_deadlock: give exactly one of avg_vel [R][B] and avg_sum [B]");
    if (B <= 0) return fail(MRF_EINVAL, "mrf_deadlock: B must be positive");
    MRF_CUDA(cudaSetDevice(h->device));
    const MrfConfig& c = h->cfg;
    const long long Rl = c.n_robots;
    DlCfg d{rec_layout ? (long long)B : 3 * (long long)B, rec_layout ? Rl * B : (long long)B, (long long)B,
            (rec_layout && c.estimate_goal && goal_est && c.estimate_robot < c.n_robots) ? c.estimate_robot : -1,
            c.n_robots, c.dl_time_wait, c.dl_time_gate, c.dl_avg_vel_constant, c.dl_dist_constant,
            c.dl_goal_weight_follower, c.dl_goal_weight_leader, c.dl_nr_goal_scale, c.dl_dist_endeff, c.dl_backoff};
    const long long dl_blocks = (B + 255) / 256;
    same_carveout(deadlock_kernel<T>);
    // Grid-stride.  As the last kernel of a sweep's post step (result tensor given) it runs next to the rollouts of the
    // following batches, where every CTA it places takes a slot from them: 16 CTAs instead of 64 cost the sweep 0.5 % less
    // (measured; fewer still lengthen the chain).  A stand-alone call wants the latency of the wider grid.
    const long long dl_grid = result != nullptr ? 16 : 64;
    deadlock_kernel<T><<<(unsigned)(dl_blocks < dl_grid ? dl_blocks : dl_grid), 256, 0, (cudaStream_t)stream>>>(
        d, x_ee, goals, weights, avg_vel, avg_sum, sm_state, time_step, tdo, st_int, st_goal, flag, goal_est, (long long)B,
        ov, result);
    MRF_CUDA(cudaGetLastError());
    h->launches += 1;
    return MRF_OK;
}

extern "C" int mrf_rollout_dev_f64(mrf_handle_t h, const double* rec, int N, double* avg_vel, double* x_ee,
                                   double* goal_est, double* qN, double* qdN, int64_t B, void* stream) {
    return rollout_dev<double>(h, rec, N, avg_vel, x_ee, goal_est, qN, qdN, B, stream);
}
extern "C" int mrf_rollout_dev_f32(mrf_handle_t h, const float* rec, int N, float* avg_vel, float* x_ee, float* goal_est,
                                   float* qN, float* qdN, int64_t B, void* stream) {
    return rollout_dev<float>(h, rec, N, avg_vel, x_ee, goal_est, qN, qdN, B, stream);
}
extern "C" int mrf_rollout_static_dev_f64(mrf_handle_t h, const double* rec, int N, int n_static, const double* stat,
                                          double* avg_vel, double* x_ee, double* goal_est, double* qN, double* qdN, int64_t B,
                                          void* stream) {
    RollExtra<double> ex{};
    ex.n_static = n_static;
    ex.stat = stat;
    return rollout_dev<double>(h, rec, N, avg_vel, x_ee, goal_est, qN, qdN, B, stream, false, 0, MRF_REC, nullptr, nullptr, ex);
}
extern "C" int mrf_rollout_static_dev_f32(mrf_handle_t h, const float* rec, int N, int n_static, const float* stat,
                                          float* avg_vel, float* x_ee, float* goal_est, float* qN, float* qdN, int64_t B,
                                          void* stream) {
    RollExtra<float> ex{};
    ex.n_static = n_static;
    ex.stat = stat;
    return rollout_dev<float>(h, rec, N, avg_vel, x_ee, goal_est, qN, qdN, B, stream, false, 0, MRF_REC, nullptr, nullptr, ex);
}
extern "C" int mrf_action_dev_f64(mrf_handle_t h, int robot_first, int n_rob, const double* rec, int S,
                                  const double* obst, double* action, int64_t B, void* stream) {
    return action_dev<double, false>(h, robot_first, n_rob, rec, S, obst, 0, action, nullptr, nullptr, B, stream);
}
extern "C" int mrf_action_dev_f32(mrf_handle_t h, int robot_first, int n_rob, const float* rec, int S, const float* obst,
                                  float* action, int64_t B, void* stream) {
    return action_dev<float, false>(h, robot_first, n_rob, rec, S, obst, 0, action, nullptr, nullptr, B, stream);
}
extern "C" int mrf_rollout_cart_dev_f64(mrf_handle_t h, int robot, const double* rec, int S, const double* obst, int N,
                                        double* avg_vel, double* qN, double* qdN, int64_t B, void* stream) {
    return action_dev<double, true>(h, robot, 1, rec, S, obst, N, avg_vel, qN, qdN, B, stream);
}
extern "C" int mrf_rollout_cart_dev_f32(mrf_handle_t h, int robot, const float* rec, int S, const float* obst, int N,
                                        float* avg_vel, float* qN, float* qdN, int64_t B, void* stream) {
    return action_dev<float, true>(h, robot, 1, rec, S, obst, N, avg_vel, qN, qdN, B, stream);
}
extern "C" int mrf_rollout_cart_all_dev_f64(mrf_handle_t h, const double* rec, int S, const double* obst, int N,
                                            double* avg_vel, double* qN, double* qdN, int64_t B, void* stream) {
    if (!h) return fail(MRF_EINVAL, "mrf_rollout_cart_all: null handle");
    return action_dev<double, true>(h, 0, h->cfg.n_robots, rec, S, obst, N, avg_vel, qN, qdN, B, stream);
}
extern "C" int mrf_rollout_cart_all_dev_f32(mrf_handle_t h, const float* rec, int S, const float* obst, int N,
                                            float* avg_vel, float* qN, float* qdN, int64_t B, void* stream) {
    if (!h) return fail(MRF_EINVAL, "mrf_rollout_cart_all: null handle");
    return action_dev<float, true>(h, 0, h->cfg.n_robots, rec, S, obst, N, avg_vel, qN, qdN, B, stream);
}
extern "C" int mrf_kinematics_dev_f64(mrf_handle_t h, const double* q, const double* qdot, double* x, double* v,
                                      double* a, int64_t B, void* stream) {
    return kinematics_dev<double>(h, q, qdot, x, v, a, B, stream);
}
extern "C" int mrf_kinematics_dev_f32(mrf_handle_t h, const float* q, const float* qdot, float* x, float* v, float* a,
                                      int64_t B, void* stream) {
    return kinematics_dev<float>(h, q, qdot, x, v, a, B, stream);
}
extern "C" int mrf_deadlock_dev_f64(mrf_handle_t h, const double* x_ee, double* goals, double* weights, const double* avg_vel,
                                    const double* avg_sum, const int32_t* sm_state, const int32_t* time_step,
                                    int32_t* time_deadlock_out, int32_t* st_int, double* st_goal, int32_t* flag, int64_t B,
                                    void* stream) {
    return deadlock_dev<double>(h, x_ee, goals, weights, avg_vel, avg_sum, sm_state, time_step, time_deadlock_out, st_int,
                             st_goal, flag, B, stream);
}
extern "C" int mrf_deadlock_dev_f32(mrf_handle_t h, const float* x_ee, float* goals, float* weights, const float* avg_vel,
                                    const float* avg_sum, const int32_t* sm_state, const int32_t* time_step,
                                    int32_t* time_deadlock_out, int32_t* st_int, float* st_goal, int32_t* flag, int64_t B,
                                    void* stream) {
    return deadlock_dev<float>(h, x_ee, goals, weights, avg_vel, avg_sum, sm_state, time_step, time_deadlock_out, st_int,
                             st_goal, flag, B, stream);
}

// deadlock step operating in place on the SoA record tensor: goals = rows MRF_G0..+2, weights = row MRF_W0
template <typename T>
static int deadlock_rec_dev(mrf_handle_t h, const T* x_ee, T* rec, const T* goal_est, const T* avg_vel, const T* avg_sum,
                            const int32_t* sm_state, const int32_t* time_step, int32_t* tdo, int32_t* st_int, T* st_goal,
                            int32_t* flag, int64_t B, void* stream) {
    if (!h || !rec) return fail(MRF_EINVAL, "mrf_deadlock_rec: null argument");
    const long long RB = (long long)h->cfg.n_robots * B;
    return deadlock_dev<T>(h, x_ee, rec + MRF_G0 * RB, rec + MRF_W0 * RB, avg_vel, avg_sum, sm_state, time_step, tdo, st_int,
                           st_goal, flag, B, stream, true, goal_est);
}
extern "C" int mrf_deadlock_rec_dev_f64(mrf_handle_t h, const double* x_ee, double* rec, const double* goal_est,
                                        const double* avg_vel, const double* avg_sum, const int32_t* sm_state,
                                        const int32_t* time_step, int32_t* time_deadlock_out, int32_t* st_int,
                                        double* st_goal, int32_t* flag, int64_t B, void* stream) {
    return deadlock_rec_dev<double>(h, x_ee, rec, goal_est, avg_vel, avg_sum, sm_state, time_step, time_deadlock_out, st_int,
                                    st_goal, flag, B, stream);
}
extern "C" int mrf_deadlock_rec_dev_f32(mrf_handle_t h, const float* x_ee, float* rec, const float* goal_est,
                                        const float* avg_vel, const float* avg_sum, const int32_t* sm_state,
                                        const int32_t* time_step, int32_t* time_deadlock_out, int32_t* st_int,
                                        float* st_goal, int32_t* flag, int64_t B, void* stream) {
    return deadlock_rec_dev<float>(h, x_ee, rec, goal_est, avg_vel, avg_sum, sm_state, time_step, time_deadlock_out, st_int,
                                   st_goal, flag, B, stream);
}

// ---------------------------------- RF-CV post step: FP64 guard re-roll + deadlock heuristic ----------------------
static int guard_reserve(mrf_handle_t h, int slot, size_t bytes) {
    if (h->guard_bytes[slot] >= bytes) return MRF_OK;
    if (h->guard_buf[slot]) MRF_CUDA(cudaFree(h->guard_buf[slot]));
    h->guard_buf[slot] = nullptr;
    h->guard_bytes[slot] = 0;
    if (cudaMalloc(&h->guard_buf[slot], bytes) != cudaSuccess) {
        cudaGetLastError();
        return fail(MRF_ENOMEM, "mrf_rfcv_post: device allocation failed");
    }
    h->guard_bytes[slot] = bytes;
    return MRF_OK;
}

template <typename T>
static int rfcv_post_dev(mrf_handle_t h, const T* rec, int N, const T* x_ee, T* rec_work, const T* goal_est,
                         const T* avg_vel, const T* risk, const int32_t* sm_state, const int32_t* time_step, int32_t* tdo,
                         int32_t* st_int, T* st_goal, int32_t* flag, T* result, int64_t B, void* stream, int slot,
                         const RollExtra<double>* src_records = nullptr) {
    // src_records: where the FP64 re-roll reads the listed scenarios' records from when that is not the SoA tensor `rec`
    // (host-record sweeps: the caller's AoS records in page-locked memory); `rec` then only has to expose the goal rows
    if (!h || !rec || !rec_work || !x_ee || !avg_vel || !sm_state || !time_step)
        return fail(MRF_EINVAL, "mrf_rfcv_post: null argument");
    if (slot < 0 || slot >= MRF_GUARD_SLOTS) return fail(MRF_EINVAL, "mrf_rfcv_post: slot out of range");
    if (B <= 0 || N <= 0) return fail(MRF_EINVAL, "mrf_rfcv_post: B and N must be positive");
    const int R = h->cfg.n_robots;
    const long long RB = (long long)R * B;
    const bool est = h->cfg.estimate_goal != 0 && goal_est != nullptr;
    const DlOverride ov{nullptr, nullptr, nullptr, nullptr, 0, nullptr};
    if (sizeof(T) == 4 && risk != nullptr) {
        if (R < 2 || R > 4) return fail(MRF_EINVAL, "mrf_rfcv_post: n_robots must be 2..4");
        MRF_CUDA(cudaSetDevice(h->device));
        cudaStream_t st = (cudaStream_t)stream;
        const long long cap = h->guard_cap > 0 ? h->guard_cap : (B / 16 > 256 ? B / 16 : 256);
        // doubles first (8-byte aligned), then the integer arrays
        const size_t n64 = (size_t)cap * ((size_t)R + 3 * R + 3);
        const size_t bytes = sizeof(double) * n64 + sizeof(int) * ((size_t)cap + (size_t)B);
        int rc = guard_reserve(h, slot, bytes);
        if (rc) return rc;
        double* avg64 = (double*)h->guard_buf[slot];
        double* xee64 = avg64 + (size_t)R * cap;
        double* gest64 = xee64 + (size_t)3 * R * cap;
        int* list = (int*)(gest64 + (size_t)3 * cap);
        int* slot_of = list + cap;
        unsigned* counters = h->d_sync + 16 + 4 * slot; // [0] is zero on entry: reset by the previous call's deadlock kernel
        GuardCfg g{R, est ? h->cfg.estimate_robot : -1, h->cfg.dl_avg_vel_constant, h->cfg.dl_dist_endeff, h->guard_band_dist,
                   {h->guard_band[0], h->guard_band[1], h->guard_band[2]}, {h->guard_rel[0], h->guard_rel[1], h->guard_rel[2]},
                   {h->guard_edge[0], h->guard_edge[1]}, (unsigned)cap};
        // the heuristic's arguments as both kernels of the post step see them (FP32 arrays)
        const MrfConfig& mc = h->cfg;
        DlPost dp{};
        dp.enabled = 1;
        dp.c = DlCfg{(long long)B, (long long)R * B, (long long)B,
                     (mc.estimate_goal && goal_est && mc.estimate_robot < mc.n_robots) ? mc.estimate_robot : -1,
                     mc.n_robots, mc.dl_time_wait, mc.dl_time_gate, mc.dl_avg_vel_constant, mc.dl_dist_constant,
                     mc.dl_goal_weight_follower, mc.dl_goal_weight_leader, mc.dl_nr_goal_scale, mc.dl_dist_endeff, mc.dl_backoff};
        dp.B = (long long)B;
        dp.x_ee = (const float*)x_ee;
        dp.goals = (float*)(rec_work + MRF_G0 * RB);
        dp.weights = (float*)(rec_work + MRF_W0 * RB);
        dp.avg_vel = (const float*)avg_vel;
        dp.sm_state = sm_state;
        dp.time_step = time_step;
        dp.tdo = tdo;
        dp.st_int = st_int;
        dp.st_goal = (float*)st_goal;
        dp.flag = flag;
        dp.goal_est = (const float*)goal_est;
        dp.result = (float*)result;
        dp.ov = DlOverride{slot_of, avg64, xee64, gest64, cap, counters};
        dp.done = h->d_sync + 16 + 4 * MRF_GUARD_SLOTS + slot;
        // kernel 1: list the scenarios to re-roll, run the heuristic for all the others
        const long long sel_blocks = (B + 255) / 256;
        same_carveout(guard_deadlock_kernel<T>);
        guard_deadlock_kernel<T><<<(unsigned)(sel_blocks < 64 ? sel_blocks : 64), 256, 0, st>>>(
            g, rec, risk, h->cfg.dl_time_gate, h->cfg.dl_dist_constant, slot_of, counters, list, dp);
        MRF_CUDA(cudaGetLastError());
        h->launches += 1;
        // kernel 2: FP64 re-roll of the listed scenarios by the throughput kernel, straight from the FP32 records through the
        // list (the kernel reads the count from device memory; grid: a few CTAs striding over the tiles), each CTA followed
        // by the heuristic for the scenarios it re-rolled
        RollExtra<double> ex{};
        if (src_records) {
            ex = *src_records;
        } else {
            ex.src = (const float*)rec;
            ex.sf = (long long)R * B;
            ex.sr = (long long)B;
            ex.sb = 1;
            ex.src_nvar = MRF_REC;
        }
        ex.n_live = counters;
        ex.list = list;
        ex.dl = dp;
        return rollout_dev<double>(h, nullptr, N, avg64, xee64, gest64, nullptr, nullptr, cap, stream, false, 0, MRF_REC, nullptr,
                                   nullptr, ex);
    }
    return deadlock_dev<T>(h, x_ee, rec_work + MRF_G0 * RB, rec_work + MRF_W0 * RB, avg_vel, nullptr, sm_state, time_step, tdo,
                           st_int, st_goal, flag, B, stream, true, goal_est, ov, result);
}
extern "C" int mrf_rfcv_post_dev_f32(mrf_handle_t h, const float* rec, int N, const float* x_ee, float* rec_work,
                                     const float* goal_est, const float* avg_vel, const float* risk,
                                     const int32_t* sm_state, const int32_t* time_step, int32_t* time_deadlock_out,
                                     int32_t* st_int, float* st_goal, int32_t* flag, float* result, int64_t B, void* stream,
                                     int slot) {
    return rfcv_post_dev<float>(h, rec, N, x_ee, rec_work, goal_est, avg_vel, risk, sm_state, time_step, time_deadlock_out,
                                st_int, st_goal, flag, result, B, stream, slot);
}
extern "C" int mrf_rfcv_post_dev_f64(mrf_handle_t h, const double* rec, int N, const double* x_ee, double* rec_work,
                                     const double* goal_est, const double* avg_vel, const double* risk,
                                     const int32_t* sm_state, const int32_t* time_step, int32_t* time_deadlock_out,
                                     int32_t* st_int, double* st_goal, int32_t* flag, double* result, int64_t B,
                                     void* stream, int slot) {
    return rfcv_post_dev<double>(h, rec, N, x_ee, rec_work, goal_est, avg_vel, risk, sm_state, time_step, time_deadlock_out,
                                 st_int, st_goal, flag, result, B, stream, slot);
}
extern "C" int mrf_rollout_risk_dev_f32(mrf_handle_t h, const float* rec, int N, float* avg_vel, float* x_ee, float* goal_est,
                                        float* risk, int64_t B, void* stream) {
    return rollout_dev<float>(h, rec, N, avg_vel, x_ee, goal_est, nullptr, nullptr, B, stream, false, 0, MRF_REC, nullptr, risk);
}
extern "C" int mrf_rollout_risk_dev_f64(mrf_handle_t h, const double* rec, int N, double* avg_vel, double* x_ee,
                                        double* goal_est, double* risk, int64_t B, void* stream) {
    return rollout_dev<double>(h, rec, N, avg_vel, x_ee, goal_est, nullptr, nullptr, B, stream, false, 0, MRF_REC, nullptr, risk);
}
extern "C" int mrf_set_guard(mrf_handle_t h, const double* bands, const double* risk_edges, double band_dist, int64_t cap) {
    if (!h) return fail(MRF_EINVAL, "mrf_set_guard: null handle");
    if (bands)
        for (int i = 0; i < 3; ++i) {
            h->guard_band[i] = bands[i];
            h->guard_rel[i] = bands[3 + i];
        }
    if (risk_edges) {
        if (!(risk_edges[0] <= risk_edges[1])) return fail(MRF_EINVAL, "mrf_set_guard: risk_edges must be ascending");
        h->guard_edge[0] = risk_edges[0];
        h->guard_edge[1] = risk_edges[1];
    }
    if (band_dist >= 0) h->guard_band_dist = band_dist;
    if (cap >= 0) h->guard_cap = cap;
    return MRF_OK;
}
extern "C" int mrf_guard_stats(mrf_handle_t h, int64_t* out) {
    if (!h || !out) return fail(MRF_EINVAL, "mrf_guard_stats: null argument");
    MRF_CUDA(cudaSetDevice(h->device));
    unsigned c[4 * MRF_GUARD_SLOTS];
    MRF_CUDA(cudaMemcpy(c, h->d_sync + 16, sizeof(c), cudaMemcpyDeviceToHost));
    out[0] = out[1] = 0;
    for (int i = 0; i < MRF_GUARD_SLOTS; ++i) {
        out[0] += c[4 * i + 2];
        out[1] += c[4 * i + 3];
    }
    out[2] = c[1];
    return MRF_OK;
}

// ---------------------------------- host-pointer entries ----------------------------------------
// Device scratch of the synchronous host entries.  Every call starts with scratch_reset and takes a distinct region
// for each array it stages; no region is reused within a call, so the staging needs no synchronisation of its own.  A
// call that outgrows the last block continues in a new one and keeps the old (its earlier regions live there).  The
// next reset frees them all -- cudaFree waits for the device, so no earlier work still reads them -- and allocates one
// block that holds the whole previous call: repeated calls with the same shapes allocate nothing.
static int scratch_grow(mrf_handle_t h, size_t bytes) {
    const size_t want = bytes + bytes / 4;
    void* p = nullptr;
    if (cudaMalloc(&p, want) != cudaSuccess) {
        cudaGetLastError();
        return fail(MRF_ENOMEM, "mrf: device allocation failed");
    }
    h->scratch.push_back(p);
    h->scratch_cap = want;
    h->scratch_off = 0;
    return MRF_OK;
}

static int scratch_reset(mrf_handle_t h) {
    const size_t used = h->scratch_used;
    h->scratch_off = h->scratch_used = 0;
    if (h->scratch.size() <= 1) return MRF_OK;
    for (void* p : h->scratch) MRF_CUDA(cudaFree(p));
    h->scratch.clear();
    h->scratch_cap = 0;
    return scratch_grow(h, used);
}

template <typename T> static int scratch_take(mrf_handle_t h, size_t n, T** out) {
    const size_t bytes = (sizeof(T) * n + 255) / 256 * 256;
    if (h->scratch_off + bytes > h->scratch_cap) {
        int rc = scratch_grow(h, h->scratch_used + bytes);
        if (rc) return rc;
    }
    *out = (T*)((char*)h->scratch.back() + h->scratch_off);
    h->scratch_off += bytes;
    h->scratch_used += bytes;
    return MRF_OK;
}

template <typename T, bool TO_DEVICE>
static int launch_layout(mrf_handle_t h, const T* in, T* out, long long B, int A, int F, cudaStream_t stream) {
    dim3 grid((unsigned)((B + 31) / 32), (unsigned)((A * F + 31) / 32)), block(32, 8);
    layout_kernel<T, TO_DEVICE><<<grid, block, 0, stream>>>(in, out, B, A, F);
    MRF_CUDA(cudaGetLastError());
    h->launches += 1;
    return MRF_OK;
}

// host [B][A][F] -> device [F][A][B] in scratch: one copy and one layout kernel on h->stream
template <typename T>
static int stage_in(mrf_handle_t h, const T* host, long long B, int A, int F, const T** dev) {
    const size_t n = (size_t)B * A * F;
    T *raw, *out;
    int rc = scratch_take(h, n, &raw);
    if (!rc) rc = scratch_take(h, n, &out);
    if (rc) return rc;
    MRF_CUDA(cudaMemcpyAsync(raw, host, sizeof(T) * n, cudaMemcpyHostToDevice, h->stream));
    *dev = out;
    return launch_layout<T, true>(h, raw, out, B, A, F, h->stream);
}

// device [F][A][B] -> host [B][A][F] on h->stream; nothing when host is null
template <typename T>
static int stage_out(mrf_handle_t h, const T* dev, long long B, int A, int F, T* host) {
    if (!host) return MRF_OK;
    const size_t n = (size_t)B * A * F;
    if (A * F > 1) { // with one field per scenario both layouts are the same array
        T* tmp;
        int rc = scratch_take(h, n, &tmp);
        if (!rc) rc = launch_layout<T, false>(h, dev, tmp, B, A, F, h->stream);
        if (rc) return rc;
        dev = tmp;
    }
    MRF_CUDA(cudaMemcpyAsync(host, dev, sizeof(T) * n, cudaMemcpyDeviceToHost, h->stream));
    return MRF_OK;
}

static int finish_timed(mrf_handle_t h) {
    MRF_CUDA(cudaStreamSynchronize(h->stream));
    float ms = 0.f;
    MRF_CUDA(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    h->last_ms = ms;
    return MRF_OK;
}

// Large batches without trajectory output: the batch is cut into chunks; the H2D copy of chunk c+1 (copy stream)
// overlaps the layout kernels + rollout + result read-back of chunk c (compute stream).
template <typename T>
static int rollout_host_pipelined(mrf_handle_t h, const T* rec, int N, T* avg_vel, T* x_ee, T* goal_est, int64_t B) {
    const int R = h->cfg.n_robots, C = B >= 32768 ? 8 : 4;
    const long long Bc = (((B + C - 1) / C) + 31) / 32 * 32; // chunk size, multiple of the CTA tile
    const size_t per = (size_t)(R + 3 * R + 3);
    T *d_aos, *d_soa, *d_res, *a_avg;
    int rc = scratch_take(h, (size_t)B * R * MRF_REC, &d_aos);               // records as uploaded
    if (!rc) rc = scratch_take(h, (size_t)Bc * C * R * MRF_REC, &d_soa);     // device layout, one block per chunk
    if (!rc) rc = scratch_take(h, per * Bc * C, &d_res);                     // device-layout results per chunk
    if (!rc) rc = scratch_take(h, per * B, &a_avg);                          // host order: avg [B][R], x_ee [B][3R], goal [B][3]
    if (rc) return rc;
    T* a_xee = a_avg + (size_t)B * R;
    T* a_goal = a_xee + (size_t)B * 3 * R;
    // make sure earlier work on the compute stream no longer reads the staging buffers the copy stream overwrites
    MRF_CUDA(cudaEventRecord(h->ev0, h->stream));
    MRF_CUDA(cudaEventRecord(h->ev_free, h->stream));
    MRF_CUDA(cudaStreamWaitEvent(h->s_copy, h->ev_free, 0));
    int used = 0;
    for (int c = 0; c < C; ++c) {
        const long long lo = (long long)c * Bc, n = (lo + Bc <= B ? Bc : B - lo);
        if (n <= 0) break;
        used = c + 1;
        // one stream per chunk: the rollout kernels of consecutive chunks overlap on the GPU (a 16k-scenario chunk
        // alone is less than one wave of CTAs), only the copy -> compute order of each chunk is enforced
        cudaStream_t cs = h->s_chunk[c];
        MRF_CUDA(cudaStreamWaitEvent(cs, h->ev_free, 0));
        T* c_aos = d_aos + (size_t)lo * R * MRF_REC;
        MRF_CUDA(cudaMemcpyAsync(c_aos, rec + (size_t)lo * R * MRF_REC, sizeof(T) * (size_t)n * R * MRF_REC,
                                 cudaMemcpyHostToDevice, h->s_copy));
        MRF_CUDA(cudaEventRecord(h->ev_up[c], h->s_copy));
        MRF_CUDA(cudaStreamWaitEvent(cs, h->ev_up[c], 0));
        T* c_soa = d_soa + (size_t)c * Bc * R * MRF_REC;
        rc = launch_layout<T, true>(h, c_aos, c_soa, n, R, MRF_REC, cs);
        if (rc) return rc;
        T* d_avg = d_res + (size_t)c * Bc * per;
        T* d_xee = d_avg + (size_t)R * n;
        T* d_goal = d_xee + (size_t)3 * R * n;
        rc = rollout_dev<T>(h, c_soa, N, d_avg, d_xee, d_goal, nullptr, nullptr, n, cs);
        if (rc) return rc;
        struct { T* src; T* dst; T* host; int F; } outs[3] = {{d_avg, a_avg + (size_t)lo * R, avg_vel, R},
                                                              {d_xee, a_xee + (size_t)lo * 3 * R, x_ee, 3 * R},
                                                              {d_goal, a_goal + (size_t)lo * 3, goal_est, 3}};
        for (auto& o : outs) {
            if (!o.host) continue;
            rc = launch_layout<T, false>(h, o.src, o.dst, n, 1, o.F, cs);
            if (rc) return rc;
            MRF_CUDA(cudaMemcpyAsync(o.host + (size_t)lo * o.F, o.dst, sizeof(T) * (size_t)n * o.F, cudaMemcpyDeviceToHost, cs));
        }
        MRF_CUDA(cudaEventRecord(h->ev_chunk[c], cs));
    }
    for (int c = 0; c < used; ++c) MRF_CUDA(cudaStreamWaitEvent(h->stream, h->ev_chunk[c], 0));
    MRF_CUDA(cudaEventRecord(h->ev1, h->stream));
    return finish_timed(h);
}

// Device view of a host pointer when it is page-locked (cudaHostAlloc / cudaHostRegister: torch pinned tensors), else
// nullptr.  With unified addressing the kernel can read and write such memory directly over PCIe.
static void* pinned_view(const void* p) {
    if (!p) return nullptr;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        (void)cudaGetLastError();
        return nullptr;
    }
    return (a.type == cudaMemoryTypeHost && ((uintptr_t)a.devicePointer & 15) == 0) ? a.devicePointer : nullptr;
}

// Page-locked records: ONE kernel launch reads the caller's records straight from host memory (record order, coalesced
// 16-byte loads per tile) and writes avg / x_ee / goal straight back -- the CTA scheduler overlaps the PCIe reads of
// later tiles with the horizons of earlier ones, so there is no staging copy, no layout kernel and no chunk pipeline.
// Results whose host buffer is not page-locked go through a device buffer and one copy.
template <typename T>
static int rollout_host_zerocopy(mrf_handle_t h, const T* rec_view, int N, T* avg_vel, T* x_ee, T* goal_est, int64_t B) {
    const int R = h->cfg.n_robots;
    struct Out { T* host; T* dev; size_t n; bool direct; } outs[3] = {{avg_vel, nullptr, (size_t)B * R, false},
                                                                      {x_ee, nullptr, (size_t)B * 3 * R, false},
                                                                      {goal_est, nullptr, (size_t)B * 3, false}};
    for (auto& o : outs) {
        if (!o.host) continue;
        o.dev = (T*)pinned_view(o.host);
        o.direct = o.dev != nullptr;
        if (!o.direct) {
            int rc = scratch_take(h, o.n, &o.dev);
            if (rc) return rc;
        }
    }
    MRF_CUDA(cudaEventRecord(h->ev0, h->stream));
    int rc = rollout_dev<T>(h, rec_view, N, outs[0].dev, outs[1].dev, outs[2].dev, nullptr, nullptr, B, h->stream, true);
    if (rc) return rc;
    MRF_CUDA(cudaEventRecord(h->ev1, h->stream));
    for (auto& o : outs)
        if (o.host && !o.direct)
            MRF_CUDA(cudaMemcpyAsync(o.host, o.dev, sizeof(T) * o.n, cudaMemcpyDeviceToHost, h->stream));
    return finish_timed(h);
}

template <typename T>
static int rollout_host(mrf_handle_t h, const T* rec, int N, T* avg_vel, T* x_ee, T* goal_est, T* qN, T* qdN, int64_t B) {
    if (!h || !rec) return fail(MRF_EINVAL, "mrf_rollout_host: null argument");
    if (B <= 0 || N <= 0) return fail(MRF_EINVAL, "mrf_rollout_host: B and N must be positive");
    MRF_CUDA(cudaSetDevice(h->device));
    const int R = h->cfg.n_robots;
    int rc = scratch_reset(h);
    if (rc) return rc;
    if (!qN && !qdN && B >= 8192) {
        if (h->zero_copy)
            if (const T* view = (const T*)pinned_view(rec)) return rollout_host_zerocopy<T>(h, view, N, avg_vel, x_ee, goal_est, B);
        return rollout_host_pipelined<T>(h, rec, N, avg_vel, x_ee, goal_est, B);
    }
    const T* d_rec;
    T *d_avg, *d_xee, *d_goal, *d_q = nullptr, *d_qd = nullptr;
    const size_t n_traj = (size_t)B * R * N * MRF_DOF;
    rc = stage_in(h, rec, B, R, MRF_REC, &d_rec);
    if (!rc) rc = scratch_take(h, (size_t)B * R, &d_avg);          // [R][B]
    if (!rc) rc = scratch_take(h, (size_t)B * 3 * R, &d_xee);      // [R][3][B]
    if (!rc) rc = scratch_take(h, (size_t)B * 3, &d_goal);         // [3][B]
    if (!rc && qN) rc = scratch_take(h, n_traj, &d_q);             // [R][N][7][B]
    if (!rc && qdN) rc = scratch_take(h, n_traj, &d_qd);
    if (rc) return rc;
    MRF_CUDA(cudaEventRecord(h->ev0, h->stream));
    rc = rollout_dev<T>(h, d_rec, N, d_avg, d_xee, d_goal, d_q, d_qd, B, h->stream);
    if (rc) return rc;
    MRF_CUDA(cudaEventRecord(h->ev1, h->stream));
    rc = stage_out(h, d_avg, B, 1, R, avg_vel);
    if (!rc) rc = stage_out(h, d_xee, B, 1, 3 * R, x_ee);
    if (!rc) rc = stage_out(h, d_goal, B, 1, 3, goal_est);
    if (!rc) rc = stage_out(h, d_q, B, 1, R * N * MRF_DOF, qN);
    if (!rc) rc = stage_out(h, d_qd, B, 1, R * N * MRF_DOF, qdN);
    if (rc) return rc;
    return finish_timed(h);
}

// Two-deep submit / wait pipeline over the in-place path, for sweeps of independent batches: while batch i computes,
// the tiles of batch i+1 are already being read over PCIe (the kernels sit on two streams and share the SMs), so the
// bus fill of one launch hides behind the tail of the previous one.  All buffers must be page-locked.
static int rollout_wait_oldest(mrf_handle_t h) {
    const int s = h->zc_oldest;
    if (!h->zc_pending[s]) return MRF_OK;
    MRF_CUDA(cudaSetDevice(h->device));
    MRF_CUDA(cudaEventSynchronize(h->ev_chunk[s]));
    h->zc_pending[s] = 0;
    h->zc_oldest = s ^ 1;
    return MRF_OK;
}
template <typename T>
static int rollout_host_submit(mrf_handle_t h, const T* rec, int N, T* avg_vel, T* x_ee, T* goal_est, int64_t B,
                               const T* shared = nullptr) {
    if (!h || !rec) return fail(MRF_EINVAL, "mrf_rollout_host_submit: null argument");
    if (B <= 0 || N <= 0) return fail(MRF_EINVAL, "mrf_rollout_host_submit: B and N must be positive");
    MRF_CUDA(cudaSetDevice(h->device));
    const T* view = (const T*)pinned_view(rec);
    T* outs[3] = {avg_vel, x_ee, goal_est};
    T* dv[3] = {nullptr, nullptr, nullptr};
    bool ok = view != nullptr;
    for (int i = 0; i < 3 && ok; ++i)
        if (outs[i]) {
            cudaPointerAttributes a;
            ok = cudaPointerGetAttributes(&a, outs[i]) == cudaSuccess && a.type == cudaMemoryTypeHost && a.devicePointer;
            if (ok) dv[i] = (T*)a.devicePointer; else (void)cudaGetLastError();
        }
    if (!ok) return fail(MRF_EINVAL, "mrf_rollout_host_submit: records and results must be page-locked host memory "
                                     "(cudaHostAlloc / cudaHostRegister, records 16-byte aligned)");
    const int s = h->zc_slot;
    if (h->zc_pending[s]) { // both slots busy: the oldest submission is the one in this slot
        int rc = rollout_wait_oldest(h);
        if (rc) return rc;
    }
    int rc;
    const T* d_tail = nullptr;
    if (shared) { // compact records: the shared trailing fields travel once per submission (R x 44 scalars)
        const size_t tb = sizeof(T) * (size_t)h->cfg.n_robots * MRF_REC;
        MRF_CUDA(cudaMemcpyAsync(h->d_tail[s], shared, tb, cudaMemcpyHostToDevice, h->s_chunk[s]));
        d_tail = (const T*)h->d_tail[s];
    }
    rc = rollout_dev<T>(h, view, N, dv[0], dv[1], dv[2], nullptr, nullptr, B, h->s_chunk[s], true, 1 + s,
                        shared ? MRF_G1 : MRF_REC, d_tail);
    if (rc) return rc;
    MRF_CUDA(cudaEventRecord(h->ev_chunk[s], h->s_chunk[s]));
    if (!h->zc_pending[s ^ 1]) h->zc_oldest = s;
    h->zc_pending[s] = 1;
    h->zc_slot = s ^ 1;
    return MRF_OK;
}
extern "C" int mrf_rollout_host_submit_f64(mrf_handle_t h, const double* rec, int N, double* avg_vel, double* x_ee,
                                           double* goal_est, int64_t B) {
    return rollout_host_submit<double>(h, rec, N, avg_vel, x_ee, goal_est, B);
}
extern "C" int mrf_rollout_host_submit_f32(mrf_handle_t h, const float* rec, int N, float* avg_vel, float* x_ee,
                                           float* goal_est, int64_t B) {
    return rollout_host_submit<float>(h, rec, N, avg_vel, x_ee, goal_est, B);
}
extern "C" int mrf_rollout_host_submit_compact_f64(mrf_handle_t h, const double* rec_var, const double* rec_shared, int N,
                                                   double* avg_vel, double* x_ee, double* goal_est, int64_t B) {
    if (!rec_shared) return fail(MRF_EINVAL, "mrf_rollout_host_submit_compact: null argument");
    return rollout_host_submit<double>(h, rec_var, N, avg_vel, x_ee, goal_est, B, rec_shared);
}
extern "C" int mrf_rollout_host_submit_compact_f32(mrf_handle_t h, const float* rec_var, const float* rec_shared, int N,
                                                   float* avg_vel, float* x_ee, float* goal_est, int64_t B) {
    if (!rec_shared) return fail(MRF_EINVAL, "mrf_rollout_host_submit_compact: null argument");
    return rollout_host_submit<float>(h, rec_var, N, avg_vel, x_ee, goal_est, B, rec_shared);
}

// One RF-CV step of a sweep END TO END from host memory: the in-place rollout kernel reads the caller's page-locked
// records over PCIe and leaves its results on the device (SoA); the post step -- guard select, FP64 re-roll of the listed
// scenarios (read from the same host records through the list), deadlock heuristic -- follows on the same stream, and
// only the per-scenario result [R+1][B] (and optionally the resolved goals / weights [4][R][B]) travels back.  Stateless:
// every batch is a fresh control step (no deadlock history: time_deadlock_out = 1000, leader / follower at their
// defaults), state-machine codes 0, one time step for the batch.
static int rf_wait_oldest(mrf_handle_t h) {
    if (h->rf_count == 0) return MRF_OK;
    const int s = (h->rf_head - h->rf_count + 8) & 3;
    MRF_CUDA(cudaSetDevice(h->device));
    MRF_CUDA(cudaEventSynchronize(h->ev_rf[s]));
    h->rf_count -= 1;
    return MRF_OK;
}

__global__ void rfcv_state_init_kernel(int32_t* __restrict__ sm, int32_t* __restrict__ ts, int32_t* __restrict__ tdo,
                                       int32_t* __restrict__ st_int, float* __restrict__ st_goal, int32_t time_step, int R,
                                       long long B) {
    for (long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x; b < B; b += (long long)gridDim.x * blockDim.x) {
        for (int r = 0; r < R; ++r) sm[(long long)r * B + b] = 0;
        ts[b] = time_step;
        tdo[b] = 1000;
        st_int[0 * B + b] = 0; st_int[1 * B + b] = 1; st_int[2 * B + b] = 0; st_int[3 * B + b] = 1;
        st_goal[0 * B + b] = 0.f; st_goal[1 * B + b] = 0.f; st_goal[2 * B + b] = 0.f;
    }
}

extern "C" int mrf_rfcv_host_submit_f32(mrf_handle_t h, const float* rec, const float* rec_shared, int N, int32_t time_step,
                                        float* result, float* goals_out, int64_t B) {
    if (!h || !rec || !result) return fail(MRF_EINVAL, "mrf_rfcv_host_submit: null argument");
    if (B <= 0 || N <= 0) return fail(MRF_EINVAL, "mrf_rfcv_host_submit: B and N must be positive");
    const int R = h->cfg.n_robots;
    if (R < 2) return fail(MRF_EINVAL, "mrf_rfcv_host_submit: the deadlock heuristic needs n_robots >= 2");
    MRF_CUDA(cudaSetDevice(h->device));
    const float* view = (const float*)pinned_view(rec);
    if (!view) return fail(MRF_EINVAL, "mrf_rfcv_host_submit: records must be page-locked host memory, 16-byte aligned");
    for (const void* p : {(const void*)result, (const void*)goals_out}) {
        if (!p) continue;
        cudaPointerAttributes a;
        if (cudaPointerGetAttributes(&a, p) != cudaSuccess || a.type != cudaMemoryTypeHost) {
            (void)cudaGetLastError();
            return fail(MRF_EINVAL, "mrf_rfcv_host_submit: result buffers must be page-locked host memory");
        }
    }
    if (h->rf_count == 4) { // four batches in flight: the oldest one is in the slot this submission takes
        int rc = rf_wait_oldest(h);
        if (rc) return rc;
    }
    const int s = h->rf_head;
    cudaStream_t st = h->s_chunk[4 + s];
    const long long RB = (long long)R * B;
    const int n_var = rec_shared ? MRF_G1 : MRF_REC;
    // per-slot device buffers: avg, risk [R][B]; x_ee [R][3][B]; goal_est [3][B]; rec_out [n_var][R][B]; st_goal [3][B];
    // result [R+1][B]; int: sm [R][B], ts, tdo, flag [B], st_int [4][B]
    const size_t nf = (size_t)(2 * RB + 3 * RB + 3 * B + (long long)n_var * RB + 3 * B + (R + 1) * B), ni = (size_t)(RB + 3 * B + 4 * B);
    if (h->rf_bytes[s] < 4 * (nf + ni)) {  // (the slot is idle: its previous batch was waited for above or long ago)
        if (h->rf_buf[s]) MRF_CUDA(cudaFree(h->rf_buf[s]));
        h->rf_buf[s] = nullptr;
        h->rf_bytes[s] = 0;
        if (cudaMalloc(&h->rf_buf[s], 4 * (nf + ni)) != cudaSuccess) {
            cudaGetLastError();
            return fail(MRF_ENOMEM, "mrf_rfcv_host_submit: device allocation failed");
        }
        h->rf_bytes[s] = 4 * (nf + ni);
    }
    float* avg = (float*)h->rf_buf[s];
    float* risk = avg + RB;
    float* xee = risk + RB;
    float* gest = xee + 3 * RB;
    float* rec_out = gest + 3 * B;
    float* st_goal = rec_out + (long long)n_var * RB;
    float* d_result = st_goal + 3 * B;
    int32_t* sm = (int32_t*)(d_result + (R + 1) * B);
    int32_t* ts = sm + RB;
    int32_t* tdo = ts + B;
    int32_t* flag = tdo + B;
    int32_t* st_int = flag + B;
    const float* d_tail = nullptr;
    if (rec_shared) {
        MRF_CUDA(cudaMemcpyAsync(h->d_tail_rf[s], rec_shared, sizeof(float) * (size_t)R * MRF_REC, cudaMemcpyHostToDevice, st));
        d_tail = (const float*)h->d_tail_rf[s];
    }
    const long long ib = (B + 255) / 256;
    rfcv_state_init_kernel<<<(unsigned)(ib < 64 ? ib : 64), 256, 0, st>>>(sm, ts, tdo, st_int, st_goal, time_step, R, (long long)B);
    MRF_CUDA(cudaGetLastError());
    h->launches += 1;
    RollExtra<float> ex{};
    ex.out_soa = 1;
    ex.rec_out = rec_out;
    // at most TWO rollout kernels share the GPU and the bus (the in-place reads are admitted tile window by tile window;
    // with four kernels resident most CTAs would spin on admission): this rollout starts when the one two batches
    // earlier has finished -- the post steps of up to four batches still overlap
    if (h->rf_roll_valid[(s + 2) & 3]) MRF_CUDA(cudaStreamWaitEvent(st, h->ev_rf_roll[(s + 2) & 3], 0));
    int rc = rollout_dev<float>(h, view, N, avg, xee, gest, nullptr, nullptr, B, st, true, 3 + s, n_var, d_tail, risk, ex);
    if (rc) return rc;
    MRF_CUDA(cudaEventRecord(h->ev_rf_roll[s], st));
    h->rf_roll_valid[s] = 1;
    // post step on the slot's HIGH-PRIORITY stream (its small kernels are placed as soon as a rollout CTA retires), reading
    // the device copy of the records: rows MRF_G0..MRF_W0 for the heuristic (in place), whole records for the re-roll
    // (fields >= n_var of compact records from the shared tail)
    cudaStream_t sp = h->s_rf_post[s];
    MRF_CUDA(cudaStreamWaitEvent(sp, h->ev_rf_roll[s], 0));
    RollExtra<double> src{};
    src.src = rec_out;
    src.sf = RB;
    src.sr = (long long)B;
    src.sb = 1;
    src.src_nvar = n_var;
    src.src_tail = d_tail;
    rc = rfcv_post_dev<float>(h, rec_out, N, xee, rec_out, gest, avg, risk, sm, ts, tdo, st_int, st_goal, flag, d_result, B, sp,
                              4 + s, &src);
    if (rc) return rc;
    MRF_CUDA(cudaMemcpyAsync(result, d_result, sizeof(float) * (size_t)(R + 1) * B, cudaMemcpyDeviceToHost, sp));
    if (goals_out)
        MRF_CUDA(cudaMemcpyAsync(goals_out, rec_out + (long long)MRF_G0 * RB, sizeof(float) * (size_t)4 * RB, cudaMemcpyDeviceToHost, sp));
    MRF_CUDA(cudaEventRecord(h->ev_rf[s], sp));
    h->rf_head = (s + 1) & 3;
    h->rf_count += 1;
    return MRF_OK;
}
extern "C" int mrf_rollout_host_wait(mrf_handle_t h, int all) {
    if (!h) return fail(MRF_EINVAL, "mrf_rollout_host_wait: null handle");
    int rc = rollout_wait_oldest(h);
    if (rc) return rc;
    rc = rf_wait_oldest(h);
    if (rc || !all) return rc;
    rc = rollout_wait_oldest(h);
    while (!rc && h->rf_count > 0) rc = rf_wait_oldest(h);
    return rc;
}

template <typename T, bool CART>
static int action_host(mrf_handle_t h, int robot_first, int n_rob, const T* rec, int S, const T* obst, int N, T* out,
                       T* qN, T* qdN, int64_t B) {
    if (!h || !rec || (S > 0 && !obst)) return fail(MRF_EINVAL, "mrf_action_host: null argument");
    if (B <= 0 || S < 0 || n_rob < 1) return fail(MRF_EINVAL, "mrf_action_host: bad sizes");
    MRF_CUDA(cudaSetDevice(h->device));
    const int R = n_rob;
    const T *d_rec, *d_obst = nullptr;
    T *d_out, *d_q = nullptr, *d_qd = nullptr;
    const size_t n_traj = CART ? (size_t)B * N * MRF_DOF : 0;
    int rc = scratch_reset(h);
    if (!rc) rc = stage_in(h, rec, B, R, MRF_REC, &d_rec);
    if (!rc && S > 0) rc = stage_in(h, obst, B, R, S * MRF_OBST, &d_obst);          // [S][10][R][B]
    if (!rc) rc = scratch_take(h, (size_t)B * (CART ? 1 : MRF_DOF * R), &d_out);    // avg_vel [B] or action [7][R][B]
    if (!rc && CART && qN) rc = scratch_take(h, n_traj, &d_q);                      // [N][7][B]
    if (!rc && CART && qdN) rc = scratch_take(h, n_traj, &d_qd);
    if (rc) return rc;
    MRF_CUDA(cudaEventRecord(h->ev0, h->stream));
    rc = action_dev<T, CART>(h, robot_first, n_rob, d_rec, S, d_obst, N, d_out, d_q, d_qd, B, h->stream);
    if (rc) return rc;
    MRF_CUDA(cudaEventRecord(h->ev1, h->stream));
    if (CART) {
        rc = stage_out(h, d_out, B, 1, 1, out);
        if (!rc) rc = stage_out(h, d_q, B, 1, N * MRF_DOF, qN);
        if (!rc) rc = stage_out(h, d_qd, B, 1, N * MRF_DOF, qdN);
    } else {
        rc = stage_out(h, d_out, B, R, MRF_DOF, out);
    }
    if (rc) return rc;
    return finish_timed(h);
}

extern "C" int mrf_rollout_host_f64(mrf_handle_t h, const double* rec, int N, double* avg_vel, double* x_ee,
                                    double* goal_est, double* qN, double* qdN, int64_t B) {
    return rollout_host<double>(h, rec, N, avg_vel, x_ee, goal_est, qN, qdN, B);
}
extern "C" int mrf_rollout_host_f32(mrf_handle_t h, const float* rec, int N, float* avg_vel, float* x_ee, float* goal_est,
                                    float* qN, float* qdN, int64_t B) {
    return rollout_host<float>(h, rec, N, avg_vel, x_ee, goal_est, qN, qdN, B);
}
extern "C" int mrf_action_host_f64(mrf_handle_t h, int robot_first, int n_rob, const double* rec, int S,
                                   const double* obst, double* action, int64_t B) {
    return action_host<double, false>(h, robot_first, n_rob, rec, S, obst, 0, action, nullptr, nullptr, B);
}
extern "C" int mrf_action_host_f32(mrf_handle_t h, int robot_first, int n_rob, const float* rec, int S, const float* obst,
                                   float* action, int64_t B) {
    return action_host<float, false>(h, robot_first, n_rob, rec, S, obst, 0, action, nullptr, nullptr, B);
}
extern "C" int mrf_rollout_cart_host_f64(mrf_handle_t h, int robot, const double* rec, int S, const double* obst, int N,
                                         double* avg_vel, double* qN, double* qdN, int64_t B) {
    return action_host<double, true>(h, robot, 1, rec, S, obst, N, avg_vel, qN, qdN, B);
}
extern "C" int mrf_rollout_cart_host_f32(mrf_handle_t h, int robot, const float* rec, int S, const float* obst, int N,
                                         float* avg_vel, float* qN, float* qdN, int64_t B) {
    return action_host<float, true>(h, robot, 1, rec, S, obst, N, avg_vel, qN, qdN, B);
}

extern "C" int mrf_kinematics_host_f64(mrf_handle_t h, const double* q, const double* qdot, double* x, double* v,
                                       double* a, int64_t B) {
    if (!h || !q || !qdot) return fail(MRF_EINVAL, "mrf_kinematics_host: null argument");
    if (B <= 0) return fail(MRF_EINVAL, "mrf_kinematics_host: B must be positive");
    MRF_CUDA(cudaSetDevice(h->device));
    const int R = h->cfg.n_robots, F = MRF_NLINKS * 3; // outputs: device [l][c][r][b], host [b][r][l][c]
    const double *d_q, *d_qd;
    double *d_x, *d_v, *d_a;
    int rc = scratch_reset(h);
    if (!rc) rc = stage_in(h, q, B, R, MRF_DOF, &d_q);
    if (!rc) rc = stage_in(h, qdot, B, R, MRF_DOF, &d_qd);
    if (!rc) rc = scratch_take(h, (size_t)B * R * F, &d_x);
    if (!rc) rc = scratch_take(h, (size_t)B * R * F, &d_v);
    if (!rc) rc = scratch_take(h, (size_t)B * R * F, &d_a);
    if (rc) return rc;
    MRF_CUDA(cudaEventRecord(h->ev0, h->stream));
    rc = kinematics_dev<double>(h, d_q, d_qd, d_x, d_v, d_a, B, h->stream);
    if (rc) return rc;
    MRF_CUDA(cudaEventRecord(h->ev1, h->stream));
    rc = stage_out(h, d_x, B, R, F, x);
    if (!rc) rc = stage_out(h, d_v, B, R, F, v);
    if (!rc) rc = stage_out(h, d_a, B, R, F, a);
    if (rc) return rc;
    return finish_timed(h);
}

// host variant of the deadlock step: arrays in the reference's order, marshalled to SoA on the host (O(B R) copies)
extern "C" int mrf_deadlock_host_f64(mrf_handle_t h, const double* x_ee, double* goals, double* weights,
                                     const double* avg_sum, const int32_t* sm_state, const int32_t* time_step,
                                     int32_t* time_deadlock_out, int32_t* st_int, double* st_goal, int32_t* flag,
                                     int64_t B) {
    if (!h || !x_ee || !goals || !weights || !avg_sum || !sm_state || !time_step || !time_deadlock_out || !st_int ||
        !st_goal)
        return fail(MRF_EINVAL, "mrf_deadlock_host: null argument");
    if (B <= 0) return fail(MRF_EINVAL, "mrf_deadlock_host: B must be positive");
    MRF_CUDA(cudaSetDevice(h->device));
    const int R = h->cfg.n_robots;
    const size_t nd = (size_t)B * (3 * R + 3 * R + R + 1 + 3), ni = (size_t)B * (R + 1 + 1 + 4 + 1);
    std::vector<double> hd(nd);
    std::vector<int32_t> hi(ni);
    double* px = hd.data();
    double* pg = px + (size_t)3 * R * B;
    double* pw = pg + (size_t)3 * R * B;
    double* pa = pw + (size_t)R * B;
    double* ps = pa + B;
    int32_t* qs = hi.data();
    int32_t* qt = qs + (size_t)R * B;
    int32_t* qo = qt + B;
    int32_t* qi = qo + B;
    int32_t* qf = qi + (size_t)4 * B;
    for (int64_t b = 0; b < B; ++b) {
        for (int r = 0; r < R; ++r) {
            for (int k = 0; k < 3; ++k) {
                px[((size_t)r * 3 + k) * B + b] = x_ee[(b * R + r) * 3 + k];
                pg[((size_t)r * 3 + k) * B + b] = goals[(b * R + r) * 3 + k];
            }
            pw[(size_t)r * B + b] = weights[b * R + r];
            qs[(size_t)r * B + b] = sm_state[b * R + r];
        }
        pa[b] = avg_sum[b];
        qt[b] = time_step[b];
        qo[b] = time_deadlock_out[b];
        for (int k = 0; k < 4; ++k) qi[(size_t)k * B + b] = st_int[b * 4 + k];
        for (int k = 0; k < 3; ++k) ps[(size_t)k * B + b] = st_goal[b * 3 + k];
    }
    double* dd;
    int32_t* di;
    int rc = scratch_reset(h);
    if (!rc) rc = scratch_take(h, nd, &dd);
    if (!rc) rc = scratch_take(h, ni, &di);
    if (rc) return rc;
    MRF_CUDA(cudaMemcpyAsync(dd, hd.data(), sizeof(double) * nd, cudaMemcpyHostToDevice, h->stream));
    MRF_CUDA(cudaMemcpyAsync(di, hi.data(), sizeof(int32_t) * ni, cudaMemcpyHostToDevice, h->stream));
    MRF_CUDA(cudaEventRecord(h->ev0, h->stream));
    rc = deadlock_dev<double>(h, dd, dd + (pg - px), dd + (pw - px), nullptr, dd + (pa - px), di, di + (qt - qs),
                              di + (qo - qs), di + (qi - qs), dd + (ps - px), di + (qf - qs), B, h->stream);
    if (rc) return rc;
    MRF_CUDA(cudaEventRecord(h->ev1, h->stream));
    MRF_CUDA(cudaMemcpyAsync(hd.data(), dd, sizeof(double) * nd, cudaMemcpyDeviceToHost, h->stream));
    MRF_CUDA(cudaMemcpyAsync(hi.data(), di, sizeof(int32_t) * ni, cudaMemcpyDeviceToHost, h->stream));
    rc = finish_timed(h);
    if (rc) return rc;
    for (int64_t b = 0; b < B; ++b) {
        for (int r = 0; r < R; ++r) {
            for (int k = 0; k < 3; ++k) goals[(b * R + r) * 3 + k] = pg[((size_t)r * 3 + k) * B + b];
            weights[b * R + r] = pw[(size_t)r * B + b];
        }
        time_deadlock_out[b] = qo[b];
        for (int k = 0; k < 4; ++k) st_int[b * 4 + k] = qi[(size_t)k * B + b];
        for (int k = 0; k < 3; ++k) st_goal[b * 3 + k] = ps[(size_t)k * B + b];
        if (flag) flag[b] = qf[b];
    }
    return MRF_OK;
}

template <typename T>
static int obstacles_dev(mrf_handle_t h, int n_per_link, const double* offsets, int vel_mode, const T* q, const T* qd,
                         T* obst, T* sx, T* sv, int64_t B, void* stream) {
    if (!h || !offsets || !q || !qd) return fail(MRF_EINVAL, "mrf_obstacles: null argument");
    if (B <= 0 || n_per_link < 1 || n_per_link > MRF_MAX_SPHERES_PER_LINK)
        return fail(MRF_EINVAL, "mrf_obstacles: n_per_link must be 1..MRF_MAX_SPHERES_PER_LINK");
    if (obst && h->cfg.n_robots < 2) return fail(MRF_EINVAL, "mrf_obstacles: obstacle lists need at least 2 robots");
    MRF_CUDA(cudaSetDevice(h->device));
    SphereOffsets<T> off;
    memset(&off, 0, sizeof(off));
    off.n = n_per_link;
    for (int l = 0; l < MRF_NLINKS; ++l)
        for (int s = 0; s < n_per_link; ++s)
            for (int k = 0; k < 3; ++k) off.t[l][s][k] = (T)offsets[((size_t)l * n_per_link + s) * 3 + k];
    const long long total = (long long)h->cfg.n_robots * B;
    obstacles_kernel<T><<<(unsigned)((total + kActThreads - 1) / kActThreads), kActThreads, 0, (cudaStream_t)stream>>>(
        devcfg<T>(h), off, vel_mode, q, qd, obst, sx, sv, (long long)B);
    MRF_CUDA(cudaGetLastError());
    h->launches += 1;
    return MRF_OK;
}
extern "C" int mrf_obstacles_dev_f64(mrf_handle_t h, int n_per_link, const double* offsets, int vel_mode, const double* q,
                                     const double* qdot, double* obst, double* spheres_x, double* spheres_v, int64_t B,
                                     void* stream) {
    return obstacles_dev<double>(h, n_per_link, offsets, vel_mode, q, qdot, obst, spheres_x, spheres_v, B, stream);
}
extern "C" int mrf_obstacles_dev_f32(mrf_handle_t h, int n_per_link, const double* offsets, int vel_mode, const float* q,
                                     const float* qdot, float* obst, float* spheres_x, float* spheres_v, int64_t B,
                                     void* stream) {
    return obstacles_dev<float>(h, n_per_link, offsets, vel_mode, q, qdot, obst, spheres_x, spheres_v, B, stream);
}

template <typename T>
static int point_action_dev(mrf_handle_t h, const T* rec, int Ss, const T* stat, int Sd, const T* dyn, T* action, int64_t B,
                            void* stream) {
    if (!h || !rec || !action || (Ss > 0 && !stat) || (Sd > 0 && !dyn)) return fail(MRF_EINVAL, "mrf_point_action: null argument");
    if (B <= 0 || Ss < 0 || Sd < 0) return fail(MRF_EINVAL, "mrf_point_action: bad sizes");
    MRF_CUDA(cudaSetDevice(h->device));
    point_action_kernel<T><<<(unsigned)((B + kActThreads - 1) / kActThreads), kActThreads, 0, (cudaStream_t)stream>>>(
        (T)h->cfg.eps, (T)h->cfg.jdot_sign, (T)(2.0 * h->cfg.exec_scale), rec, Ss, stat, Sd, dyn, action, (long long)B);
    MRF_CUDA(cudaGetLastError());
    h->launches += 1;
    return MRF_OK;
}
extern "C" int mrf_point_action_dev_f64(mrf_handle_t h, const double* rec, int Ss, const double* stat, int Sd,
                                        const double* dyn, double* action, int64_t B, void* stream) {
    return point_action_dev<double>(h, rec, Ss, stat, Sd, dyn, action, B, stream);
}
extern "C" int mrf_point_action_dev_f32(mrf_handle_t h, const float* rec, int Ss, const float* stat, int Sd,
                                        const float* dyn, float* action, int64_t B, void* stream) {
    return point_action_dev<float>(h, rec, Ss, stat, Sd, dyn, action, B, stream);
}
// host variant: rec [B][10], stat [B][Ss][4], dyn [B][Sd][7] -> action [B][3]
extern "C" int mrf_point_action_host_f64(mrf_handle_t h, const double* rec, int Ss, const double* stat, int Sd,
                                         const double* dyn, double* action, int64_t B) {
    if (!h || !rec || !action || (Ss > 0 && !stat) || (Sd > 0 && !dyn)) return fail(MRF_EINVAL, "mrf_point_action_host: null argument");
    if (B <= 0) return fail(MRF_EINVAL, "mrf_point_action_host: B must be positive");
    MRF_CUDA(cudaSetDevice(h->device));
    const double *d_rec, *d_stat = nullptr, *d_dyn = nullptr;
    double* d_act;
    int rc = scratch_reset(h);
    if (!rc) rc = stage_in(h, rec, B, 1, 10, &d_rec);
    if (!rc && Ss > 0) rc = stage_in(h, stat, B, 1, Ss * 4, &d_stat);
    if (!rc && Sd > 0) rc = stage_in(h, dyn, B, 1, Sd * 7, &d_dyn);
    if (!rc) rc = scratch_take(h, (size_t)B * 3, &d_act);
    if (rc) return rc;
    MRF_CUDA(cudaEventRecord(h->ev0, h->stream));
    rc = point_action_dev<double>(h, d_rec, Ss, d_stat, Sd, d_dyn, d_act, B, h->stream);
    if (rc) return rc;
    MRF_CUDA(cudaEventRecord(h->ev1, h->stream));
    rc = stage_out(h, d_act, B, 1, 3, action);
    if (rc) return rc;
    return finish_timed(h);
}

template <typename T>
static int point_episode_run_dev(mrf_handle_t h, const MrfPointEpisode* ep, int64_t B, int32_t n_steps, void* stream) {
    if (!h || !ep) return fail(MRF_EINVAL, "mrf_point_episode_run: null argument");
    if (ep->struct_size != (int32_t)sizeof(MrfPointEpisode))
        return fail(MRF_EINVAL, "mrf_point_episode_run: MrfPointEpisode size mismatch");
    const int R = ep->n_robots;
    if (R < 2 || R > MRF_MAX_POINT_ROBOTS) return fail(MRF_EINVAL, "mrf_point_episode_run: n_robots must be 2..MRF_MAX_POINT_ROBOTS");
    if (ep->n_scene < 0 || ep->n_scene > MRF_MAX_STATIC) return fail(MRF_EINVAL, "mrf_point_episode_run: n_scene must be 0..MRF_MAX_STATIC");
    if (ep->dynamic != 0 && ep->dynamic != 1) return fail(MRF_EINVAL, "mrf_point_episode_run: dynamic must be 0 or 1");
    if (!ep->state || !ep->goal || !ep->weight || !ep->radius || (ep->n_scene > 0 && !ep->scene) || !ep->time_step ||
        !ep->done_at || !ep->nonfinite_steps || !ep->min_clear_robots || !ep->min_clear_scene)
        return fail(MRF_EINVAL, "mrf_point_episode_run: null state pointer");
    if (B <= 0) return fail(MRF_EINVAL, "mrf_point_episode_run: B must be positive");
    if (n_steps < 1) return fail(MRF_EINVAL, "mrf_point_episode_run: n_steps must be positive");
    MRF_CUDA(cudaSetDevice(h->device));
    const int W = R <= 2 ? 2 : (R <= 4 ? 4 : 8), spb = kPointThreads / W;
    const unsigned grid = (unsigned)((B + spb - 1) / spb);
    const size_t smem = sizeof(T) * (size_t)spb * ep->n_scene * 4;
    auto kern = ep->dynamic ? point_episode_kernel<T, true> : point_episode_kernel<T, false>;
    kern<<<grid, kPointThreads, smem, (cudaStream_t)stream>>>(
        (T)h->cfg.eps, (T)h->cfg.jdot_sign, (T)(2.0 * h->cfg.exec_scale), (T)h->cfg.dt, (T)ep->epsilon, R, W, ep->n_scene,
        n_steps, (T*)ep->state, (const T*)ep->goal, (const T*)ep->weight, (const T*)ep->radius, (const T*)ep->scene,
        ep->time_step, ep->done_at, ep->nonfinite_steps, (T*)ep->min_clear_robots, (T*)ep->min_clear_scene, (T*)ep->traj,
        (long long)B);
    MRF_CUDA(cudaGetLastError());
    h->launches += 1;
    return MRF_OK;
}
extern "C" int mrf_point_episode_run_dev_f64(mrf_handle_t h, const MrfPointEpisode* ep, int64_t B, int32_t n_steps, void* stream) {
    return point_episode_run_dev<double>(h, ep, B, n_steps, stream);
}
extern "C" int mrf_point_episode_run_dev_f32(mrf_handle_t h, const MrfPointEpisode* ep, int64_t B, int32_t n_steps, void* stream) {
    return point_episode_run_dev<float>(h, ep, B, n_steps, stream);
}

template <typename T>
static int fsm_dev(mrf_handle_t h, const int32_t* nr_blocks, const T* x_ee, const T* q_grip, const T* goal_block,
                   const T* start_goal, T* goal, T* above, T* weight, int32_t* st, T* grip_action, int64_t B, void* stream) {
    if (!h || !nr_blocks || !x_ee || !q_grip || !goal_block || !start_goal || !goal || !above || !weight || !st)
        return fail(MRF_EINVAL, "mrf_fsm: null argument");
    if (B <= 0) return fail(MRF_EINVAL, "mrf_fsm: B must be positive");
    MRF_CUDA(cudaSetDevice(h->device));
    FsmCfg c;
    c.R = h->cfg.n_robots;
    for (int r = 0; r < MRF_MAX_ROBOTS; ++r) c.nr_blocks[r] = r < c.R ? nr_blocks[r] : 0;
    const long long total = (long long)c.R * B;
    fsm_kernel<T><<<(unsigned)((total + 127) / 128), 128, 0, (cudaStream_t)stream>>>(c, x_ee, q_grip, goal_block, start_goal,
                                                                                      goal, above, weight, st, grip_action,
                                                                                      (long long)B);
    MRF_CUDA(cudaGetLastError());
    h->launches += 1;
    return MRF_OK;
}
extern "C" int mrf_fsm_dev_f64(mrf_handle_t h, const int32_t* nr_blocks, const double* x_ee, const double* q_grip,
                               const double* goal_block, const double* start_goal, double* goal, double* above,
                               double* weight, int32_t* st, double* grip_action, int64_t B, void* stream) {
    return fsm_dev<double>(h, nr_blocks, x_ee, q_grip, goal_block, start_goal, goal, above, weight, st, grip_action, B, stream);
}
extern "C" int mrf_fsm_dev_f32(mrf_handle_t h, const int32_t* nr_blocks, const float* x_ee, const float* q_grip,
                               const float* goal_block, const float* start_goal, float* goal, float* above, float* weight,
                               int32_t* st, float* grip_action, int64_t B, void* stream) {
    return fsm_dev<float>(h, nr_blocks, x_ee, q_grip, goal_block, start_goal, goal, above, weight, st, grip_action, B, stream);
}

// ------------------------------------------------------------------------------------------------
// closed-loop control step (examples/example_pandas_Jointspace.py:280-458) for B independent scenarios: the
// bookkeeping between the rollout / deadlock / obstacle / action kernels as three small kernels, so one control step is
// seven launches on one stream (CUDA-graph friendly) instead of ~45 framework launches
// ------------------------------------------------------------------------------------------------
struct EpLimits {
    double v[MRF_DOF];
};
// :288 velocity clip of the measured state; goals / weights of this step start from the task's own (:352-368).
// goal0 == nullptr: the clip only.  kin != nullptr (decoupled Cartesian rollouts): kin_scratch [3][8][3][R][B] of the
// clipped state; robot est_robot's goal is the RF-CV estimate x_hand + est_h * J qdot when `estimate` is set
// (example_pandas_cartesian.py:355-357), and goal_est [3][B] receives the goal that robot's rollout uses.
template <typename T>
__global__ void episode_pre_kernel(T* __restrict__ rec, const T* __restrict__ goal0, const T* __restrict__ w0, EpLimits lim,
                                   T w1, int R, long long B, const T* __restrict__ kin = nullptr, int est_robot = -1,
                                   int estimate = 0, T est_h = T(0), T* __restrict__ goal_est = nullptr) {
    const long long RB = (long long)R * B, idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= RB) return;
    const int r = (int)(idx / B);
    const long long b = idx - (long long)r * B;
#pragma unroll
    for (int i = 0; i < MRF_DOF; ++i) {
        T* p = rec + (MRF_QD + i) * RB + idx;
        const T l = (T)lim.v[i], v = *p;
        *p = v < -l ? -l : (v > l ? l : v); // NaN stays NaN, like np.clip
    }
    if (goal0 == nullptr) return;
    const bool est_here = kin != nullptr && r == est_robot;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        T g = goal0[((long long)r * 3 + c) * B + b];
        if (est_here) {
            if (estimate) {
                const T* hand = kin + (long long)(MRF_NLINKS - 1) * 3 * RB; // x of link 8; its v rows follow 8 * 3 rows on
                g = hand[c * RB + idx] + hand[(long long)MRF_NLINKS * 3 * RB + c * RB + idx] * est_h;
            }
            if (goal_est != nullptr) goal_est[(long long)c * B + b] = g;
        }
        rec[(MRF_G0 + c) * RB + idx] = g;
    }
    rec[MRF_W0 * RB + idx] = w0[idx];
    rec[MRF_W1 * RB + idx] = w1;
}
// between the rollouts and the executed action: RF-CV goal (when the deadlock kernel has not already applied it, :346-348)
// and weight_goal_1 of the executed planner (:427)
template <typename T>
__global__ void episode_mid_kernel(T* __restrict__ rec, const T* __restrict__ goal_est, int est_robot, T w1, int R, long long B) {
    const long long RB = (long long)R * B, idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= RB) return;
    const int r = (int)(idx / B);
    const long long b = idx - (long long)r * B;
    rec[MRF_W1 * RB + idx] = w1;
    if (goal_est != nullptr && r == est_robot) {
#pragma unroll
        for (int c = 0; c < 3; ++c) rec[(MRF_G0 + c) * RB + idx] = goal_est[(long long)c * B + b];
    }
}
// hand position at the measured state (for the state machine and, with decoupled Cartesian rollouts, the deadlock
// heuristic) and, in the pick-and-place task (:289-303, blocks != nullptr), the block each robot goes for next -- block
// number nr_blocks_success of its own stack, grasp height 0.1 above the block (:302-303)
template <typename T>
__global__ void episode_blocks_kernel(const T* __restrict__ hand, T* __restrict__ x_ee, const T* __restrict__ blocks, int n_blocks,
                                      const int32_t* __restrict__ st, T* __restrict__ goal_block, int R, long long B) {
    const long long RB = (long long)R * B, idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= RB) return;
    const int r = (int)(idx / B);
    const long long b = idx - (long long)r * B;
    const int n_ok = blocks != nullptr ? st[1 * RB + idx] : n_blocks;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        x_ee[((long long)r * 3 + c) * B + b] = hand[((long long)c * R + r) * B + b];
        if (n_ok < n_blocks)
            goal_block[((long long)r * 3 + c) * B + b] = blocks[(((long long)n_ok * R + r) * 3 + c) * B + b] + (c == 2 ? T(0.1) : T(0));
    }
}
// :453-470 clip the action, kinematic environment step (urdfenvs 'vel' mode stand-in), reach / clearance / deadlock metrics
template <typename T>
__global__ void episode_post_kernel(T* __restrict__ rec, const T* __restrict__ act, const T* __restrict__ x_ee, int xee_link_major,
                                    const T* __restrict__ goal0, const T* __restrict__ sx, int S, const int32_t* __restrict__ flag,
                                    EpLimits lim, T dt, T eps, T rsum, int32_t* __restrict__ tstep, int32_t* __restrict__ done_at,
                                    int32_t* __restrict__ deadlock_steps, T* __restrict__ min_clear, int R, long long B,
                                    const int32_t* __restrict__ sm, T* __restrict__ q_grip, const T* __restrict__ grip_action,
                                    int32_t* __restrict__ nonfinite_steps) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const long long RB = (long long)R * B;
    bool reached = true, bad = false;
    for (int r = 0; r < R; ++r) {
        const long long idx = (long long)r * B + b;
        const int state = sm != nullptr ? sm[idx] : 0;
#pragma unroll
        for (int i = 0; i < MRF_DOF; ++i) {
            const T l = (T)lim.v[i];
            T a = act[(long long)i * RB + idx];
            a = a < -l ? -l : (a > l ? l : a);
            if (!(a - a == T(0))) { a = T(0); bad = true; } // non-finite action: hold still, and count the step
            if (state == 3 || state == 5) a = T(0); // gripping / releasing: the arm holds still (:418-419)
            rec[(MRF_QD + i) * RB + idx] = a;
            rec[(MRF_Q + i) * RB + idx] += a * dt;
        }
        if (q_grip != nullptr) { // finger joints follow the state machine's gripper velocity inside their limits [0, 0.04]
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                T* g = q_grip + ((long long)r * 2 + k) * B + b;
                T v = *g + dt * grip_action[((long long)r * 2 + k) * B + b];
                *g = v < T(0) ? T(0) : (v > T(0.04) ? T(0.04) : v);
            }
        }
        if (sm != nullptr) { // pick-and-place: done when every state machine reports "all blocks picked" (:305-312)
            reached = reached && state == 10;
            continue;
        }
        T d2 = T(0);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const T x = xee_link_major ? x_ee[((long long)c * R + r) * B + b] : x_ee[((long long)r * 3 + c) * B + b];
            const T d = x - goal0[((long long)r * 3 + c) * B + b];
            d2 += d * d;
        }
        reached = reached && (Mth<T>::sqrt(d2) < eps);
    }
    const int32_t t = tstep[b];
    if (reached && done_at[b] < 0) done_at[b] = t;
    if (sx != nullptr) {
        T mc = min_clear[b];
        for (int ra = 0; ra < R; ++ra)
            for (int rb = ra + 1; rb < R; ++rb)
                for (int i = 0; i < S; ++i) {
                    const T ax = sx[((long long)(i * 3 + 0) * R + ra) * B + b], ay = sx[((long long)(i * 3 + 1) * R + ra) * B + b],
                            az = sx[((long long)(i * 3 + 2) * R + ra) * B + b];
                    for (int j = 0; j < S; ++j) {
                        const T dx = ax - sx[((long long)(j * 3 + 0) * R + rb) * B + b], dy = ay - sx[((long long)(j * 3 + 1) * R + rb) * B + b],
                                dz = az - sx[((long long)(j * 3 + 2) * R + rb) * B + b];
                        const T c = Mth<T>::sqrt(dx * dx + dy * dy + dz * dz) - rsum;
                        mc = c < mc ? c : mc;
                    }
                }
        min_clear[b] = mc;
    }
    if (flag != nullptr && deadlock_steps != nullptr) deadlock_steps[b] += flag[b];
    if (nonfinite_steps != nullptr && bad) nonfinite_steps[b] += 1;
    tstep[b] = t + 1;
}

template <typename T> static int episode_step_dev(mrf_handle_t h, const MrfEpisode* ep, int64_t B, void* stream) {
    if (!h || !ep) return fail(MRF_EINVAL, "mrf_episode_step: null argument");
    if (ep->struct_size != (int32_t)sizeof(MrfEpisode)) return fail(MRF_EINVAL, "mrf_episode_step: MrfEpisode size mismatch");
    if (!ep->rec || !ep->goal0 || !ep->w0 || !ep->x_ee || (h->cfg.n_robots > 1 && !ep->obst) || !ep->spheres_x || !ep->action ||
        !ep->offsets || !ep->time_step || !ep->done_at || !ep->min_clearance)
        return fail(MRF_EINVAL, "mrf_episode_step: null state pointer");
    if (ep->n_per_link < 1 || ep->n_per_link > MRF_MAX_SPHERES_PER_LINK) return fail(MRF_EINVAL, "mrf_episode_step: bad n_per_link");
    if (ep->rollout_fabrics && (!ep->avg_vel || !ep->goal_est || ep->n_horizon <= 0))
        return fail(MRF_EINVAL, "mrf_episode_step: rollouts need avg_vel, goal_est and n_horizon > 0");
    if (ep->rollout_fabrics && ep->resolve_deadlocks &&
        ((!ep->sm_state && !ep->pick_and_place) || !ep->time_deadlock_out || !ep->st_int || !ep->st_goal || !ep->flag ||
         !ep->deadlock_steps))
        return fail(MRF_EINVAL, "mrf_episode_step: deadlock resolution needs its state arrays");
    if (!ep->rollout_fabrics && !ep->kin_scratch) return fail(MRF_EINVAL, "mrf_episode_step: MRDF mode needs kin_scratch");
    if (ep->rollout_fabrics && ep->rollout_model != 0 && ep->rollout_model != 1)
        return fail(MRF_EINVAL, "mrf_episode_step: rollout_model must be 0 (coupled joint-space) or 1 (decoupled Cartesian)");
    const bool cart = ep->rollout_fabrics && ep->rollout_model == 1;
    if (cart && !ep->kin_scratch) return fail(MRF_EINVAL, "mrf_episode_step: Cartesian rollouts need kin_scratch");
    if (B <= 0) return fail(MRF_EINVAL, "mrf_episode_step: B must be positive");
    MRF_CUDA(cudaSetDevice(h->device));
    const int R = h->cfg.n_robots;
    const long long RB = (long long)R * B;
    cudaStream_t st = (cudaStream_t)stream;
    T* rec = (T*)ep->rec;
    EpLimits lim;
    for (int i = 0; i < MRF_DOF; ++i) lim.v[i] = ep->vel_limit[i];
    const unsigned g_rb = (unsigned)((RB + 255) / 256), g_b = (unsigned)((B + 127) / 128);
    const bool est = h->cfg.estimate_goal != 0 && R > 1;
    const bool pnp = ep->pick_and_place != 0;
    const int32_t* sm_state = ep->sm_state;
    if (cart) { // the velocity clip first: the kinematics below (hand, J qdot of the estimate) read the clipped state
        episode_pre_kernel<T><<<g_rb, 256, 0, st>>>(rec, nullptr, nullptr, lim, T(0), R, (long long)B);
        MRF_CUDA(cudaGetLastError());
        h->launches += 1;
    }
    if (pnp) {
        if (!ep->kin_scratch || !ep->blocks || !ep->q_grip || !ep->start_goal || !ep->goal_block || !ep->fsm_above || !ep->fsm_st ||
            !ep->grip_action || ep->n_blocks < 1)
            return fail(MRF_EINVAL, "mrf_episode_step: pick-and-place needs its state arrays");
        T* kx = (T*)ep->kin_scratch;
        const size_t n = (size_t)MRF_NLINKS * 3 * RB;
        int rc0 = kinematics_dev<T>(h, rec + MRF_Q * RB, rec + MRF_QD * RB, kx, kx + n, kx + 2 * n, B, stream);
        if (rc0) return rc0;
        episode_blocks_kernel<T><<<g_rb, 256, 0, st>>>(kx + (size_t)(MRF_NLINKS - 1) * 3 * RB, (T*)ep->x_ee, (const T*)ep->blocks,
                                                       ep->n_blocks, ep->fsm_st, (T*)ep->goal_block, R, (long long)B);
        MRF_CUDA(cudaGetLastError());
        h->launches += 1;
        int nb[MRF_MAX_ROBOTS];
        for (int r = 0; r < MRF_MAX_ROBOTS; ++r) nb[r] = ep->n_blocks;
        // the state machine rewrites this step's task goal and weight_goal_0 (goal0 / w0) and the gripper command
        rc0 = fsm_dev<T>(h, nb, (const T*)ep->x_ee, (const T*)ep->q_grip, (const T*)ep->goal_block, (const T*)ep->start_goal,
                         (T*)ep->goal0, (T*)ep->fsm_above, (T*)ep->w0, ep->fsm_st, (T*)ep->grip_action, B, stream);
        if (rc0) return rc0;
        sm_state = ep->fsm_st; // row 0 of [6][R][B] = state codes
    } else if (cart) {
        T* kx = (T*)ep->kin_scratch;
        const size_t n = (size_t)MRF_NLINKS * 3 * RB;
        int rc0 = kinematics_dev<T>(h, rec + MRF_Q * RB, rec + MRF_QD * RB, kx, kx + n, kx + 2 * n, B, stream);
        if (rc0) return rc0;
        episode_blocks_kernel<T><<<g_rb, 256, 0, st>>>(kx + (size_t)(MRF_NLINKS - 1) * 3 * RB, (T*)ep->x_ee, nullptr, 0,
                                                       nullptr, nullptr, R, (long long)B);
        MRF_CUDA(cudaGetLastError());
        h->launches += 1;
    }
    const int est_robot = (h->cfg.estimate_robot >= 0 && h->cfg.estimate_robot < R) ? h->cfg.estimate_robot : -1;
    episode_pre_kernel<T><<<g_rb, 256, 0, st>>>(rec, (const T*)ep->goal0, (const T*)ep->w0, lim,
                                                (T)(ep->rollout_fabrics ? ep->w1_rollout : ep->w1_action), R, (long long)B,
                                                cart ? (const T*)ep->kin_scratch : nullptr, est_robot, est ? 1 : 0,
                                                (T)h->cfg.estimate_horizon, cart ? (T*)ep->goal_est : nullptr);
    MRF_CUDA(cudaGetLastError());
    h->launches += 1;
    int rc;
    const T* xee = (const T*)ep->x_ee;
    int link_major = 0;
    const int S1 = MRF_NLINKS * ep->n_per_link;
    if (ep->rollout_fabrics) {
        if (cart) {
            // example_pandas_cartesian.py:343-352: each robot's rollout sees the other robots' spheres with their true
            // velocities J_sphere qdot (compute_x_obsts_dyn_0, utils_apply_fk.py:3-33), moving at constant velocity over the
            // horizon.  The executed action below keeps the joint-space loop's staging (link-origin velocities): the
            // Cartesian example's action-side assembly is taken to be the same as the joint-space example's.
            rc = obstacles_dev<T>(h, ep->n_per_link, ep->offsets, 1, rec + MRF_Q * RB, rec + MRF_QD * RB, (T*)ep->obst, nullptr,
                                  nullptr, B, stream);
            if (rc) return rc;
            rc = action_dev<T, true>(h, 0, R, rec, S1 * (R - 1), (const T*)ep->obst, ep->n_horizon, (T*)ep->avg_vel, nullptr,
                                     nullptr, B, stream);
        } else {
            rc = rollout_dev<T>(h, rec, ep->n_horizon, (T*)ep->avg_vel, (T*)ep->x_ee, (T*)ep->goal_est, nullptr, nullptr, B,
                                stream);
        }
        if (rc) return rc;
        // Cartesian: the estimate already sits in the record's goal rows (episode_pre_kernel)
        const T* gest = (est && !cart) ? (const T*)ep->goal_est : nullptr;
        if (ep->resolve_deadlocks && R >= 2) { // the heuristic is defined on robot pairs
            rc = deadlock_rec_dev<T>(h, (const T*)ep->x_ee, rec, gest, (const T*)ep->avg_vel, nullptr, sm_state, ep->time_step,
                                     ep->time_deadlock_out, ep->st_int, (T*)ep->st_goal, ep->flag, B, stream);
            if (rc) return rc;
        }
        episode_mid_kernel<T><<<g_rb, 256, 0, st>>>(rec, !ep->resolve_deadlocks ? gest : nullptr, h->cfg.estimate_robot,
                                                    (T)ep->w1_action, R, (long long)B);
        MRF_CUDA(cudaGetLastError());
        h->launches += 1;
    } else if (!pnp) {
        T* kx = (T*)ep->kin_scratch;
        const size_t n = (size_t)MRF_NLINKS * 3 * RB;
        rc = kinematics_dev<T>(h, rec + MRF_Q * RB, rec + MRF_QD * RB, kx, kx + n, kx + 2 * n, B, stream);
        if (rc) return rc;
        xee = kx + (size_t)(MRF_NLINKS - 1) * 3 * RB; // hand rows [3][R][B]
        link_major = 1;
    }
    rc = obstacles_dev<T>(h, ep->n_per_link, ep->offsets, 0, rec + MRF_Q * RB, rec + MRF_QD * RB, (T*)ep->obst, (T*)ep->spheres_x,
                          nullptr, B, stream);
    if (rc) return rc;
    rc = action_dev<T, false>(h, 0, R, rec, S1 * (R - 1), (const T*)ep->obst, 0, (T*)ep->action, nullptr, nullptr, B, stream,
                              pnp ? sm_state : nullptr);
    if (rc) return rc;
    episode_post_kernel<T><<<g_b, 128, 0, st>>>(
        rec, (const T*)ep->action, xee, link_major, (const T*)ep->goal0, R > 1 ? (const T*)ep->spheres_x : nullptr, S1,
        (ep->rollout_fabrics && ep->resolve_deadlocks && R >= 2) ? ep->flag : nullptr, lim, (T)h->cfg.dt, (T)ep->epsilon,
        (T)ep->clearance_radius_sum, ep->time_step, ep->done_at, ep->deadlock_steps, (T*)ep->min_clearance, R, (long long)B,
        pnp ? sm_state : nullptr, pnp ? (T*)ep->q_grip : nullptr, pnp ? (const T*)ep->grip_action : nullptr,
        ep->nonfinite_steps);
    MRF_CUDA(cudaGetLastError());
    h->launches += 1;
    return MRF_OK;
}
extern "C" int mrf_episode_step_dev_f64(mrf_handle_t h, const MrfEpisode* ep, int64_t B, void* stream) {
    return episode_step_dev<double>(h, ep, B, stream);
}
extern "C" int mrf_episode_step_dev_f32(mrf_handle_t h, const MrfEpisode* ep, int64_t B, void* stream) {
    return episode_step_dev<float>(h, ep, B, stream);
}

template <typename T> static int fma_peak(mrf_handle_t h, double* tflops) {
    MRF_CUDA(cudaSetDevice(h->device));
    cudaDeviceProp prop;
    MRF_CUDA(cudaGetDeviceProperties(&prop, h->device));
    const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 1 << 15;
    T* out;
    int rc = scratch_reset(h);
    if (!rc) rc = scratch_take(h, (size_t)blocks * threads, &out);
    if (rc) return rc;
    double best = 0.0;
    for (int rep = 0; rep < 6; ++rep) {
        MRF_CUDA(cudaEventRecord(h->ev0, h->stream));
        fma_peak_kernel<T><<<blocks, threads, 0, h->stream>>>(out, iters, T(0.999), T(1e-3));
        MRF_CUDA(cudaGetLastError());
        MRF_CUDA(cudaEventRecord(h->ev1, h->stream));
        MRF_CUDA(cudaStreamSynchronize(h->stream));
        float ms = 0.f;
        MRF_CUDA(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
        double tf = 2.0 * 8.0 * (double)iters * blocks * threads / (ms * 1e-3) / 1e12;
        if (rep > 0 && tf > best) best = tf;
    }
    if (sizeof(T) == 4) { // the FP32 pipe peak is reached with packed FFMA2 (scalar FFMA is issue-limited to ~93 %)
        for (int rep = 0; rep < 6; ++rep) {
            MRF_CUDA(cudaEventRecord(h->ev0, h->stream));
            fma2_peak_kernel<<<blocks, threads, 0, h->stream>>>((float*)out, iters, 0.999f, 1e-3f);
            MRF_CUDA(cudaGetLastError());
            MRF_CUDA(cudaEventRecord(h->ev1, h->stream));
            MRF_CUDA(cudaStreamSynchronize(h->stream));
            float ms = 0.f;
            MRF_CUDA(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
            double tf = 2.0 * 8.0 * (double)iters * blocks * threads / (ms * 1e-3) / 1e12;
            if (rep > 0 && tf > best) best = tf;
        }
    }
    *tflops = best;
    return MRF_OK;
}
extern "C" int mrf_fma_peak(mrf_handle_t h, int is_f64, double* tflops) {
    if (!h || !tflops) return fail(MRF_EINVAL, "mrf_fma_peak: null argument");
    return is_f64 ? fma_peak<double>(h, tflops) : fma_peak<float>(h, tflops);
}
