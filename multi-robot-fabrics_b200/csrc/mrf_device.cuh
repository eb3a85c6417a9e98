// mrf_device.cuh -- per-thread device code of the multi-robot fabric hot path (sm_100a).
//
// One thread owns one (scenario, robot).  Its joint state, joint axes and the 7x7 metric stay in registers
// for the whole horizon; its five distinct moving link points (x, v, Jdot*qdot) and its parameter block
// live in shared memory, where the other robots of the same scenario (same lane, other warps of the CTA)
// read them every rollout step.  No tensor cores: the work is tiny per-robot solves and scalar leaf algebra.
//
// What is computed (reference call sites; arithmetic restated from fabrics 0.9.5, see DESIGN.md):
//   chain_forward   fk / jac / jac_dot functions   multi_robot_fabrics/utils/utils.py:16-54
//   fabric_action   planner._funs._function        examples/example_pandas_Jointspace.py:64-134,417-445
//   (the rollout loop around them is in mrf_kernels.cu)
//
// The functions are MRF_HD so that tests/emul can run the same source on the host as a debugging aid;
// the shipped library only ever calls them from __global__ kernels.
#pragma once

#include <stdint.h>

#if defined(__CUDACC__)
#define MRF_HD __host__ __device__ __forceinline__
#else
#define MRF_HD inline
#include <cmath>
#endif

#include "../../include/mrf_b200.h"

namespace mrf {

template <int N> struct Int {
    static constexpr int value = N;
};

constexpr int kDof = 7;
constexpr int kEgo = 5;        // distinct moving link points: link3, link4, link5(==link6), link7, link8
constexpr int kPts = kEgo + 1; // + the constant point link1 == link2 (slot 5), so readers need no special case
// x, v, c per point; then, for FP64 only, the six joint axes of the thread's own robot.  They are needed only at the
// pullbacks; keeping them out of the register file across the leaf loops removes the FP64 kernel's spills (36
// registers; measured +2.7 %), while for FP32 (18 registers, no spills) the extra shared-memory reads cost 1.3 %.
constexpr int kZ = kPts * 9;
#ifdef MRF_AXES_SMEM_F32
template <typename T> constexpr bool kAxesInSmem = true;
#else
template <typename T> constexpr bool kAxesInSmem = sizeof(T) == 8;
#endif
template <typename T> constexpr int kKinRows = kPts * 9 + (kAxesInSmem<T> ? 18 : 0);
constexpr int kMaxEnt = 8 * (MRF_MAX_ROBOTS - 1); // sphere entries one robot sees (all links of all other robots)
// parameter block (per thread, shared memory)
enum { P_G0 = 0, P_W0 = 3, P_G1 = 4, P_W1 = 7, P_G2 = 8, P_W2 = 9, P_ANG = 10, P_NH = 19, P_DN = 22, P_RB = 23, P_RISK = 29, P_N = 30 };

// ------------------------------------------------------------------------------------------------
// math
// ------------------------------------------------------------------------------------------------
template <typename T> struct Mth;
template <> struct Mth<float> {
    static MRF_HD float sqrt(float x) { return ::sqrtf(x); }
    // FP32 throughput path: single MUFU.RSQ / MUFU.RCP (2^-22 relative error, below the FP32 rounding that the
    // stated FP32 tolerance already covers); an IEEE 1.0f/x costs ~8 extra instructions and was 20 % of all stalls
    static MRF_HD float rsqrt(float x) {
#if defined(__CUDA_ARCH__)
        float r;
        asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
        return r;
#else
        return 1.0f / ::sqrtf(x);
#endif
    }
    static MRF_HD float rcp(float x) {
#if defined(__CUDA_ARCH__)
        float r;
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
        return r;
#else
        return 1.0f / x;
#endif
    }
    // exp / tanh through MUFU.EX2 (2 ulp): ~1e-7 relative on exp; tanh = (t-1)/(t+1), t = 2^(2x log2 e), absolute
    // error < 3e-7 (argument clamped so t stays finite).  Used 7 times per action; ::expf / ::tanhf cost ~30 each.
    static MRF_HD float exp(float x) {
#if defined(__CUDA_ARCH__)
        float r;
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x * 1.4426950408889634f));
        return r;
#else
        return ::expf(x);
#endif
    }
    static MRF_HD float tanh(float x) {
#if defined(__CUDA_ARCH__)
        float xc = ::fminf(::fmaxf(x, -15.0f), 15.0f), t;
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(xc * 2.8853900817779268f));
        return (t - 1.0f) * rcp(t + 1.0f);
#else
        return ::tanhf(x);
#endif
    }
    // Joint angles are bounded by the Panda limits (|q| < 3.8 rad): Cody-Waite reduction by pi/2 and degree-7/8
    // minimax polynomials on [-pi/4, pi/4] (~1e-7 abs error) in ~22 instructions, without the argument-reduction slow
    // path that ::sincosf drags into every call site (it was 2 % of instructions and much more of the code size).
    static MRF_HD void sincos(float x, float* s, float* c) {
        float k = ::rintf(x * 0.636619772f);
        float r = ::fmaf(k, -1.57079601e+00f, x);
        r = ::fmaf(k, -3.13916473e-07f, r);
        r = ::fmaf(k, -5.39030253e-15f, r);
        float r2 = r * r;
        float sp = ::fmaf(::fmaf(::fmaf(-1.9515295891e-4f, r2, 8.3321608736e-3f), r2, -1.6666654611e-1f), r2 * r, r);
        float cp = ::fmaf(::fmaf(::fmaf(2.443315711809948e-5f, r2, -1.388731625493765e-3f), r2, 4.166664568298827e-2f),
                          r2 * r2, ::fmaf(-0.5f, r2, 1.0f));
        int q = (int)k;
        float ss = (q & 1) ? cp : sp, cc = (q & 1) ? sp : cp;
        *s = (q & 2) ? -ss : ss;
        *c = ((q + 1) & 2) ? -cc : cc;
    }
    static MRF_HD float fma(float a, float b, float c) { return ::fmaf(a, b, c); } // explicit: never re-associated
    static MRF_HD float abs(float x) { return ::fabsf(x); }
    static MRF_HD float max(float a, float b) { return ::fmaxf(a, b); }
};
template <> struct Mth<double> {
    static MRF_HD double sqrt(double x) { return ::sqrt(x); }
    // FP64 reciprocal / reciprocal square root: the library sequences (::rsqrt, IEEE division) carry special-case handling
    // the leaf arguments never need (finite, far from the denormal range); the native 20-bit seeds MUFU.RCP64H /
    // MUFU.RSQ64H plus two Newton steps give ~1 ulp in 5 / 8 FP64 instructions.  Measured on B200: FP64 rollout 4.07 -> 3.23 ms
    // (-DMRF_IEEE_F64_RECIP restores the library sequences).  0, inf and NaN arguments end in NaN, as the degenerate cases of
    // the reference do (0/0 at an exactly reached goal).
    static MRF_HD double rsqrt(double x) {
#if defined(__CUDA_ARCH__) && !defined(MRF_IEEE_F64_RECIP)
        double y;
        asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
        const double h = 0.5 * x;
        double t = ::fma(-(h * y), y, 0.5);
        y = ::fma(y, t, y);
        t = ::fma(-(h * y), y, 0.5);
        return ::fma(y, t, y);
#elif defined(__CUDA_ARCH__)
        return ::rsqrt(x);
#else
        return 1.0 / ::sqrt(x);
#endif
    }
    static MRF_HD double rcp(double x) {
#if defined(__CUDA_ARCH__) && !defined(MRF_IEEE_F64_RECIP)
        double r;
        asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
        double e = ::fma(-x, r, 1.0);
        r = ::fma(r, e, r);
        e = ::fma(-x, r, 1.0);
        return ::fma(r, e, r);
#else
        return 1.0 / x;
#endif
    }
    // FP64 exp / tanh / sincos on the device: the same story as the reciprocals -- the library versions spend a third of
    // their instructions on argument ranges this path never sees (|q| of a few radians, |x| of tens).  Cody-Waite reduction
    // with the 1.5 x 2^52 rounding constant, the fdlibm kernel polynomials for sin / cos on [-pi/4, pi/4] and a degree-13
    // Taylor polynomial for exp on [-ln2/2, ln2/2]: |error| <= 2.3e-16 absolute for sin / cos / tanh and relative for exp
    // (checked against numpy over 2e6 arguments each).  -DMRF_IEEE_F64_MATH restores the library calls.
#if defined(__CUDA_ARCH__) && !defined(MRF_IEEE_F64_MATH)
    static __device__ __forceinline__ double exp(double x0) {
        const double x = x0 < -700.0 ? -700.0 : (x0 > 700.0 ? 700.0 : x0); // NaN passes through the comparisons
        const double t = ::fma(x, 1.4426950408889634, 6755399441055744.0);
        const double k = t - 6755399441055744.0;
        double r = ::fma(-k, 6.93147180369123816490e-01, x);
        r = ::fma(-k, 1.90821492927058770002e-10, r);
        double p = 1.6059043836821613e-10;                     // 1/13!
        p = ::fma(p, r, 2.08767569878681e-09);                 // 1/12!
        p = ::fma(p, r, 2.505210838544172e-08);
        p = ::fma(p, r, 2.755731922398589e-07);
        p = ::fma(p, r, 2.7557319223985893e-06);
        p = ::fma(p, r, 2.48015873015873e-05);
        p = ::fma(p, r, 1.984126984126984e-04);
        p = ::fma(p, r, 1.388888888888889e-03);
        p = ::fma(p, r, 8.333333333333333e-03);
        p = ::fma(p, r, 4.1666666666666664e-02);
        p = ::fma(p, r, 1.6666666666666666e-01);
        p = ::fma(p, r, 0.5);
        const double er = ::fma(r * r, p, r) + 1.0;
        const double e2k = __hiloint2double(__double2hiint(er) + (__double2loint(t) << 20), __double2loint(er)); // er * 2^k
        return x0 != x0 ? x0 : e2k;
    }
    static __device__ __forceinline__ double tanh(double x) {
        const double t = exp(-2.0 * ::fabs(x));
        const double r = (1.0 - t) * rcp(1.0 + t);
        return ::copysign(r, x);
    }
    static __device__ __forceinline__ void sincos(double x0, double* s, double* c) {
        // joint angles are a few radians; a rollout that has blown up stays finite and bounded (the quadrant counter is the
        // low word of t: valid below 2^31 quarter turns), NaN passes through the comparisons
        const double x = x0 > 1.0e9 ? 1.0e9 : (x0 < -1.0e9 ? -1.0e9 : x0);
        const double t = ::fma(x, 0.6366197723675814, 6755399441055744.0);
        const double k = t - 6755399441055744.0;
        const int q = __double2loint(t);
        double r = ::fma(-k, 1.5707963267948966, x);
        r = ::fma(-k, 6.123233995736766e-17, r);
        const double z = r * r;
        double ps = 1.58969099521155010221e-10;
        ps = ::fma(ps, z, -2.50507602534068634195e-08);
        ps = ::fma(ps, z, 2.75573137070700676789e-06);
        ps = ::fma(ps, z, -1.98412698298579493134e-04);
        ps = ::fma(ps, z, 8.33333333332248946124e-03);
        ps = ::fma(ps, z, -1.66666666666666324348e-01);
        const double sr = ::fma(r * z, ps, r);
        double pc = -1.13596475577881948265e-11;
        pc = ::fma(pc, z, 2.08757232129817482790e-09);
        pc = ::fma(pc, z, -2.75573143513906633035e-07);
        pc = ::fma(pc, z, 2.48015872894767294178e-05);
        pc = ::fma(pc, z, -1.38888888888741095749e-03);
        pc = ::fma(pc, z, 4.16666666666666019037e-02);
        const double cr = ::fma(z * z, pc, ::fma(-0.5, z, 1.0));
        const double ss = (q & 1) ? cr : sr, cc = (q & 1) ? sr : cr;
        *s = (q & 2) ? -ss : ss;
        *c = ((q + 1) & 2) ? -cc : cc;
    }
#else
    static MRF_HD double exp(double x) { return ::exp(x); }
    static MRF_HD double tanh(double x) { return ::tanh(x); }
    static MRF_HD void sincos(double x, double* s, double* c) {
#if defined(__CUDA_ARCH__)
        ::sincos(x, s, c);
#else
        *s = ::sin(x);
        *c = ::cos(x);
#endif
    }
#endif
    static MRF_HD double fma(double a, double b, double c) { return ::fma(a, b, c); }
    static MRF_HD double abs(double x) { return ::fabs(x); }
    static MRF_HD double max(double a, double b) { return ::fmax(a, b); }
};

template <typename T> struct V3 {
    T x, y, z;
};
template <typename T> MRF_HD V3<T> mk(T x, T y, T z) { return V3<T>{x, y, z}; }
template <typename T> MRF_HD V3<T> operator+(V3<T> a, V3<T> b) { return V3<T>{a.x + b.x, a.y + b.y, a.z + b.z}; }
template <typename T> MRF_HD V3<T> operator-(V3<T> a, V3<T> b) { return V3<T>{a.x - b.x, a.y - b.y, a.z - b.z}; }
template <typename T> MRF_HD V3<T> operator*(V3<T> a, T s) { return V3<T>{a.x * s, a.y * s, a.z * s}; }
template <typename T> MRF_HD T dot(V3<T> a, V3<T> b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
template <typename T> MRF_HD V3<T> cross(V3<T> a, V3<T> b) {
    return V3<T>{a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x};
}

// c + a x b as two chained multiply-adds per component (cross() followed by an addition costs three)
template <typename T> MRF_HD V3<T> cross_add(V3<T> a, V3<T> b, V3<T> c) {
    return V3<T>{(c.x + a.y * b.z) - a.z * b.y, (c.y + a.z * b.x) - a.x * b.z, (c.z + a.x * b.y) - a.y * b.x};
}
// c + a.b and c - a.b as three chained multiply-adds (a separate dot() costs a fourth instruction for the final add)
template <typename T> MRF_HD T dot_add(V3<T> a, V3<T> b, T c) { return ((c + a.z * b.z) + a.y * b.y) + a.x * b.x; }
template <typename T> MRF_HD T dot_sub(V3<T> a, V3<T> b, T c) { return ((c - a.z * b.z) - a.y * b.y) - a.x * b.x; }

// ------------------------------------------------------------------------------------------------
// configuration as the kernels see it (passed by value as a __grid_constant__ kernel parameter)
// ------------------------------------------------------------------------------------------------
template <typename T> struct DevCfg {
    int n_robots, mode, static_or_dyn, has_coll, estimate_goal, estimate_robot;
    T est_h, dt, eps, sigma, sref, s2;
    T R0[MRF_MAX_ROBOTS][9];   // mount rotation, row-major
    T p0[MRF_MAX_ROBOTS][3];   // mount translation
    T link1[MRF_MAX_ROBOTS][3]; // constant origin of panda_link1 == panda_link2
    T lim[kDof][2];
    T r_link[MRF_MAX_ROBOTS][MRF_NLINKS]; // sphere radius of each link as seen by the other robots
    // spheres robot r sees in a coupled rollout, flattened over the other robots (ascending) and their distinct
    // points with multiplicity: link1==link2 and link5==link6 share a point and are merged into one entry of weight
    // 2 when their radii agree.  ent_off = kinematics-table offset (point * 9 * NT + other_robot * 32).
    // per distinct point of robot j (slot order link3, link4, link5==6, link7, link8, link1==2): the radii of the one or
    // two links sharing it; pt_n = 1 with weight 2 when both radii agree (used by the cooperative low-latency kernel)
    int pt_n[MRF_MAX_ROBOTS][kPts];
    T pt_w[MRF_MAX_ROBOTS][kPts];
    T pt_rad[MRF_MAX_ROBOTS][kPts][2];
    int ego_mask[MRF_MAX_ROBOTS]; // bit k: panda_link(3+k) of robot r carries collision leaves (collision_links_nr)
    int uniform_obst;           // every r_robots[j][l] equal and every link of every robot in its collision set ->
                                // SmemSrcUniform fast path with radius r_obst
    T r_obst;
    int ent_n[MRF_MAX_ROBOTS];
    int ent_rob[MRF_MAX_ROBOTS][kMaxEnt];
    int ent_src[MRF_MAX_ROBOTS][kMaxEnt];
    T ent_rad[MRF_MAX_ROBOTS][kMaxEnt];
    T ent_w[MRF_MAX_ROBOTS][kMaxEnt];
};

// Self-collision pairs of each robot (mrf_set_self_collision), resolved to point-table slots: pt = slot of each link's
// point (link1/2 -> 5, 3 -> 0, 4 -> 1, 5/6 -> 2, 7 -> 3, 8/hand -> 4), K = Jacobian columns of that point (0 for the
// constant link1 origin).  Only the kernels instantiated with self-collision take it (DevCfgSelf), so the parameter
// block of every other kernel is unchanged.
constexpr int kMaxSelfPairs = MRF_MAX_SELF_PAIRS;
template <typename T> struct SelfTab {
    int n[MRF_MAX_ROBOTS];
    int pt[MRF_MAX_ROBOTS][kMaxSelfPairs][2];
    int K[MRF_MAX_ROBOTS][kMaxSelfPairs][2];
    T rho[MRF_MAX_ROBOTS][kMaxSelfPairs];
    T kg, kf;            // geometry / Finsler coefficients
    int pg, pf;          // exponents of 1/x
    int gg, gf;          // sign gates
};
template <typename T> struct DevCfgSelf : DevCfg<T> {
    SelfTab<T> self;
};
struct NoSelf {};
template <typename S> constexpr bool kIsSelf = true;
template <> constexpr bool kIsSelf<NoSelf> = false;
template <typename T, bool SELF> struct CfgSel { using type = DevCfg<T>; };
template <typename T> struct CfgSel<T, true> { using type = DevCfgSelf<T>; };
template <typename T, bool SELF> using CfgOf = typename CfgSel<T, SELF>::type;

// per-thread state that persists over the horizon (registers)
template <typename T> struct Chain {
    V3<T> z[6]; // world axes of joints 1..6 (joint 7 moves no collision point)
};
// axis j of the thread's robot / origin of joint j+1 (joints 1,2 at link1; 3 at link3; 4 at link4; 5,6 at link5)
template <typename T> MRF_HD V3<T> axis_of(const Chain<T>& ch, const T* kin, int NT, int tid, int j) {
    if (kAxesInSmem<T>) {
        const T* k = kin + (kZ + 3 * j) * NT + tid;
        return V3<T>{k[0], k[NT], k[2 * NT]};
    }
    return ch.z[j];
}

// ------------------------------------------------------------------------------------------------
// chain_forward: Panda FK with velocity / acceleration propagation (qdd = 0).
// URDF constants: examples/simulation_environments/urdfs/panda_with_finger.urdf:98-106,150-158,201-209,
// 253-261,326-334,378-386,451-465.  Writes x, v = J qdot, c = d(J qdot)/dq qdot of link3,4,5,7,8 to
// kin[(e*9+comp)*NT + tid].
// ------------------------------------------------------------------------------------------------
template <typename T> struct Frame {
    V3<T> a, b, n; // columns of the rotation
    V3<T> p, w, al, v, ac;
};

template <typename T> MRF_HD void fr_advance(Frame<T>& f, V3<T> r) {
    V3<T> t = cross(f.w, r);
    f.ac = cross_add(f.w, t, cross_add(f.al, r, f.ac));
    f.v = f.v + t;
    f.p = f.p + r;
}
// roll = +1: Rx(+pi/2), -1: Rx(-pi/2), 0: none; then Rz(q) with joint velocity qd.  Returns joint axis.
template <typename T, int ROLL> MRF_HD V3<T> fr_joint(Frame<T>& f, T q, T qd) {
    if (ROLL == 1) {
        V3<T> t = f.b;
        f.b = f.n;
        f.n = t * T(-1);
    } else if (ROLL == -1) {
        V3<T> t = f.b;
        f.b = f.n * T(-1);
        f.n = t;
    }
    T s, c;
    Mth<T>::sincos(q, &s, &c);
    V3<T> a = f.a * c + f.b * s;
    V3<T> b = f.b * c - f.a * s;
    f.a = a;
    f.b = b;
    V3<T> zq = f.n * qd;
    f.al = cross_add(f.w, zq, f.al);
    f.w = f.w + zq;
    return f.n;
}
// Point table layout.  FP64: kin[(e * 9 + c) * NT + tid].  FP32: the points are stored in PAIRS (2pp, 2pp + 1) interleaved
// per thread, kin[(((e >> 1) * 9 + c) * NT + tid) * 2 + (e & 1)], so that a reader fetches component c of two points of
// another robot with ONE 64-bit shared-memory load straight into the register pair the packed FP32x2 leaf consumes
// (half the LDS instructions of the leaf loop and no pack moves); a warp's 32 x 8 B are contiguous, conflict-free.
template <typename T> constexpr bool kPairLayout = sizeof(T) == 4;
template <typename T> MRF_HD int kin_index(int NT, int tid, int e, int c) {
    return kPairLayout<T> ? (((e >> 1) * 9 + c) * NT + tid) * 2 + (e & 1) : (e * 9 + c) * NT + tid;
}
template <typename T> constexpr int kKinStride = kPairLayout<T> ? 2 : 1; // x NT: distance between components of a point
template <typename T> MRF_HD void kin_store(T* kin, int NT, int tid, int e, const Frame<T>& f) {
    T* k = kin + kin_index<T>(NT, tid, e, 0);
    const int s = kKinStride<T> * NT;
    k[0 * s] = f.p.x; k[1 * s] = f.p.y; k[2 * s] = f.p.z;
    k[3 * s] = f.v.x; k[4 * s] = f.v.y; k[5 * s] = f.v.z;
    k[6 * s] = f.ac.x; k[7 * s] = f.ac.y; k[8 * s] = f.ac.z;
}
template <typename T> MRF_HD V3<T> kin_load(const T* kin, int NT, int tid, int e, int c) {
    const T* k = kin + kin_index<T>(NT, tid, e, c);
    const int s = kKinStride<T> * NT;
    return V3<T>{k[0], k[s], k[2 * s]};
}

template <typename T>
MRF_HD void chain_forward(const DevCfg<T>& cfg, int r, const T* q, const T* qd, Chain<T>& ch, T* kin, int NT, int tid) {
    Frame<T> f;
    const T* R = cfg.R0[r];
    f.a = mk(R[0], R[3], R[6]);
    f.b = mk(R[1], R[4], R[7]);
    f.n = mk(R[2], R[5], R[8]);
    f.p = mk(cfg.link1[r][0], cfg.link1[r][1], cfg.link1[r][2]); // p0 + R0 (0,0,0.333): base is fixed
    f.w = mk(T(0), T(0), T(0));
    f.al = f.w; f.v = f.w; f.ac = f.w;
    kin_store(kin, NT, tid, 5, f);                                   // link1 == link2 (constant, v = c = 0)
    ch.z[0] = fr_joint<T, 0>(f, q[0], qd[0]);                       // joint1
    ch.z[1] = fr_joint<T, -1>(f, q[1], qd[1]);                      // joint2 (zero offset)
    fr_advance(f, f.b * T(-0.316));                                  // joint3 origin (0,-0.316,0)
    kin_store(kin, NT, tid, 0, f);                                   // link3
    ch.z[2] = fr_joint<T, 1>(f, q[2], qd[2]);
    fr_advance(f, f.a * T(0.0825));                                  // joint4 origin (0.0825,0,0)
    kin_store(kin, NT, tid, 1, f);                                   // link4
    ch.z[3] = fr_joint<T, 1>(f, q[3], qd[3]);
    fr_advance(f, f.a * T(-0.0825) + f.b * T(0.384));                // joint5 origin (-0.0825,0.384,0)
    kin_store(kin, NT, tid, 2, f);                                   // link5 == link6
    ch.z[4] = fr_joint<T, -1>(f, q[4], qd[4]);
    ch.z[5] = fr_joint<T, 1>(f, q[5], qd[5]);                        // joint6 (zero offset)
    fr_advance(f, f.a * T(0.088));                                   // joint7 origin (0.088,0,0)
    kin_store(kin, NT, tid, 3, f);                                   // link7
    // joint7 turns about the very axis the hand sits on (fixed joint8 (0,0,0.107) along it): hand position, velocity and
    // d(J qdot)/dq qdot do not depend on q7 / qdot7 (the angular terms cancel identically), so only the roll of the joint
    // frame is applied -- its axis is -b -- and the joint itself (sincos, angular updates) is skipped
    fr_advance(f, f.b * T(-0.107));                                  // hand == link8
    kin_store(kin, NT, tid, 4, f);                                   // link8
    if (kAxesInSmem<T>) {
#pragma unroll
        for (int j = 0; j < 6; ++j) {
            T* k = kin + (kZ + 3 * j) * NT + tid;
            k[0] = ch.z[j].x; k[NT] = ch.z[j].y; k[2 * NT] = ch.z[j].z;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// P2<T>: two independent values processed together.  For float on sm_100a the arithmetic maps to the packed
// FP32x2 instructions FFMA2 / FMUL2 / FADD2 (__ffma2_rn ...): one issue slot for two FMAs.  The rollout kernel is
// issue-bound (ncu: 76 % issue slots busy at 59 % FMA-pipe utilisation), so evaluating two sphere leaves per
// instruction stream removes ~30 % of its issued instructions; measured on B200 (tools/micro/ffma2_probe.cu):
// FFMA2 reaches the same pipe peak as scalar FFMA (74 TFLOP/s) with half the issue slots.  For double (and on the
// host) the pair is two scalars.
// ------------------------------------------------------------------------------------------------
#if !defined(__CUDACC__)
struct float2 {
    float x, y;
};
static inline float2 make_float2(float x, float y) { return float2{x, y}; }
#endif
template <typename T> struct P2;
template <> struct P2<float> {
    float2 v;
};
template <> struct P2<double> {
    double a, b;
};
MRF_HD P2<float> pmk(float a, float b) { return P2<float>{make_float2(a, b)}; }
MRF_HD P2<double> pmk(double a, double b) { return P2<double>{a, b}; }
MRF_HD P2<float> psplat(float a) { return pmk(a, a); }
MRF_HD P2<double> psplat(double a) { return pmk(a, a); }
MRF_HD float plo(P2<float> x) { return x.v.x; }
MRF_HD float phi(P2<float> x) { return x.v.y; }
MRF_HD double plo(P2<double> x) { return x.a; }
MRF_HD double phi(P2<double> x) { return x.b; }
MRF_HD P2<float> pmul(P2<float> x, P2<float> y) {
#if defined(__CUDA_ARCH__)
    return P2<float>{__fmul2_rn(x.v, y.v)};
#else
    return pmk(x.v.x * y.v.x, x.v.y * y.v.y);
#endif
}
MRF_HD P2<float> padd(P2<float> x, P2<float> y) {
#if defined(__CUDA_ARCH__)
    return P2<float>{__fadd2_rn(x.v, y.v)};
#else
    return pmk(x.v.x + y.v.x, x.v.y + y.v.y);
#endif
}
MRF_HD P2<float> pfma(P2<float> x, P2<float> y, P2<float> z) {
#if defined(__CUDA_ARCH__)
    return P2<float>{__ffma2_rn(x.v, y.v, z.v)};
#else
    return pmk(x.v.x * y.v.x + z.v.x, x.v.y * y.v.y + z.v.y);
#endif
}
MRF_HD P2<double> pmul(P2<double> x, P2<double> y) { return pmk(x.a * y.a, x.b * y.b); }
MRF_HD P2<double> padd(P2<double> x, P2<double> y) { return pmk(x.a + y.a, x.b + y.b); }
MRF_HD P2<double> pfma(P2<double> x, P2<double> y, P2<double> z) { return pmk(x.a * y.a + z.a, x.b * y.b + z.b); }
template <typename T> MRF_HD P2<T> prsqrt(P2<T> x) { return pmk(Mth<T>::rsqrt(plo(x)), Mth<T>::rsqrt(phi(x))); }
template <typename T> MRF_HD P2<T> prcp(P2<T> x) { return pmk(Mth<T>::rcp(plo(x)), Mth<T>::rcp(phi(x))); }
template <typename T> MRF_HD P2<T> pdot(const V3<P2<T>>& a, const V3<P2<T>>& b) {
    return pfma(a.z, b.z, pfma(a.y, b.y, pmul(a.x, b.x)));
}

// components c..c+2 of the point pair (2pp, 2pp + 1) of thread `tid`: FP32 one 64-bit load per component
MRF_HD V3<P2<float>> kin_load_pair(const float* kin, int NT, int tid, int pp, int c) {
    const float2* k = reinterpret_cast<const float2*>(kin) + (pp * 9 + c) * NT + tid;
    return V3<P2<float>>{P2<float>{k[0]}, P2<float>{k[NT]}, P2<float>{k[2 * NT]}};
}
MRF_HD V3<P2<double>> kin_load_pair(const double* kin, int NT, int tid, int pp, int c) {
    const double* a = kin + ((2 * pp) * 9 + c) * NT + tid;
    const double* b = a + 9 * NT;
    return V3<P2<double>>{pmk(a[0], b[0]), pmk(a[NT], b[NT]), pmk(a[2 * NT], b[2 * NT])};
}

// ------------------------------------------------------------------------------------------------
// accumulators
// ------------------------------------------------------------------------------------------------
template <typename T> struct Sym3 {
    T xx, xy, xz, yy, yz, zz;
};
template <typename T> struct PointAcc {
    Sym3<T> A;   // sum M_l g g^T
    V3<T> b;     // sum g (f_l + M_l (sigma curv - g.a_o))
};
template <typename T> MRF_HD V3<T> symmul(const Sym3<T>& A, V3<T> u) {
    return V3<T>{A.xx * u.x + A.xy * u.y + A.xz * u.z, A.xy * u.x + A.yy * u.y + A.yz * u.z,
                 A.xz * u.x + A.yz * u.y + A.zz * u.z};
}

// Spec in joint space: 6x6 upper triangle + decoupled joint 7 (no collision point or task map moves with q7)
template <typename T> struct Spec {
    T M[6][6]; // fabric_action accumulates the NEGATED metric here (see chol_solve6n)
    T m7;
    T f[kDof];
};

// One sphere leaf (collision_geometry "-0.5/x^4 xdot^2", collision_finsler "0.01/x^4 xdot^2",
// examples/example_pandas_Jointspace.py:88-89) of ego point (p, v, c) against sphere (xo, vo, ao), in the
// point's task space.  wt = multiplicity of identical leaves.  Same arrangement of the algebra as the packed
// sphere_leaf2 below (the FP64 kernels are bound by the FP64 pipe's issue rate, so operations count there too).
// IRHO: every leaf of the caller's loop has the same rho and the caller passes irho = 1 / rho.
template <typename T, bool IRHO = false>
MRF_HD void sphere_leaf(V3<T> p, V3<T> v, V3<T> cc, V3<T> xo, V3<T> vo, V3<T> co, T vref, T aref, T rho, T wt,
                        T sigma, PointAcc<T>& acc, T& num, T irho = T(0)) {
    // obstacle velocity = vref * vo, obstacle acceleration = aref * co (the scalars are applied to dot products)
    V3<T> d = p - xo;
    V3<T> w = mk(v.x - vref * vo.x, v.y - vref * vo.y, v.z - vref * vo.z);
    T n2 = dot(d, d);
    T in1 = Mth<T>::rsqrt(n2);
    T gs, ix;
    if (IRHO) {
        gs = in1 * irho;                                   // 1/(n rho): g = d * gs is the gradient of x w.r.t. the point
        ix = Mth<T>::rcp(Mth<T>::fma(n2, gs, T(-1)));      // 1/x, x = n/rho - 1 = n^2/(n rho) - 1
    } else {
        // x = n/rho - 1.  One reciprocal u = 1/(n rho (n - rho)) gives both 1/(n rho) (gradient scale) and 1/x.
        T n = n2 * in1;
        T t = n - rho;
        T nr = n * rho;
        T u = Mth<T>::rcp(nr * t);
        gs = u * t;
        ix = (u * nr) * rho;                               // 1/x = rho/(n - rho)
    }
    T dw = dot(d, w), da = dot(d, co), dv = dot(d, v);
    T wc = dot_add(d, cc, dot(w, w));                      // |w|^2 + d.c
    T ix2 = ix * ix, ix4 = ix2 * ix2;
    T Ml = (T(0.02) * wt) * ix4;                           // d2L/dxdot2 (x multiplicity)
    T Mg = Ml * gs;
    T k = Mg * gs;
    T u1 = k * (dw * dw);                                  // M xdot^2, xdot = (d.w) gs
    T hh = T(-0.5) * ix4;
    T fl = u1 * hh;                                        // M h, h = -0.5 xdot^2 / x^4
    T fd = u1 * Mth<T>::fma(T(2), ix, hh);                 // f_l - f_e,l (Euler-Lagrange force of the leaf energy: -2 M xdot^2 / x)
    // X = M |grad x| (kappa + g.c) = Mg (|w|^2 + d.c) - Mg (d.w)^2 / n^2, and Mg (d.w)^2 / n^2 = u1 rho / n
    T X = Mth<T>::fma(-u1, rho * in1, Mg * wc);
    T fq = Mth<T>::fma(sigma, X, Mth<T>::fma(-aref, Mg * da, fl));
    num = Mth<T>::fma(dv * gs, Mth<T>::fma(sigma - T(1), X, fd), num);
    V3<T> Md = d * k;
    acc.A.xx += Md.x * d.x; acc.A.xy += Md.x * d.y; acc.A.xz += Md.x * d.z;
    acc.A.yy += Md.y * d.y; acc.A.yz += Md.y * d.z; acc.A.zz += Md.z * d.z;
    acc.b = acc.b + d * (gs * fq);
}

// Two sphere leaves of the same ego point at once (obstacle points A and B packed in P2): same algebra as
// sphere_leaf, every operation on pairs.
template <typename T> struct PointAcc2 {
    Sym3<P2<T>> A;
    V3<P2<T>> b;
    V3<P2<T>> nv; // sum of d * gs * (f - f_e terms): dotted with the ego point's velocity once per point -> num
};
template <typename T> MRF_HD void acc2_zero(PointAcc2<T>& a) {
    const P2<T> z = psplat(T(0));
    a.A = Sym3<P2<T>>{z, z, z, z, z, z};
    a.b = V3<P2<T>>{z, z, z};
    a.nv = V3<P2<T>>{z, z, z};
}
// cM = 0.02 x multiplicity (d2L/dxdot2 coefficient of the leaf).  IRHO: every leaf of the loop has the same rho, the
// caller passes irho = 1 / rho (one reciprocal per ego point instead of the combined-reciprocal trick per leaf).
// The FP32 rollout spends two thirds of its FMA-pipe cycles here (a packed instruction occupies the pipe for two
// cycles: packing halves the issue slots, not the pipe time), so the algebra is arranged for the fewest operations:
// 58 packed instructions + 4 MUFU per pair of leaves.
template <typename T, bool IRHO>
MRF_HD void sphere_leaf2(const V3<P2<T>>& p, const V3<P2<T>>& v, const V3<P2<T>>& cc, const V3<P2<T>>& xo,
                         const V3<P2<T>>& vo, const V3<P2<T>>& co, T vref, T aref, P2<T> rho, P2<T> irho, P2<T> cM, T sigma,
                         PointAcc2<T>& acc) {
    const P2<T> m1 = psplat(T(-1)), nvref = psplat(-vref);
    V3<P2<T>> d{pfma(xo.x, m1, p.x), pfma(xo.y, m1, p.y), pfma(xo.z, m1, p.z)};
    V3<P2<T>> w{pfma(vo.x, nvref, v.x), pfma(vo.y, nvref, v.y), pfma(vo.z, nvref, v.z)};
    P2<T> n2 = pdot(d, d);
    P2<T> in1 = prsqrt(n2);
    P2<T> gs, ix, nrin;
    if (IRHO) {
        gs = pmul(in1, irho);                   // 1/(n rho): g = d * gs is the gradient of x w.r.t. the point
        ix = prcp(pfma(n2, gs, m1));            // 1/x, x = n/rho - 1 = n^2/(n rho) - 1
        nrin = pmul(in1, rho);                  // caller passes rho = -(r_o + r_b) on this path: -rho/n
    } else {
        // one reciprocal u = 1/(n rho (n - rho)) gives both 1/(n rho) and 1/x
        P2<T> n = pmul(n2, in1);
        P2<T> t = pfma(rho, m1, n);
        P2<T> nr = pmul(n, rho);
        P2<T> u = prcp(pmul(nr, t));
        gs = pmul(u, t);
        ix = pmul(pmul(u, nr), rho);
        nrin = pmul(pmul(in1, rho), m1);
    }
    P2<T> dw = pdot(d, w), da = pdot(d, co);
    P2<T> wc = pfma(d.z, cc.z, pfma(d.y, cc.y, pfma(d.x, cc.x, pdot(w, w)))); // |w|^2 + d.c
    P2<T> ix2 = pmul(ix, ix), ix4 = pmul(ix2, ix2);
    P2<T> Ml = pmul(cM, ix4);                                     // d2L/dxdot2 = 0.02 w / x^4
    P2<T> Mg = pmul(Ml, gs);
    P2<T> k = pmul(Mg, gs);
    P2<T> u1 = pmul(k, pmul(dw, dw));                             // M xdot^2, xdot = (d.w) gs
    P2<T> hh = pmul(ix4, psplat(T(-0.5)));
    P2<T> fl = pmul(u1, hh);                                      // M h, h = -0.5 xdot^2 / x^4
    P2<T> fd = pmul(u1, pfma(ix, psplat(T(2)), hh));              // f_l - f_e,l (Euler-Lagrange force -2 M xdot^2 / x)
    // X = M |grad x| (kappa + g.c) = Mg (|w|^2 + d.c) - Mg (d.w)^2 / n^2, and Mg (d.w)^2 / n^2 = u1 rho / n
    P2<T> X = pfma(u1, nrin, pmul(Mg, wc));
    P2<T> fq = pfma(X, psplat(sigma), pfma(pmul(Mg, da), psplat(-aref), fl));
    P2<T> ge = pmul(gs, pfma(X, psplat(sigma - T(1)), fd));
    acc.nv.x = pfma(d.x, ge, acc.nv.x); acc.nv.y = pfma(d.y, ge, acc.nv.y); acc.nv.z = pfma(d.z, ge, acc.nv.z);
    V3<P2<T>> Md{pmul(d.x, k), pmul(d.y, k), pmul(d.z, k)};
    acc.A.xx = pfma(Md.x, d.x, acc.A.xx); acc.A.xy = pfma(Md.x, d.y, acc.A.xy); acc.A.xz = pfma(Md.x, d.z, acc.A.xz);
    acc.A.yy = pfma(Md.y, d.y, acc.A.yy); acc.A.yz = pfma(Md.y, d.z, acc.A.yz); acc.A.zz = pfma(Md.z, d.z, acc.A.zz);
    P2<T> gf = pmul(gs, fq);
    acc.b.x = pfma(d.x, gf, acc.b.x); acc.b.y = pfma(d.y, gf, acc.b.y); acc.b.z = pfma(d.z, gf, acc.b.z);
}

// ------------------------------------------------------------------------------------------------
// Shared robot-robot leaves (FP32 throughput rollout of three robots with one sphere radius).  A leaf between point a
// of robot i and point b of robot j is evaluated by both robots; swapping the roles gives d -> -d, w -> -w and leaves
// n, g_s, 1/x, M_l, k = M_g g_s, u1, f_l and f_d unchanged when rho is the same on both sides.  The curvature term
// becomes X_b = M_g (|w|^2 - d.c_b) + u1 rho' / n, and with vref = 1, aref = sigma (dynamic mode, jdot_sign ==
// jdot_ref_sign) g_s f_q is the same on both sides: robot j's increments are A += k d d^T, b += g_s f_q d' with
// d' = -d, and its energy term (d'.v_b) g_s ((sigma - 1) X_b + f_d) is one scalar.  So each leaf is evaluated once:
// stage 1 (pair_leaves_eval) -- robot r against robot r+1, (k, g_s f_q) stored per leaf --, a CTA barrier, stage 2
// (pair_leaves_rebuild inside fabric_action) -- every robot rebuilds its point accumulators from its own slots and from
// robot r-1's.  -DMRF_NO_PAIR_LEAVES builds the kernels without it (every robot evaluates all its leaves).
// ------------------------------------------------------------------------------------------------
#ifdef MRF_NO_PAIR_LEAVES
constexpr bool kPairLeaves = false;
#else
constexpr bool kPairLeaves = true;
#endif
constexpr int kTile = 32;                            // scenarios per CTA in the rollout kernel (one lane each)
constexpr int kPairSlots = kEgo * (kPts / 2) * 2;    // per thread: (k, g_s f_q) of 5 ego points x 3 point pairs, as pairs
constexpr int kPairRows = 2 * kPairSlots + 1;        // scalars per thread: the slots + the partner's energy sum
template <typename T, int R, bool UNIFORM> constexpr bool kPairPath = kPairLeaves && UNIFORM && R == 3 && sizeof(T) == 4;

// slot s of thread t holds a pair: scalars [(s * NT + t) * 2 + 0/1], one 64-bit access for FP32
MRF_HD void pl_put(float* pl, int NT, int t, int s, P2<float> x) { reinterpret_cast<float2*>(pl)[s * NT + t] = x.v; }
MRF_HD void pl_put(double* pl, int NT, int t, int s, P2<double> x) {
    pl[(s * NT + t) * 2] = x.a;
    pl[(s * NT + t) * 2 + 1] = x.b;
}
MRF_HD P2<float> pl_get(const float* pl, int NT, int t, int s) { return P2<float>{reinterpret_cast<const float2*>(pl)[s * NT + t]}; }
MRF_HD P2<double> pl_get(const double* pl, int NT, int t, int s) { return pmk(pl[(s * NT + t) * 2], pl[(s * NT + t) * 2 + 1]); }
template <typename T> MRF_HD T pl_half(const T* pl, int NT, int t, int s, int h) { return pl[(s * NT + t) * 2 + h]; }

// The leaf slots follow the parameter blocks: prm + P_N * NT, kPairRows * NT scalars.
template <typename T> struct PairLeaves {
    T num;   // energy terms of the robot's leaves evaluated in stage 1, by itself and by robot r-1
    bool on; // this lane's scenario takes the shared-leaf path (pair_leaves_lane)
};

// Configuration side of the condition: dynamic mode, sigma == aref, collision leaves on, three robots.
template <typename T> MRF_HD bool pair_leaves_cfg(const DevCfg<T>& cfg) {
    return cfg.n_robots == 3 && cfg.uniform_obst != 0 && cfg.has_coll != 0 && cfg.static_or_dyn != 0 && cfg.sigma == cfg.sref;
}
// Scenario side (per lane, so that a scenario's result never depends on its tile neighbours): every body radius of the
// three robots is the same, so rho = r_obst + radius_body is one value for both sides of every leaf.
template <typename T> MRF_HD bool pair_leaves_lane(const T* prm, int NT, int lane) {
    const T r0 = prm[P_RB * NT + lane];
    bool eq = true;
    for (int j = 0; j < 3; ++j)
#pragma unroll
        for (int l = 0; l < 6; ++l) eq = eq && prm[(P_RB + l) * NT + j * kTile + lane] == r0;
    return eq;
}

// Two leaves of the same ego point whose other sides are points of robot r+1 (dynamic mode, aref == sigma, rho passed
// as in sphere_leaf2<T, true>): sphere_leaf2's algebra without the accumulation into A and b; returns k and g_s f_q,
// accumulates the ego energy vector like sphere_leaf2 and the partner's energy term (d.v_b) g_e,b (negated by the caller).
template <typename T>
MRF_HD void sphere_leaf2_shared(const V3<P2<T>>& p, const V3<P2<T>>& v, const V3<P2<T>>& cc, const V3<P2<T>>& xo,
                                const V3<P2<T>>& vo, const V3<P2<T>>& co, P2<T> nrho, P2<T> irho, P2<T> cM, T sigma,
                                P2<T>& k, P2<T>& gf, V3<P2<T>>& nv, P2<T>& nvb) {
    const P2<T> m1 = psplat(T(-1));
    V3<P2<T>> d{pfma(xo.x, m1, p.x), pfma(xo.y, m1, p.y), pfma(xo.z, m1, p.z)};
    V3<P2<T>> w{pfma(vo.x, m1, v.x), pfma(vo.y, m1, v.y), pfma(vo.z, m1, v.z)};
    P2<T> n2 = pdot(d, d);
    P2<T> in1 = prsqrt(n2);
    P2<T> gs = pmul(in1, irho);
    P2<T> ix = prcp(pfma(n2, gs, m1));
    P2<T> nrin = pmul(in1, nrho);
    P2<T> dw = pdot(d, w), da = pdot(d, co);
    P2<T> ww = pdot(w, w);
    P2<T> wc = pfma(d.z, cc.z, pfma(d.y, cc.y, pfma(d.x, cc.x, ww))); // |w|^2 + d.c_a
    P2<T> wcb = pfma(da, m1, ww);                                      // |w|^2 + d'.c_b
    P2<T> ix2 = pmul(ix, ix), ix4 = pmul(ix2, ix2);
    P2<T> Ml = pmul(cM, ix4);
    P2<T> Mg = pmul(Ml, gs);
    k = pmul(Mg, gs);
    P2<T> u1 = pmul(k, pmul(dw, dw));
    P2<T> hh = pmul(ix4, psplat(T(-0.5)));
    P2<T> fl = pmul(u1, hh);
    P2<T> fd = pmul(u1, pfma(ix, psplat(T(2)), hh));
    P2<T> X = pfma(u1, nrin, pmul(Mg, wc));
    P2<T> Xb = pfma(u1, nrin, pmul(Mg, wcb));
    P2<T> fq = pfma(X, psplat(sigma), pfma(pmul(Mg, da), psplat(-sigma), fl));
    const P2<T> s1 = psplat(sigma - T(1));
    P2<T> ge = pmul(gs, pfma(X, s1, fd));
    nv.x = pfma(d.x, ge, nv.x); nv.y = pfma(d.y, ge, nv.y); nv.z = pfma(d.z, ge, nv.z);
    P2<T> geb = pmul(gs, pfma(Xb, s1, fd));
    nvb = pfma(pdot(d, vo), geb, nvb); // the constant point of robot r+1 has v = 0: no partner term
    gf = pmul(gs, fq);
}

// Stage 1, thread (r, lane) of a pair lane: the 5 x 6 leaves of robot r's ego points against robot r+1's points (25
// shared, 5 one-sided against r+1's constant link1==2 point) as sphere_leaf2 pairs; (k, g_s f_q) to the slots
// (e * 3 + pp) * 2 + 0 / 1, the partner's energy sum to row 2 * kPairSlots.  Returns robot r's own energy terms.
template <typename T>
MRF_HD T pair_leaves_eval(const DevCfg<T>& cfg, int r, const T* kin, const T* prm, T* pl, int NT, int tid, int lane) {
    const int t = (r == 2 ? 0 : r + 1) * kTile + lane;
    const T rho = cfg.r_obst + prm[P_RB * NT + tid];
    const P2<T> irho = psplat(Mth<T>::rcp(rho)), nrho = psplat(-rho);
    T num = T(0);
    P2<T> nvb = psplat(T(0));
#pragma unroll 1
    for (int e = 0; e < kEgo; ++e) {
        const V3<T> p = kin_load(kin, NT, tid, e, 0), v = kin_load(kin, NT, tid, e, 3), cc = kin_load(kin, NT, tid, e, 6);
        const V3<P2<T>> p2{psplat(p.x), psplat(p.y), psplat(p.z)}, v2{psplat(v.x), psplat(v.y), psplat(v.z)},
            c2{psplat(cc.x), psplat(cc.y), psplat(cc.z)};
        const T cw = T(0.02) * (e == 2 ? T(2) : T(1)); // link5 == link6
        V3<P2<T>> nv{psplat(T(0)), psplat(T(0)), psplat(T(0))};
#pragma unroll
        for (int pp = 0; pp < kPts / 2; ++pp) {
            P2<T> k, gf;
            sphere_leaf2_shared(p2, v2, c2, kin_load_pair(kin, NT, t, pp, 0), kin_load_pair(kin, NT, t, pp, 3),
                                kin_load_pair(kin, NT, t, pp, 6), nrho, irho,
                                pmk(pp == 1 ? T(2) * cw : cw, pp == 2 ? T(2) * cw : cw), cfg.sigma, k, gf, nv, nvb);
            pl_put(pl, NT, tid, (e * 3 + pp) * 2, k);
            pl_put(pl, NT, tid, (e * 3 + pp) * 2 + 1, gf);
        }
        num = Mth<T>::fma(v.x, plo(nv.x) + phi(nv.x),
                          Mth<T>::fma(v.y, plo(nv.y) + phi(nv.y), Mth<T>::fma(v.z, plo(nv.z) + phi(nv.z), num)));
    }
    pl[2 * kPairSlots * NT + tid] = -(plo(nvb) + phi(nvb));
    return num;
}

// Stage 2, ego point e of thread (r, lane) of a pair lane, after the barrier: the one-sided leaf against robot r-1's
// constant point (evaluated here), then the leaves e shares with robot r+1 (this thread's slots) and with robot r-1
// (r-1's slots for its points 0..4 against point e) rebuilt from k and g_s f_q with d = p - x_o from the point table.
template <typename T>
MRF_HD void pair_leaves_rebuild(const DevCfg<T>& cfg, int r, const T* kin, const T* pl, int NT, int tid, int lane, int e,
                                V3<T> p, V3<T> v, V3<T> cc, T rb, T we, PointAcc<T>& acc, T& num) {
    const int tn = (r == 2 ? 0 : r + 1) * kTile + lane, tp = (r == 0 ? 2 : r - 1) * kTile + lane;
    const V3<P2<T>> x2p = kin_load_pair(kin, NT, tp, 2, 0); // robot r-1's link8 | link1==2
    const T rho = cfg.r_obst + rb;
    const V3<T> z0 = mk(T(0), T(0), T(0));
    sphere_leaf<T, true>(p, v, cc, mk(phi(x2p.x), phi(x2p.y), phi(x2p.z)), z0, z0, T(0), T(0), rho, T(2) * we, cfg.sigma,
                         acc, num, Mth<T>::rcp(rho));
    const int pe = e >> 1, he = e & 1; // point e in the point-pair numbering of the slots
    {
        const V3<T> d = p - mk(plo(x2p.x), plo(x2p.y), plo(x2p.z));
        const int s = (4 * 3 + pe) * 2;
        const T k = pl_half(pl, NT, tp, s, he), gf = pl_half(pl, NT, tp, s + 1, he);
        const V3<T> Md = d * k;
        acc.A.xx = Mth<T>::fma(Md.x, d.x, acc.A.xx); acc.A.xy = Mth<T>::fma(Md.x, d.y, acc.A.xy);
        acc.A.xz = Mth<T>::fma(Md.x, d.z, acc.A.xz); acc.A.yy = Mth<T>::fma(Md.y, d.y, acc.A.yy);
        acc.A.yz = Mth<T>::fma(Md.y, d.z, acc.A.yz); acc.A.zz = Mth<T>::fma(Md.z, d.z, acc.A.zz);
        acc.b.x = Mth<T>::fma(d.x, gf, acc.b.x); acc.b.y = Mth<T>::fma(d.y, gf, acc.b.y); acc.b.z = Mth<T>::fma(d.z, gf, acc.b.z);
    }
    // the scalar sums seed the lo halves of the pair accumulators (as in fabric_action's sphere_leaf2 path)
    const P2<T> m1 = psplat(T(-1));
    Sym3<P2<T>> A{pmk(acc.A.xx, T(0)), pmk(acc.A.xy, T(0)), pmk(acc.A.xz, T(0)), pmk(acc.A.yy, T(0)), pmk(acc.A.yz, T(0)),
                  pmk(acc.A.zz, T(0))};
    V3<P2<T>> b{pmk(acc.b.x, T(0)), pmk(acc.b.y, T(0)), pmk(acc.b.z, T(0))};
    const V3<P2<T>> p2{psplat(p.x), psplat(p.y), psplat(p.z)};
    auto add = [&](const V3<P2<T>>& xo, P2<T> k, P2<T> gf) {
        const V3<P2<T>> d{pfma(xo.x, m1, p2.x), pfma(xo.y, m1, p2.y), pfma(xo.z, m1, p2.z)};
        const V3<P2<T>> Md{pmul(d.x, k), pmul(d.y, k), pmul(d.z, k)};
        A.xx = pfma(Md.x, d.x, A.xx); A.xy = pfma(Md.x, d.y, A.xy); A.xz = pfma(Md.x, d.z, A.xz);
        A.yy = pfma(Md.y, d.y, A.yy); A.yz = pfma(Md.y, d.z, A.yz); A.zz = pfma(Md.z, d.z, A.zz);
        b.x = pfma(d.x, gf, b.x); b.y = pfma(d.y, gf, b.y); b.z = pfma(d.z, gf, b.z);
    };
#pragma unroll
    for (int pp = 0; pp < kPts / 2; ++pp)
        add(kin_load_pair(kin, NT, tn, pp, 0), pl_get(pl, NT, tid, (e * 3 + pp) * 2), pl_get(pl, NT, tid, (e * 3 + pp) * 2 + 1));
#pragma unroll
    for (int pp = 0; pp < 2; ++pp) {
        const int s0 = ((2 * pp) * 3 + pe) * 2, s1 = ((2 * pp + 1) * 3 + pe) * 2;
        add(kin_load_pair(kin, NT, tp, pp, 0), pmk(pl_half(pl, NT, tp, s0, he), pl_half(pl, NT, tp, s1, he)),
            pmk(pl_half(pl, NT, tp, s0 + 1, he), pl_half(pl, NT, tp, s1 + 1, he)));
    }
    acc.A.xx = plo(A.xx) + phi(A.xx); acc.A.xy = plo(A.xy) + phi(A.xy); acc.A.xz = plo(A.xz) + phi(A.xz);
    acc.A.yy = plo(A.yy) + phi(A.yy); acc.A.yz = plo(A.yz) + phi(A.yz); acc.A.zz = plo(A.zz) + phi(A.zz);
    acc.b.x = plo(b.x) + phi(b.x); acc.b.y = plo(b.y) + phi(b.y); acc.b.z = plo(b.z) + phi(b.z);
}

// Plane leaf (geometry_plane_constraint "10*(1/(1+exp(-10x))-1) xdot^2", example_pandas_Jointspace.py:87;
// finsler "0.1/x^2 s xdot^2", fabrics default)
template <typename T>
MRF_HD void plane_leaf(V3<T> p, V3<T> v, V3<T> cc, V3<T> nh, T dn, T rb, T wt, T sigma, PointAcc<T>& acc, T& num) {
    T x = dot(nh, p) + dn - rb;
    T xd = dot(nh, v);
    T s = xd > T(0) ? T(0) : (xd < T(0) ? T(1) : T(0.5)); // -0.5 (sign(xdot) - 1)
    T ix = Mth<T>::rcp(x);
    T xd2 = xd * xd;
    T Ml = ((T(0.2) * wt) * s) * ix * ix;                  // d2L/dxdot2 = 0.2 s / x^2
    T u = Ml * xd2;                                         // f_e = -u / x
    T h = T(-10) * xd2 * Mth<T>::rcp(T(1) + Mth<T>::exp(T(10) * x));
    T fl = Ml * h;
    T X = Ml * dot(nh, cc);
    T fq = fl + sigma * X;
    num += xd * ((fl + u * ix) + (sigma - T(1)) * X);
    V3<T> Mg = nh * Ml;
    acc.A.xx += Mg.x * nh.x; acc.A.xy += Mg.x * nh.y; acc.A.xz += Mg.x * nh.z;
    acc.A.yy += Mg.y * nh.y; acc.A.yz += Mg.y * nh.z; acc.A.zz += Mg.z * nh.z;
    acc.b = acc.b + nh * fq;
}

// Jacobian columns of a point p that rides on joints 1..K: z_j x (p - o_j).  Joint origins: o_1 = o_2 = link1,
// o_3 = link3, o_4 = link4, o_5 = o_6 = link5.
template <typename T, int K, typename Org>
MRF_HD void jac_cols(const Chain<T>& ch, const T* kin, int NT, int tid, V3<T> p, const Org& org, V3<T>* Jc) {
#pragma unroll
    for (int j = 0; j < K; ++j) Jc[j] = cross(axis_of(ch, kin, NT, tid, j), p - org(j));
}

template <typename T, int K> MRF_HD void pullback(const V3<T>* Jc, const PointAcc<T>& acc, Spec<T>& S) {
#pragma unroll
    for (int j = 0; j < K; ++j) {
        V3<T> AJ = symmul(acc.A, Jc[j]);
        S.f[j] += dot(Jc[j], acc.b);
#pragma unroll
        for (int i = 0; i <= j; ++i) S.M[i][j] += dot(Jc[i], AJ);
    }
}

// In-place Cholesky of the 6x6 upper triangle (M + eps I) and solve; returns x = (M + eps I)^-1 b.
template <typename T> MRF_HD void chol_solve6(T (&M)[6][6], T eps, const T* b, T* x) {
    T inv[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        T s = M[j][j] + eps;
#pragma unroll
        for (int k = 0; k < j; ++k) s -= M[k][j] * M[k][j];
        T r = Mth<T>::rsqrt(s);
        inv[j] = r;
        M[j][j] = s * r;
#pragma unroll
        for (int i = j + 1; i < 6; ++i) {
            T t = M[j][i];
#pragma unroll
            for (int k = 0; k < j; ++k) t -= M[k][j] * M[k][i];
            M[j][i] = t * r; // U[j][i], M = U^T U
        }
    }
    T y[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) { // U^T y = b
        T s = b[i];
#pragma unroll
        for (int k = 0; k < i; ++k) s -= M[k][i] * y[k];
        y[i] = s * inv[i];
    }
#pragma unroll
    for (int i = 5; i >= 0; --i) { // U x = y
        T s = y[i];
#pragma unroll
        for (int k = i + 1; k < 6; ++k) s -= M[i][k] * x[k];
        x[i] = s * inv[i];
    }
}

// The geometry and the forced system factored together as pairs (lo = G, hi = F): one dependent chain instead of two,
// packed FP32x2 arithmetic on sm_100a.
template <typename T> MRF_HD void chol_solve6_pair(P2<T> (&M)[6][6], T eps, const P2<T>* b, P2<T>* x) {
    P2<T> inv[6];
    const P2<T> m1 = psplat(T(-1)), e2 = psplat(eps);
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        P2<T> s = padd(M[j][j], e2);
#pragma unroll
        for (int k = 0; k < j; ++k) s = pfma(pmul(M[k][j], m1), M[k][j], s);
        P2<T> r = prsqrt(s);
        inv[j] = r;
#pragma unroll
        for (int i = j + 1; i < 6; ++i) {
            P2<T> t = M[j][i];
#pragma unroll
            for (int k = 0; k < j; ++k) t = pfma(pmul(M[k][j], m1), M[k][i], t);
            M[j][i] = pmul(t, r);
        }
    }
    P2<T> y[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        P2<T> s = b[i];
#pragma unroll
        for (int k = 0; k < i; ++k) s = pfma(pmul(M[k][i], m1), y[k], s);
        y[i] = pmul(s, inv[i]);
    }
#pragma unroll
    for (int i = 5; i >= 0; --i) {
        P2<T> s = y[i];
#pragma unroll
        for (int k = i + 1; k < 6; ++k) s = pfma(pmul(M[i][k], m1), x[k], s);
        x[i] = pmul(s, inv[i]);
    }
}

// Negated convention: the caller accumulates N = -M (free: the subtraction folds into the FMA's operand sign) and the
// factor is kept as U' = -U, so that every update of the factorisation and of the two triangular solves is a plain
// multiply-add -- the packed FP32x2 FMA has no operand negation, and the positive convention above spends one FMUL2 per
// update on it (65 of ~240 packed instructions).  N_jj - eps + sum U'_kj^2 = -s;  U'_ji = (N_ji + sum U'_kj U'_ki) r,
// r = rsqrt(s);  U^T y = b -> y_i = (b_i + sum U'_ki y_k) r_i;  U x = y -> x_i = (y_i + sum U'_ik x_k) r_i.
template <typename T> MRF_HD void chol_solve6n(T (&N)[6][6], T eps, const T* b, T* x) {
    T inv[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        T s = N[j][j] - eps;
#pragma unroll
        for (int k = 0; k < j; ++k) s += N[k][j] * N[k][j];
        T r = Mth<T>::rsqrt(-s);
        inv[j] = r;
#pragma unroll
        for (int i = j + 1; i < 6; ++i) {
            T t = N[j][i];
#pragma unroll
            for (int k = 0; k < j; ++k) t += N[k][j] * N[k][i];
            N[j][i] = t * r;
        }
    }
    T y[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        T s = b[i];
#pragma unroll
        for (int k = 0; k < i; ++k) s += N[k][i] * y[k];
        y[i] = s * inv[i];
    }
#pragma unroll
    for (int i = 5; i >= 0; --i) {
        T s = y[i];
#pragma unroll
        for (int k = i + 1; k < 6; ++k) s += N[i][k] * x[k];
        x[i] = s * inv[i];
    }
}
template <typename T> MRF_HD void chol_solve6n_pair(P2<T> (&N)[6][6], T eps, const P2<T>* b, P2<T>* x) {
    P2<T> inv[6];
    const P2<T> ne = psplat(-eps);
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        P2<T> s = padd(N[j][j], ne);
#pragma unroll
        for (int k = 0; k < j; ++k) s = pfma(N[k][j], N[k][j], s);
        P2<T> r = pmk(Mth<T>::rsqrt(-plo(s)), Mth<T>::rsqrt(-phi(s)));
        inv[j] = r;
#pragma unroll
        for (int i = j + 1; i < 6; ++i) {
            P2<T> t = N[j][i];
#pragma unroll
            for (int k = 0; k < j; ++k) t = pfma(N[k][j], N[k][i], t);
            N[j][i] = pmul(t, r);
        }
    }
    P2<T> y[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        P2<T> s = b[i];
#pragma unroll
        for (int k = 0; k < i; ++k) s = pfma(N[k][i], y[k], s);
        y[i] = pmul(s, inv[i]);
    }
#pragma unroll
    for (int i = 5; i >= 0; --i) {
        P2<T> s = y[i];
#pragma unroll
        for (int k = i + 1; k < 6; ++k) s = pfma(N[i][k], x[k], s);
        x[i] = pmul(s, inv[i]);
    }
}

template <typename T> MRF_HD void attractor_scalars(T n, T w, T& dpsi, T& m2) {
    // attractor_potential 5(|x| + 0.1 log(1 + exp(-20|x|))): d/d|x| = 5 tanh(10|x|);
    // attractor_metric (1.7 exp(-(0.75|x|)^2) + 0.3) I, L = xdot^T m xdot -> M = 2 m I
    dpsi = T(5) * w * Mth<T>::tanh(T(10) * n);
    m2 = T(2) * (T(1.7) * Mth<T>::exp(T(-0.5625) * n * n) + T(0.3));
}

// ------------------------------------------------------------------------------------------------
// fabric_action: energised geometry + forcing + damper for one robot.  `src.each(f)` enumerates the obstacle
// spheres: f(xo, vo, co, radius, weight) with velocity src.vref * vo and acceleration src.aref * co.  q, qd in registers; own kinematics in kin[..tid]; parameters in
// prm[k*NT + tid].  Writes act[7] (velocity in 'vel' mode, acceleration in 'acc' mode).
// ------------------------------------------------------------------------------------------------
template <typename T, typename Src, typename Self = NoSelf>
MRF_HD void fabric_action(const DevCfg<T>& cfg, int r, const T* q, const T* qd, const Chain<T>& ch, const T* kin,
                          const T* prm, int NT, int tid, const Src& src, T* act, T* stiff = nullptr,
                          const PairLeaves<T>* pair = nullptr, const Self& self = Self{}) {
    const T sigma = cfg.sigma;
    // shared robot-robot leaves (pair_leaves_eval has run for this step): the sphere leaves come from the slots
    const bool pair_on = kPairLeaves && Src::kUniformRadius && pair != nullptr && pair->on;
    // stiffness indicator of this evaluation: sum over the ego points of trace(A_e) = sum over the collision leaves of
    // M_l |grad x|^2 (sphere leaf: 0.02 w / (x^4 rho^2), plane leaf: 0.2 s / x^2).  Near contact it explodes like 1/x^4;
    // the FP32 rollouts use its maximum over the horizon to decide which scenarios are re-rolled in FP64 (mrf_rfcv_post).
    T stiff_sum = T(0);
    Spec<T> G;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
#pragma unroll
        for (int j = 0; j < 6; ++j) G.M[i][j] = T(0);
        G.M[i][i] = T(-0.2); // base_energy 0.5*0.2*qd.qd (G.M, F.M hold -M)
        G.f[i] = T(0);
    }
    G.m7 = T(0.2);
    G.f[6] = T(0);
    T num = pair_on ? pair->num : T(0); // qdot . (f_g - f_e,g)

    // ---- joint-limit leaves (limit_geometry "-0.1/x xdot^2", limit_finsler "0.1/x s xdot^2") ----
    // lower and upper leaf of a joint as one pair (x = q - lo | hi - q, xdot = qd | -qd):
    //   M = 0.2 s/x,  f = M h = -0.02 s xdot^2/x^2,  f - f_e = 0.08 s xdot^2/x^2
#pragma unroll
    for (int i = 0; i < kDof; ++i) {
        const P2<T> x2 = pmk(q[i] - cfg.lim[i][0], cfg.lim[i][1] - q[i]);
        const T sl = qd[i] > T(0) ? T(0) : (qd[i] < T(0) ? T(1) : T(0.5)); // lower side switch; upper = 1 - sl
        const P2<T> ix = prcp(x2);
        const P2<T> t = pmul(pmk(sl, T(1) - sl), ix);                          // s/x
        const P2<T> u = pmul(pmul(psplat(qd[i] * qd[i]), ix), t);              // s xdot^2/x^2
        const T Ml = T(0.2) * (plo(t) + phi(t));
        if (i < 6) G.M[i][i] -= Ml; else G.m7 += Ml;
        const T du = plo(u) - phi(u);                                           // lower pushes +, upper -
        G.f[i] += T(-0.02) * du;
        num += qd[i] * (T(0.08) * du);
    }


    // joint origins: FP64 re-reads them from the point table where a Jacobian column is formed (not held across the
    // leaves); FP32 keeps them in registers
    V3<T> org_[6];
    if (!kAxesInSmem<T>) {
        org_[0] = mk(cfg.link1[r][0], cfg.link1[r][1], cfg.link1[r][2]);
        org_[1] = org_[0];
        org_[2] = kin_load(kin, NT, tid, 0, 0);
        org_[3] = kin_load(kin, NT, tid, 1, 0);
        org_[4] = kin_load(kin, NT, tid, 2, 0);
        org_[5] = org_[4];
    }
    auto org = [&](int j) -> V3<T> {
        if (!kAxesInSmem<T>) return org_[j];
        return j < 2 ? mk(cfg.link1[r][0], cfg.link1[r][1], cfg.link1[r][2]) : kin_load(kin, NT, tid, j < 4 ? j - 2 : 2, 0);
    };

    // Jacobian columns of the point being pulled back.  FP32: function scope, so that the hand's columns (link8, the last
    // point of the loop) are still there for the attractors; FP64 recomputes them (18 doubles held across the attractor
    // scalars would spill).
    constexpr bool kKeepJ8 = sizeof(T) == 4;
    V3<T> Jc[6];
    bool have_j8 = false;
    // ---- collision leaves per distinct ego point (runtime loop: one copy of the leaf code keeps the kernel
    //      inside the instruction cache; the column count K of each point is warp-uniform) ----
    if (src.collide(cfg.has_coll != 0)) {
        const V3<T> nh = mk(prm[(P_NH + 0) * NT + tid], prm[(P_NH + 1) * NT + tid], prm[(P_NH + 2) * NT + tid]);
        const T dn = prm[P_DN * NT + tid];
        // Obstacle-major accumulation for sources that stream the spheres from global memory (executed action,
        // Cartesian rollout): every sphere is loaded ONCE and evaluated against the six ego links as three packed
        // pairs (link3|link4, link5|link6, link7|link8) -- the ego-major loop below would re-read the list five times
        // (measured: the S = 64 action was bound by that traffic).  FP32 only (pairs in registers).
        constexpr bool kObstMajor = Src::kObstacleMajor && sizeof(T) == 4;
        // which of panda_link3..8 carry leaves (collision_links_nr of set_planner_panda); the uniform fast path is only
        // taken when every link of every robot is in its set
        int em = 0x3F;
        if constexpr (!Src::kFullLinks) em = cfg.ego_mask[r];
        PointAcc2<T> om[3];
        if (kObstMajor) {
            V3<P2<T>> pp[3], vv[3], cp[3];
            P2<T> rbp[3];
#pragma unroll
            for (int ps = 0; ps < 3; ++ps) {
                const int ea = ps == 0 ? 0 : (ps == 1 ? 2 : 3), eb = ps == 0 ? 1 : (ps == 1 ? 2 : 4);
                V3<T> pa = kin_load(kin, NT, tid, ea, 0), pb = kin_load(kin, NT, tid, eb, 0);
                V3<T> va = kin_load(kin, NT, tid, ea, 3), vb = kin_load(kin, NT, tid, eb, 3);
                V3<T> ca = kin_load(kin, NT, tid, ea, 6), cb = kin_load(kin, NT, tid, eb, 6);
                pp[ps] = V3<P2<T>>{pmk(pa.x, pb.x), pmk(pa.y, pb.y), pmk(pa.z, pb.z)};
                vv[ps] = V3<P2<T>>{pmk(va.x, vb.x), pmk(va.y, vb.y), pmk(va.z, vb.z)};
                cp[ps] = V3<P2<T>>{pmk(ca.x, cb.x), pmk(ca.y, cb.y), pmk(ca.z, cb.z)};
                rbp[ps] = pmk(prm[(P_RB + 2 * ps) * NT + tid], prm[(P_RB + 2 * ps + 1) * NT + tid]);
                acc2_zero(om[ps]);
            }
            src.each([&](V3<T> xo, V3<T> vo, V3<T> co, T ro, T wo) {
                const V3<P2<T>> xo2{psplat(xo.x), psplat(xo.y), psplat(xo.z)}, vo2{psplat(vo.x), psplat(vo.y), psplat(vo.z)},
                    co2{psplat(co.x), psplat(co.y), psplat(co.z)};
                const P2<T> ro2 = psplat(ro);
#pragma unroll
                for (int ps = 0; ps < 3; ++ps)
                    sphere_leaf2<T, false>(pp[ps], vv[ps], cp[ps], xo2, vo2, co2, src.vref, src.aref, padd(ro2, rbp[ps]), ro2,
                                           pmk(T(0.02) * wo * T((em >> (2 * ps)) & 1), T(0.02) * wo * T((em >> (2 * ps + 1)) & 1)),
                                           sigma, om[ps]);
            });
        }
        // FP64 with a global-memory source: obstacle-major as well, one scalar leaf per (sphere, ego point), the five task-space
        // accumulators in registers and the ego points re-read from shared memory -- the list is fetched once instead of
        // five times and the five leaves of a sphere are independent instruction streams for the FP64 pipe
#ifdef MRF_NO_OBSTMAJOR_F64
        constexpr bool kObstMajorD = false;
#else
        constexpr bool kObstMajorD = Src::kObstacleMajor && sizeof(T) == 8;
#endif
        PointAcc<T> od[kEgo];
        if (kObstMajorD) {
            T rbv[6], wl[6];
#pragma unroll
            for (int l = 0; l < 6; ++l) {
                rbv[l] = prm[(P_RB + l) * NT + tid];
                wl[l] = T((em >> l) & 1);
            }
            if (wl[2] > T(0) && wl[3] > T(0) && rbv[2] == rbv[3]) { // link5 == link6: one leaf of weight 2
                wl[2] = T(2);
                wl[3] = T(0);
            }
#pragma unroll
            for (int e = 0; e < kEgo; ++e) {
                od[e].A = Sym3<T>{T(0), T(0), T(0), T(0), T(0), T(0)};
                od[e].b = mk(T(0), T(0), T(0));
            }
            src.each([&](V3<T> xo, V3<T> vo, V3<T> co, T ro, T wo) {
#pragma unroll
                for (int e = 0; e < kEgo; ++e) {
                    const int l = e + (e > 2 ? 1 : 0);
                    const V3<T> pe = kin_load(kin, NT, tid, e, 0), ve = kin_load(kin, NT, tid, e, 3), ce = kin_load(kin, NT, tid, e, 6);
                    sphere_leaf(pe, ve, ce, xo, vo, co, src.vref, src.aref, ro + rbv[l], wl[l] * wo, sigma, od[e], num);
                    if (e == 2 && wl[3] > T(0))
                        sphere_leaf(pe, ve, ce, xo, vo, co, src.vref, src.aref, ro + rbv[3], wl[3] * wo, sigma, od[e], num);
                }
            });
        }
#pragma unroll 1
        for (int e = 0; e < kEgo; ++e) {
            const int K = e < 3 ? e + 2 : 6;           // link3: 2, link4: 3, link5/6: 4, link7: 6, link8: 6 joints
            const int rb_first = e + (e > 2 ? 1 : 0);  // index into radius_body_panda_link3..8
            V3<T> p = kin_load(kin, NT, tid, e, 0), v = kin_load(kin, NT, tid, e, 3), cc = kin_load(kin, NT, tid, e, 6);
            PointAcc<T> acc;
            acc.A = Sym3<T>{T(0), T(0), T(0), T(0), T(0), T(0)};
            acc.b = mk(T(0), T(0), T(0));
            T rb = prm[(P_RB + rb_first) * NT + tid];
            T we = T(1);
            int passes = 1;
            if (e == 2) { // link5 and link6 share the point; identical leaves if their radii agree
                T rb2 = prm[(P_RB + rb_first + 1) * NT + tid];
                if (Src::kFullLinks || ((em >> rb_first) & 3) == 3) {
                    if (rb2 == rb) we = T(2); else passes = 2;
                } else if ((em >> (rb_first + 1)) & 1) {
                    rb = rb2;                       // only link6 is a collision link
                } else if (!((em >> rb_first) & 1)) {
                    passes = 0;                     // neither
                }
            } else if (!Src::kFullLinks && !((em >> rb_first) & 1)) {
                passes = 0;
            }
            if (!Src::kFullLinks && passes == 0) continue; // no collision link at this point: no leaves, nothing to pull back
            if (kObstMajor) {
                // pick this point's accumulators from the pair slots: link3 = slot0.lo, link4 = slot0.hi,
                // link5 + link6 = slot1.lo + slot1.hi (same point), link7 = slot2.lo, link8 = slot2.hi
                auto pick = [&](const P2<T>& s0, const P2<T>& s1, const P2<T>& s2) {
                    return e == 0 ? plo(s0) : e == 1 ? phi(s0) : e == 2 ? plo(s1) + phi(s1) : e == 3 ? plo(s2) : phi(s2);
                };
                acc.A.xx = pick(om[0].A.xx, om[1].A.xx, om[2].A.xx); acc.A.xy = pick(om[0].A.xy, om[1].A.xy, om[2].A.xy);
                acc.A.xz = pick(om[0].A.xz, om[1].A.xz, om[2].A.xz); acc.A.yy = pick(om[0].A.yy, om[1].A.yy, om[2].A.yy);
                acc.A.yz = pick(om[0].A.yz, om[1].A.yz, om[2].A.yz); acc.A.zz = pick(om[0].A.zz, om[1].A.zz, om[2].A.zz);
                acc.b.x = pick(om[0].b.x, om[1].b.x, om[2].b.x); acc.b.y = pick(om[0].b.y, om[1].b.y, om[2].b.y);
                acc.b.z = pick(om[0].b.z, om[1].b.z, om[2].b.z);
                num += dot(v, mk(pick(om[0].nv.x, om[1].nv.x, om[2].nv.x), pick(om[0].nv.y, om[1].nv.y, om[2].nv.y),
                                 pick(om[0].nv.z, om[1].nv.z, om[2].nv.z)));
            }
            if (kObstMajorD) {
                auto pk = [&](T a0, T a1, T a2, T a3, T a4) { return e == 0 ? a0 : e == 1 ? a1 : e == 2 ? a2 : e == 3 ? a3 : a4; };
                acc.A.xx = pk(od[0].A.xx, od[1].A.xx, od[2].A.xx, od[3].A.xx, od[4].A.xx);
                acc.A.xy = pk(od[0].A.xy, od[1].A.xy, od[2].A.xy, od[3].A.xy, od[4].A.xy);
                acc.A.xz = pk(od[0].A.xz, od[1].A.xz, od[2].A.xz, od[3].A.xz, od[4].A.xz);
                acc.A.yy = pk(od[0].A.yy, od[1].A.yy, od[2].A.yy, od[3].A.yy, od[4].A.yy);
                acc.A.yz = pk(od[0].A.yz, od[1].A.yz, od[2].A.yz, od[3].A.yz, od[4].A.yz);
                acc.A.zz = pk(od[0].A.zz, od[1].A.zz, od[2].A.zz, od[3].A.zz, od[4].A.zz);
                acc.b.x = pk(od[0].b.x, od[1].b.x, od[2].b.x, od[3].b.x, od[4].b.x);
                acc.b.y = pk(od[0].b.y, od[1].b.y, od[2].b.y, od[3].b.y, od[4].b.y);
                acc.b.z = pk(od[0].b.z, od[1].b.z, od[2].b.z, od[3].b.z, od[4].b.z);
            }
            // scalar leaves first (plane, static spheres; every sphere for FP64) ...
            constexpr bool kPackedSpheres = sizeof(T) == 4 && !kObstMajor;
            const T rb0 = rb;
            for (int pass = 0; pass < passes; ++pass) {
                if (pass == 1) rb = prm[(P_RB + rb_first + 1) * NT + tid];
                if (!kPackedSpheres && !kObstMajor && !kObstMajorD && !pair_on) {
                    // FP64: no packed instructions exist and pairing doubles the live registers -> one leaf at a time
                    if constexpr (Src::kUniformRadius) {
                        const T rho = src.ro + rb, irho = Mth<T>::rcp(rho); // one rho for every leaf of this ego point
                        src.each([&](V3<T> xo, V3<T> vo, V3<T> co, T, T wo) {
                            sphere_leaf<T, true>(p, v, cc, xo, vo, co, src.vref, src.aref, rho, we * wo, sigma, acc, num, irho);
                        });
                    } else {
                        src.each([&](V3<T> xo, V3<T> vo, V3<T> co, T ro, T wo) {
                            sphere_leaf(p, v, cc, xo, vo, co, src.vref, src.aref, ro + rb, we * wo, sigma, acc, num);
                        });
                    }
                }
                // static spheres of the rollout planners (x_obst_i, radius_obst_i; forward_planner_Jointspace.py:319-322):
                // the same leaf with a sphere at rest
                if constexpr (Src::kHasStatic)
                    src.each_static([&](V3<T> xo, T ro) {
                        const V3<T> z0 = mk(T(0), T(0), T(0));
                        sphere_leaf(p, v, cc, xo, z0, z0, T(0), T(0), ro + rb, we, sigma, acc, num);
                    });
                plane_leaf(p, v, cc, nh, dn, rb, we, sigma, acc, num);
            }
            if (pair_on) {
                pair_leaves_rebuild(cfg, r, kin, prm + P_N * NT, NT, tid, tid % kTile, e, p, v, cc, rb0, we, acc, num);
            } else if (kPackedSpheres) {
                // ... then the FP32 sphere leaves two at a time with packed FP32x2 instructions (sm_100a FFMA2 / FMUL2); the
                // scalar sums seed the lo halves of the pair accumulators, so folding the pairs is one addition per entry
                PointAcc2<T> acc2;
                acc2.A = Sym3<P2<T>>{pmk(acc.A.xx, T(0)), pmk(acc.A.xy, T(0)), pmk(acc.A.xz, T(0)),
                                     pmk(acc.A.yy, T(0)), pmk(acc.A.yz, T(0)), pmk(acc.A.zz, T(0))};
                acc2.b = V3<P2<T>>{pmk(acc.b.x, T(0)), pmk(acc.b.y, T(0)), pmk(acc.b.z, T(0))};
                acc2.nv = V3<P2<T>>{psplat(T(0)), psplat(T(0)), psplat(T(0))};
                const V3<P2<T>> p2{psplat(p.x), psplat(p.y), psplat(p.z)}, v2{psplat(v.x), psplat(v.y), psplat(v.z)},
                    c2{psplat(cc.x), psplat(cc.y), psplat(cc.z)};
                const P2<T> cw = psplat(T(0.02) * we);
                rb = rb0;
                for (int pass = 0; pass < passes; ++pass) {
                    if (pass == 1) rb = prm[(P_RB + rb_first + 1) * NT + tid];
                    if constexpr (Src::kUniformRadius) {
                        // one rho for every leaf of this ego point: 1/rho and -rho go in
                        const P2<T> irho = psplat(Mth<T>::rcp(src.ro + rb)), nrho = psplat(-(src.ro + rb));
                        src.each2([&](const V3<P2<T>>& xo, const V3<P2<T>>& vo, const V3<P2<T>>& co, P2<T>, P2<T> wo) {
                            sphere_leaf2<T, true>(p2, v2, c2, xo, vo, co, src.vref, src.aref, nrho, irho, pmul(wo, cw), sigma, acc2);
                        });
                    } else {
                        src.each2([&](const V3<P2<T>>& xo, const V3<P2<T>>& vo, const V3<P2<T>>& co, P2<T> ro, P2<T> wo) {
                            sphere_leaf2<T, false>(p2, v2, c2, xo, vo, co, src.vref, src.aref, padd(ro, psplat(rb)), ro,
                                                   pmul(wo, cw), sigma, acc2);
                        });
                    }
                }
                acc.A.xx = plo(acc2.A.xx) + phi(acc2.A.xx); acc.A.xy = plo(acc2.A.xy) + phi(acc2.A.xy);
                acc.A.xz = plo(acc2.A.xz) + phi(acc2.A.xz); acc.A.yy = plo(acc2.A.yy) + phi(acc2.A.yy);
                acc.A.yz = plo(acc2.A.yz) + phi(acc2.A.yz); acc.A.zz = plo(acc2.A.zz) + phi(acc2.A.zz);
                acc.b.x = plo(acc2.b.x) + phi(acc2.b.x); acc.b.y = plo(acc2.b.y) + phi(acc2.b.y);
                acc.b.z = plo(acc2.b.z) + phi(acc2.b.z);
                // explicit multiply-adds: the compiler's choice of which products of a scalar sum to contract differed between
                // two instantiations of the rollout kernel (host-record / device layouts must stay bitwise identical)
                num = Mth<T>::fma(v.x, plo(acc2.nv.x) + phi(acc2.nv.x),
                                  Mth<T>::fma(v.y, plo(acc2.nv.y) + phi(acc2.nv.y), Mth<T>::fma(v.z, plo(acc2.nv.z) + phi(acc2.nv.z), num)));
            }
            stiff_sum += (acc.A.xx + acc.A.yy) + acc.A.zz;
            if (kKeepJ8 && e == kEgo - 1) have_j8 = true;
#pragma unroll
            for (int j = 0; j < 6; ++j)
                if (j < K) Jc[j] = cross(axis_of(ch, kin, NT, tid, j), p - org(j));
#pragma unroll
            for (int j = 0; j < 6; ++j) {
                if (j < K) {
                    V3<T> AJ = symmul(acc.A, Jc[j]);
                    G.f[j] = dot_add(Jc[j], acc.b, G.f[j]);
#pragma unroll
                    for (int i = 0; i <= j; ++i) G.M[i][j] = dot_sub(Jc[i], AJ, G.M[i][j]);
                }
            }
        }
    }

    if (stiff != nullptr) *stiff = stiff_sum;

    // ---- self-collision leaves (every planner of the handle, grasp planner included): the sphere leaf's closed form on
    //      the relative point d = p_a - p_b, w = v_a - v_b, c = c_a - c_b with columns J_a - J_b, one rank-1 update each.
    //      M = 2 k_f s_f / x^p_f, f = M h with h = k_g s_g xdot^2 / x^p_g, f_e = -(p_f / 2) M xdot^2 / x ----
    if constexpr (kIsSelf<Self>) {
#pragma unroll 1
        for (int k = 0; k < self.n[r]; ++k) {
            const int ea = self.pt[r][k][0], eb = self.pt[r][k][1], Ka = self.K[r][k][0], Kb = self.K[r][k][1];
            const V3<T> pa = kin_load(kin, NT, tid, ea, 0), pb = kin_load(kin, NT, tid, eb, 0);
            const V3<T> d = pa - pb;
            const V3<T> w = kin_load(kin, NT, tid, ea, 3) - kin_load(kin, NT, tid, eb, 3);
            const V3<T> c = kin_load(kin, NT, tid, ea, 6) - kin_load(kin, NT, tid, eb, 6);
            const T rho = self.rho[r][k];
            const T n2 = dot(d, d);
            const T n = Mth<T>::sqrt(n2);
            const T gs = Mth<T>::rcp(n * rho);                 // g = d * gs is the gradient of x w.r.t. the relative point
            const T ix = rho * Mth<T>::rcp(n - rho);            // 1/x
            const T dw = dot(d, w);
            const T xd = dw * gs;                               // xdot
            const T s = xd > T(0) ? T(0) : (xd < T(0) ? T(1) : T(0.5));
            T ipf = T(1), ipg = T(1);
            for (int i = 0; i < self.pf; ++i) ipf *= ix;
            for (int i = 0; i < self.pg; ++i) ipg *= ix;
            const T Ml = T(2) * self.kf * (self.gf ? s : T(1)) * ipf;
            const T hh = self.kg * (self.gg ? s : T(1)) * ipg;  // h = hh xdot^2
            const T Mg = Ml * gs;
            const T kk = Mg * gs;
            const T u1 = Ml * (xd * xd);                        // M xdot^2
            const T fl = u1 * hh;                               // f = M h
            const T fd = u1 * (hh + T(0.5) * T(self.pf) * ix);  // f - f_e
            // X = M (J-dot qdot of x without sigma) = Mg (|w|^2 + d.c) - u1 rho / n
            const T X = Mg * (dot(w, w) + dot(d, c)) - u1 * rho * Mth<T>::rcp(n);
            const T fq = sigma * X + fl;
            num += xd * ((sigma - T(1)) * X + fd);
            T u[6];
#pragma unroll
            for (int j = 0; j < 6; ++j) {
                const V3<T> z = axis_of(ch, kin, NT, tid, j), o = org(j);
                T uj = T(0);
                if (j < Ka) uj += dot(d, cross(z, pa - o));
                if (j < Kb) uj -= dot(d, cross(z, pb - o));
                u[j] = uj;
            }
            const T gf = gs * fq;
#pragma unroll
            for (int j = 0; j < 6; ++j) {
                G.f[j] += u[j] * gf;
                const T ku = kk * u[j];
#pragma unroll
                for (int i = 0; i <= j; ++i) G.M[i][j] -= u[i] * ku;
            }
        }
    }

    // ---- q^T M_g q ----
    T qMq = G.m7 * qd[6] * qd[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) { // row sums first: one multiply-add per entry
        T row = G.M[i][i] * qd[i];
#pragma unroll
        for (int j = i + 1; j < 6; ++j) row += G.M[i][j] * (qd[j] + qd[j]);
        qMq -= row * qd[i];
    }
    const T e = cfg.eps;
    const T a_geom = -num * Mth<T>::rcp(e + qMq);

    // ---- forced spec = geometry + attractors (goal struct example_pandas_Jointspace.py:25-62) ----
    Spec<T> F = G;
    T xpsi;
    {
        V3<T> p8 = kin_load(kin, NT, tid, 4, 0), c8 = kin_load(kin, NT, tid, 4, 6);
        V3<T> p7 = kin_load(kin, NT, tid, 3, 0), c7 = kin_load(kin, NT, tid, 3, 6);
        // sub-goal 0: world -> panda_hand
        V3<T> x0 = p8 - mk(prm[(P_G0 + 0) * NT + tid], prm[(P_G0 + 1) * NT + tid], prm[(P_G0 + 2) * NT + tid]);
        T n0 = Mth<T>::sqrt(dot(x0, x0));
        xpsi = n0;
        T dpsi0, m0;
        attractor_scalars(n0, prm[P_W0 * NT + tid], dpsi0, m0);
        V3<T> t0 = (x0 * (dpsi0 * Mth<T>::rcp(n0)) + c8 * sigma) * m0;
        // sub-goal 1: angle_goal_1 (hand - link7) - x_goal_1
        T Rg[9];
#pragma unroll
        for (int k = 0; k < 9; ++k) Rg[k] = prm[(P_ANG + k) * NT + tid];
        auto rot = [&](V3<T> u) {
            return V3<T>{Rg[0] * u.x + Rg[1] * u.y + Rg[2] * u.z, Rg[3] * u.x + Rg[4] * u.y + Rg[5] * u.z,
                         Rg[6] * u.x + Rg[7] * u.y + Rg[8] * u.z};
        };
        V3<T> d87 = p8 - p7;
        V3<T> x1 = rot(d87) - mk(prm[(P_G1 + 0) * NT + tid], prm[(P_G1 + 1) * NT + tid], prm[(P_G1 + 2) * NT + tid]);
        T n1 = Mth<T>::sqrt(dot(x1, x1));
        T dpsi1, m1;
        attractor_scalars(n1, prm[P_W1 * NT + tid], dpsi1, m1);
        V3<T> t1 = (x1 * (dpsi1 * Mth<T>::rcp(n1)) + rot(c8 - c7) * sigma) * m1;
        // Both attractors are point loads.  Sub-goal 0 acts at the hand: columns J8_j, metric m0 I, force t0.  Sub-goal 1
        // acts on the direction hand - link7, columns Jd_j = z_j x (p8 - p7), metric m1 R^T R, force R^T t1 (the rotation
        // angle_goal_1 is folded into metric and force once instead of rotating every column).
        const V3<T> u1{Rg[0] * t1.x + Rg[3] * t1.y + Rg[6] * t1.z, Rg[1] * t1.x + Rg[4] * t1.y + Rg[7] * t1.z,
                       Rg[2] * t1.x + Rg[5] * t1.y + Rg[8] * t1.z};
        const T nm1 = -m1, nm0 = -m0;
        const Sym3<T> nW{nm1 * (Rg[0] * Rg[0] + Rg[3] * Rg[3] + Rg[6] * Rg[6]), nm1 * (Rg[0] * Rg[1] + Rg[3] * Rg[4] + Rg[6] * Rg[7]),
                         nm1 * (Rg[0] * Rg[2] + Rg[3] * Rg[5] + Rg[6] * Rg[8]), nm1 * (Rg[1] * Rg[1] + Rg[4] * Rg[4] + Rg[7] * Rg[7]),
                         nm1 * (Rg[1] * Rg[2] + Rg[4] * Rg[5] + Rg[7] * Rg[8]), nm1 * (Rg[2] * Rg[2] + Rg[5] * Rg[5] + Rg[8] * Rg[8])};
        if (!kKeepJ8 || !have_j8) jac_cols<T, 6>(ch, kin, NT, tid, p8, org, Jc);
        V3<T> Jd[6];
#pragma unroll
        for (int j = 0; j < 6; ++j) Jd[j] = cross(axis_of(ch, kin, NT, tid, j), d87);
#pragma unroll
        for (int j = 0; j < 6; ++j) {
            const V3<T> A0 = Jc[j] * nm0, A1 = symmul(nW, Jd[j]);
            F.f[j] = dot_add(Jc[j], t0, dot_add(Jd[j], u1, F.f[j]));
#pragma unroll
            for (int i = 0; i <= j; ++i) F.M[i][j] = dot_add(Jc[i], A0, dot_add(Jd[i], A1, F.M[i][j]));
        }
        // sub-goal 2: joint 7 -> x_goal_2
        T x2 = q[6] - prm[P_G2 * NT + tid];
        T dpsi2, m2;
        attractor_scalars(Mth<T>::abs(x2), prm[P_W2 * NT + tid], dpsi2, m2);
        F.f[6] += m2 * dpsi2 * (x2 > T(0) ? T(1) : (x2 < T(0) ? T(-1) : T(0)));
        F.m7 += m2;
    }

    // ---- solves and speed-control damper ----
    T hg[kDof], hf[kDof];
    if (sizeof(T) == 4) {
        P2<T> M2[6][6], b2[6], x2[6];
#pragma unroll
        for (int j = 0; j < 6; ++j) {
            b2[j] = pmk(G.f[j], F.f[j]);
#pragma unroll
            for (int i = 0; i <= j; ++i) M2[i][j] = pmk(G.M[i][j], F.M[i][j]);
        }
        chol_solve6n_pair(M2, e, b2, x2);
#pragma unroll
        for (int j = 0; j < 6; ++j) {
            hg[j] = plo(x2[j]);
            hf[j] = phi(x2[j]);
        }
    } else {
        chol_solve6n(G.M, e, G.f, hg);
        chol_solve6n(F.M, e, F.f, hf);
    }
    hg[6] = G.f[6] * Mth<T>::rcp(G.m7 + e);
    hf[6] = F.f[6] * Mth<T>::rcp(F.m7 + e);
    T qq = T(0), qhg = T(0), qhf = T(0);
#pragma unroll
    for (int i = 0; i < kDof; ++i) {
        qq += qd[i] * qd[i];
        qhg += qd[i] * hg[i];
        qhf += qd[i] * hf[i];
    }
    const T iden = Mth<T>::rcp(e + cfg.s2 * qq);
    const T a_ex0 = -cfg.s2 * qhg * iden, a_exf = -cfg.s2 * qhf * iden;
    const T eta = T(0.5) * (Mth<T>::tanh(T(-0.45) * qq - T(0.5)) + T(1)); // damper_eta
    const T a_ex = eta * a_ex0 + (T(1) - eta) * a_exf;
    const T beta = T(0.5) * (Mth<T>::tanh(T(-0.5) * (xpsi - T(0.02))) + T(1)) * T(6.5) + T(0.01) +
                   Mth<T>::max(T(0), a_geom - a_ex); // damper_beta
    const T damp = a_ex + beta;
#pragma unroll
    for (int i = 0; i < kDof; ++i) {
        T qdd = -hf[i] - damp * qd[i];
        act[i] = cfg.mode == 1 ? qd[i] + cfg.dt * qdd : qdd;
    }
}

// ------------------------------------------------------------------------------------------------
// obstacle sources for fabric_action
// ------------------------------------------------------------------------------------------------
// other robots of the same scenario, read from the CTA's shared kinematics table (generic: table driven, any radii)
template <typename T> struct SmemSrc {
    static constexpr bool kUniformRadius = false;
    static constexpr bool kFullLinks = false;     // ego leaves follow cfg.ego_mask
    static constexpr bool kHasStatic = true;      // + n_static spheres at rest per robot, staged at stat[(o*4+c)*NT + tid]
    template <typename F> MRF_HD void each_static(F f) const {
        for (int o = 0; o < n_static; ++o) {
            const T* b = stat + (o * 4) * NT + tid_s;
            f(mk(b[0], b[NT], b[2 * NT]), b[3 * NT]);
        }
    }
    static constexpr bool kObstacleMajor = false; // shared-memory points: re-reading per ego point is cheap
    MRF_HD bool collide(bool has) const { return has; }
    const DevCfg<T>& cfg;
    const T* kin;
    int NT, lane, r;
    T vref, aref;
    const T* stat = nullptr;
    int n_static = 0, tid_s = 0;
    template <typename F> MRF_HD void each(F f) const {
        const int ne = cfg.ent_n[r];
#pragma unroll 2
        for (int k = 0; k < ne; ++k) {
            const int t = cfg.ent_rob[r][k] * kTile + lane, e = cfg.ent_src[r][k];
            f(kin_load(kin, NT, t, e, 0), kin_load(kin, NT, t, e, 3), kin_load(kin, NT, t, e, 6), cfg.ent_rad[r][k],
              cfg.ent_w[r][k]);
        }
    }
    // pairs of entries; an odd tail is paired with itself at weight 0
    template <typename F> MRF_HD void each2(F f) const {
        const int ne = cfg.ent_n[r];
        for (int k = 0; k < ne; k += 2) {
            const int k1 = k + 1 < ne ? k + 1 : k;
            const int ta = cfg.ent_rob[r][k] * kTile + lane, tb = cfg.ent_rob[r][k1] * kTile + lane;
            const int ea = cfg.ent_src[r][k], eb = cfg.ent_src[r][k1];
            const V3<T> xa = kin_load(kin, NT, ta, ea, 0), va = kin_load(kin, NT, ta, ea, 3), ca = kin_load(kin, NT, ta, ea, 6);
            const V3<T> xb = kin_load(kin, NT, tb, eb, 0), vb = kin_load(kin, NT, tb, eb, 3), cb = kin_load(kin, NT, tb, eb, 6);
            f(V3<P2<T>>{pmk(xa.x, xb.x), pmk(xa.y, xb.y), pmk(xa.z, xb.z)},
              V3<P2<T>>{pmk(va.x, vb.x), pmk(va.y, vb.y), pmk(va.z, vb.z)},
              V3<P2<T>>{pmk(ca.x, cb.x), pmk(ca.y, cb.y), pmk(ca.z, cb.z)},
              pmk(cfg.ent_rad[r][k], cfg.ent_rad[r][k1]), pmk(cfg.ent_w[r][k], k1 == k ? T(0) : cfg.ent_w[r][k1]));
        }
    }
};

// same, specialised to the reference's set-up in which every robot sphere has the same radius
// (parameters_manipulators.py:23,37-43): no table look-ups, the six distinct points of each other robot are unrolled
// with their multiplicities (link3, link4, link5==6 [x2], link7, link8, link1==2 [x2]) as compile-time constants.
template <typename T, int R> struct SmemSrcUniform {
    static constexpr bool kUniformRadius = true;  // every sphere has radius ro: rho = ro + radius_body is per ego point
    static constexpr bool kFullLinks = true;      // all of panda_link3..8 carry leaves (the reference's set-up)
    static constexpr bool kHasStatic = false;
    static constexpr bool kObstacleMajor = false;
    MRF_HD bool collide(bool has) const { return has; }
    const T* kin;
    int lane, r;
    T vref, aref, ro;
    template <typename F> MRF_HD void each(F f) const {
        constexpr int NT = kTile * R;
        // runtime loops (pairs of leaves unrolled for ILP): a fully unrolled body overflows the instruction cache
        // (measured: stall_no_inst 46 % with 12 inlined leaves vs 7 % with 2)
#pragma unroll 1
        for (int j = 0; j < R; ++j) {
            if (j == r) continue;
            const int t = j * kTile + lane;
#pragma unroll 2
            for (int pt = 0; pt < kPts; ++pt) {
                f(kin_load(kin, NT, t, pt, 0), kin_load(kin, NT, t, pt, 3), kin_load(kin, NT, t, pt, 6), ro,
                  (pt == 2 || pt == 5) ? T(2) : T(1));
            }
        }
    }
    // point pairs (link3, link4), (link5==6 [x2], link7), (link8, link1==2 [x2]) of every other robot
    template <typename F> MRF_HD void each2(F f) const {
        constexpr int NT = kTile * R;
        const P2<T> ro2 = psplat(ro);
#ifdef MRF_EACH2_UNROLL
#pragma unroll
#else
#pragma unroll 1
#endif
        for (int j = 0; j < R; ++j) {
            if (j == r) continue;
            const int t = j * kTile + lane;
#pragma unroll
            for (int pp = 0; pp < kPts / 2; ++pp) { // 3 independent packed leaves in flight (ILP); 64-bit pair loads
                f(kin_load_pair(kin, NT, t, pp, 0), kin_load_pair(kin, NT, t, pp, 3), kin_load_pair(kin, NT, t, pp, 6), ro2,
                  pmk(pp == 1 ? T(2) : T(1), pp == 2 ? T(2) : T(1)));
            }
        }
    }
};

// caller-supplied spheres in global memory, SoA [S][MRF_OBST][stride]; tk > 0 extrapolates x + tk * xdot.
// On the device the list is streamed through a per-thread ring in shared memory with cp.async (LDGSTS): kObstRing - 1
// spheres (ten scalars each) are in flight per thread without holding registers, which is what hides the HBM latency
// at the 8-12 warps per SM this kernel runs with (ncu before: 45 % of stall samples on the register-prefetched loads,
// 1.4 TB/s).  ring == nullptr (host emulation) reads directly.
#ifndef MRF_OBST_RING
#define MRF_OBST_RING 4
#endif
constexpr int kObstRing = MRF_OBST_RING; // power of two
#if defined(__CUDA_ARCH__)
template <typename T> __device__ __forceinline__ void cp_async_scalar(T* smem_dst, const T* gsrc) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    if (sizeof(T) == 4)
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(gsrc) : "memory");
    else
        asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
#endif
template <typename T, bool CART> struct GlobalSrc {
    static constexpr bool kUniformRadius = false;
    static constexpr bool kFullLinks = false;
    static constexpr bool kHasStatic = false;     // static spheres arrive in the same list with zero velocity
    static constexpr bool kObstacleMajor = true; // global-memory spheres: load each once (see fabric_action)
    const T* obst;
    long long stride, off;
    int S;
    T tk;
    T vref, aref;
    T* ring;   // shared memory, kObstRing * MRF_OBST * NT scalars (element [slot][c][tid]); nullptr on the host
    int NT, tid;
    bool grasp = false; // this thread evaluates the obstacle-free grasp planner (example_pandas_Jointspace.py:160-166,440)
    MRF_HD bool collide(bool has) const { return has && !grasp; }
    template <typename F> MRF_HD void emit(const T* cur, F& f) const {
        V3<T> xo = mk(cur[0], cur[1], cur[2]);
        V3<T> vo = mk(cur[3], cur[4], cur[5]);
        V3<T> ao;
        if (CART) {
            xo = xo + vo * tk;
            ao = mk(T(0), T(0), T(0));
        } else {
            ao = mk(cur[6], cur[7], cur[8]);
        }
        f(xo, vo, ao, cur[9], T(1));
    }
    template <typename F> MRF_HD void each(F f) const {
        if (S <= 0) return;
#if defined(__CUDA_ARCH__)
        if (ring != nullptr) {
            auto issue = [&](int o) {
                if (o < S) {
                    const T* b = obst + (long long)o * MRF_OBST * stride + off;
                    T* d = ring + (o & (kObstRing - 1)) * MRF_OBST * NT + tid;
#pragma unroll
                    for (int c = 0; c < MRF_OBST; ++c) cp_async_scalar(d + c * NT, b + c * stride);
                }
                cp_async_commit(); // an empty group past the end keeps the wait count uniform
            };
#pragma unroll
            for (int o = 0; o < kObstRing - 1; ++o) issue(o);
            for (int o = 0; o < S; ++o) {
                issue(o + kObstRing - 1); // refills the slot consumed at o - 1
                cp_async_wait<kObstRing - 1>();
                const T* d = ring + (o & (kObstRing - 1)) * MRF_OBST * NT + tid;
                T cur[MRF_OBST];
#pragma unroll
                for (int c = 0; c < MRF_OBST; ++c) cur[c] = d[c * NT];
                emit(cur, f);
            }
            cp_async_wait<0>();
            return;
        }
#endif
        for (int o = 0; o < S; ++o) {
            const T* b = obst + (long long)o * MRF_OBST * stride + off;
            T cur[MRF_OBST];
#pragma unroll
            for (int c = 0; c < MRF_OBST; ++c) cur[c] = b[c * stride];
            emit(cur, f);
        }
    }
    template <typename F> MRF_HD void each2(F f) const {
        for (int o = 0; o < S; o += 2) {
            const int o1 = o + 1 < S ? o + 1 : o;
            const T* a = obst + (long long)o * MRF_OBST * stride + off;
            const T* b = obst + (long long)o1 * MRF_OBST * stride + off;
            V3<P2<T>> xo{pmk(a[0], b[0]), pmk(a[stride], b[stride]), pmk(a[2 * stride], b[2 * stride])};
            V3<P2<T>> vo{pmk(a[3 * stride], b[3 * stride]), pmk(a[4 * stride], b[4 * stride]), pmk(a[5 * stride], b[5 * stride])};
            V3<P2<T>> ao;
            if (CART) {
                const P2<T> tk2 = psplat(tk);
                xo = V3<P2<T>>{pfma(vo.x, tk2, xo.x), pfma(vo.y, tk2, xo.y), pfma(vo.z, tk2, xo.z)};
                ao = V3<P2<T>>{psplat(T(0)), psplat(T(0)), psplat(T(0))};
            } else {
                ao = V3<P2<T>>{pmk(a[6 * stride], b[6 * stride]), pmk(a[7 * stride], b[7 * stride]), pmk(a[8 * stride], b[8 * stride])};
            }
            f(xo, vo, ao, pmk(a[9 * stride], b[9 * stride]), pmk(T(1), o1 == o ? T(0) : T(1)));
        }
    }
};

// load the parameter block of one record into shared memory
template <typename T, typename L> MRF_HD void load_params(L ld, T* prm, int NT, int tid) {
#pragma unroll
    for (int k = 0; k < 3; ++k) prm[(P_G0 + k) * NT + tid] = ld(MRF_G0 + k);
    prm[P_W0 * NT + tid] = ld(MRF_W0);
#pragma unroll
    for (int k = 0; k < 3; ++k) prm[(P_G1 + k) * NT + tid] = ld(MRF_G1 + k);
    prm[P_W1 * NT + tid] = ld(MRF_W1);
    prm[P_G2 * NT + tid] = ld(MRF_G2);
    prm[P_W2 * NT + tid] = ld(MRF_W2);
#pragma unroll
    for (int k = 0; k < 9; ++k) prm[(P_ANG + k) * NT + tid] = ld(MRF_ANG + k);
    T c0 = ld(MRF_CON), c1 = ld(MRF_CON + 1), c2 = ld(MRF_CON + 2), c3 = ld(MRF_CON + 3);
    T inv = Mth<T>::rsqrt(c0 * c0 + c1 * c1 + c2 * c2);
    prm[(P_NH + 0) * NT + tid] = c0 * inv;
    prm[(P_NH + 1) * NT + tid] = c1 * inv;
    prm[(P_NH + 2) * NT + tid] = c2 * inv;
    prm[P_DN * NT + tid] = c3 * inv;
#pragma unroll
    for (int k = 0; k < 6; ++k) prm[(P_RB + k) * NT + tid] = ld(MRF_RB + k);
}


} // namespace mrf
