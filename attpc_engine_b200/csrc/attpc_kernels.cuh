// Device code of the AT-TPC detector-simulation hot path for B200 (sm_100a).
//
// Stages (one kernel each, all launched on the handle's stream; see DESIGN.md for the data layout):
//   track_plan_*      longest-first launch order of the tracks (expected lifetime), stable four-class partition.
//   track_kernel      Lorentz force + energy loss, Dormand-Prince 5(4) on the reference's 0.1 ns grid: a lane owns a
//                     track (dynamic work cursor), the warp shares the grid points of all accepted steps; fused Fano
//                     electrons, >=1 mask, gain, z -> time bucket (detector/solver.py:19-76, 243-305, 308-347, 386-398).
//   replay_kernel     the same electron/mask/gain/time arithmetic from GIVEN trajectory rows and normals, in the
//                     reference's exact operation order (parity part (a)).
//   point_scan/order  per-event work units, points into (event, rank, arrival) order, sigma_t and the pad-table rows and
//                     columns of the 10x10 mesh of every point (detector/transporter.py:78-120, 217-226, 301).
//   sub_*             longitudinal diffusion only (off by default, not in the reference): every point becomes one
//                     record per time bucket of its window ("sub-points"), which the deposit kernel takes as points.
//   deposit_kernel    persistent CTAs that pull work units, one lane per mesh row: pad lookup, bivariate-normal share,
//                     accumulation per (pad, time bucket) in a shared-memory open-addressing table that is appended to
//                     the event's entry list in dense segments (detector/transporter.py:11-41, 123-249, 252-317; pairing.py:6-28).
//   collect/scan/emit TB wiggle, 0 <= tb < 512 mask, canonical (ascending time bucket, pad) order, CSR compaction
//                     (detector/simulator.py:19-49, 104-115); optional Spyral rows (detector/writer.py:61-112).
//
// Arithmetic that decides a pad id, a time bucket or an integer charge is written with the _rn intrinsics so that
// nvcc cannot contract it into FMAs: it must round exactly like the reference's numpy/numba code.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include <type_traits>

#include "philox.cuh"

#ifndef ATTPC_FIN_THREADS
#define ATTPC_FIN_THREADS 512  // threads of a finalize CTA (one event)
#endif
#ifndef ATTPC_FIN_MIN_CTAS
#define ATTPC_FIN_MIN_CTAS 2   // CTAs per SM the register allocation of order_kernel aims at
#endif
#ifndef ATTPC_FIN_ITEMS
#define ATTPC_FIN_ITEMS 8192   // longest entry list order_kernel orders in shared memory (12 B per entry; two CTAs per SM)
#endif

namespace attpc {

constexpr int MAX_SPECIES = 8;
constexpr int MAX_TRACKS_PER_EVENT = 16;
constexpr int GRID_POINTS = 10001;        // detector/solver.py:16
constexpr double GRID_DT = 1.0e-10;       // s
constexpr double C_LIGHT = 299792458.0;   // detector/constants.py
constexpr double KE_LIMIT = 1.0e-6;       // MeV, detector/solver.py:14
constexpr double Z_HI = 1.0, Z_LO = 0.0, RHO_MAX = 0.292;  // detector/solver.py:160,200,240
constexpr int MESH_N = 10;                // detector/transporter.py:8
constexpr int NUM_TB = 512;               // detector/constants.py:23
constexpr unsigned FULL = 0xFFFFFFFFu;

struct SpeciesDev {
    double mass;     // MeV/c^2
    double qm_c;     // Z e / (m_kg c)  [1/(T s)]
    int32_t z;
    int32_t table;   // offset (in doubles) of this species' deceleration table
    double ke_eq;    // kinetic energy [MeV] of the terminal drift along the field: drag(ke_eq) == q E / m
};

// Scalars every kernel reads; passed by value as a __grid_constant__ parameter.
struct SimParams {
    double length, dv, mm_edge, win_edge, diffusion, efield, fano, ev_per_w;
    double B, E;  // negated fields, detector/solver.py:298-299
    long long gain;
    double grid_low, grid_high;
    int32_t lut_origin, lut_n;
    double adc_threshold;
    double rtol, atol, freeze_ke;
    int32_t lm, e_min, n_oct, n_nodes;
    int32_t n_species, n_pads, n_response, pad0;
    SpeciesDev sp[MAX_SPECIES];
    const int16_t* lut;
    const double* tables;  // [n_species][n_nodes]: dE/dx * MEV_2_JOULE * density * 100 / (m_kg c)  -> d(gamma beta)/dt
    const double* stop_ns; // [n_species][n_nodes]: time [ns] an ion of that energy needs to slow down to the first node
    const double* pad_xy;
    const double* pad_scale;
    const double* response;
    const double* resp_sorted;   // response sorted descending
    const double* resp_prefix;   // prefix sums of resp_sorted, [n_response + 1]
    double resp_max;
    long long e_keep_min;     // smallest electron count whose amplitude min(resp_max * e, 4095) exceeds adc_threshold
    double mesh_w[MESH_N * MESH_N];  // (2 / (9 pi)) exp(-(a_i^2 + a_j^2) / 2), a_i = -3 + 6 i / 9: pdf * step^2 of the mesh
    double mesh_w_unique[MESH_N * MESH_N];  // its distinct values (15 for the symmetric 10 x 10 mesh)
    int32_t n_mesh_w_unique, pad1;
    double long_diffusion;  // V, longitudinal diffusion coefficient (0: off, every point stays in one time bucket)
};

// Active track points (>= 1 electron).  The track kernels append them per event group in arrival order and number
// them inside their (event, rank) list; order_points_kernel then scatters them into (event, rank, arrival) order so
// that the deposit kernel of an event reads one contiguous run per track.
struct PointBuf {
    double* x;
    double* y;
    double* t;          // exact time bucket (float), detector/solver.py:396-398
    long long* q;       // electrons after mpgd_gain
    int32_t* ev;        // event slot inside the launch batch
    int32_t* rank;      // position of the track in `indices`
    uint32_t* j;        // arrival index inside the (event, rank) list
    unsigned* count;    // [n_groups] points appended per group
    unsigned* cnt;      // [launch events * ranks] points per (event, rank)
    unsigned* start;    // [launch events * ranks] first position of the list inside the group's ordered run
    double* geom;       // ordered: GEOM_DOUBLES per point, the per-point constants of the drift mesh (exact path)
    uint32_t* rec;      // ordered: REC_WORDS per point, what the deposit kernel reads (see make_point)
    // work units of the deposit kernel (one CTA each): a slice of <= UNIT_POINTS points of one event
    int32_t* unit_event;   // [max_units] event index inside the group
    int32_t* unit_first;   // [max_units] first point of the slice inside the event's ordered run
    int32_t* unit_count;   // [max_units]
    int32_t* unit_order;   // [max_units] units by decreasing size (longest first)
    int32_t* n_units;      // [n_groups]
    int64_t group_cap;  // points per group
    int32_t group_events;
    int32_t ranks;      // tracks per event
    int32_t max_units;  // capacity of the unit arrays per group
    int32_t unit_points;  // longest slice of one event handled by one CTA of the deposit kernel (<= UNIT_POINTS)
};

// Per-launch counters (one set per in-flight launch; zeroed when the launch starts).
struct Counters {
    unsigned long long track_cursor;
    unsigned long long traj_points, active_points, primary_electrons, deposits, keys, probes, flushes;
    // overflow_sub: the sub-points of longitudinal diffusion did not fit (raised together with overflow_points, which
    // voids the launch; the host then grows the sub-point buffers instead of the point buffers)
    int overflow_points, overflow_hash, overflow_out, replay_miss, overflow_charge, overflow_sub;
    // integrator probes: Dormand-Prince steps tried / rejected, and the most loop passes any one track needed (the
    // serial critical path of a launch)
    unsigned long long rk_steps, rk_rejects, max_track_passes;
};

// Publish a launch's counters and the running CSR totals into mapped host memory.  A copy-engine transfer would
// queue behind the (large) device-to-host copy of the previous launch's rows and stall the compute stream.
__global__ void publish_kernel(const Counters* ctr, const unsigned long long* csr, Counters* host_ctr,
                               unsigned long long* host_csr) {
    *host_ctr = *ctr;
    host_csr[0] = csr[0];
    host_csr[1] = csr[1];
    host_csr[2] = csr[2];
    __threadfence_system();
}

// Running CSR total after a chunk of groups, published for the host so that it can start copying the finished rows.
__global__ void publish_total_kernel(const unsigned long long* csr, unsigned long long* host_slot) {
    host_slot[0] = csr[0];  // cloud rows so far
    host_slot[1] = csr[2];  // Spyral rows so far
    __threadfence_system();
}

struct HashEntry {
    unsigned key1;   // compact key ((time bucket << 15) | pad) + 1, 0 = empty (the Szudzik id is formed on output)
    unsigned rank;   // highest track rank that touched the key (label precedence, transporter.py:247-249)
    unsigned long long charge;
};

// ------------------------------------------------------------------------------------------------ block scans
// Exclusive scan of one value per thread of a CTA of T threads; returns the thread's prefix, `total` for everybody.
// Every thread calls it, and the last read of s_warp [T / 32] must be behind a barrier; one barrier.
template <int T, typename V>
__device__ __forceinline__ V block_scan(V v, V& total, V* s_warp) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    V incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const V t = __shfl_up_sync(FULL, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    V base = incl - v;
    total = 0;
#pragma unroll
    for (int w = 0; w < T / 32; ++w) {
        const V t = s_warp[w];
        if (w < warp) base += t;
        total += t;
    }
    return base;
}

// Exclusive scan of load(0), ..., load(n - 1) on top of `base` in tiles of T values: store(i, base + sum of the values
// before i).  Every thread of the CTA calls it and gets the final sum.  Value i is loaded and stored by one thread.
template <int T, typename V, typename Load, typename Store>
__device__ __forceinline__ V scan_tiles(int n, V base, V* s_warp, Load load, Store store) {
    for (int start = 0; start < n; start += T) {
        const int i = start + (int)threadIdx.x;
        V total;
        __syncthreads();  // (the previous tile is done with s_warp)
        const V before = block_scan<T>(i < n ? load(i) : V(0), total, s_warp);
        if (i < n) store(i, base + before);
        base += total;
    }
    return base;
}

// ----------------------------------------------------------------------------------------------- stopping power
struct TableView {
    const double* t;
    double ke_min, inv_ke_min;
    int32_t hi_min, shift, last;
    double frac_scale;
};

__device__ __forceinline__ TableView make_table_view(const SimParams& P, const double* base) {
    TableView v;
    v.t = base;
    v.shift = 52 - P.lm;
    v.hi_min = (1023 + P.e_min) << P.lm;
    v.last = P.n_nodes - 1;
    v.ke_min = __longlong_as_double((long long)(1023 + P.e_min) << 52);
    v.inv_ke_min = 1.0 / v.ke_min;
    v.frac_scale = __longlong_as_double((long long)(1023 - v.shift) << 52);  // 2^-shift
    return v;
}

// attpc_engine_b200/target.py:DedxTable.__call__ on the pre-scaled table.
__device__ __forceinline__ double table_eval(const TableView& v, double ke) {
    if (!(ke >= v.ke_min)) return ke > 0.0 ? v.t[0] * sqrt(ke * v.inv_ke_min) : 0.0;
    const long long bits = __double_as_longlong(ke);
    const int i = (int)(bits >> v.shift) - v.hi_min;
    if (i >= v.last) return v.t[v.last];
    const double f = (double)(bits & ((1LL << v.shift) - 1)) * v.frac_scale;
    const double lo = v.t[i];
    return fma(f, v.t[i + 1] - lo, lo);
}

// -------------------------------------------------------------------------------------------- equation of motion
struct State {
    double x, y, z, ux, uy, uz;
};

struct TrackConst {
    double mass, qmB, qmE;  // qm_c * B, qm_c * E
    double ke_eq;
    TableView tab;
};

// Can this ion still make an electron?  (Production-only shortcut; the reference integrates a stalled ion to 1 us
// and throws those rows away at detector/solver.py:387.)  A stopped ion relaxes to a drift along the field with
// kinetic energy ke_eq: the transverse motion only decays and, once the ion already moves in the drift direction, the
// parallel motion approaches the drift speed monotonically.  The total variation left in KE is then at most
// KE_perp + |KE_par - ke_eq|; if twice that cannot give one grid step the `budget` = n* W needed for
// int(n + sqrt(F n) z) >= 1 with |z| <= NORMAL_ABS_MAX, every later row has zero electrons.
__device__ __forceinline__ bool inert_forever(double mass, double qmE, double ke_eq, const State& s, double ke,
                                              double budget) {
    if (!(budget > 0.0)) return false;
    if (qmE == 0.0) return ke < budget;  // no field to re-accelerate the ion
    if (!(s.uz * qmE > 0.0)) return false;
    const double k_par = 0.5 * mass * s.uz * s.uz;
    const double k_perp = 0.5 * mass * (s.ux * s.ux + s.uy * s.uy);
    return 2.0 * (k_perp + fabs(k_par - ke_eq)) < budget;
}

__device__ __forceinline__ double kinetic_energy(double mass, double ux, double uy, double uz) {
    const double g2 = ux * ux + uy * uy + uz * uz;
    return mass * g2 / (sqrt(1.0 + g2) + 1.0);  // m (gamma - 1) without the cancellation
}

// detector/solver.py:52-76 with u = gamma*beta:  v = u c / gamma,  du/dt = (q/m (v x B + E) - a u_hat) / c
__device__ __forceinline__ State rhs(const TrackConst& c, const State& s) {
    const double g2 = s.ux * s.ux + s.uy * s.uy + s.uz * s.uz;
    const double gamma = sqrt(1.0 + g2);
    const double ke = c.mass * g2 / (gamma + 1.0);
    const double a = table_eval(c.tab, ke);
    const double c_over_gamma = C_LIGHT / gamma;
    const double drag = g2 > 0.0 ? a * rsqrt(g2) : 0.0;
    State d;
    d.x = s.ux * c_over_gamma;
    d.y = s.uy * c_over_gamma;
    d.z = s.uz * c_over_gamma;
    d.ux = c.qmB * d.y - drag * s.ux;
    d.uy = -c.qmB * d.x - drag * s.uy;
    d.uz = c.qmE - drag * s.uz;
    return d;
}

#define ATTPC_COMBINE(dst, base, h, expr)   \
    dst.x = base.x + (h) * (expr(x));       \
    dst.y = base.y + (h) * (expr(y));       \
    dst.z = base.z + (h) * (expr(z));       \
    dst.ux = base.ux + (h) * (expr(ux));    \
    dst.uy = base.uy + (h) * (expr(uy));    \
    dst.uz = base.uz + (h) * (expr(uz));

// Coefficients of the 4th-order continuous extension of the step (Shampine's interpolant, the one scipy's RK45
// uses): y(t0 + theta h) = y0 + h theta (q0 + theta (q1 + theta (q2 + theta q3))).
struct Dense {
    State q0, q1, q2, q3;
};

// One Dormand-Prince 5(4) step of size h from (y, k1 = f(y)).  Returns the scaled RMS error (<= 1 accepts).
__device__ __forceinline__ double dopri5_step(const TrackConst& c, const State& y, const State& k1, double h,
                                              double rtol, double atol, State& ynew, State& knew, Dense& dense) {
    State t, k2, k3, k4, k5, k6;
#define E2(f) (0.2 * k1.f)
    ATTPC_COMBINE(t, y, h, E2)
    k2 = rhs(c, t);
#define E3(f) (3.0 / 40.0 * k1.f + 9.0 / 40.0 * k2.f)
    ATTPC_COMBINE(t, y, h, E3)
    k3 = rhs(c, t);
#define E4(f) (44.0 / 45.0 * k1.f - 56.0 / 15.0 * k2.f + 32.0 / 9.0 * k3.f)
    ATTPC_COMBINE(t, y, h, E4)
    k4 = rhs(c, t);
#define E5(f) (19372.0 / 6561.0 * k1.f - 25360.0 / 2187.0 * k2.f + 64448.0 / 6561.0 * k3.f - 212.0 / 729.0 * k4.f)
    ATTPC_COMBINE(t, y, h, E5)
    k5 = rhs(c, t);
#define E6(f)                                                                                              \
    (9017.0 / 3168.0 * k1.f - 355.0 / 33.0 * k2.f + 46732.0 / 5247.0 * k3.f + 49.0 / 176.0 * k4.f - \
     5103.0 / 18656.0 * k5.f)
    ATTPC_COMBINE(t, y, h, E6)
    k6 = rhs(c, t);
#define E7(f) \
    (35.0 / 384.0 * k1.f + 500.0 / 1113.0 * k3.f + 125.0 / 192.0 * k4.f - 2187.0 / 6784.0 * k5.f + 11.0 / 84.0 * k6.f)
    ATTPC_COMBINE(ynew, y, h, E7)
    knew = rhs(c, ynew);
#define EE(f)                                                                                                  \
    (71.0 / 57600.0 * k1.f - 71.0 / 16695.0 * k3.f + 71.0 / 1920.0 * k4.f - 17253.0 / 339200.0 * k5.f + \
     22.0 / 525.0 * k6.f - 1.0 / 40.0 * knew.f)
    double acc = 0.0;
#define ERRTERM(f)                                                              \
    {                                                                           \
        const double sc = atol + rtol * fmax(fabs(y.f), fabs(ynew.f));          \
        const double e = h * (EE(f)) / sc;                                      \
        acc += e * e;                                                           \
    }
    ERRTERM(x) ERRTERM(y) ERRTERM(z) ERRTERM(ux) ERRTERM(uy) ERRTERM(uz)
    // dense-output polynomial: q_j = sum_i k_i P[i][j]  (P of scipy/integrate/_ivp/rk.py: RK45.P; row 2 is zero)
#define Q0(f) (k1.f)
#define Q1(f)                                                                                                       \
    (-8048581381.0 / 2820520608.0 * k1.f + 131558114200.0 / 32700410799.0 * k3.f - 1754552775.0 / 470086768.0 * k4.f + \
     127303824393.0 / 49829197408.0 * k5.f - 282668133.0 / 205662961.0 * k6.f + 40617522.0 / 29380423.0 * knew.f)
#define Q2(f)                                                                                                        \
    (8663915743.0 / 2820520608.0 * k1.f - 68118460800.0 / 10900136933.0 * k3.f + 14199869525.0 / 1410260304.0 * k4.f - \
     318862633887.0 / 49829197408.0 * k5.f + 2019193451.0 / 616988883.0 * k6.f - 110615467.0 / 29380423.0 * knew.f)
#define Q3(f)                                                                                                          \
    (-12715105075.0 / 11282082432.0 * k1.f + 87487479700.0 / 32700410799.0 * k3.f - 10690763975.0 / 1880347072.0 * k4.f + \
     701980252875.0 / 199316789632.0 * k5.f - 1453857185.0 / 822651844.0 * k6.f + 69997945.0 / 29380423.0 * knew.f)
#define SETQ(f)           \
    dense.q0.f = Q0(f);   \
    dense.q1.f = Q1(f);   \
    dense.q2.f = Q2(f);   \
    dense.q3.f = Q3(f);
    SETQ(x) SETQ(y) SETQ(z) SETQ(ux) SETQ(uy) SETQ(uz)
#undef Q0
#undef Q1
#undef Q2
#undef Q3
#undef SETQ
#undef E2
#undef E3
#undef E4
#undef E5
#undef E6
#undef E7
#undef EE
#undef ERRTERM
    return sqrt(acc * (1.0 / 6.0));
}

__device__ __forceinline__ State dense_eval(const State& y0, const Dense& d, double h, double theta) {
    State r;
    const double ht = h * theta;
#define DE(f) r.f = fma(ht, fma(theta, fma(theta, fma(theta, d.q3.f, d.q2.f), d.q1.f), d.q0.f), y0.f);
    DE(x) DE(y) DE(z) DE(ux) DE(uy) DE(uz)
#undef DE
    return r;
}

constexpr double MAX_STEP_CELLS = 64.0;  // a step never spans more than 64 grid cells (6.4 ns)

// Standard step-size controller of an order-5 pair: factor = 0.9 err^(-1/5), limited to [0.2, 5].
__device__ __forceinline__ double step_factor(double err) {
    if (!(err > 1e-10)) return 5.0;
    return (double)fminf(5.0f, fmaxf(0.2f, 0.9f * exp2f(-0.2f * log2f((float)err))));  // step control needs no FP64
}

// scipy's event rule (scipy/integrate/_ivp/ivp.py: find_active_events) applied per grid cell, with the
// reference's directions (detector/solver.py:276-283).
__device__ __forceinline__ bool crossed_up(double g0, double g1) { return g0 <= 0.0 && g1 >= 0.0; }
__device__ __forceinline__ bool crossed_down(double g0, double g1) { return g0 >= 0.0 && g1 <= 0.0; }

// Terminal events between two consecutive grid points a -> b.  The radial bound is tested on rho^2 - R^2, which has
// the sign of rho - R; all four tests are evaluated (bitwise or) so that the warp does not diverge on them.
__device__ __forceinline__ bool terminal_event(double ax, double ay, double az, double ke_a, double bx, double by,
                                               double bz, double ke_b) {
    const double ra = ax * ax + ay * ay - RHO_MAX * RHO_MAX, rb = bx * bx + by * by - RHO_MAX * RHO_MAX;
    return crossed_down(ke_a - KE_LIMIT, ke_b - KE_LIMIT) | crossed_up(az - Z_HI, bz - Z_HI) |
           crossed_down(az - Z_LO, bz - Z_LO) | crossed_up(ra, rb);
}

__device__ __forceinline__ unsigned lanemask_lt() {
    unsigned m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

// Append of one active point (replay kernel: one thread per trajectory row).
__device__ __forceinline__ void append_point(const PointBuf& pb, Counters* ctr, bool emit, int ev, int rank,
                                             double x, double y, double t, long long q) {
    if (!emit) return;
    const int g = ev / pb.group_events;
    const unsigned pos = atomicAdd(&pb.count[g], 1u);
    if ((int64_t)pos >= pb.group_cap) {
        ctr->overflow_points = 1;
        return;
    }
    const int64_t i = (int64_t)g * pb.group_cap + pos;
    pb.x[i] = x;
    pb.y[i] = y;
    pb.t[i] = t;
    pb.q[i] = q;
    pb.ev[i] = ev;
    pb.rank[i] = rank;
    pb.j[i] = atomicAdd(&pb.cnt[(int64_t)ev * pb.ranks + rank], 1u);
}

struct TrackBatch {
    const double* momenta;   // [n_events, n_nuclei, 4]
    const double* vertices;  // [n_events, 3]
    int64_t n_events;
    int32_t n_nuclei, n_tracks_per_event;
    int32_t nucleus[MAX_TRACKS_PER_EVENT];
    int32_t species[MAX_TRACKS_PER_EVENT];
    uint64_t seed;
    int64_t first_event;  // global id of event slot 0
    const int32_t* order; // longest-first order of the tracks (track_plan kernels), or null = as they come
    // trajectory recording (attpc_trajectories): one track per "event", rows to rec_points
    const int32_t* rec_species;  // [n_events]
    double* rec_points;          // [n_events, rec_max, 6]
    int32_t* rec_counts;         // [n_events]
    int32_t rec_stride, rec_max;
};

// ---- longest first.  The track kernel is bound by its longest tracks (a stopping light ion takes ten times the
// steps of an exiting one), so the tracks that are expected to live long must start at once, not when a lane happens
// to reach them.  Expected lifetime = min(time to slow down, time to reach the end wall at the initial speed); four
// classes, stable partition (tracks keep their event order inside a class, which keeps the appends of a warp in one
// event group for all but the long classes).
constexpr int PLAN_CLASSES = 4;
constexpr int PLAN_THREADS = 256;

__device__ __forceinline__ int track_class(const SimParams& P, const TrackBatch& tb, int64_t track) {
    const int ev = (int)(track / tb.n_tracks_per_event), rank = (int)(track % tb.n_tracks_per_event);
    const int sp = tb.species[rank];
    if (sp < 0) return PLAN_CLASSES - 1;
    const SpeciesDev& S = P.sp[sp];
    const double* m4 = tb.momenta + ((int64_t)ev * tb.n_nuclei + tb.nucleus[rank]) * 4;
    const double ux = m4[0] / S.mass, uy = m4[1] / S.mass, uz = m4[2] / S.mass;
    const double g2 = ux * ux + uy * uy + uz * uz;
    const double gamma = sqrt(1.0 + g2);
    const double ke = S.mass * g2 / (gamma + 1.0);
    const TableView v = make_table_view(P, P.stop_ns + S.table);
    double life = table_eval(v, ke);                                // ns to slow down
    const double z = tb.vertices[(int64_t)ev * 3 + 2];
    const double vz = uz * C_LIGHT / gamma * 1e-9;                  // m / ns
    if (vz > 0.0) life = fmin(life, (Z_HI - z) / vz);
    if (vz < 0.0) life = fmin(life, (Z_LO - z) / vz);
    return life > 120.0 ? 0 : life > 40.0 ? 1 : life > 12.0 ? 2 : 3;
}

// (1) class of every track, per-CTA class counts
__global__ void __launch_bounds__(PLAN_THREADS)
track_plan_count_kernel(const __grid_constant__ SimParams P, const __grid_constant__ TrackBatch tb, uint8_t* cls,
                        unsigned* cta_counts) {
    __shared__ unsigned s_cnt[PLAN_CLASSES];
    if (threadIdx.x < PLAN_CLASSES) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    const int64_t n_tracks = tb.n_events * tb.n_tracks_per_event;
    const int64_t t = (int64_t)blockIdx.x * PLAN_THREADS + threadIdx.x;
    if (t < n_tracks) {
        const int c = track_class(P, tb, t);
        cls[t] = (uint8_t)c;
        atomicAdd(&s_cnt[c], 1u);
    }
    __syncthreads();
    if (threadIdx.x < PLAN_CLASSES) cta_counts[(int64_t)threadIdx.x * gridDim.x + blockIdx.x] = s_cnt[threadIdx.x];
}

// (2) exclusive scan of the counts, class-major (one CTA)
__global__ void __launch_bounds__(1024) track_plan_scan_kernel(unsigned* cta_counts, int n) {
    __shared__ unsigned s_warp[32];
    scan_tiles<1024>(n, 0u, s_warp, [&](int i) { return cta_counts[i]; },
                     [&](int i, unsigned s) { cta_counts[i] = s; });
}

// (3) stable scatter: position = start of (class, CTA) + tracks of the same class before this one in the CTA
__global__ void __launch_bounds__(PLAN_THREADS)
track_plan_scatter_kernel(const uint8_t* cls, const unsigned* cta_starts, int64_t n_tracks, int32_t* order) {
    __shared__ unsigned s_warp[PLAN_CLASSES][PLAN_THREADS / 32];
    const int64_t t = (int64_t)blockIdx.x * PLAN_THREADS + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c = t < n_tracks ? (int)cls[t] : -1;
    unsigned below = 0;
#pragma unroll
    for (int k = 0; k < PLAN_CLASSES; ++k) {
        const unsigned m = __ballot_sync(FULL, c == k);
        if (c == k) below = __popc(m & ((1u << lane) - 1u));
        if (lane == 0) s_warp[k][warp] = __popc(m);
    }
    __syncthreads();
    if (c >= 0) {
        unsigned idx = cta_starts[(int64_t)c * gridDim.x + blockIdx.x] + below;  // class-major, stable
        for (int w = 0; w < warp; ++w) idx += s_warp[c][w];
        // Spread the long classes (0, 1) over the warps instead of packing them: every S-th position of the order is
        // a long track, the positions between are filled with the others in their order.  A warp full of long tracks
        // would make every one of them pay for the grid points of 31 others at every step.
        const unsigned n_long = cta_starts[(int64_t)2 * gridDim.x];
        const unsigned S = n_long > 0 ? min(32u, (unsigned)(n_tracks / n_long)) : 0u;
        unsigned pos = idx;
        if (S >= 2u) {
            if (idx < n_long) {
                pos = idx * S;
            } else {
                const unsigned k = idx - n_long, block = k / (S - 1u);
                pos = block < n_long ? block * S + k % (S - 1u) + 1u : n_long * S + (k - n_long * (S - 1u));
            }
        }
        order[pos] = (int32_t)t;
    }
}

// Step slot: what the lanes of a warp need to turn one accepted step of ONE track into its 0.1 ns grid points.
// Every warp has 32 slots (one per lane = per track in flight), stored field-major in shared memory
// (field k of slot o at [k * 32 + o]) so that owners write and evaluators read without bank conflicts.
enum {
    SF_Y = 0,     // state at the start of the step (6)
    SF_Q = 6,     // continuous extension q0..q3 (4 x 6)
    SF_YN = 30,   // state at the end of the step (6)
    SF_H = 36, SF_TC = 37, SF_HC = 38,
    SF_PX = 39, SF_PY = 40, SF_PZ = 41, SF_PKE = 42,  // last grid point of the track so far: position and KE
    SF_MASS = 43, SF_QME = 44, SF_KEEQ = 45,
    SF_DOUBLES = 46
};
enum { SI_STEP = 0, SI_EV, SI_RANK, SI_NUC, SI_NOUT, SI_CUT, SI_TRACK, SI_INTS = 8 };
constexpr int TRACK_THREADS = 384;  // at most: 12 warps, one CTA per SM (65536 registers / 384 = 170 per thread)
// + per lane one staged active point (x, y, time, electrons, event, rank, arrival index) waiting for its position
constexpr int STAGE_DOUBLES = 4, STAGE_INTS = 4;
constexpr size_t TRACK_SLOT_BYTES_PER_WARP =
    32 * ((SF_DOUBLES + STAGE_DOUBLES) * sizeof(double) + (SI_INTS + STAGE_INTS) * sizeof(int));

// One lane OWNS one track at a time (and pulls the next from a global cursor when it finishes, so exiting tracks
// do not wait for the stopping tracks of the same warp); the warp SHARES the per-grid-point work.  A pass of the
// warp is
//   A  every owner takes one Dormand-Prince step (error controlled, <= 64 grid cells);
//   B  the grid points inside all accepted steps of the warp are laid out as one flat list and evaluated 32 at a
//      time, whoever owns them: continuous extension, kinetic energy, the four terminal events against the
//      previous grid point, |dKE| / W, the Fano normal, the >= 1 mask, gain, z -> time bucket, and a coalesced
//      append.  Everything a point needs from its neighbour comes from the lane below (or the previous round).
//      The append position comes from one global atomic per round whose result is only consumed a round later
//      (the points wait in shared memory), so its latency is off the critical path.
// The serial critical path of a track is then its number of steps (tens), not its number of grid points (thousands),
// and the per-point code always runs with full warps.
template <bool TAB_SMEM, bool RECORD>
__global__ void __launch_bounds__(TRACK_THREADS, 1)
track_kernel(const __grid_constant__ SimParams P, const __grid_constant__ TrackBatch tb, PointBuf pb, Counters* ctr) {
    extern __shared__ __align__(16) double s_dyn[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    double* sf = s_dyn + (size_t)warp * (SF_DOUBLES + STAGE_DOUBLES) * 32;
    double* stage_d = sf + SF_DOUBLES * 32;  // [STAGE_DOUBLES][32]
    int* si = reinterpret_cast<int*>(s_dyn + (size_t)n_warps * (SF_DOUBLES + STAGE_DOUBLES) * 32) +
              warp * (SI_INTS + STAGE_INTS) * 32;
    int* stage_i = si + SI_INTS * 32;        // [STAGE_INTS][32]
    double* s_tab = s_dyn + (size_t)n_warps * ((SF_DOUBLES + STAGE_DOUBLES) * 32 + (SI_INTS + STAGE_INTS) * 32 / 2);
    if (TAB_SMEM) {
        const int n = P.n_species * P.n_nodes;
        for (int i = threadIdx.x; i < n; i += blockDim.x) s_tab[i] = P.tables[i];
        __syncthreads();
    }
    const double* tab_base = TAB_SMEM ? s_tab : P.tables;
    const int64_t n_tracks = tb.n_events * tb.n_tracks_per_event;
    const unsigned lanes_below = lanemask_lt();

    bool have = false, done = false;
    TrackConst c;
    State y, k;                  // integrator state at time tc and its derivative
    State yn, kn;                // end state of the accepted step whose grid points are being emitted
    double gx = 0.0, gy = 0.0, gz = 0.0, ke = 0.0;  // position and kinetic energy at the last grid point
    double h = 0.0, err = 0.0, t_end = 0.0;
    int pending = 0;             // grid points inside the accepted step
    int n_out = 0;               // active points this track has produced so far
    double tc = 0.0, hc = 1.0;   // time and step size in units of grid cells (0.1 ns)
    int step = 0, ev = 0, rank = 0, nucleus = 0;
    int64_t track = 0;
    unsigned long long n_traj = 0, n_active = 0, n_prim = 0;
    unsigned n_steps = 0, n_rejects = 0, passes = 0, max_passes = 0;
    // Points staged by the previous round (warp-uniform mask of the lanes that hold one) and the still pending result
    // of the atomic that reserved their positions: in the leader's register (one atomic for the warp, leader >= 0)
    // or in every lane's own (tracks of several event groups in one round, leader < 0).
    unsigned staged_mask = 0, staged_first = 0, staged_prefix = 0, staged_peers = 0;
    int staged_leader = 0;
    auto store_staged = [&]() {  // whole warp; the first read of staged_first waits for the atomic issued a round ago
        if (staged_mask == 0u) return;
        unsigned pos = 0;
        if (staged_leader >= 0) {
            pos = __shfl_sync(FULL, staged_first, staged_leader) + staged_prefix;
        } else if ((staged_mask >> lane) & 1u) {  // one atomic per event group: its result sits in the group's first lane
            pos = __shfl_sync(staged_peers, staged_first, __ffs(staged_peers) - 1) + staged_prefix;
        }
        if ((staged_mask >> lane) & 1u) {
            const int gi = stage_i[0 * 32 + lane] / pb.group_events;
            if ((int64_t)pos >= pb.group_cap) {
                ctr->overflow_points = 1;
            } else {
                const int64_t i = (int64_t)gi * pb.group_cap + pos;
                pb.x[i] = stage_d[0 * 32 + lane];
                pb.y[i] = stage_d[1 * 32 + lane];
                pb.t[i] = stage_d[2 * 32 + lane];
                pb.q[i] = __double_as_longlong(stage_d[3 * 32 + lane]);
                pb.ev[i] = stage_i[0 * 32 + lane];
                pb.rank[i] = stage_i[1 * 32 + lane];
                pb.j[i] = (unsigned)stage_i[2 * 32 + lane];
            }
        }
        staged_mask = 0u;
    };

    while (true) {
        if (!have && !done) {
            track = (int64_t)atomicAdd(&ctr->track_cursor, 1ULL);
            if (track >= n_tracks) {
                done = true;
            } else {
                if (!RECORD && tb.order) track = tb.order[track];
                ev = (int)(track / tb.n_tracks_per_event);
                rank = (int)(track % tb.n_tracks_per_event);
                const int sp = RECORD ? tb.rec_species[track] : tb.species[rank];
                nucleus = RECORD ? 0 : tb.nucleus[rank];
                if (sp >= 0) {
                    const SpeciesDev& S = P.sp[sp];
                    const double* m4 = tb.momenta + ((int64_t)ev * tb.n_nuclei + nucleus) * 4;
                    const double* vx = tb.vertices + (int64_t)ev * 3;
                    c.mass = S.mass;
                    c.qmB = S.qm_c * P.B;
                    c.qmE = S.qm_c * P.E;
                    c.ke_eq = S.ke_eq;
                    c.tab = make_table_view(P, tab_base + S.table);
                    y.x = vx[0];
                    y.y = vx[1];
                    y.z = vx[2];
                    y.ux = m4[0] / S.mass;  // detector/solver.py:270-273
                    y.uy = m4[1] / S.mass;
                    y.uz = m4[2] / S.mass;
                    k = rhs(c, y);
                    gx = y.x;
                    gy = y.y;
                    gz = y.z;
                    ke = kinetic_energy(c.mass, y.ux, y.uy, y.uz);
                    step = 0;
                    tc = 0.0;
                    hc = 1.0;
                    pending = 0;
                    n_out = 0;
                    passes = 0;
                    have = true;
                    n_traj += 1;  // grid point 0 (never active: detector/solver.py:338-339)
                    if (RECORD && tb.rec_max > 0) {
                        double* o = tb.rec_points + (int64_t)track * tb.rec_max * 6;
                        o[0] = y.x; o[1] = y.y; o[2] = y.z; o[3] = y.ux; o[4] = y.uy; o[5] = y.uz;
                    }
                } else if (RECORD) {
                    tb.rec_counts[track] = 0;
                }
            }
        }
        if (__all_sync(FULL, done)) break;

        // ---- phase A: every owner tries one Dormand-Prince step of hc grid cells from tc
        passes += have;
        if (have) {
            Dense dense;
            h = hc * GRID_DT;
            err = dopri5_step(c, y, k, h, P.rtol, P.atol, yn, kn, dense);
            n_steps += 1;
            if (!(err <= 1.0) && hc > 1.0 / 4096.0) {  // reject: retry with a smaller step
                n_rejects += 1;
                hc *= (err == err) ? fmin(0.9, step_factor(err)) : 0.2;
            } else {
                t_end = tc + hc;
                pending = max(0, (int)floor(t_end + 1e-9) - step);  // grid points inside (tc, tc + hc]
                if (pending == 0) {  // step ends before the next grid point: just advance
                    tc = t_end;
                    y = yn;
                    k = kn;
                    hc = fmin(MAX_STEP_CELLS, hc * step_factor(err));
                } else {  // hand the step to the warp
#define PUT(field, value) sf[(field) * 32 + lane] = (value)
                    PUT(SF_Y + 0, y.x); PUT(SF_Y + 1, y.y); PUT(SF_Y + 2, y.z);
                    PUT(SF_Y + 3, y.ux); PUT(SF_Y + 4, y.uy); PUT(SF_Y + 5, y.uz);
#define PUTQ(n, q) \
    PUT(SF_Q + 6 * n + 0, q.x); PUT(SF_Q + 6 * n + 1, q.y); PUT(SF_Q + 6 * n + 2, q.z); \
    PUT(SF_Q + 6 * n + 3, q.ux); PUT(SF_Q + 6 * n + 4, q.uy); PUT(SF_Q + 6 * n + 5, q.uz);
                    PUTQ(0, dense.q0) PUTQ(1, dense.q1) PUTQ(2, dense.q2) PUTQ(3, dense.q3)
#undef PUTQ
                    PUT(SF_YN + 0, yn.x); PUT(SF_YN + 1, yn.y); PUT(SF_YN + 2, yn.z);
                    PUT(SF_YN + 3, yn.ux); PUT(SF_YN + 4, yn.uy); PUT(SF_YN + 5, yn.uz);
                    PUT(SF_H, h); PUT(SF_TC, tc); PUT(SF_HC, hc);
                    PUT(SF_PX, gx); PUT(SF_PY, gy); PUT(SF_PZ, gz); PUT(SF_PKE, ke);
                    PUT(SF_MASS, c.mass); PUT(SF_QME, c.qmE); PUT(SF_KEEQ, c.ke_eq);
#undef PUT
                    si[SI_STEP * 32 + lane] = step;
                    si[SI_EV * 32 + lane] = ev;
                    si[SI_RANK * 32 + lane] = rank;
                    si[SI_NUC * 32 + lane] = nucleus;
                    si[SI_NOUT * 32 + lane] = n_out;
                    si[SI_CUT * 32 + lane] = INT_MAX;
                    si[SI_TRACK * 32 + lane] = (int)track;
                }
            }
        }
        // ---- phase B: the grid points of all accepted steps of the warp, 32 at a time
        const bool emitting = have && pending > 0;
        const int mine = emitting ? pending : 0;
        int incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl += v;
        }
        const int excl = incl - mine;
        const int total = __shfl_sync(FULL, incl, 31);
        if (total == 0) continue;  // warp-uniform
        __syncwarp();
        double carry_x = 0.0, carry_y = 0.0, carry_z = 0.0, carry_ke = 0.0;  // lane 31 of the previous round
        for (int base = 0; base < total; base += 32) {
            const int f = base + lane;
            const bool valid = f < total;
            int o = 0;  // owner of flat point f: the number of lanes whose inclusive count is <= f
#pragma unroll
            for (int s = 16; s > 0; s >>= 1) {
                const int v = __shfl_sync(FULL, incl, o + s - 1);
                if (v <= f) o += s;
            }
            const int j = f - __shfl_sync(FULL, excl, o);  // position inside the owner's step
#define GET(field) sf[(field) * 32 + o]
            const int s_idx = si[SI_STEP * 32 + o] + 1 + j;  // grid step of this point
            const double hc_o = GET(SF_HC);
            const double theta = fmin(1.0, ((double)s_idx - GET(SF_TC)) / hc_o);
            State g;
            if (theta >= 1.0) {
                g.x = GET(SF_YN + 0); g.y = GET(SF_YN + 1); g.z = GET(SF_YN + 2);
                g.ux = GET(SF_YN + 3); g.uy = GET(SF_YN + 4); g.uz = GET(SF_YN + 5);
            } else {
                const double ht = GET(SF_H) * theta;
#define DE(f, i) \
    g.f = fma(ht, fma(theta, fma(theta, fma(theta, GET(SF_Q + 18 + i), GET(SF_Q + 12 + i)), GET(SF_Q + 6 + i)), GET(SF_Q + i)), GET(SF_Y + i));
                DE(x, 0) DE(y, 1) DE(z, 2) DE(ux, 3) DE(uy, 4) DE(uz, 5)
#undef DE
            }
            const double mass = GET(SF_MASS);
            const double ke_g = kinetic_energy(mass, g.ux, g.uy, g.uz);
            // the previous grid point of the same track: the lane below, the last lane of the previous round, or
            // (first point of the step) what the owner left in the slot
            double px = __shfl_up_sync(FULL, g.x, 1), py = __shfl_up_sync(FULL, g.y, 1);
            double pz = __shfl_up_sync(FULL, g.z, 1), pke = __shfl_up_sync(FULL, ke_g, 1);
            if (lane == 0) {
                px = carry_x; py = carry_y; pz = carry_z; pke = carry_ke;
            }
            if (j == 0) {
                px = GET(SF_PX); py = GET(SF_PY); pz = GET(SF_PZ); pke = GET(SF_PKE);
            }
            // the track ends BEFORE this point (terminal event in the cell) or AFTER it (time limit, inert ion)
            const bool term = valid && terminal_event(px, py, pz, pke, g.x, g.y, g.z, ke_g);
            const bool after = valid && !term &&
                               (s_idx >= GRID_POINTS - 1 ||
                                inert_forever(mass, GET(SF_QME), GET(SF_KEEQ), g, ke_g, P.freeze_ke));
            if (term | after) atomicMin(&si[SI_CUT * 32 + o], term ? j : j + 1);
            __syncwarp();
            const bool live = valid && j < si[SI_CUT * 32 + o];  // a row of the trajectory
            const int ev_o = si[SI_EV * 32 + o];
            bool emit = false;
            long long n_e = 0;
            if (RECORD) {
                if (live && s_idx % tb.rec_stride == 0 && s_idx / tb.rec_stride < tb.rec_max) {
                    double* r = tb.rec_points + ((int64_t)si[SI_TRACK * 32 + o] * tb.rec_max + s_idx / tb.rec_stride) * 6;
                    r[0] = g.x; r[1] = g.y; r[2] = g.z; r[3] = g.ux; r[4] = g.uy; r[5] = g.uz;
                }
            } else if (live) {
                // detector/solver.py:338-346: mean = |dKE| / W, Gaussian with variance F * mean, truncation
                const double mean = fabs(ke_g - pke) * P.ev_per_w;
                const double spread = sqrt(P.fano * mean);
                if (mean + spread * NORMAL_ABS_MAX >= 1.0) {
                    const double zn = philox_normal(tb.seed, (uint64_t)(tb.first_event + ev_o),
                                                    (uint32_t)si[SI_NUC * 32 + o], (uint32_t)s_idx);
                    n_e = (long long)(mean + spread * zn);
                    emit = n_e >= 1;  // detector/solver.py:387
                }
            }
            n_traj += live;
            const unsigned emit_mask = __ballot_sync(FULL, emit);
            // arrival index inside the track: emitted points of the same owner below this lane
            const int seg_start = max(0, lane - j);
            const int before = __popc(emit_mask & lanes_below & ~((1u << seg_start) - 1u));
            const int n_out_o = si[SI_NOUT * 32 + o];
            const int o_next = __shfl_down_sync(FULL, o, 1);
            const int live_next = __shfl_down_sync(FULL, (int)live, 1);
            const bool same_next = lane < 31 && f + 1 < total && o_next == o;
            __syncwarp();  // every read of this round's slot fields is done
            if (valid && !same_next) si[SI_NOUT * 32 + o] = n_out_o + before + (int)emit;
            if (live && !(same_next && live_next)) {  // the last row so far of this track
                sf[SF_PX * 32 + o] = g.x;
                sf[SF_PY * 32 + o] = g.y;
                sf[SF_PZ * 32 + o] = g.z;
                sf[SF_PKE * 32 + o] = ke_g;
            }
#undef GET
            store_staged();  // the points of the previous round: their positions have arrived by now
            if (emit_mask) {  // warp-uniform: one atomic on the group counter per round (tracks of a warp almost
                              // always belong to the same event group); the lanes keep their points in shared
                              // memory until the next round
                const int gi = emit ? ev_o / pb.group_events : -1;
                const int leader = __ffs(emit_mask) - 1;
                const int g0 = __shfl_sync(FULL, gi, leader);
                const bool uniform = __all_sync(FULL, !emit || gi == g0);
                staged_mask = emit_mask;
                staged_leader = uniform ? leader : -1;
                staged_prefix = (unsigned)__popc(emit_mask & lanes_below);
                if (uniform) {
                    if (lane == leader) staged_first = atomicAdd(&pb.count[g0], (unsigned)__popc(emit_mask));
                } else {  // tracks of several event groups (the long tracks run first, whatever their event):
                          // one atomic per group present in the round
                    staged_peers = __match_any_sync(FULL, gi) & emit_mask;
                    if (emit) {
                        staged_prefix = (unsigned)__popc(staged_peers & lanes_below);
                        if (lane == __ffs(staged_peers) - 1)
                            staged_first = atomicAdd(&pb.count[gi], (unsigned)__popc(staged_peers));
                    }
                }
                if (emit) {
                    stage_d[0 * 32 + lane] = g.x;
                    stage_d[1 * 32 + lane] = g.y;
                    stage_d[2 * 32 + lane] = (P.length - g.z) / P.dv + P.mm_edge;  // detector/solver.py:396-398
                    stage_d[3 * 32 + lane] = __longlong_as_double(n_e * P.gain);     // detector/solver.py:392
                    stage_i[0 * 32 + lane] = ev_o;
                    stage_i[1 * 32 + lane] = si[SI_RANK * 32 + o];
                    stage_i[2 * 32 + lane] = n_out_o + before;
                    n_active += 1;
                    n_prim += (unsigned long long)n_e;
                }
            }
            carry_x = __shfl_sync(FULL, g.x, 31);
            carry_y = __shfl_sync(FULL, g.y, 31);
            carry_z = __shfl_sync(FULL, g.z, 31);
            carry_ke = __shfl_sync(FULL, ke_g, 31);
            __syncwarp();  // the slot updates of this round are visible to the first reads of the next
        }
        __syncwarp();
        if (emitting) {  // owners take their tracks back
            const int cut = si[SI_CUT * 32 + lane];
            const bool finished = cut <= pending;
            step += min(pending, cut);
            n_out = si[SI_NOUT * 32 + lane];
            gx = sf[SF_PX * 32 + lane];
            gy = sf[SF_PY * 32 + lane];
            gz = sf[SF_PZ * 32 + lane];
            ke = sf[SF_PKE * 32 + lane];
            pending = 0;
            if (!finished) {  // all grid points of the step are out: advance the integrator
                tc = t_end;
                y = yn;
                k = kn;
                hc = fmin(MAX_STEP_CELLS, hc * step_factor(err));
            } else {
                have = false;
                max_passes = max(max_passes, passes);
                if (RECORD) tb.rec_counts[track] = step + 1;
                else pb.cnt[(int64_t)ev * pb.ranks + rank] = (unsigned)n_out;  // length of this track's list
            }
        }
        __syncwarp();
    }
    store_staged();
    // per-warp statistics
    for (int o = 16; o > 0; o >>= 1) {
        n_traj += __shfl_xor_sync(FULL, n_traj, o);
        n_active += __shfl_xor_sync(FULL, n_active, o);
        n_prim += __shfl_xor_sync(FULL, n_prim, o);
    }
    n_steps = __reduce_add_sync(FULL, n_steps);
    n_rejects = __reduce_add_sync(FULL, n_rejects);
    max_passes = __reduce_max_sync(FULL, max_passes);
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&ctr->traj_points, n_traj);
        atomicAdd(&ctr->active_points, n_active);
        atomicAdd(&ctr->primary_electrons, n_prim);
        atomicAdd(&ctr->rk_steps, (unsigned long long)n_steps);
        atomicAdd(&ctr->rk_rejects, (unsigned long long)n_rejects);
        atomicMax(&ctr->max_track_passes, (unsigned long long)max_passes);
    }
}

// --------------------------------------------------------------------------------------------------- replay
struct ReplayBatch {
    const int64_t* track_offsets;  // [n_tracks + 1]
    const double* rows;            // [n_rows, 6]
    const double* normals;         // [n_rows]
    const int32_t* track_event;
    const int32_t* track_rank;
    const int32_t* track_species;
    int64_t n_tracks, n_rows;
    long long* electrons_out;      // may be null
};

// detector/solver.py:332-335 in numpy's operation order (norm = sqrt((a*a + b*b) + c*c)).
__device__ __forceinline__ double reference_ke(const double* r, double mass) {
    const double gv =
        __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(r[3], r[3]), __dmul_rn(r[4], r[4])), __dmul_rn(r[5], r[5])));
    const double g2 = __dmul_rn(gv, gv);
    const double beta = __dsqrt_rn(__ddiv_rn(g2, __dadd_rn(1.0, g2)));
    const double gamma = __ddiv_rn(gv, beta);
    return __dmul_rn(mass, __dsub_rn(gamma, 1.0));
}

__global__ void __launch_bounds__(256)
replay_kernel(const __grid_constant__ SimParams P, ReplayBatch rb, PointBuf pb, Counters* ctr) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rb.n_rows) return;
    // locate the track of row r
    int64_t lo = 0, hi = rb.n_tracks;
    while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (rb.track_offsets[mid] <= r) lo = mid; else hi = mid;
    }
    const int64_t t = lo;
    const int sp = rb.track_species[t];
    long long n_e = 0;
    if (sp >= 0) {
        const double mass = P.sp[sp].mass;
        double mean = 0.0;  // row 0 of a track: electrons[0] = 0 (detector/solver.py:338-339)
        if (r > rb.track_offsets[t]) {
            const double ke1 = reference_ke(rb.rows + r * 6, mass);
            const double ke0 = reference_ke(rb.rows + (r - 1) * 6, mass);
            mean = __dmul_rn(fabs(__dsub_rn(ke1, ke0)), P.ev_per_w);
        }
        // rng.normal(mean, sqrt(F mean)) == mean + sqrt(F mean) * standard_normal  (numpy legacy-free Generator)
        const double draw = __dadd_rn(mean, __dmul_rn(__dsqrt_rn(__dmul_rn(P.fano, mean)), rb.normals[r]));
        n_e = (long long)draw;  // C truncation, like ndarray.astype(int64)
        atomicAdd(&ctr->traj_points, 1ULL);
    }
    if (rb.electrons_out) rb.electrons_out[r] = n_e;
    if (n_e >= 1) {
        const double* row = rb.rows + r * 6;
        const double time = __dadd_rn(__ddiv_rn(__dsub_rn(P.length, row[2]), P.dv), P.mm_edge);
        append_point(pb, ctr, true, rb.track_event[t], rb.track_rank[t], row[0], row[1], time, n_e * P.gain);
        atomicAdd(&ctr->active_points, 1ULL);
        atomicAdd(&ctr->primary_electrons, (unsigned long long)n_e);
    }
}

// ----------------------------------------------------------------------------------------------- pad lookup
// detector/transporter.py:78-120 then pad_grid[ix, iy] and the beam-pad veto (:165, :237), all folded into the
// 1 mm lookup table built by the host (engine.build_pad_lut).  Returns -1 for "no deposit".
__device__ __forceinline__ int lookup_pad(const SimParams& P, double x_m, double y_m) {
    const double fx = floor(__dmul_rn(x_m, 1000.0));
    const double fy = floor(__dmul_rn(y_m, 1000.0));
    if (fx >= P.grid_high || fy >= P.grid_high) return -1;
    if (fx < P.grid_low || fy < P.grid_low) return -1;
    if (!(fx == fx) || !(fy == fy)) return -1;  // NaN positions never index the table
    const int ix = (int)fx - P.lut_origin, iy = (int)fy - P.lut_origin;
    if ((unsigned)ix >= (unsigned)P.lut_n || (unsigned)iy >= (unsigned)P.lut_n) return -1;
    return (int)__ldg(P.lut + (int64_t)ix * P.lut_n + iy);
}

__global__ void lookup_kernel(const __grid_constant__ SimParams P, const double* xy, int64_t n, int32_t* out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = lookup_pad(P, xy[2 * i], xy[2 * i + 1]);
}

// detector/pairing.py:6-28
__device__ __forceinline__ unsigned szudzik_pair(unsigned tb, unsigned pad) {
    return tb >= pad ? tb * tb + tb + pad : pad * pad + tb;
}

// detector/pairing.py:31-55 in integers
__device__ __forceinline__ void szudzik_unpair(unsigned key, unsigned& tb, unsigned& pad) {
    unsigned s = (unsigned)sqrt((double)key);
    while (s * s > key) --s;
    while ((s + 1) * (s + 1) <= key) ++s;
    const unsigned rem = key - s * s;
    if (rem < s) {
        tb = rem;
        pad = s;
    } else {
        tb = s;
        pad = rem - s;
    }
}

// ------------------------------------------------------------------------------------------------- accumulate
// points[id] = (charge + q, label) of detector/transporter.py:166-169, 247-249: integer adds commute and the label
// is "last track in indices order", i.e. the maximum rank, so the result does not depend on thread order.
struct GroupView {
    int32_t first_slot;   // first event slot of the group inside the launch batch
    int32_t n_events;     // events in this group
    int32_t group;        // group index (selects the PointBuf region)
    int32_t hash_cap;     // entries per event region (power of two)
    HashEntry* tables;    // [chunk events][hash_cap]: entry list of every event
    unsigned* n_entries;  // [launch events] entries of the list (zeroed before the deposit kernel)
    unsigned* mode;       // [launch events] 0 = every key once, 1 = a key may appear several times (the event was
                          // deposited in several segments: dense event, or split over several units)
    int32_t exact_mesh;   // ATTPC_EXACT_MESH: every pixel through the reference's own expression (validation)
    int32_t group_events; // events per full group
    int32_t chunk_e0;     // first event of the group inside the chunk (row of `tables` and of the sort scratch)
    int32_t spill_keys;   // keys in a CTA's shared-memory table that trigger a segment append (<= SMEM_SPILL_AT)
};

// The host describes a CHUNK of consecutive groups (first_slot / group / n_events of the whole chunk) and launches
// every group kernel once per chunk with one grid row (or, for point_scan_kernel, one CTA) per group.
__device__ __forceinline__ GroupView sub_group(GroupView gv, int dy) {
    const int skip = dy * gv.group_events;
    gv.group += dy;
    gv.first_slot += skip;
    gv.n_events = max(0, min(gv.group_events, gv.n_events - skip));
    gv.chunk_e0 = skip;
    return gv;
}

// ------------------------------------------------------------------------------------------- ordering of points
constexpr int UNIT_POINTS = 1024;   // longest slice of one event handled by one CTA of the deposit kernel
constexpr int MAX_UNITS_SORT = 8192;
constexpr int GEOM_DOUBLES = 12;

// Per group, single CTA: (1) exclusive scan of the (event, rank) list lengths -> start of every list in the group's
// ordered run; (2) split every event into work units of <= UNIT_POINTS points; (3) order the units by decreasing
// size so that the longest start first (the per-event cost varies by 100x between a short recoil and a stopped ion).
__global__ void __launch_bounds__(1024) point_scan_kernel(PointBuf pb, GroupView chunk, const Counters* ctr) {
    const GroupView gv = sub_group(chunk, blockIdx.x);
    __shared__ unsigned s_warp[32];
    __shared__ uint32_t s_sort[MAX_UNITS_SORT];
    const int tid = threadIdx.x;
    if (ctr->overflow_points) {  // the point lists are incomplete: the host will redo the launch with bigger buffers
        if (tid == 0) pb.n_units[gv.group] = 0;
        return;
    }
    const int n = gv.n_events * pb.ranks;
    const int64_t first = (int64_t)gv.first_slot * pb.ranks;
    int32_t* u_event = pb.unit_event + (int64_t)gv.group * pb.max_units;
    int32_t* u_first = pb.unit_first + (int64_t)gv.group * pb.max_units;
    int32_t* u_count = pb.unit_count + (int64_t)gv.group * pb.max_units;
    int32_t* u_order = pb.unit_order + (int64_t)gv.group * pb.max_units;
    scan_tiles<1024>(n, 0u, s_warp, [&](int i) { return pb.cnt[first + i]; },
                     [&](int i, unsigned s) { pb.start[first + i] = s; });
    // units: event e has ceil(points / UNIT_POINTS) of them (at least one, so that empty events still get their
    // zero-length entry list written)
    const unsigned up = (unsigned)pb.unit_points;
    unsigned pts = 0, nu = 0;  // of the thread's event: scan_tiles loads and stores it on the same thread
    const unsigned n_units = scan_tiles<1024>(
        gv.n_events, 0u, s_warp,
        [&](int e) {
            pts = 0;
            for (int r = 0; r < pb.ranks; ++r) pts += pb.cnt[first + (int64_t)e * pb.ranks + r];
            nu = max(1u, (pts + up - 1u) / up);
            return nu;
        },
        [&](int e, unsigned u0) {
            gv.mode[gv.first_slot + e] = nu > 1 ? 1u : 0u;  // several units: a key may be listed once per unit
            for (unsigned k = 0; k < nu; ++k) {
                const unsigned u = u0 + k;
                if (u < (unsigned)pb.max_units) {
                    u_event[u] = e;
                    u_first[u] = (int32_t)(k * up);
                    u_count[u] = (int32_t)min(up, pts - min(pts, k * up));
                }
            }
        });
    __syncthreads();  // (the sort reads the unit counts of every thread)
    const int total = min((int)n_units, pb.max_units);
    if (tid == 0) pb.n_units[gv.group] = total;
    // longest first: bitonic sort of (UNIT_POINTS - count) << 16 | unit ... only when it fits the sort buffer
    if (total <= MAX_UNITS_SORT) {
        int n2 = 1;
        while (n2 < total) n2 <<= 1;
        for (int i = tid; i < n2; i += 1024)
            s_sort[i] = i < total ? ((uint32_t)(UNIT_POINTS - u_count[i]) << 16) | (uint32_t)i : 0xFFFFFFFFu;
        __syncthreads();
        for (int k = 2; k <= n2; k <<= 1)
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int i = tid; i < n2; i += 1024) {
                    const int l = i ^ j;
                    if (l > i) {
                        const uint32_t a = s_sort[i], b = s_sort[l];
                        if ((a > b) == ((i & k) == 0)) {
                            s_sort[i] = b;
                            s_sort[l] = a;
                        }
                    }
                }
                __syncthreads();
            }
        for (int i = tid; i < total; i += 1024) u_order[i] = (int32_t)(s_sort[i] & 0xFFFFu);
    } else {
        for (int i = tid; i < total; i += 1024) u_order[i] = i;
    }
}

// ------------------------------------------------------------------------------------------------- drift geometry
// Per-point constants of detector/transporter.py:172-249, in the reference's operation order.
// geom[] = cx, cy, lo_x, hi_x, dx, lo_y, hi_y, dy, sigma, guard, qd, (unused)
//
// `guard` bounds the relative distance between the reference's floating-point value of
//     pdf * (step_x * step_y) * electrons                      (detector/transporter.py:240-246)
// and the exact-arithmetic value  (2 / (9 pi)) exp(-(a_i^2 + a_j^2) / 2) * electrons,  a_i = -3 + 6 i / 9,  which does
// not depend on sigma or on the mesh centre.  Error budget in units of u = 2^-53, with M = max(|cx|, |cy|) + 3 sigma
// the largest magnitude that is rounded while the pixel coordinates are formed:
//   * pixel - centre: numba's linspace rounds lo, hi, (hi - lo) / 9, i * d and lo + i * d: |err| <= (4 M + 21 sigma) u
//   * exponent (-1 / 2 / sigma^2) * (dx^2 + dy^2): |err| <= 6 (4 M + 21 sigma) u / sigma + 54 u   (|exponent| <= 9)
//   * c1, exp (<= 1 ulp), the two products, the constant table: < 40 u
// => relative error <= (24 M / sigma + 220) u.  The deposit kernel uses the table whenever the product is further
// than twice that bound from an integer (so the truncation of transporter.py:240 cannot differ) and evaluates the
// reference's own expression otherwise.
constexpr double MESH_GUARD_U = 1.1102230246251565e-16;  // 2^-53

// detector/transporter.py:102-120 on one coordinate: floor(mm), range test, row / column of the 1 mm pad table
__device__ __forceinline__ int lut_index(const SimParams& P, double coord_m) {
    const double f = floor(__dmul_rn(coord_m, 1000.0));
    if (!(f < P.grid_high) || !(f >= P.grid_low)) return -1;  // also NaN
    const int idx = (int)f - P.lut_origin;
    return (unsigned)idx < (unsigned)P.lut_n ? idx : -1;
}

// Record of one ordered point as the deposit kernel reads it (64 B):
//   word 0      time bucket | careful << 29 | kind << 30   (kind 0: nothing, 1: single deposit, 2: 10x10 mesh;
//               careful: some pixel's share is so close to an integer that the table weight might round it differently
//               from the reference's expression -- the deposit kernel then tests every pixel of the point)
//   word 1      guard as float, rounded up
//   words 2-3   electrons after gain as double
//   words 4-8   int16 iy[10]: pad-table column of mesh column j (-1 = outside), kind 1: iy[0] of the point itself
//   words 9-13  int16 ix[10]: pad-table row of mesh row i
//   word 14     rank of the track (position in `indices`)
constexpr int REC_WORDS = 16;

// `tb` is the time bucket of the record: (int)time (detector/transporter.py:165, 238), or one bucket of the
// longitudinal window of the point (sub_point_kernel); `q` its electrons.
__device__ __forceinline__ void make_point(const SimParams& P, double cx, double cy, double time, int tb, long long q,
                                           bool exact_mesh, double* g, uint32_t* rec) {
    g[0] = cx;
    g[1] = cy;
    g[10] = (double)q;
#pragma unroll
    for (int k = 0; k < REC_WORDS; ++k) rec[k] = 0u;
    rec[2] = (uint32_t)__double2loint(g[10]);
    rec[3] = (uint32_t)__double2hiint(g[10]);
    // detector/transporter.py:301, evaluated left to right
    const double sigma = __dsqrt_rn(__ddiv_rn(__dmul_rn(__dmul_rn(__dmul_rn(2.0, P.diffusion), P.dv), time), P.efield));
    if (tb < 0 || tb >= 8192 || !(sigma == sigma)) return;  // kind 0: never reached for 0 <= z <= length + mm_edge*dv (tb <= windows_edge)
    if (sigma == 0.0) {  // kind 1: single deposit, transporter.py:123-169
        rec[0] = (uint32_t)tb | (1u << 30);
        rec[4] = (uint32_t)(uint16_t)(int16_t)lut_index(P, cy);
        rec[9] = (uint32_t)(uint16_t)(int16_t)lut_index(P, cx);
        return;
    }
    // detector/transporter.py:217-226 with numba's linspace (numba/np/arrayobj.py: linspace)
    const double three_sigma = __dmul_rn(3.0, sigma);
    g[2] = __dsub_rn(cx, three_sigma);
    g[3] = __dadd_rn(cx, three_sigma);
    g[4] = __ddiv_rn(__dsub_rn(g[3], g[2]), (double)(MESH_N - 1));
    g[5] = __dsub_rn(cy, three_sigma);
    g[6] = __dadd_rn(cy, three_sigma);
    g[7] = __ddiv_rn(__dsub_rn(g[6], g[5]), (double)(MESH_N - 1));
    g[8] = sigma;
    const double big = fmax(fabs(cx), fabs(cy)) + three_sigma;
    g[9] = 2.0 * (24.0 * big / sigma + 220.0) * MESH_GUARD_U;
    rec[0] = (uint32_t)tb | (2u << 30);
    const float guard_f = __double2float_ru(g[9]);
    rec[1] = __float_as_uint(guard_f);
    // can the constant-weight shortcut change any of the 100 truncations of this point?  (same test, same operands
    // as the deposit kernel's per-pixel one, on the distinct weights)
    bool careful = exact_mesh;
    const double guard = (double)guard_f;
    for (int k = 0; k < P.n_mesh_w_unique; ++k) {
        const double v = __dmul_rn(P.mesh_w_unique[k], g[10]);
        careful = careful || !(fabs(__dsub_rn(v, rint(v))) > __dmul_rn(guard, v));
    }
    if (careful) rec[0] |= 1u << 29;
#pragma unroll
    for (int a = 0; a < MESH_N; ++a) {
        const double px = (a == MESH_N - 1) ? g[3] : __dadd_rn(g[2], __dmul_rn((double)a, g[4]));
        const double py = (a == MESH_N - 1) ? g[6] : __dadd_rn(g[5], __dmul_rn((double)a, g[7]));
        const uint32_t ix = (uint32_t)(uint16_t)(int16_t)lut_index(P, px), iy = (uint32_t)(uint16_t)(int16_t)lut_index(P, py);
        rec[4 + a / 2] |= iy << (16 * (a & 1));
        rec[9 + a / 2] |= ix << (16 * (a & 1));
    }
}

// The reference's own arithmetic for one mesh pixel (i, j): detector/transporter.py:36-41, 217-226, 240-246.
__device__ __noinline__ long long exact_share(const double* g, int i, int j) {
    const double px = (i == MESH_N - 1) ? g[3] : __dadd_rn(g[2], __dmul_rn((double)i, g[4]));
    const double py = (j == MESH_N - 1) ? g[6] : __dadd_rn(g[5], __dmul_rn((double)j, g[7]));
    const double ddx = __dsub_rn(px, g[0]), ddy = __dsub_rn(py, g[1]);
    const double r2 = __dadd_rn(__dmul_rn(ddx, ddx), __dmul_rn(ddy, ddy));
    const double sigma = g[8];
    const double cell = __ddiv_rn(__dmul_rn(6.0, sigma), (double)(MESH_N - 1));
    const double cell2 = __dmul_rn(cell, cell);
    const double s2 = __dmul_rn(sigma, sigma);
    const double norm = __ddiv_rn(__ddiv_rn(0.5, 3.141592653589793), s2);  // 1 / 2 / pi / sigma**2
    const double c2 = __ddiv_rn(-0.5, s2);                                 // -1 / 2 / sigma**2
    const double pdf = __dmul_rn(norm, exp(__dmul_rn(c2, r2)));
    return (long long)__dmul_rn(__dmul_rn(pdf, cell2), g[10]);
}

// The record of a point of track rank `rank` (make_point's arguments) at ordered position d of `pb`, with its mesh
// constants when the record is careful.
__device__ __forceinline__ void put_point(const SimParams& P, const PointBuf& pb, int64_t d, double cx, double cy,
                                          double time, int tb, long long q, int rank, bool exact_mesh) {
    double g[GEOM_DOUBLES];
    uint32_t rec[REC_WORDS];
#pragma unroll
    for (int k = 0; k < GEOM_DOUBLES; ++k) g[k] = 0.0;
    make_point(P, cx, cy, time, tb, q, exact_mesh, g, rec);
    rec[14] = (uint32_t)rank;
    if ((rec[0] >> 29) & 1u) {  // only the exact path of the deposit kernel reads the mesh constants
        double2* out = reinterpret_cast<double2*>(pb.geom + d * GEOM_DOUBLES);
#pragma unroll
        for (int k = 0; k < GEOM_DOUBLES / 2; ++k) out[k] = make_double2(g[2 * k], g[2 * k + 1]);
    }
    uint4* out_rec = reinterpret_cast<uint4*>(pb.rec + d * REC_WORDS);
#pragma unroll
    for (int k = 0; k < REC_WORDS / 4; ++k)
        out_rec[k] = make_uint4(rec[4 * k], rec[4 * k + 1], rec[4 * k + 2], rec[4 * k + 3]);
}

// Scatter the group's points into (event, rank, arrival) order and compute their mesh constants (one thread each).
__global__ void __launch_bounds__(256) point_order_kernel(const __grid_constant__ SimParams P, PointBuf pb,
                                                          GroupView chunk, const Counters* ctr) {
    if (ctr->overflow_points) return;
    const GroupView gv = sub_group(chunk, blockIdx.y);
    const int64_t n = min((int64_t)pb.count[gv.group], pb.group_cap);
    const int64_t base = (int64_t)gv.group * pb.group_cap;
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = base + p;
        const int64_t d = base + pb.start[(int64_t)pb.ev[i] * pb.ranks + pb.rank[i]] + pb.j[i];
        put_point(P, pb, d, pb.x[i], pb.y[i], pb.t[i], (int)pb.t[i], pb.q[i], pb.rank[i], gv.exact_mesh != 0);
    }
}

// ------------------------------------------------------------------------------------- longitudinal diffusion
// (an extension outside the reference, DESIGN.md §3a; launched only when SimParams.long_diffusion > 0)
// A point of drift time `time` [time buckets] spreads over the buckets k0..k1 = floor(time -+ 3 sigma_L) (k < 0
// dropped) with sigma_L = sqrt(2 D_L dv time / E) / dv, the transverse expression of detector/transporter.py:301 over
// dv.  Bucket k receives (int64)(f_k q), f_k = Phi((k + 1 - time) / sigma_L) - Phi((k - time) / sigma_L), and every
// bucket of the window becomes a record of its own ("sub-point") with the point's position and transverse sigma, so
// the deposit kernel runs unchanged on one time bucket and at most 100 keys per record.  The window depends on the
// correctly rounded sqrt and floor only; erfc decides the charges, not which keys exist.
// sigma_L <= 0 or NaN (time <= 0): the point keeps its single bucket (int)time and all its electrons.
__device__ __forceinline__ double long_sigma(const SimParams& P, double time) {
    return __ddiv_rn(__dsqrt_rn(__ddiv_rn(__dmul_rn(__dmul_rn(__dmul_rn(2.0, P.long_diffusion), P.dv), time), P.efield)),
                     P.dv);
}

__device__ __forceinline__ void long_window(const SimParams& P, double time, double& sl, int& k0, int& k1) {
    sl = long_sigma(P, time);
    if (!(sl > 0.0)) {
        k0 = k1 = (int)time;
        return;
    }
    const double w = __dmul_rn(3.0, sl);
    k0 = max(0, (int)floor(__dsub_rn(time, w)));
    k1 = (int)floor(__dadd_rn(time, w));
}

__device__ __forceinline__ double long_phi(double x) {  // 0.5 erfc(-x / sqrt(2))
    return __dmul_rn(0.5, erfc(__ddiv_rn(-x, 1.4142135623730951)));
}

__device__ __forceinline__ long long long_electrons(double time, double sl, int k, long long q) {
    const double f = __dsub_rn(long_phi(__ddiv_rn(__dsub_rn((double)(k + 1), time), sl)),
                               long_phi(__ddiv_rn(__dsub_rn((double)k, time), sl)));
    return (long long)__dmul_rn(f, (double)q);
}

// (1) sub-points of every point, stored at the point's position in the (event, rank, arrival) order
__global__ void __launch_bounds__(256) sub_count_kernel(const __grid_constant__ SimParams P, PointBuf pb,
                                                        GroupView chunk, const Counters* ctr, unsigned* nsub) {
    if (ctr->overflow_points) return;
    const GroupView gv = sub_group(chunk, blockIdx.y);
    const int64_t n = min((int64_t)pb.count[gv.group], pb.group_cap);
    const int64_t base = (int64_t)gv.group * pb.group_cap;
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = base + p;
        double sl;
        int k0, k1;
        long_window(P, pb.t[i], sl, k0, k1);
        nsub[base + pb.start[(int64_t)pb.ev[i] * pb.ranks + pb.rank[i]] + pb.j[i]] = k1 >= k0 ? (unsigned)(k1 - k0 + 1) : 0u;
    }
}

// (2) one warp per (event, rank) list: exclusive scan of the list's sub-point counts in place (the offset of each
// point's first sub-point inside the list) and the list's total in sb.cnt, which point_scan_kernel then turns into
// sub-point list starts and work units.  The group's total is checked against the sub-point capacity sb.group_cap.
__global__ void __launch_bounds__(256) sub_scan_kernel(PointBuf pb, PointBuf sb, GroupView chunk, Counters* ctr,
                                                       unsigned* nsub, unsigned long long* sub_total) {
    if (ctr->overflow_points) return;
    const GroupView gv = sub_group(chunk, blockIdx.y);
    const int lane = threadIdx.x & 31;
    const int n = gv.n_events * pb.ranks;
    const int64_t first = (int64_t)gv.first_slot * pb.ranks;
    const int64_t base = (int64_t)gv.group * pb.group_cap;
    const int n_warps = gridDim.x * (blockDim.x / 32);
    for (int l = blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5); l < n; l += n_warps) {
        const int64_t s = base + pb.start[first + l];
        const unsigned c = pb.cnt[first + l];
        unsigned run = 0;
        for (unsigned o = 0; o < c; o += 32) {
            const unsigned idx = o + (unsigned)lane;
            const unsigned v = idx < c ? nsub[s + idx] : 0u;
            unsigned x = v;
#pragma unroll
            for (int k = 1; k < 32; k <<= 1) {
                const unsigned y = __shfl_up_sync(FULL, x, k);
                if (lane >= k) x += y;
            }
            if (idx < c) nsub[s + idx] = run + x - v;
            run += __shfl_sync(FULL, x, 31);
        }
        if (lane == 0) {
            sb.cnt[first + l] = run;
            const unsigned long long before = run ? atomicAdd(&sub_total[blockIdx.y], (unsigned long long)run) : 0ull;
            if (before + run > (unsigned long long)sb.group_cap) {  // the host grows the sub-point buffers and redoes the launch
                ctr->overflow_sub = 1;
                ctr->overflow_points = 1;
            }
        }
    }
}

// (3) after point_scan_kernel on sb: the records of every sub-point, (event, rank, arrival, bucket) order.  `sb`
// addresses the chunk's groups from 0 (its records exist for one chunk at a time).
__global__ void __launch_bounds__(256) sub_point_kernel(const __grid_constant__ SimParams P, PointBuf pb, PointBuf sb,
                                                        GroupView chunk, const Counters* ctr, const unsigned* nsub) {
    if (ctr->overflow_points) return;
    const GroupView gv = sub_group(chunk, blockIdx.y);
    const int64_t n = min((int64_t)pb.count[gv.group], pb.group_cap);
    const int64_t base = (int64_t)gv.group * pb.group_cap;
    const int64_t sbase = (int64_t)blockIdx.y * sb.group_cap;
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = base + p;
        const int64_t l = (int64_t)pb.ev[i] * pb.ranks + pb.rank[i];
        const double time = pb.t[i], cx = pb.x[i], cy = pb.y[i];
        const long long q = pb.q[i];
        double sl;
        int k0, k1;
        long_window(P, time, sl, k0, k1);
        int64_t d = sbase + sb.start[l] + nsub[base + pb.start[l] + pb.j[i]];
        for (int k = k0; k <= k1; ++k, ++d)
            put_point(P, sb, d, cx, cy, time, k, sl > 0.0 ? long_electrons(time, sl, k, q) : q, pb.rank[i],
                      gv.exact_mesh != 0);
    }
}

// ---------------------------------------------------------------------------------------- shared-memory accumulate
constexpr int DEPOSIT_THREADS = 256;
constexpr int DEPOSIT_WARPS = DEPOSIT_THREADS / 32;
constexpr int POINTS_PER_WARP = 3;   // three active points per warp pass: 3 x 10 mesh rows on 30 lanes
constexpr int POINTS_PER_ITER = DEPOSIT_WARPS * POINTS_PER_WARP;
constexpr int QUEUE_SLOTS = 64;      // per-warp ring of finished (key, charge) runs waiting for a full 32-lane insert
constexpr int SMEM_SLOTS = 4864;     // per-CTA table in shared memory: 10 B per slot = 47.5 KB, four CTAs per SM
// fill check once per pass of the CTA: a pass adds at most 100 keys per point plus what the rings still hold
constexpr int SMEM_SPILL_AT = SMEM_SLOTS - 100 * POINTS_PER_ITER - DEPOSIT_WARPS * QUEUE_SLOTS - 512;
// That is the highest safe threshold.  The default is lower: a table at 30 % load answers most inserts with one probe,
// and the appends it costs are cheap (measured optimum over the four workloads; AttpcConfig.table_spill_keys).
constexpr int SMEM_SPILL_DEFAULT = 2000 < SMEM_SPILL_AT ? 2000 : SMEM_SPILL_AT;
constexpr size_t DEPOSIT_SMEM_BYTES = (size_t)SMEM_SLOTS * (2 * sizeof(unsigned) + sizeof(uint16_t));
constexpr unsigned SMEM_KEY_MASK = 0x0FFFFFFFu;  // low 28 bits: ((tb << 15) | pad) + 1; top 4 bits: track rank

// Slot word = compact key (time bucket < 8192, pad id < 32768) + 1 in the low 28 bits, 0 = empty, and in the top four
// bits the rank of the last track that touched the slot.  Tracks are processed in rank order, so the rank is kept
// current with a plain store of the whole word (every writer of a phase stores the same value; a concurrent CAS on
// a non-empty word simply fails and re-reads it).  The charge is a 48-bit sum: 32 low bits + 16 high bits packed two
// per word (max 2.8e14 electrons per pad and time bucket, far above anything physical; overflow is flagged).
struct SmemTable {
    unsigned* word;   // key + rank
    unsigned* lo;     // charge bits 0..31
    unsigned* hi2;    // charge bits 32..47, two slots per 32-bit word
};

__device__ __forceinline__ unsigned smem_key(unsigned tb, unsigned pad) { return ((tb << 15) | pad) + 1u; }

__device__ __forceinline__ unsigned smem_home(unsigned key1) {
    return __umulhi(key1 * 2654435761u, (unsigned)SMEM_SLOTS);  // multiply-shift range reduction, no division
}

// Find the slot of `key1`, claiming an empty one if it is new (counted in the lane's `n_new`; the warp publishes the
// sum before every fill check).  The table is flushed long before it can fill.
__device__ __forceinline__ unsigned smem_find(const SmemTable& t, unsigned key1, unsigned rank, unsigned& n_new,
                                              unsigned& probes) {
    unsigned slot = smem_home(key1);
#pragma unroll 1
    for (unsigned probe = 0; probe < (unsigned)SMEM_SLOTS; ++probe) {
        unsigned w = *(volatile unsigned*)&t.word[slot];
        if ((w & SMEM_KEY_MASK) == key1) break;  // the common case: the key is there, at its home slot
        if (w == 0u) {
            w = atomicCAS(&t.word[slot], 0u, key1 | (rank << 28));
            if (w == 0u) {
                n_new += 1u;
                break;
            }
            if ((w & SMEM_KEY_MASK) == key1) break;
        }
        probes += 1u;  // (extra probes; the first probe of every insert is counted from the number of pushes)
        slot = slot + 1u == (unsigned)SMEM_SLOTS ? 0u : slot + 1u;
    }
    return slot;
}

// Exact accumulate from native 32-bit shared-memory atomics (carry into the 16-bit high part).
__device__ __forceinline__ void smem_charge(const SmemTable& t, unsigned slot, unsigned long long q, int* overflow) {
    const unsigned vlo = (unsigned)q, vhi = (unsigned)(q >> 32);
    unsigned carry = 0u;
    if (vlo) carry = atomicAdd(&t.lo[slot], vlo) > ~vlo ? 1u : 0u;
    const unsigned add = vhi + carry;
    if (add) {
        const unsigned shift = (slot & 1u) * 16u;
        const unsigned old = (atomicAdd(&t.hi2[slot >> 1], add << shift) >> shift) & 0xFFFFu;
        if (add > 0xFFFFu || old + add > 0xFFFFu) *overflow = 1;
    }
}

__device__ __forceinline__ unsigned long long smem_charge_of(const SmemTable& t, unsigned slot) {
    const unsigned hi = (t.hi2[slot >> 1] >> ((slot & 1u) * 16u)) & 0xFFFFu;
    return ((unsigned long long)hi << 32) | t.lo[slot];
}

// Persistent CTAs, as many as are resident at once: each pulls work units from `cursor` (zeroed before every launch),
// the chunk's groups one after the other and every group's units in its longest-first unit_order.  A unit is a slice
// of one event's points, all tracks together; label = last track in `indices` order to touch a key,
// detector/transporter.py:166-169, 247-249 = the highest rank, kept with an atomicMax.  The table is cleared once
// when the CTA starts; every segment append clears the slots it reads, so each unit leaves the table empty.
//
// A warp takes three active points per pass; lane (s, i) owns row i (one x of the 10x10 mesh) of point s and walks
// the ten y of that row in the reference's pixel order.  Neighbouring pixels of a row usually fall on the same pad, so
// the lane sums the integer shares of such a run in registers (integer adds commute and every share is truncated
// on its own first, exactly as transporter.py:240-248 does) and only a finished run (key, charge) is pushed into the
// warp's ring in shared memory.  Whenever the ring holds 32 runs, all 32 lanes insert one each into the CTA's
// open-addressing table: the insert code (probe loop, two atomics) runs once per 32 runs instead of once per 32
// pixels.  The table is appended to the event's entry list as a dense segment whenever it reaches the spill threshold
// and at the end; events deposited in several segments (dense events, events split over several units) may then list
// a key several times, which order_kernel merges after sorting.
__global__ void __launch_bounds__(DEPOSIT_THREADS, 4)
deposit_kernel(const __grid_constant__ SimParams P, PointBuf pb, GroupView chunk, int n_groups, unsigned* cursor,
               Counters* ctr) {
    extern __shared__ __align__(16) unsigned s_raw[];
    __shared__ unsigned s_nkeys, s_out, s_flush, s_base;
    __shared__ unsigned s_qkey[DEPOSIT_WARPS][QUEUE_SLOTS], s_qlo[DEPOSIT_WARPS][QUEUE_SLOTS],
        s_qhi[DEPOSIT_WARPS][QUEUE_SLOTS];
    // the unit the CTA works on: group s_group of the chunk, entry s_unit of its unit_order; cursor values
    // [s_group_first, s_group_end) are the units of group s_group (thread 0's walk over the groups)
    __shared__ int s_group, s_unit;
    __shared__ unsigned s_group_first, s_group_end;
    SmemTable t;
    t.word = s_raw;
    t.lo = s_raw + SMEM_SLOTS;
    t.hi2 = s_raw + 2 * SMEM_SLOTS;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    {
        constexpr int TABLE_VEC4 = (2 * SMEM_SLOTS + SMEM_SLOTS / 2) / 4;
        uint4* v = reinterpret_cast<uint4*>(s_raw);
        for (int i = threadIdx.x; i < TABLE_VEC4; i += blockDim.x) v[i] = make_uint4(0u, 0u, 0u, 0u);
    }
    if (threadIdx.x == 0) {
        s_nkeys = 0;
        s_out = 0;
        s_flush = 0;
        s_group = -1;
        s_group_first = 0;
        s_group_end = 0;
    }
    const int sub = lane / MESH_N;                                  // point of the warp's triple; 3 = idle lanes 30, 31
    const int row = lane - sub * MESH_N;                            // mesh row (x index) of this lane
    // constant mesh weights: the rows differ from lane to lane, so they are read from shared memory (row stride 11
    // doubles: the ten rows start in ten different bank pairs), not through the constant cache
    __shared__ double s_w[MESH_N][MESH_N + 1];
    for (int k = threadIdx.x; k < MESH_N * MESH_N; k += blockDim.x) s_w[k / MESH_N][k % MESH_N] = P.mesh_w[k];
    const double* wrow = s_w[row];
    const bool exact_mesh = chunk.exact_mesh != 0;
    unsigned* qkey = s_qkey[warp];
    unsigned* qlo = s_qlo[warp];
    unsigned* qhi = s_qhi[warp];
    const unsigned lanes_below = lanemask_lt();
    static_assert(SMEM_SLOTS % DEPOSIT_THREADS == 0, "segment appends give every warp whole 32-slot blocks");
    static_assert(sizeof(HashEntry) == 16 && offsetof(HashEntry, charge) == 8, "appends store entries as uint4");
    constexpr unsigned NO_ROOM = ~0u;  // s_base of a segment that does not fit the event's region

    while (true) {
        if (threadIdx.x == 0) {  // pull the next unit
            const unsigned c = atomicAdd(cursor, 1u);
            int g = s_group;
            unsigned first = s_group_first, end = s_group_end;
            while (c >= end && ++g < n_groups) {
                first = end;
                end += (unsigned)pb.n_units[chunk.group + g];
            }
            s_group = g;
            s_group_first = first;
            s_group_end = end;
            s_unit = (int)(c - first);
        }
        __syncthreads();  // (the first one also publishes the cleared table and the staged weights)
        if (s_group >= n_groups) break;
        const GroupView gv = sub_group(chunk, s_group);
        const int64_t ubase = (int64_t)gv.group * pb.max_units;
        const int unit = pb.unit_order[ubase + s_unit];
        const int e = pb.unit_event[ubase + unit];
        const int u_first = pb.unit_first[ubase + unit], u_count = pb.unit_count[ubase + unit];
        const int slot_event = gv.first_slot + e;
        HashEntry* region = gv.tables + (int64_t)(gv.chunk_e0 + e) * gv.hash_cap;
        const int64_t base = (int64_t)gv.group * pb.group_cap;
        unsigned n_dep = 0, n_probe = 0, n_new = 0;
        unsigned q_head = 0, q_tail = 0;  // warp-uniform ring positions

        auto drain = [&](unsigned n) {  // whole warp: insert ring entries [q_head, q_head + n), n <= 32
            __syncwarp();
            if ((unsigned)lane < n) {
                const unsigned at = (q_head + (unsigned)lane) & (QUEUE_SLOTS - 1);
                const unsigned kw = qkey[at];
                const unsigned long long q = ((unsigned long long)qhi[at] << 32) | qlo[at];
                const unsigned slot = smem_find(t, kw & SMEM_KEY_MASK, kw >> 28, n_new, n_probe);
                smem_charge(t, slot, q, &ctr->overflow_charge);
                atomicMax(&t.word[slot], kw);  // same key bits: the highest rank wins (transporter.py:247-249)
            }
            __syncwarp();
            q_head += n;
        };
        auto publish_new_keys = [&]() {  // whole warp, before a barrier that precedes a read of s_nkeys
            const unsigned total = __reduce_add_sync(FULL, n_new);
            if (lane == 0 && total) atomicAdd(&s_nkeys, total);
            n_new = 0;
        };

        // Append the table as one dense SEGMENT to the event's entry list and clear it in the same pass (all threads,
        // after a barrier that follows every warp's publish_new_keys).  The position comes from the event's entry
        // counter, which the units of a split event share.  A key can then sit in several segments of the list:
        // gv.mode marks such events and order_kernel merges the copies after sorting (integer adds commute, the label
        // is a maximum), and it sorts every list, so the order of the entries inside a segment is free.  Every warp
        // compacts blocks of 32 consecutive slots: one shared atomic reserves the block's keys, the lanes write them
        // as consecutive 16 B entries and zero their slots (the 16 hi2 words of a block belong to no other block).
        auto append_segment = [&](bool last) {
            if (threadIdx.x == 0) {
                const unsigned n = s_nkeys;
                const unsigned seg0 = atomicAdd(&gv.n_entries[slot_event], n);
                s_base = seg0 + n > (unsigned)gv.hash_cap ? NO_ROOM : seg0;
                if (s_base == NO_ROOM) ctr->overflow_hash = 1;  // the host grows the regions and redoes the launch
                if (!last) {
                    gv.mode[slot_event] = 1u;
                    atomicAdd(&ctr->flushes, 1ULL);
                }
                s_nkeys = 0;  // (every warp read it before the barrier that precedes this call)
                s_out = 0;
            }
            __syncthreads();
            const unsigned seg0 = s_base;
#pragma unroll 1
            for (int b = warp * 32; b < SMEM_SLOTS; b += DEPOSIT_THREADS) {
                const unsigned slot = (unsigned)(b + lane);
                const unsigned w = t.word[slot];
                const unsigned long long q = smem_charge_of(t, slot);
                __syncwarp();  // every lane has read its hi2 word
                t.word[slot] = 0u;
                t.lo[slot] = 0u;
                if (lane < 16) t.hi2[b / 2 + lane] = 0u;
                const unsigned m = __ballot_sync(FULL, w != 0u);
                if (m && seg0 != NO_ROOM) {  // warp-uniform
                    unsigned at = 0;
                    if (lane == 0) at = atomicAdd(&s_out, (unsigned)__popc(m));
                    at = seg0 + __shfl_sync(FULL, at, 0) + __popc(m & lanes_below);
                    if (w)  // one 16 B store (region rows are 16 B aligned; HashEntry is only 8 B aligned)
                        reinterpret_cast<uint4*>(region)[at] =
                            make_uint4(w & SMEM_KEY_MASK, w >> 28, (unsigned)q, (unsigned)(q >> 32));
                }
            }
            if (threadIdx.x == 0) s_flush = 0;  // (every warp read it before the barrier above)
            __syncthreads();
        };

        // The unit's slice [u_first, u_first + u_count) of the event's run, all tracks together: the label of a key is
        // the highest rank that touched it (atomicMax on the slot word), so points need no ordering.  Warps run
        // freely: a warp that sees the table filling up raises s_flush, every warp notices at its next pass boundary
        // and only then do they meet at a barrier (every barrier inside a unit is followed by the same uniform
        // decision on s_flush, whichever call site a warp arrives from).
        const int64_t run0 = pb.start[(int64_t)slot_event * pb.ranks];
        const int end = u_first + u_count;
        for (int p0 = u_first; p0 < end; p0 += POINTS_PER_ITER) {
            const int w0 = p0 + warp * POINTS_PER_WARP;
            if (w0 < end) {  // warp-uniform
                const int pp = w0 + sub;
                const bool have = sub < POINTS_PER_WARP && pp < end;
                const int64_t p = base + run0 + (have ? pp : w0);
                const uint4* rp = reinterpret_cast<const uint4*>(pb.rec + p * REC_WORDS);
                uint4 head = __ldg(rp);
                if (!have) head.x = 0u;
                const unsigned r = __ldg(pb.rec + p * REC_WORDS + 14);  // rank of the point's track
                const int kind = (int)(head.x >> 30), tb = (int)(head.x & 0x1FFFFFFFu);
                const bool careful_point = (head.x >> 29) & 1u;
                const unsigned keybase = (((unsigned)tb << 15) + 1u) | (r << 28);  // + pad = slot word
                const double qd = kind == 2 ? __hiloint2double((int)head.w, (int)head.z) : 0.0;
                const double guard = exact_mesh ? 2.0 : (double)__uint_as_float(head.y);
                int cur = -1;         // pad of the run being summed
                long long acc = 0;    // its charge so far
                int pad[MESH_N];
#pragma unroll
                for (int j = 0; j < MESH_N; ++j) pad[j] = -1;
                if (kind != 0) {
                    // pad-table row of this lane's mesh row, columns of the ten mesh columns (make_point)
                    const uint4 cols = __ldg(rp + 1);
                    const uint2 tail = __ldg(reinterpret_cast<const uint2*>(rp + 2));  // iy[8], iy[9] | ix[0], ix[1]
                    const int ix = (int)__ldg(reinterpret_cast<const int16_t*>(rp) + 18 + row);
                    const unsigned cw[5] = {cols.x, cols.y, cols.z, cols.w, tail.x};
                    const int16_t* lut_row = P.lut + (int64_t)max(ix, 0) * P.lut_n;
                    if (kind == 2) {
#pragma unroll
                        for (int j = 0; j < MESH_N; ++j) {  // all pad lookups first: independent loads in flight
                            const int iy = (j & 1) ? (int)cw[j / 2] >> 16 : (int)(int16_t)(cw[j / 2] & 0xFFFFu);
                            if (ix >= 0 && iy >= 0) pad[j] = (int)__ldg(lut_row + iy);
                        }
                    } else if (row == 0) {  // detector/transporter.py:123-169: all electrons on one pad
                        const int iy = (int)(int16_t)(cw[0] & 0xFFFFu);
                        if (ix >= 0 && iy >= 0) cur = (int)__ldg(lut_row + iy);
                        acc = (long long)__hiloint2double((int)head.w, (int)head.z);
                        n_dep += cur >= 0;
                    }
                }
                // detector/transporter.py:240-246: int(pdf * step^2 * electrons).  pdf * step^2 is the constant mesh
                // weight up to rounding (see make_point); the reference's own expression is evaluated only where the
                // rounding could change the truncation -- rare, so the warp then takes a second copy of the loop.
                unsigned risky = 0u;
                const bool careful_warp = __any_sync(FULL, careful_point);
                if (careful_warp && careful_point) {
#pragma unroll
                    for (int j = 0; j < MESH_N; ++j) {
                        const double v = __dmul_rn(wrow[j], qd);
                        if (!(fabs(__dsub_rn(v, rint(v))) > __dmul_rn(guard, v)) && pad[j] >= 0) risky |= 1u << j;
                    }
                }
                const double* g = pb.geom + p * GEOM_DOUBLES;
                auto walk_row = [&](auto careful) {
                    // j == MESH_N is the sentinel that pushes the last run of the row
#pragma unroll
                    for (int j = 0; j <= MESH_N; ++j) {
                        const int pj = j < MESH_N ? pad[j] : -1;
                        long long share = 0;  // (of a pixel without pad: added to a run that is never pushed)
                        if (j < MESH_N) {
                            share = (long long)__dmul_rn(wrow[j], qd);
                            if (decltype(careful)::value) {
                                if ((risky >> j) & 1u) share = exact_share(g, row, j);
                            }
                            n_dep += pj >= 0;
                        }
                        const bool change = pj != cur;
                        const bool push = change && cur >= 0;
                        const unsigned m = __ballot_sync(FULL, push);
                        if (m) {  // warp-uniform
                            if (push) {
                                const unsigned at = (q_tail + __popc(m & lanes_below)) & (QUEUE_SLOTS - 1);
                                qkey[at] = keybase + (unsigned)cur;
                                qlo[at] = (unsigned)acc;
                                qhi[at] = (unsigned)((unsigned long long)acc >> 32);
                            }
                            q_tail += __popc(m);
                            if (q_tail - q_head >= 32u) drain(32u);
                        }
                        if (change) {
                            cur = pj;
                            acc = 0;
                        }
                        acc += share;
                    }
                };
                if (careful_warp && __any_sync(FULL, risky != 0u)) walk_row(std::true_type{});
                else walk_row(std::false_type{});
            }
            publish_new_keys();
            if (*(volatile unsigned*)&s_nkeys > (unsigned)gv.spill_keys) *(volatile unsigned*)&s_flush = 1u;
            if (__any_sync(FULL, *(volatile unsigned*)&s_flush != 0u)) {
                __syncthreads();
                append_segment(false);
            }
        }
        while (q_tail != q_head) drain(min(32u, q_tail - q_head));
        publish_new_keys();
        if (*(volatile unsigned*)&s_nkeys > (unsigned)gv.spill_keys) *(volatile unsigned*)&s_flush = 1u;
        while (true) {
            __syncthreads();
            if (*(volatile unsigned*)&s_flush == 0u) break;
            append_segment(false);
        }
        append_segment(true);  // leaves the table empty and s_nkeys, s_out, s_flush zero for the next unit
        unsigned long long n_dep64 = n_dep, n_probe64 = n_probe + (lane == 0 ? q_tail : 0u);  // q_tail: runs pushed = inserts
        for (int o = 16; o > 0; o >>= 1) {
            n_dep64 += __shfl_xor_sync(FULL, n_dep64, o);
            n_probe64 += __shfl_xor_sync(FULL, n_probe64, o);
        }
        if (lane == 0 && n_dep64) {
            atomicAdd(&ctr->deposits, n_dep64);
            atomicAdd(&ctr->probes, n_probe64);
        }
    }
}

// ---------------------------------------------------------------------------------------------------- finalize
struct ReplayUniforms {
    const int64_t* offsets;  // [n_events + 1] or null
    const int64_t* keys;
    const double* vals;
};

// Where Spyral rows go: the eight float64 columns of detector/writer.py:97-110 and the labels, or
// (ATTPC_SPYRAL_COLUMNS: pad != null) what those are functions of: pad, time bucket Q16.16, electrons as 32 low +
// 16 high bits, label.
// Amplitude and integral follow from the electrons alone, x / y / pad size from the pad id and z from the time bucket,
// so the host rebuilds the eight columns bit for bit (Engine.rows_from_columns).
struct SpyralSink {
    double* rows;  // [rows, 8]
    int64_t* row_labels;
    int16_t* pad;
    uint32_t* tb_q16;
    uint32_t* e_lo;
    uint16_t* e_hi;
    int8_t* label;
};

struct FinalizeArgs {
    uint64_t seed;
    int64_t first_event;      // global id of event slot 0 of the launch batch
    uint32_t flags;
    int32_t n_tracks_per_event;
    int32_t label_of_rank[MAX_TRACKS_PER_EVENT];
    const int32_t* label_of_event_rank;  // replay: [n_events, n_tracks_per_event] or null
    ReplayUniforms replay;
    uint64_t* sort_items;     // [chunk events][scratch_stride] scratch of the events whose lists do not fit shared memory
    unsigned* kept;           // [launch events] rows kept per event
    int64_t* offsets;         // [launch events + 1] CSR offsets (global across groups of the launch)
    double* cloud;            // [out_cap, 3]
    int64_t* labels;          // [out_cap]
    int64_t out_cap;
    // optional columnar copy of the same rows in their natural types (15 B instead of 32 B per row on the wire).
    // col_tb_q16 = (time bucket << 16) | (wiggle * 2^16): time bucket + wiggle == col_tb_q16 / 65536 exactly for the
    // library's own 16-bit wiggle; a replayed 53-bit uniform is truncated to 16 bits there (replay tests read the
    // float64 cloud).
    int16_t* col_pad;
    uint32_t* col_tb_q16;
    int64_t* col_electrons;
    int8_t* col_label;
    // compact electrons column: the low 32 bits of every count, plus a list of (row, count) for the counts that
    // need more (rare for light ions; the host falls back to col_electrons when the list overflows)
    uint32_t* col_electrons32;
    int64_t* big_rows;
    int64_t* big_electrons;
    unsigned long long* big_count;  // running number of exceptions of the call (also counts what did not fit)
    int64_t big_cap;
    // packed columns (ATTPC_COLUMNS_PACKED): col_pad = pad | rank << rank_shift, the wiggle alone, rows per time
    // bucket and event; col_tb_q16 / col_label are then null
    uint16_t* col_wiggle;
    uint16_t* tb_counts;      // [launch events][NUM_TB]
    int32_t rank_shift, pad2_;
    unsigned long long* csr_total;  // running totals of the call {cloud rows, electron counts >= 2^32, Spyral rows}
    uint4* staged;            // [chunk events][hash_cap] ordered rows of every event, 16 B each (order_kernel -> emit_kernel):
                              //   x = time bucket << 16 | wiggle (16 bit);  y = electrons, low 32 bits;
                              //   z = electrons bits 32..47 | pad << 16 | above-ADC-threshold << 31;  w = track rank | z-order place << 4
    int64_t scratch_stride;   // 64-bit words of sort_items per event
    // events queued by order_kernel for the kernels with more shared memory per event (list == null: tier not in use);
    // count and cursor are zeroed per chunk
    struct Queue {
        unsigned* list;   // [chunk events]
        unsigned* count;
        unsigned* cursor;
    } big, far;  // big: second shared-memory tier; far: lists ordered in global scratch
    // Spyral rows of the same events (detector/writer.py:61-112, 232-238), thresholded and in z order, into rsink
    bool spyral;
    unsigned* row_kept;       // [launch events] rows above the ADC threshold
    int64_t* row_offsets;     // [launch events + 1]
    SpyralSink rsink;         // [out_cap] rows
};

constexpr uint32_t F_KEEP_ALL_TB = 1u, F_SPYRAL = 2u, F_NO_WIGGLE = 4u;
constexpr int TB_BINS = 1024;  // counting-sort bins over the integer time bucket (last bin collects tb >= 1023)

// Exclusive scan, in place, of a[at(0)], a[at(1)], ..., a[at(TB_BINS - 1)]; every thread of the CTA calls it after a
// barrier that completed `a`; returns the total; ends with a barrier.
template <int T, typename Map>
__device__ __forceinline__ unsigned scan_bins(unsigned* a, Map at, unsigned* s_warp) {
    constexpr int PER = TB_BINS / T;
    const int tid = threadIdx.x;
    unsigned local[PER], sum = 0;
#pragma unroll
    for (int k = 0; k < PER; ++k) {
        local[k] = a[at(tid * PER + k)];
        sum += local[k];
    }
    unsigned total;
    unsigned base = block_scan<T>(sum, total, s_warp);
#pragma unroll
    for (int k = 0; k < PER; ++k) {
        a[at(tid * PER + k)] = base;
        base += local[k];
    }
    __syncthreads();
    return total;
}

__device__ __forceinline__ double wiggle_of(const FinalizeArgs& fa, int slot_event, unsigned key, Counters* ctr) {
    if (fa.flags & F_NO_WIGGLE) return 0.0;
    if (fa.replay.offsets) {
        int64_t lo = fa.replay.offsets[slot_event], hi = fa.replay.offsets[slot_event + 1];
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            const int64_t k = fa.replay.keys[mid];
            if (k == (int64_t)key) return fa.replay.vals[mid];
            if (k < (int64_t)key) lo = mid + 1; else hi = mid;
        }
        ctr->replay_miss = 1;
        return 0.0;
    }
    return philox_uniform16(fa.seed, (uint64_t)(fa.first_event + slot_event), STREAM_WIGGLE, key);
}

// ------------------------------------------------------------------------------------------------ Spyral rows
struct SpyralArgs {
    const int64_t* offsets;   // [n_events + 1] input cloud CSR
    const double* cloud;      // [n, 3]
    const int64_t* labels;    // [n]
    int64_t n_events;         // events of this pass: first .. first + n_events - 1 of the arrays below
    int64_t first;
    unsigned long long* total;  // running number of rows before event `first` (device; updated by the scan)
    int64_t scratch_rows;     // rows of sort_keys / sort_idx per half
    const Counters* ctr;      // launch counters (null: none): a launch that overflowed a buffer is void and will be redone
    int64_t cloud_cap;        // rows the cloud buffer holds
    unsigned* kept;           // [n_events]
    int64_t* row_offsets;     // [n_events + 1]
    SpyralSink sink;          // [n] rows (capacity = input points)
    uint64_t* sort_keys;      // [n] scratch (order-preserving bits of z)
    uint32_t* sort_idx;       // [n] scratch
    int32_t keep_all;         // 1: every row, input order (plain convert_to_spyral, detector/writer.py:61-112)
};

// detector/response.py:35-57: amplitude = max(min(r_i e, 4095)), integral = sum(min(r_i e, 4095)).
// max commutes with the monotone map r -> min(fl(r e), 4095), so amplitude = min(fl(r_max e), 4095) exactly.  The
// integral uses the descending-sorted response and its prefix sums: entries with r_i e > 4095 form a prefix.
__device__ __forceinline__ void shaped(const SimParams& P, double electrons, double& amp, double& integral) {
    const double top = __dmul_rn(P.resp_max, electrons);
    amp = fmin(top, 4095.0);
    int lo = 0, hi = top > 4095.0 ? P.n_response : 0;  // first index whose scaled response is <= 4095 (0: none clipped)
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (__dmul_rn(P.resp_sorted[mid], electrons) > 4095.0) lo = mid + 1; else hi = mid;
    }
    // (explicitly rounded operations: the host rebuilds this value from the typed columns and must get the same bits)
    integral = __dadd_rn(__dmul_rn(4095.0, (double)lo),
                         __dmul_rn(electrons, __dsub_rn(P.resp_prefix[P.n_response], P.resp_prefix[lo])));
}

// detector/writer.py:101-103: (window_edge - tb) / (window_edge - mm_edge) * length * 1000.0 (explicitly rounded, like
// the amplitude: the host rebuilds it from the typed columns)
__device__ __forceinline__ double spyral_z(const SimParams& P, double tbf) {
    const double span = (double)(P.win_edge - P.mm_edge);
    return __dmul_rn(__dmul_rn(__ddiv_rn(__dsub_rn(P.win_edge, tbf), span), P.length), 1000.0);
}

// Spyral row `at` of `sink` (detector/writer.py:97-110) from a cloud row: `pad` and `electrons` as the float64 cloud
// holds them, `tbf` the time bucket with its wiggle and `tb_q16` that value in Q16.16.
__device__ __forceinline__ void put_spyral_row(const SimParams& P, const SpyralSink& sink, int64_t at, double pad,
                                               double tbf, uint32_t tb_q16, double electrons, int64_t label) {
    const int p = (int)pad;
    if (sink.pad) {
        const unsigned long long q = (unsigned long long)(long long)electrons;
        sink.pad[at] = (int16_t)p;
        sink.tb_q16[at] = tb_q16;
        sink.e_lo[at] = (uint32_t)q;
        sink.e_hi[at] = (uint16_t)(q >> 32);
        sink.label[at] = (int8_t)label;
        return;
    }
    double amp, integral;
    shaped(P, electrons, amp, integral);
    double* row = sink.rows + at * 8;
    row[0] = P.pad_xy[2 * p];
    row[1] = P.pad_xy[2 * p + 1];
    row[2] = spyral_z(P, tbf);
    row[3] = amp;
    row[4] = integral;
    row[5] = pad;
    row[6] = tbf;
    row[7] = P.pad_scale[p];
    sink.row_labels[at] = label;
}

__device__ __forceinline__ uint64_t orderable(double v) {
    const uint64_t b = (uint64_t)__double_as_longlong(v);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ULL);
}

// pass 1: per point amplitude/threshold (detector/writer.py:232), count kept rows per event
__global__ void __launch_bounds__(256) spyral_count_kernel(const __grid_constant__ SimParams P, SpyralArgs sa) {
    const int64_t e = sa.first + blockIdx.x;
    __shared__ unsigned s_n;
    if (threadIdx.x == 0) s_n = 0;
    __syncthreads();
    const int64_t a = sa.offsets[e], b = sa.offsets[e + 1];
    const bool bad = (sa.ctr && (sa.ctr->overflow_points | sa.ctr->overflow_hash | sa.ctr->overflow_out)) || b > sa.cloud_cap;
    if (bad) {  // the rows of this attempt were never written
        if (threadIdx.x == 0) sa.kept[e] = 0;
        return;
    }
    unsigned mine = 0;
    for (int64_t i = a + threadIdx.x; i < b; i += blockDim.x) {
        const double amp = fmin(__dmul_rn(P.resp_max, sa.cloud[i * 3 + 2]), 4095.0);
        if (sa.keep_all || amp > P.adc_threshold) mine += 1;
    }
    atomicAdd(&s_n, mine);
    __syncthreads();
    if (threadIdx.x == 0) sa.kept[e] = s_n;
}

__global__ void __launch_bounds__(1024) spyral_scan_kernel(SpyralArgs sa) {
    __shared__ unsigned long long s_warp[32];
    const unsigned* kept = sa.kept + sa.first;
    int64_t* row_offsets = sa.row_offsets + sa.first;
    const unsigned long long total =
        scan_tiles<1024>((int)sa.n_events, *sa.total, s_warp, [&](int i) { return (unsigned long long)kept[i]; },
                         [&](int i, unsigned long long s) { row_offsets[i] = (int64_t)s; });
    if (threadIdx.x == 0) {
        row_offsets[sa.n_events] = (int64_t)total;
        *sa.total = total;
    }
}

constexpr int SPYRAL_SMEM_ITEMS = 4096;  // 48 KB: 8 B z-bits + 4 B point index each

// pass 2: one CTA per event: keep rows above threshold, order by z (detector/writer.py:236; ties, which numpy's
// unstable argsort leaves unspecified, are broken by input order), write the 8 columns of detector/writer.py:97-110.
// z falls as the time bucket rises, so the order is a counting sort on the integer time bucket (descending) plus
// an insertion sort inside each bucket.
__global__ void __launch_bounds__(256)
spyral_rows_kernel(const __grid_constant__ SimParams P, SpyralArgs sa) {
    extern __shared__ uint64_t s_k[];
    uint32_t* s_v = (uint32_t*)(s_k + SPYRAL_SMEM_ITEMS);
    __shared__ unsigned s_hist[TB_BINS + 1];
    __shared__ unsigned s_fill[TB_BINS];
    __shared__ unsigned s_n;
    __shared__ unsigned s_warp[8];
    const int64_t e = sa.first + blockIdx.x;
    const int64_t a = sa.offsets[e], b = sa.offsets[e + 1];
    const int64_t out0 = sa.row_offsets[e];
    const int n = (int)sa.kept[e];
    if (n == 0) return;
    const int64_t total = sa.scratch_rows;
    uint64_t* stash_k = sa.sort_keys + a;           // unordered survivors
    uint32_t* stash_v = sa.sort_idx + a;
    const bool in_smem = n <= SPYRAL_SMEM_ITEMS;
    uint64_t* keys = in_smem ? s_k : sa.sort_keys + total + a;  // ordered
    uint32_t* idx = in_smem ? s_v : sa.sort_idx + total + a;
    if (!sa.keep_all) {
        for (int i = threadIdx.x; i <= TB_BINS; i += blockDim.x) s_hist[i] = 0;
        if (threadIdx.x == 0) s_n = 0;
        __syncthreads();
        for (int64_t i = a + threadIdx.x; i < b; i += blockDim.x) {
            const double amp = fmin(__dmul_rn(P.resp_max, sa.cloud[i * 3 + 2]), 4095.0);
            if (amp > P.adc_threshold) {
                const double tbf = sa.cloud[i * 3 + 1];
                const unsigned pos = atomicAdd(&s_n, 1u);
                stash_k[pos] = orderable(spyral_z(P, tbf));
                stash_v[pos] = (uint32_t)(i - a);
                const int tbi = min(max((int)tbf, 0), TB_BINS - 1);
                atomicAdd(&s_hist[TB_BINS - 1 - tbi], 1u);
            }
        }
        __syncthreads();
        const unsigned kept = scan_bins<256>(s_hist, [](int b) { return b; }, s_warp);
        for (int i = threadIdx.x; i < TB_BINS; i += blockDim.x) s_fill[i] = s_hist[i];
        if (threadIdx.x == 0) s_hist[TB_BINS] = kept;
        __syncthreads();
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            const uint32_t id = stash_v[i];
            const int tbi = min(max((int)sa.cloud[(a + id) * 3 + 1], 0), TB_BINS - 1);
            const unsigned pos = atomicAdd(&s_fill[TB_BINS - 1 - tbi], 1u);
            keys[pos] = stash_k[i];
            idx[pos] = id;
        }
        __syncthreads();
    }
    // One thread per kept row.  Its place inside its time bucket is the number of rows of the bucket that sort before
    // it ((z, index) order: detector/writer.py:236 sorts by z, equal z keep their cloud order), so the z-sort costs a
    // handful of shared-memory reads per row.
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const uint32_t id = sa.keep_all ? (uint32_t)i : idx[i];
        const int64_t src = a + id;
        const double padf = sa.cloud[src * 3 + 0], tbf = sa.cloud[src * 3 + 1], el = sa.cloud[src * 3 + 2];
        int place = i;
        if (!sa.keep_all) {
            const int bin = TB_BINS - 1 - min(max((int)tbf, 0), TB_BINS - 1);
            const int lo = (int)s_hist[bin], hi = (int)s_hist[bin + 1];
            const uint64_t kv = keys[i];
            int before = 0;
            for (int j = lo; j < hi; ++j) before += keys[j] < kv || (keys[j] == kv && idx[j] < id);
            place = lo + before;
        }
        // (tb_q16 is exact for the library's 16-bit wiggle)
        put_spyral_row(P, sa.sink, out0 + place, padf, tbf, (uint32_t)(tbf * 65536.0), el, sa.labels[src]);
    }
}

// ---------------------------------------------------------------------------------------------------- finalize
// detector/simulator.py:19-49 (dict_to_points), :104-115 (time-bucket wiggle and mask) and, when asked for,
// detector/response.py:35-57 + detector/writer.py:232-238 (amplitude, ADC threshold, z order) on the entry lists that
// deposit_kernel left, in four launches per chunk of events:
//
// order_kernel / order_queue_kernel, one CTA per event at a time, no event waits for another:
//   1  histogram of the entries over the integer time bucket (mask applied), keys staged in shared memory
//   2  exclusive scan -> bucket starts;  3  entries into their buckets (items = pad | list index)
//   4  rank by counting inside each bucket -> canonical order, ascending (time bucket, pad); copies of a key that sit
//      in different segments of the list (events deposited in several segments) become neighbours, ordered by index
//   5  the first copy of every key is the row: bit mask of the rows + running count (events with copies only)
//   6  charge / label gathered while the list is still in L2, wiggle drawn, rows staged (16 B) in canonical order
//   7  Spyral: kept rows per bucket -> suffix sums (z falls as the time bucket rises), rank inside the bucket by the
//      wiggle -> place of every kept row in z order, stored with the staged row
// offsets_kernel: running CSR offsets from the row counts.   emit_kernel: streams the staged rows to the sinks.
//
// Everything an event needs stays in shared memory: lists of up to FIN_ITEMS entries in order_kernel (two CTAs per SM),
// longer ones, up to FIN_BIG_ITEMS, in order_queue_kernel (queued by order_kernel; persistent CTAs, one per SM);
// beyond that
// (or with more than 2^17 entries per list allowed) the same code runs on a scratch region in global memory with
// 64-bit items.
constexpr int FIN_THREADS = ATTPC_FIN_THREADS;
constexpr int FIN_ITEMS = ATTPC_FIN_ITEMS;
constexpr size_t FIN_SMEM_BYTES = (size_t)(3 * FIN_ITEMS + 2 * (FIN_ITEMS / 32)) * sizeof(uint32_t);
// second shared-memory tier: the events whose lists exceed FIN_ITEMS are queued by order_kernel and taken by persistent
// CTAs of order_queue_kernel, one per SM with (nearly) all of its shared memory, up to 16384 entries
constexpr int FIN_BIG_THREADS = 1024;
constexpr int FIN_BIG_ITEMS = 16384;
constexpr size_t FIN_BIG_SMEM_BYTES = (size_t)(3 * FIN_BIG_ITEMS + 2 * (FIN_BIG_ITEMS / 32)) * sizeof(uint32_t);
constexpr unsigned long long SCAN_AGGREGATE = 1ULL << 62, SCAN_PREFIX = 2ULL << 62, SCAN_VALUE = (1ULL << 62) - 1ULL;
static_assert(TB_BINS % FIN_THREADS == 0 && FIN_ITEMS % 32 == 0 && TB_BINS % FIN_BIG_THREADS == 0, "finalize tiling");

struct FinShared {
    unsigned hist[TB_BINS + 1];  // bucket starts (sorted positions)
    unsigned fill[TB_BINS];      // fill cursors, then kept rows per bucket, then kept rows in the later buckets
    unsigned warp[32];
    unsigned keys, next;
};

template <typename Item, bool SMEM, int T>
__device__ __forceinline__ void order_event(const SimParams& P, const FinalizeArgs& fa, const GroupView& chunk,
                                               Counters* ctr, FinShared& sh, const int L, const int limit,
                                               const HashEntry* __restrict__ tab, Item* A, Item* B, uint32_t* C,
                                               unsigned* H, unsigned* HP) {
    constexpr int SH = SMEM ? 17 : 32;  // item = (pad << SH) | index in the list
    constexpr Item IDX_MASK = ((Item)1 << SH) - 1;
    const int tid = threadIdx.x, lane = tid & 31;
    const int slot_event = chunk.first_slot + L;
    const bool dup = chunk.mode[slot_event] != 0u;  // the list may hold a key several times
    auto key_of = [&](unsigned i) -> unsigned { return SMEM ? C[i] : tab[i].key1; };
    auto bin_of = [](unsigned key1) -> unsigned { return min((key1 - 1u) >> 15, (unsigned)TB_BINS - 1u); };
    // detector/simulator.py:108-113: keep 0 <= tb + u < 512 with u in [0, 1).  Only the last bucket needs u (a replayed
    // 53-bit uniform can round 511 + u up to 512.0)
    auto masked = [&](unsigned key1) -> unsigned {
        const unsigned tb = (key1 - 1u) >> 15;
        if ((fa.flags & F_KEEP_ALL_TB) || tb < (unsigned)NUM_TB - 1u) return key1;
        if (tb != (unsigned)NUM_TB - 1u) return 0u;
        const unsigned pad = (key1 - 1u) & 0x7FFFu;
        return (double)tb + wiggle_of(fa, slot_event, szudzik_pair(tb, pad), ctr) < (double)NUM_TB ? key1 : 0u;
    };

    // 1: histogram over the time bucket
    unsigned occupied = 0;
    for (int i0 = tid; i0 < limit; i0 += 4 * T) {  // four loads in flight per thread
        unsigned k[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = i0 + u * T;
            k[u] = i < limit ? tab[i].key1 : 0u;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = i0 + u * T;
            if (i >= limit) break;
            unsigned key1 = k[u];
            if (key1) {
                occupied += 1;
                key1 = masked(key1);
            }
            if (SMEM) C[i] = key1;
            if (key1) atomicAdd(&sh.hist[bin_of(key1)], 1u);
        }
    }
    if (occupied) atomicAdd(&sh.keys, occupied);
    __syncthreads();
    // 2: bucket starts
    const int n = (int)scan_bins<T>(sh.hist, [](int b) { return b; }, sh.warp);
    for (int b = tid; b < TB_BINS; b += T) sh.fill[b] = sh.hist[b];
    if (tid == 0) {
        sh.hist[TB_BINS] = (unsigned)n;
        if (sh.keys) atomicAdd(&ctr->keys, (unsigned long long)sh.keys);
    }
    __syncthreads();
    // 3: entries into their buckets
    for (int i = tid; i < limit; i += T) {
        unsigned key1 = SMEM ? C[i] : tab[i].key1;
        if (!SMEM && key1) key1 = masked(key1);
        if (key1) A[atomicAdd(&sh.fill[bin_of(key1)], 1u)] = ((Item)((key1 - 1u) & 0x7FFFu) << SH) | (Item)(unsigned)i;
    }
    __syncthreads();
    // 4: order every bucket: one thread per item counts the smaller items of its bucket (a bucket holds the pads hit in
    // one time bucket, a handful for most tracks; neighbouring threads walk the same items, the reads are broadcasts)
    for (int i = tid; i < n; i += T) {
        const Item v = A[i];
        const unsigned kv = key_of((unsigned)(v & IDX_MASK));
        const unsigned bin = bin_of(kv);
        const int lo = (int)sh.hist[bin], hi = (int)sh.hist[bin + 1];
        int rank = 0;
        if (bin != (unsigned)TB_BINS - 1u) {  // one time bucket: (pad, index) decides
#pragma unroll 4
            for (int j = lo; j < hi; ++j) rank += A[j] < v;
        } else {  // time buckets >= 1023 share the last bin (ATTPC_KEEP_ALL_TB only): compare the whole key
            for (int j = lo; j < hi; ++j) {
                const Item w = A[j];
                const unsigned kj = key_of((unsigned)(w & IDX_MASK));
                rank += kj < kv || (kj == kv && w < v);
            }
        }
        B[lo + rank] = v;
    }
    for (int b = tid; b < TB_BINS; b += T) sh.fill[b] = 0u;  // (kept rows per bucket, step 7)
    __syncthreads();
    // 5: rows = first copies
    int n_rows = n;
    if (dup) {
        for (int p = tid; p - lane < n; p += T) {  // (warp-uniform trip count)
            bool head = false;
            if (p < n) head = p == 0 || key_of((unsigned)(B[p] & IDX_MASK)) != key_of((unsigned)(B[p - 1] & IDX_MASK));
            const unsigned m = __ballot_sync(FULL, head);
            if (lane == 0) H[p >> 5] = m;
        }
        __syncthreads();
        n_rows = (int)scan_tiles<T>((n + 31) >> 5, 0u, sh.warp, [&](int w) { return (unsigned)__popc(H[w]); },
                                    [&](int w, unsigned s) { HP[w] = s; });
        __syncthreads();
    }
    auto is_row = [&](int p) -> bool { return !dup || ((H[p >> 5] >> (p & 31)) & 1u); };
    if (tid == 0) fa.kept[slot_event] = (unsigned)n_rows;
    // 6: the rows, in canonical order, into the event's staging region (16 B each; emit_kernel streams them to the
    // sinks once the offsets of all events are known).  Charge and label of a row fold the copies of its key:
    // integer adds commute, the label is the highest rank (detector/transporter.py:166-169, 247-249).
    uint4* staged = fa.staged + (int64_t)L * chunk.hash_cap;
    const bool spy = fa.spyral;
    const bool draw = fa.replay.offsets == nullptr;  // (replayed uniforms have 53 bits: emit_kernel looks them up)
    for (int p = tid; p < n; p += T) {
        Item w_out = 0;
        if (is_row(p)) {
            const uint4 en = __ldg(reinterpret_cast<const uint4*>(tab + (unsigned)(B[p] & IDX_MASK)));
            const unsigned key1 = en.x;
            unsigned rk = en.y;
            unsigned long long q = ((unsigned long long)en.w << 32) | en.z;
            if (dup)
                for (int j = p + 1; j < n && !((H[j >> 5] >> (j & 31)) & 1u); ++j) {
                    const uint4 o = __ldg(reinterpret_cast<const uint4*>(tab + (unsigned)(B[j] & IDX_MASK)));
                    q += ((unsigned long long)o.w << 32) | o.z;
                    rk = max(rk, o.y);
                }
            if (q >> 48) ctr->overflow_charge = 1;
            const unsigned tb = (key1 - 1u) >> 15, pad = (key1 - 1u) & 0x7FFFu;
            const uint32_t u16 = draw ? (uint32_t)(wiggle_of(fa, slot_event, szudzik_pair(tb, pad), ctr) * 65536.0) : 0u;
            // amplitude above the ADC threshold (detector/writer.py:232) <=> electrons >= e_keep_min
            const unsigned keep = spy && (long long)q >= P.e_keep_min ? 1u : 0u;
            const int r = dup ? (int)(HP[p >> 5] + __popc(H[p >> 5] & ((1u << (p & 31)) - 1u))) : p;
            staged[r] = make_uint4((tb << 16) | u16, (unsigned)q, (unsigned)(q >> 32) | (pad << 16) | (keep << 31), rk);
            if (spy) {
                const unsigned bin = min(tb, (unsigned)TB_BINS - 1u);
                w_out = (Item)((rk << 27) | (bin << 17) | (keep << 16) | u16);
                if (keep) atomicAdd(&sh.fill[bin], 1u);
            }
        }
        if (spy) A[p] = w_out;
    }
    if (!spy) return;
    // 7: place of every kept row in z order.  z falls as the time bucket rises (detector/writer.py:101-103, 236):
    //   (kept rows of the later buckets) + (kept rows of its bucket with a larger wiggle, or the same and a lower position)
    __syncthreads();
    const unsigned n_kept = scan_bins<T>(sh.fill, [](int b) { return TB_BINS - 1 - b; }, sh.warp);
    if (tid == 0) fa.row_kept[slot_event] = n_kept;
    for (int p = tid; p < n; p += T) {
        const unsigned w = (unsigned)A[p];
        if (!((w >> 16) & 1u)) continue;  // below the ADC threshold, or not a row
        const unsigned bin = (w >> 17) & 0x3FFu, wp = w & 0x1FFFFu;
        const int lo = (int)sh.hist[bin], hi = (int)sh.hist[bin + 1];
        unsigned within = 0;
#pragma unroll 4
        for (int j = lo; j < hi; ++j) {
            const unsigned wj = (unsigned)A[j] & 0x1FFFFu;  // (not kept: below 0x10000, never counted)
            within += wj > wp || (wj == wp && j < p);
        }
        const int r = dup ? (int)(HP[p >> 5] + __popc(H[p >> 5] & ((1u << (p & 31)) - 1u)) ) : p;
        reinterpret_cast<unsigned*>(staged + r)[3] = (w >> 27) | ((sh.fill[bin] + within) << 4);
    }
}

// Kernel A of finalize: order the entry list of every event of the chunk (one CTA per event, no event waits for
// another) and stage its rows.  Lists that do not fit this kernel's shared memory are queued for order_queue_kernel:
// for its second shared-memory tier when the call uses it and the list fits, for its global-scratch tier otherwise.
__global__ void __launch_bounds__(FIN_THREADS, ATTPC_FIN_MIN_CTAS)
order_kernel(const __grid_constant__ SimParams P, const __grid_constant__ FinalizeArgs fa,
             const __grid_constant__ GroupView chunk, Counters* ctr) {
    extern __shared__ __align__(16) uint32_t s_fin[];
    __shared__ FinShared sh;
    const int tid = threadIdx.x;
    const int L = (int)blockIdx.x;
    const int slot_event = chunk.first_slot + L;
    // an attempt that overflowed a buffer is void (the host redoes the launch)
    const bool void_attempt = (ctr->overflow_points | ctr->overflow_hash) != 0;
    const int limit = void_attempt ? 0 : (int)min(chunk.n_entries[slot_event], (unsigned)chunk.hash_cap);
    const bool narrow = chunk.hash_cap <= (1 << 17);  // list indices fit the 32-bit items
    if (limit > FIN_ITEMS || !narrow) {  // not for this kernel's shared memory: queue the event
        const FinalizeArgs::Queue& q = narrow && fa.big.list && limit <= FIN_BIG_ITEMS ? fa.big : fa.far;
        if (tid == 0) q.list[atomicAdd(q.count, 1u)] = (unsigned)L;
        return;
    }
    if (tid == 0) sh.keys = 0;
    for (int b = tid; b <= TB_BINS; b += FIN_THREADS) sh.hist[b] = 0;
    __syncthreads();
    const HashEntry* tab = chunk.tables + (int64_t)L * chunk.hash_cap;
    uint32_t* H = s_fin + 3 * FIN_ITEMS;
    order_event<uint32_t, true, FIN_THREADS>(P, fa, chunk, ctr, sh, L, limit, tab, s_fin, s_fin + FIN_ITEMS,
                                             s_fin + 2 * FIN_ITEMS, H, H + FIN_ITEMS / 32);
}

// The queued long lists (dense events): persistent CTAs that take events from the queue until it is empty.
template <int T, int ITEMS, int MIN_CTAS>
__global__ void __launch_bounds__(T, MIN_CTAS)
order_queue_kernel(const __grid_constant__ SimParams P, const __grid_constant__ FinalizeArgs fa,
                   const __grid_constant__ GroupView chunk, Counters* ctr, const FinalizeArgs::Queue q) {
    extern __shared__ __align__(16) uint32_t s_fin[];
    __shared__ FinShared sh;
    const int tid = threadIdx.x;
    const unsigned n_queued = *q.count;
    for (;;) {
        __syncthreads();  // (the previous event is done with the shared memory)
        if (tid == 0) {
            sh.next = atomicAdd(q.cursor, 1u);
            sh.keys = 0;
        }
        for (int b = tid; b <= TB_BINS; b += T) sh.hist[b] = 0;
        __syncthreads();
        if (sh.next >= n_queued) return;
        const int L = (int)q.list[sh.next];
        const int slot_event = chunk.first_slot + L;
        // (an attempt that overflowed a buffer is void: its lists may be incomplete, the host redoes the launch)
        const bool void_attempt = (ctr->overflow_points | ctr->overflow_hash) != 0;
        const int limit = void_attempt ? 0 : (int)min(chunk.n_entries[slot_event], (unsigned)chunk.hash_cap);
        const HashEntry* tab = chunk.tables + (int64_t)L * chunk.hash_cap;
        if (ITEMS > 0) {  // shared-memory tier
            uint32_t* H = s_fin + 3 * ITEMS;
            order_event<uint32_t, true, T>(P, fa, chunk, ctr, sh, L, limit, tab, s_fin, s_fin + ITEMS, s_fin + 2 * ITEMS,
                                           H, H + ITEMS / 32);
        } else {  // global scratch, 64-bit items: no dynamic shared memory, the L1 cache keeps its full size
            uint64_t* scratch = fa.sort_items + (int64_t)L * fa.scratch_stride;
            unsigned* H = reinterpret_cast<unsigned*>(scratch + 2 * (int64_t)chunk.hash_cap);
            order_event<uint64_t, false, T>(P, fa, chunk, ctr, sh, L, limit, tab, scratch, scratch + chunk.hash_cap,
                                            nullptr, H, H + chunk.hash_cap / 32 + 1);
        }
    }
}

// Running CSR offsets of the chunk's events from their row counts (cloud rows and, when asked for, Spyral rows), on
// top of the totals of the call so far.  One CTA: a thread sums a run of consecutive events, the CTA scans the sums.
__global__ void __launch_bounds__(1024) offsets_kernel(FinalizeArgs fa, GroupView chunk, Counters* ctr) {
    __shared__ unsigned long long s_warp[2][32];
    const int tid = threadIdx.x;
    const int n = chunk.n_events;
    const int per = (n + 1023) / 1024;
    const int e0 = min(n, tid * per), e1 = min(n, e0 + per);
    const bool spy = fa.spyral;
    const unsigned* kept = fa.kept + chunk.first_slot;
    const unsigned* rkept = fa.row_kept + chunk.first_slot;
    unsigned long long sum[2] = {0ULL, 0ULL}, base[2], total[2];
    for (int e = e0; e < e1; ++e) {
        sum[0] += kept[e];
        if (spy) sum[1] += rkept[e];
    }
#pragma unroll
    for (int c = 0; c < 2; ++c) {
        base[c] = fa.csr_total[2 * c] + block_scan<1024>(sum[c], total[c], s_warp[c]);
        total[c] += fa.csr_total[2 * c];
    }
    __syncthreads();  // (every thread has read csr_total)
    int64_t* offsets = fa.offsets + chunk.first_slot;
    int64_t* roffsets = fa.row_offsets + chunk.first_slot;
    for (int e = e0; e < e1; ++e) {
        offsets[e] = (int64_t)base[0];
        base[0] += kept[e];
        if (spy) {
            roffsets[e] = (int64_t)base[1];
            base[1] += rkept[e];
        }
    }
    if (tid == 0) {
        offsets[n] = (int64_t)total[0];
        fa.csr_total[0] = total[0];
        if ((int64_t)total[0] > fa.out_cap) ctr->overflow_out = 1;
        if (spy) {
            roffsets[n] = (int64_t)total[1];
            fa.csr_total[2] = total[1];
            if ((int64_t)total[1] > fa.out_cap) ctr->overflow_out = 1;
        }
    }
}

// Kernel B of finalize: stream the staged rows of every event to the sinks (one CTA per event): [pad, tb + u,
// electrons] rows and labels (detector/simulator.py:19-49, 104-115), the typed columns, and the Spyral rows
// (detector/response.py:35-57, detector/writer.py:61-112, 232-238) at their place in z order.
constexpr int EMIT_THREADS = 256;
__global__ void __launch_bounds__(EMIT_THREADS)
emit_kernel(const __grid_constant__ SimParams P, const __grid_constant__ FinalizeArgs fa,
            const __grid_constant__ GroupView chunk, Counters* ctr) {
    const int L = (int)blockIdx.x;
    const int slot_event = chunk.first_slot + L;
    const int n = (int)fa.kept[slot_event];
    const int64_t off = fa.offsets[slot_event];
    if (off + n > fa.out_cap) return;  // (offsets_kernel has raised overflow_out)
    const bool spy = fa.spyral && fa.row_offsets[slot_event] + (int64_t)fa.row_kept[slot_event] <= fa.out_cap;
    const int64_t roff = fa.spyral ? fa.row_offsets[slot_event] : 0;
    const uint4* staged = fa.staged + (int64_t)L * chunk.hash_cap;
    const bool replayed = fa.replay.offsets != nullptr;
    const bool packed = fa.col_wiggle != nullptr;
    __shared__ unsigned s_tb[NUM_TB];  // packed columns: rows of the event per time bucket
    if (packed) {
        for (int b = threadIdx.x; b < NUM_TB; b += EMIT_THREADS) s_tb[b] = 0u;
        __syncthreads();
    }
    const int lane = threadIdx.x & 31;
    for (int i0 = threadIdx.x - lane; i0 < n; i0 += EMIT_THREADS) {  // (warp-uniform trip count)
        const int i = i0 + lane;
        const bool valid = i < n;
        const uint4 s = valid ? __ldcs(staged + i) : make_uint4(0xFFFF0000u, 0u, 0u, 0u);
        const unsigned tb = s.x >> 16, pad = (s.z >> 16) & 0x7FFFu, rk = s.w & 0xFu;
        if (packed) {  // rows come in time-bucket order: a warp sees a few runs, one shared-memory add per run
            const unsigned peers = __match_any_sync(FULL, tb);
            if (valid && lane == __ffs(peers) - 1) atomicAdd(&s_tb[min(tb, (unsigned)NUM_TB - 1u)], (unsigned)__popc(peers));
        }
        if (!valid) continue;
        const unsigned long long q = ((unsigned long long)(s.z & 0xFFFFu) << 32) | s.y;
        uint32_t u16 = s.x & 0xFFFFu;
        double u = (double)u16 * (1.0 / 65536.0);
        if (replayed) {
            u = wiggle_of(fa, slot_event, szudzik_pair(tb, pad), ctr);
            u16 = (uint32_t)(u * 65536.0);
        }
        const double tbf = (double)tb + u;
        const int64_t label = fa.label_of_event_rank
                                  ? (int64_t)fa.label_of_event_rank[(int64_t)slot_event * fa.n_tracks_per_event + rk]
                                  : (int64_t)fa.label_of_rank[rk];
        const int64_t r = off + i;
        if (fa.cloud) {  // (null: typed columns only, nobody reads the float64 rows)
            double* row = fa.cloud + r * 3;
            row[0] = (double)pad;
            row[1] = tbf;
            row[2] = (double)(long long)q;
            fa.labels[r] = label;
        }
        if (fa.col_pad) {  // only the columns that will be copied are written
            if (packed) {
                fa.col_pad[r] = (int16_t)(pad | (rk << fa.rank_shift));
                fa.col_wiggle[r] = (uint16_t)u16;
            } else {
                fa.col_pad[r] = (int16_t)pad;
                fa.col_tb_q16[r] = (tb << 16) | u16;
                fa.col_label[r] = (int8_t)label;
            }
            if (fa.col_electrons) fa.col_electrons[r] = (long long)q;
            if (fa.col_electrons32) {
                fa.col_electrons32[r] = (uint32_t)q;
                if (q >> 32) {
                    const unsigned long long k = atomicAdd(fa.big_count, 1ULL);
                    if ((int64_t)k < fa.big_cap) {
                        fa.big_rows[k] = r;
                        fa.big_electrons[k] = (long long)q;
                    }
                }
            }
        }
        if (spy && (s.z >> 31))
            put_spyral_row(P, fa.rsink, roff + (s.w >> 4), (double)pad, tbf, (tb << 16) | u16, (double)(long long)q,
                           label);
    }
    if (packed) {
        __syncthreads();
        uint16_t* counts = fa.tb_counts + (int64_t)slot_event * NUM_TB;
        for (int b = threadIdx.x; b < NUM_TB; b += EMIT_THREADS) counts[b] = (uint16_t)s_tb[b];
    }
}

}  // namespace attpc
