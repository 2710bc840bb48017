/*
 * attpc_b200.h -- C ABI of libattpc_b200.so, the B200 (sm_100a) implementation of the
 * detector-simulation hot path of ATTPC/attpc_engine v0.9.0.
 *
 * The reference is pure Python; the functions below are what a reference-side binding (ctypes, see
 * INTEGRATION.md) would call instead of the numba/scipy code named beside each entry.  Paths are
 * relative to /root/reference/src/attpc_engine/.  Plain pointers and sizes only; all pointers are HOST
 * pointers unless the name ends in `_dev`.  Inputs are borrowed for the duration of the call.  Outputs
 * are library-owned pinned host buffers that stay valid until the next call on the same handle (or
 * attpc_destroy).  One handle per GPU; a handle must not be used from two threads at once; different
 * handles are independent.  Every function returns 0 on success or a negative ATTPC_E_* code;
 * attpc_last_error() gives the message.  Nothing here ever falls back to a CPU path.
 */
#ifndef ATTPC_B200_H
#define ATTPC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ATTPC_ABI_VERSION 8

enum {
    ATTPC_OK = 0,
    ATTPC_E_BADARG = -1,   /* null pointer, negative size, inconsistent indices */
    ATTPC_E_CUDA = -2,     /* a CUDA runtime call or kernel failed              */
    ATTPC_E_CAPACITY = -3, /* an internal buffer is still too small after the automatic retries */
    ATTPC_E_NOMEM = -4
};

/* flags for attpc_simulate / attpc_simulate_replay */
enum {
    ATTPC_KEEP_ALL_TB = 1u << 0,   /* skip the 0 <= tb < 512 mask of detector/simulator.py:111-113 (tests) */
    ATTPC_SPYRAL_ROWS = 1u << 1,   /* also produce the 8-column Spyral rows (detector/writer.py:61-112,232-238) */
    ATTPC_NO_WIGGLE = 1u << 2,     /* add 0 instead of U[0,1) to the time bucket (tests) */
    ATTPC_SKIP_HOST_COPY = 1u << 3,/* leave results in device memory only (device-resident benchmarking) */
    ATTPC_ROWS_KEEP_ALL = 1u << 4, /* attpc_convert_to_spyral: every row, input order (no threshold, no sort) */
    ATTPC_SKIP_CLOUD_COPY = 1u << 5,/* with ATTPC_SPYRAL_ROWS: copy offsets and rows to the host, not the raw cloud */
    ATTPC_COLUMNS = 1u << 6,       /* host result as typed columns (col_* of AttpcResult, 15 B/row) instead of the
                                      float64 cloud + int64 labels (32 B/row); same rows, same order */
    ATTPC_COLUMNS32 = 1u << 8,     /* with ATTPC_COLUMNS: electrons as uint32 (low 32 bits) + a list of the (row, count)
                                      pairs that need more: 11 B/row.  A call with more than 2^20 such rows returns
                                      the int64 column instead (and so do the later calls on the handle) */
    ATTPC_SPYRAL_COLUMNS = 1u << 9,/* the Spyral rows (after ADC threshold, z-sorted) as typed columns instead of float64
                                      [M, 8]: row_col_* of AttpcResult, 13 B/row.  x, y, pad size follow from the pad id,
                                      z from the time bucket, amplitude and integral from the electrons: the host rebuilds
                                      the eight columns bit for bit */
    ATTPC_COLUMNS_PACKED = 1u << 10,/* with ATTPC_COLUMNS: 8 B/row + 1 KB/event instead of 11 B/row.  Rows are in ascending
                                      time-bucket order, so the integer time bucket travels as the number of rows per
                                      time bucket and event (tb_counts [n_events, 512] uint16), the wiggle as col_wiggle
                                      (uint16, k / 65536), and the track rank in the two bits above the 14-bit pad id
                                      (pad_rank_shift = 14; label = the nucleus index of that rank).  Only when pad ids
                                      are below 16384, at most four tracks per event, the library's own wiggle and the
                                      time-bucket mask are in force; otherwise the call returns the columns above */
    ATTPC_EXACT_MESH = 1u << 7     /* validation: evaluate every mesh pixel with the reference's own expression
                                      (detector/transporter.py:36-41, 240-246).  The default reads pdf * step^2 from
                                      the constant 10x10 weight table and falls back to that expression only where
                                      rounding could change the integer share; both give identical results */
};

/* Scalars of DetectorParams / ElectronicsParams / Config (detector/parameters.py:10-76,164-174). */
typedef struct AttpcConfig {
    double length;          /* m */
    double efield;          /* V/m (positive; negated internally like detector/solver.py:299) */
    double bfield;          /* T   (positive; negated internally like detector/solver.py:298) */
    int64_t mpgd_gain;
    double diffusion;       /* V */
    double fano_factor;
    double w_value;         /* eV */
    double gas_density;     /* g/cm^3, GasTarget.density */
    int32_t micromegas_edge;
    int32_t windows_edge;   /* <= 8191: attpc_create returns ATTPC_E_BADARG otherwise */
    double adc_threshold;
    double drift_velocity;  /* m / time bucket, Config.drift_velocity */
    double grid_low_mm;     /* pad_grid_edges[0] */
    double grid_high_mm;    /* pad_grid_edges[1] */
    int32_t lut_origin_mm;  /* integer mm coordinate of LUT row/col 0 */
    int32_t lut_n;          /* LUT is lut_n x lut_n */
    /* integrator controls (no counterpart in the reference, which uses scipy Radau defaults) */
    double ode_rtol;
    double ode_atol;
    double freeze_ke_mev;   /* energy budget n* W [MeV] of the "can never make another electron" test that ends a
                               stalled track early (0 = integrate to 1 us like the reference) */
    /* capacities (0 = library default); they grow automatically on overflow */
    int32_t max_events_per_launch;
    int32_t hash_capacity;          /* slots per event, power of two */
    int32_t copy_events_per_launch; /* events per host-copy chunk: rows are copied while later groups compute */
    /* stress knobs for tests (0 = library default; values above the default are clamped): results never depend on them */
    int32_t unit_points;            /* points of one event handled by one CTA of the deposit kernel (default 1024) */
    int32_t table_spill_keys;       /* keys in a CTA's shared-memory table that trigger an append to the event's list */
    /* longitudinal diffusion (an extension: the reference has none), V, same meaning as `diffusion`; 0 = off, the
       reference's behaviour.  A point of drift time t [time buckets] is spread over the buckets
       floor(t -+ 3 sigma_L), sigma_L = sqrt(2 D_L dv t / efield) / dv, bucket k receiving
       (int64)(q (Phi((k + 1 - t) / sigma_L) - Phi((k - t) / sigma_L))) electrons; every bucket of the window
       then goes through the transverse 10x10 mesh like a point of its own ("sub-point").  Must be finite, >= 0. */
    double longitudinal_diffusion;
} AttpcConfig;

/* One ion species: the dE/dx table of attpc_engine_b200/target.py:DedxTable (pseudo-log grid). */
typedef struct AttpcSpecies {
    int32_t z;
    int32_t a;
    double mass;            /* nuclear mass, MeV/c^2 */
    int32_t lm;             /* log2(nodes per octave) */
    int32_t e_min;          /* binary exponent of the first node */
    int32_t n_oct;          /* octaves covered; table has n_oct * 2^lm + 1 values */
    int32_t reserved0;
    const double* dedx;     /* MeV/(g/cm^2), replaces GasTarget.get_dedx (detector/solver.py:64-66) */
} AttpcSpecies;

/* Optional replay of the reference's random numbers (SURVEY.md App. A). */
typedef struct AttpcReplay {
    /* TB-wiggle uniforms, keyed by Szudzik id: for event e the pairs
       (u_keys[i], u_vals[i]), u_offsets[e] <= i < u_offsets[e+1], sorted by key. */
    const int64_t* u_offsets; /* [n_events + 1] */
    const int64_t* u_keys;
    const double* u_vals;
} AttpcReplay;

/* Result of one batch (all pointers are library-owned pinned host memory unless *_dev). */
typedef struct AttpcResult {
    int64_t n_events;
    int64_t n_points;           /* rows in cloud / labels */
    const int64_t* offsets;     /* [n_events + 1] row range of each event */
    const double* cloud;        /* [n_points, 3] = pad, time bucket (float), electrons -- detector/simulator.py:104-115 */
    const int64_t* labels;      /* [n_points] index of the nucleus that last touched the point */
    int64_t n_rows;             /* Spyral rows (ATTPC_SPYRAL_ROWS), after ADC threshold, z-sorted per event */
    const int64_t* row_offsets; /* [n_events + 1] */
    const double* rows;         /* [n_rows, 8] = x, y, z, amplitude, integral, pad, tb, pad size */
    const int64_t* row_labels;  /* [n_rows] */
    /* device copies of the same arrays (valid until the next call) */
    const int64_t* offsets_dev;
    const double* cloud_dev;
    const int64_t* labels_dev;
    /* workload statistics of the batch */
    int64_t n_tracks;            /* charged tracks integrated */
    int64_t n_trajectory_points; /* 0.1 ns grid points emitted by the integrator */
    int64_t n_active_points;     /* points with >= 1 electron (detector/solver.py:387) */
    int64_t n_primary_electrons; /* sum of those electrons before mpgd_gain */
    int64_t n_deposits;          /* pixel deposits attempted (100 per active point when sigma > 0; with longitudinal
                                    diffusion 100 per sub-point, i.e. per time bucket of each point's window) */
    int64_t n_keys;              /* distinct (pad, tb) keys before the time-bucket mask */
    /* device time of each stage in ms (CUDA events on the library's stream) */
    float ms_h2d, ms_tracks, ms_deposit, ms_finalize, ms_d2h, ms_total;
    int32_t n_kernel_launches;
    int32_t n_retries;           /* capacity retries that happened inside the call */
    int32_t n_track_launches;    /* launches of the track (or replay) kernel */
    int32_t n_group_launches;    /* launches of the deposit kernel (= event groups processed) */
    int64_t n_hash_probes;       /* table slots inspected by the deposits (n_hash_probes / n_deposits ~ 1 is healthy) */
    int32_t hash_capacity;       /* slots per event in use at the end of the call */
    int32_t reserved1;
    int64_t n_table_flushes;     /* shared-memory tables appended to an event's entry list before the end of their work unit */
    /* ATTPC_COLUMNS: the rows of `cloud` / `labels` as typed columns (pinned host memory) */
    const int16_t* col_pad;      /* [n_points] pad id */
    const uint32_t* col_tb_q16;  /* [n_points] time bucket + wiggle as Q16.16 fixed point: cloud[:, 1] == col_tb_q16 / 65536
                                    exactly (the library's wiggle has 16 bits; a replayed 53-bit uniform is truncated here) */
    const int64_t* col_electrons;/* [n_points] electrons (after gain) */
    const int8_t* col_label;     /* [n_points] index of the nucleus that last touched the point */
    /* integrator statistics (SURVEY.md 8d: right-hand-side evaluations = 6 * n_rk_steps + n_tracks) */
    int64_t n_rk_steps;          /* Dormand-Prince steps tried (accepted + rejected) */
    int64_t n_rk_rejects;        /* of which rejected by the error control */
    int64_t max_track_passes;    /* most step/emit passes any single track needed: the serial critical path */
    /* ATTPC_COLUMNS32: either col_electrons32 (+ the exceptions) or col_electrons is set, never both */
    const uint32_t* col_electrons32; /* [n_points] electrons modulo 2^32 */
    int64_t n_big;                   /* rows whose count is >= 2^32 */
    const int64_t* big_rows;         /* [n_big] row index (unordered) */
    const int64_t* big_electrons;    /* [n_big] full count of that row */
    float ms_order;              /* device time of the point ordering kernels (scan + scatter, and with longitudinal
                                    diffusion the split into sub-points) before the deposit kernel;
                                    ms_deposit is the deposit kernel alone */
    float reserved2;
    /* ATTPC_SPYRAL_COLUMNS: rows [row_offsets[e], row_offsets[e+1]) of event e, in the order of `rows` */
    const int16_t* row_col_pad;      /* [n_rows] pad id */
    const uint32_t* row_col_tb_q16;  /* [n_rows] time bucket + wiggle, Q16.16 */
    const uint32_t* row_col_e_lo;    /* [n_rows] electrons (after gain), bits 0..31 */
    const uint16_t* row_col_e_hi;    /* [n_rows] electrons, bits 32..47 */
    const int8_t* row_col_label;     /* [n_rows] */
    /* ATTPC_COLUMNS_PACKED (set only when the call could use it; col_tb_q16 and col_label are then null):
       col_pad = pad | rank << pad_rank_shift */
    const uint16_t* col_wiggle;      /* [n_points] wiggle * 65536 */
    const uint16_t* tb_counts;       /* [n_events, 512] rows of event e in time bucket t */
    int32_t pad_rank_shift;          /* 14, or 0 when the call is not packed */
    int32_t reserved3;
} AttpcResult;

typedef struct AttpcSim AttpcSim;

/* Version of this ABI (ATTPC_ABI_VERSION) -- lets a binding refuse a mismatched library. */
int attpc_abi_version(void);

/* Number of CUDA devices visible, or a negative error code. */
int attpc_device_count(void);

/* Build a simulator on CUDA device `device`.
 * Replaces the per-run setup of detector/parameters.py:145-261 (Config) plus the tables the hot loop
 * reads: pad_lut = the 1 mm sub-lattice of Config.pad_grid actually addressed by
 * detector/transporter.py:102-120, with beam pads (detector/beam_pads.py) and holes folded to -1;
 * pad_xy / pad_scale = Config.pad_centers / Config.pad_sizes; response = detector/response.py:8-32. */
int attpc_create(const AttpcConfig* cfg, const int16_t* pad_lut, const double* pad_xy, const double* pad_scale,
                 int32_t n_pads, const double* response, int32_t n_response, const AttpcSpecies* species,
                 int32_t n_species, int32_t device, AttpcSim** out);

void attpc_destroy(AttpcSim* sim);

/* Message of the last error on this handle (never NULL).  With sim == NULL: last attpc_create error. */
const char* attpc_last_error(const AttpcSim* sim);

/* The whole hot path for a batch of events:
 * detector/simulator.py:52-115 (simulate) applied to events first_event .. first_event + n_events - 1, i.e.
 * detector/solver.py:243-305 (trajectory), :308-347 (electrons), :386-398 (mask, gain, z -> tb),
 * detector/transporter.py:252-317 (drift + pad lookup + accumulate), detector/simulator.py:19-49,104-115.
 *   momenta        [n_events, n_nuclei, 4]  (px, py, pz, E) in MeV
 *   vertices       [n_events, 3]            m
 *   track_nucleus  [n_tracks_per_event]     index into the n_nuclei axis, in `indices` order
 *   track_species  [n_tracks_per_event]     index into the species array of attpc_create, or -1 to skip
 *                                           (the reference skips Z == 0, detector/simulator.py:97)
 * Random numbers: Philox4x32-10 keyed by (seed; global event id, nucleus index, grid step) for the Fano
 * normals and (seed; global event id, Szudzik key) for the time-bucket wiggle, so results do not depend on
 * batching or on which GPU ran the event. */
int attpc_simulate(AttpcSim* sim, const double* momenta, const double* vertices, int64_t n_events, int32_t n_nuclei,
                   const int32_t* track_nucleus, const int32_t* track_species, int32_t n_tracks_per_event,
                   uint64_t seed, int64_t first_event, uint32_t flags, AttpcResult* result);

/* Same, with inputs already in device memory (pointers from cudaMalloc on the handle's device). */
int attpc_simulate_dev(AttpcSim* sim, const double* momenta_dev, const double* vertices_dev, int64_t n_events,
                       int32_t n_nuclei, const int32_t* track_nucleus, const int32_t* track_species,
                       int32_t n_tracks_per_event, uint64_t seed, int64_t first_event, uint32_t flags,
                       AttpcResult* result);

/* Parity entry: everything after the trajectory, from GIVEN trajectory points and GIVEN random numbers --
 * detector/solver.py:308-347,386-398 + detector/transporter.py:252-317 + detector/simulator.py:104-115.
 *   track_offsets [n_tracks + 1]   row range of each track in `points`
 *   points        [n_rows, 6]      (x, y, z, gbx, gby, gbz) rows as returned by generate_trajectory
 *   normals       [n_rows]         standard normals z_k: electrons_k = (int64)(n_k + sqrt(F n_k) z_k)
 *   track_event   [n_tracks]       event slot 0 .. n_events-1
 *   track_rank    [n_tracks]       position of the track in the event's `indices` list (label precedence)
 *   track_label   [n_tracks]       label value written for the track (the nucleus index)
 *   track_species [n_tracks]
 *   electrons_out [n_rows] or NULL receives electrons_k (before the >= 1 mask and the gain) */
int attpc_simulate_replay(AttpcSim* sim, const int64_t* track_offsets, const double* points, const double* normals,
                          const int32_t* track_event, const int32_t* track_rank, const int32_t* track_label,
                          const int32_t* track_species, int64_t n_tracks, int64_t n_events,
                          const AttpcReplay* replay, uint32_t flags, int64_t* electrons_out, AttpcResult* result);

/* Trajectories only (tests of the integrator against scipy): detector/solver.py:243-305.
 *   momenta [n_tracks, 4], vertices [n_tracks, 3], species [n_tracks]
 *   out_points [n_tracks, max_points, 6] receives rows for grid steps 0, stride, 2*stride, ...
 *   out_counts [n_tracks] receives the number of 0.1 ns grid points of the track (like len(track)). */
int attpc_trajectories(AttpcSim* sim, const double* momenta, const double* vertices, const int32_t* species,
                       int64_t n_tracks, int32_t stride, int32_t max_points, double* out_points, int32_t* out_counts);

/* detector/writer.py:61-112 + :232-238 on a host cloud: rows, ADC threshold, per-event z-sort.
 *   offsets [n_events+1], cloud [n_points,3], labels [n_points]; results in result->rows etc.
 *   flags: ATTPC_ROWS_KEEP_ALL = plain convert_to_spyral (detector/writer.py:61-112 only).
 * Needs no species: a handle created with n_species == 0 can only convert. */
int attpc_convert_to_spyral(AttpcSim* sim, const int64_t* offsets, const double* cloud, const int64_t* labels,
                            int64_t n_events, uint32_t flags, AttpcResult* result);

/* Pad lookup of detector/transporter.py:78-120 + the veto of :165,237 for n positions (metres). */
int attpc_lookup_pads(AttpcSim* sim, const double* xy, int64_t n, int32_t* pads_out);

/* Copy n_bytes from one of the *_dev arrays of the handle's last result into host memory (results of a call made with
 * ATTPC_SKIP_HOST_COPY stay on the device; this is how a caller without a CUDA binding of its own reads them). */
int attpc_read_device(AttpcSim* sim, const void* dev, void* host, int64_t n_bytes);

#ifdef __cplusplus
}
#endif
#endif /* ATTPC_B200_H */
