// libattpc_b200.so -- host side of the C ABI declared in include/attpc_b200.h.
//
// One AttpcSim per GPU.  A call to attpc_simulate* walks the batch in "launches" (many events, so the
// latency-bound track integrator has tens of thousands of lanes in flight) and each launch in "groups" of a few
// hundred events whose accumulation tables (hash_cap x 16 B per event) fit the 126 MB L2 together: the deposit
// and finalize kernels of a group therefore never touch HBM except for the compact CSR they emit.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <utility>
#include <vector>

#include "../../include/attpc_b200.h"
#include "attpc_kernels.cuh"

using namespace attpc;

namespace {

thread_local std::string g_create_error = "";

constexpr double E_CHARGE = 1.602176634e-19;
constexpr double MEV_2_JOULE = E_CHARGE * 1.0e6;
constexpr double MEV_2_KG = (E_CHARGE / (C_LIGHT * C_LIGHT)) * 1.0e6;

template <typename T>
struct DevArray {
    T* p = nullptr;
    int64_t n = 0;
    DevArray() = default;
    DevArray(const DevArray&) = delete;
    DevArray& operator=(const DevArray&) = delete;
    DevArray(DevArray&& o) noexcept : p(std::exchange(o.p, nullptr)), n(std::exchange(o.n, 0)) {}
    DevArray& operator=(DevArray&& o) noexcept {
        if (this != &o) {
            release();
            p = std::exchange(o.p, nullptr);
            n = std::exchange(o.n, 0);
        }
        return *this;
    }
    ~DevArray() { release(); }
    cudaError_t reserve(int64_t want, bool keep = false, cudaStream_t s = 0) {
        if (want <= n) return cudaSuccess;
        T* q = nullptr;
        cudaError_t e = cudaMalloc((void**)&q, (size_t)want * sizeof(T));
        if (e != cudaSuccess) return e;
        if (keep && p && n > 0) {
            e = cudaMemcpyAsync(q, p, (size_t)n * sizeof(T), cudaMemcpyDeviceToDevice, s);
            if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        }
        if (p) cudaFree(p);
        p = q;
        n = want;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
    }
};

template <typename T>
struct PinnedArray {
    T* p = nullptr;
    int64_t n = 0;
    PinnedArray() = default;
    PinnedArray(const PinnedArray&) = delete;
    PinnedArray& operator=(const PinnedArray&) = delete;
    PinnedArray(PinnedArray&& o) noexcept : p(std::exchange(o.p, nullptr)), n(std::exchange(o.n, 0)) {}
    PinnedArray& operator=(PinnedArray&& o) noexcept {
        if (this != &o) {
            release();
            p = std::exchange(o.p, nullptr);
            n = std::exchange(o.n, 0);
        }
        return *this;
    }
    ~PinnedArray() { release(); }
    cudaError_t reserve(int64_t want, bool keep = false) {
        if (want <= n) return cudaSuccess;
        want += want / 4;  // pinning is slow (~0.5 s/GB): grow with slack so that it is rare
        T* q = nullptr;
        cudaError_t e = cudaHostAlloc((void**)&q, (size_t)want * sizeof(T), cudaHostAllocMapped);
        if (e != cudaSuccess) return e;
        if (keep && p && n > 0) memcpy(q, p, (size_t)n * sizeof(T));
        if (p) cudaFreeHost(p);
        p = q;
        n = want;
        return e;
    }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        n = 0;
    }
};

// An output with one row per cloud row or per Spyral row: the device array the kernels write, the pinned mirror its
// rows are copied to, and the bytes of one row.  Sink<T, W> (W values of type T per row) gives typed access.
struct RowSink {
    DevArray<char> dev;
    PinnedArray<char> host;
    const int64_t row_bytes;
    explicit RowSink(int64_t bytes) : row_bytes(bytes) {}
    cudaError_t reserve(int64_t rows, bool keep, cudaStream_t s) { return dev.reserve(rows * row_bytes, keep, s); }
    cudaError_t reserve_host(int64_t rows, bool keep) { return host.reserve(rows * row_bytes, keep); }
    cudaError_t copy_to_host(int64_t first, int64_t rows, cudaStream_t s) {
        return cudaMemcpyAsync(host.p + first * row_bytes, dev.p + first * row_bytes, (size_t)(rows * row_bytes),
                               cudaMemcpyDeviceToHost, s);
    }
};

template <typename T, int W = 1>
struct Sink : RowSink {
    Sink() : RowSink(W * (int64_t)sizeof(T)) {}
    T* d() const { return reinterpret_cast<T*>(dev.p); }
    T* h() const { return reinterpret_cast<T*>(host.p); }
};

}  // namespace

constexpr int64_t ATTPC_BIG_CAP = 1 << 20;  // (row, count) exceptions of the compact electrons column per call
// Groups per chunk when points are split into sub-points: bounds the sub-point records (160 B each, up to
// long_buckets per point) held at once, at the price of more (shorter) launches
constexpr int64_t SUB_CHUNK_GROUPS = 4;

struct AttpcSim {
    int device = 0;
    cudaStream_t stream = nullptr;
    SimParams P{};
    AttpcConfig cfg{};
    std::string error;
    int sm_count = 148;
    bool tables_in_smem = true;
    int track_warps_max = TRACK_THREADS / 32;  // warps per track CTA that fit beside the tables in shared memory
    size_t table_smem_bytes = 0;

    // constants
    DevArray<int16_t> lut;
    DevArray<double> pad_xy, pad_scale, response, resp_sorted, resp_prefix, tables, stop_ns;
    DevArray<uint8_t> plan_cls;
    DevArray<unsigned> plan_counts;
    DevArray<int32_t> plan_order;

    // sizing
    int32_t launch_events = 32768;
    int32_t copy_launch_events = 4096;  // rows go to the host in chunks of this many events (measured optimum, tools/run_r2_e2e_sweep.sh)
    int32_t group_events = 2048;
    int32_t chunk_groups = 16;  // groups per kernel launch when the rows stay on the device
    int32_t unit_points = UNIT_POINTS;     // test knobs (AttpcConfig.unit_points / table_spill_keys)
    int32_t spill_keys = SMEM_SPILL_DEFAULT;
    int64_t big_cap = ATTPC_BIG_CAP;             // exceptions accepted before a call returns the int64 column (<= ATTPC_BIG_CAP)
    int32_t hash_cap = 16384;
    int64_t group_point_cap = 0;

    // work buffers; the arrays the track kernel fills exist twice so that the track kernel of launch i+1 can run
    // (on its own stream) while the deposit / finalize kernels of launch i consume the other set
    struct LaunchSlot {
        DevArray<double> px, py, pt;
        DevArray<long long> pq;
        DevArray<int32_t> pev, prank;
        DevArray<uint32_t> pj;
        DevArray<unsigned> group_count, pcnt;
        DevArray<Counters> counters;
        PinnedArray<Counters> counters_host;
        void release_points() {
            px.release(); py.release(); pt.release(); pq.release(); pev.release(); prank.release(); pj.release();
        }
    } slot[2];
    cudaStream_t stream_t = nullptr, stream_c = nullptr;  // track kernels, device-to-host copies
    std::vector<cudaEvent_t> sync_events;                 // untimed events for cross-stream ordering
    size_t sync_used = 0;
    DevArray<unsigned long long> csr_total;
    PinnedArray<unsigned long long> csr_host;
    PinnedArray<unsigned long long> chunk_totals;  // running CSR total after each chunk of groups (mapped)
    DevArray<double> geom;
    DevArray<uint32_t> rec;
    DevArray<int32_t> unit_event, unit_first, unit_count, unit_order, n_units;
    DevArray<unsigned> pstart, n_entries, mode;
    int32_t ranks = 1;
    int32_t max_units = 0;
    int deposit_ctas = 0;                 // persistent deposit CTAs: as many as are resident at once
    DevArray<unsigned> deposit_cursor;    // next work unit of the chunk, zeroed before every deposit launch
    // longitudinal diffusion (P.long_diffusion > 0): geom / rec then hold the SUB-POINTS (one per time bucket of a
    // point's window) of one chunk of at most SUB_CHUNK_GROUPS groups, sub_cap per group
    int64_t sub_cap = 0;
    int32_t long_buckets = 0;   // most buckets one point can spread over: floor(6 sigma_L) + 2 at windows_edge + 1
    int32_t sub_max_units = 0;  // work units per group over sub-points
    DevArray<unsigned> nsub, sub_cnt, sub_start;  // per point: sub-point offset in its list; per (event, rank) list
    DevArray<unsigned long long> sub_total;       // [SUB_CHUNK_GROUPS] sub-points per group of the chunk
    DevArray<HashEntry> hash;
    DevArray<uint64_t> sort_items;
    DevArray<uint4> staged;  // ordered rows of the chunk's events between order_kernel and emit_kernel
    DevArray<unsigned> big_list;  // events queued for order_queue_kernel: two lists of [chunk events] + 2 x {count, cursor}
    int64_t big_list_events = 0;
    DevArray<unsigned> kept;
    DevArray<double> in_momenta, in_vertices;

    // outputs.  The row-indexed ones are sinks, reserved and copied through the lists of an OutputPlan; every sink a
    // call uses holds out_rows rows (the Spyral rows of an event are a subset of its cloud rows).
    int64_t out_rows = 0;
    Sink<double, 3> cloud;
    Sink<int64_t> labels;
    Sink<int16_t> col_pad;
    Sink<uint32_t> col_tbq, col_q32;
    Sink<int64_t> col_q;
    Sink<int8_t> col_label;
    Sink<uint16_t> col_wig;  // ATTPC_COLUMNS_PACKED: wiggle
    Sink<double, 8> rows;    // thresholded, z-ordered Spyral rows
    Sink<int64_t> row_labels;
    Sink<int16_t> rcol_pad;  // ... as typed columns (ATTPC_SPYRAL_COLUMNS)
    Sink<uint32_t> rcol_tbq, rcol_elo;
    Sink<uint16_t> rcol_ehi;
    Sink<int8_t> rcol_label;
    DevArray<int64_t> offsets_dev, row_offsets_dev, big_rows_dev, big_q_dev;
    PinnedArray<int64_t> offsets_host, row_offsets_host, big_rows_host, big_q_host;
    DevArray<uint16_t> tbc_dev;  // ATTPC_COLUMNS_PACKED: rows per (event, time bucket)
    PinnedArray<uint16_t> tbc_host;
    bool q32_off = false;  // sticky: a call overflowed the exception list (heavy ions): later calls copy int64 directly
    DevArray<unsigned> row_kept;
    DevArray<uint64_t> row_sort_keys;
    DevArray<uint32_t> row_sort_idx;

    std::vector<cudaEvent_t> events;
    size_t events_used = 0;
    int launches = 0;

    ~AttpcSim() {  // the arrays free themselves after this
        for (cudaStream_t s : {stream, stream_t, stream_c})
            if (s) cudaStreamSynchronize(s);
        for (auto e : events) cudaEventDestroy(e);
        for (auto e : sync_events) cudaEventDestroy(e);
        for (cudaStream_t s : {stream, stream_t, stream_c})
            if (s) cudaStreamDestroy(s);
    }

    int fail(int code, const char* fmt, ...) {
        char buf[512];
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(buf, sizeof buf, fmt, ap);
        va_end(ap);
        error = buf;
        return code;
    }
    cudaEvent_t mark(cudaStream_t s = nullptr) {
        if (events_used == events.size()) {
            cudaEvent_t e;
            cudaEventCreate(&e);
            events.push_back(e);
        }
        cudaEvent_t e = events[events_used++];
        cudaEventRecord(e, s ? s : stream);
        return e;
    }
    cudaEvent_t fence(cudaStream_t s) {  // untimed event recorded on s
        if (sync_used == sync_events.size()) {
            cudaEvent_t e;
            cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
            sync_events.push_back(e);
        }
        cudaEvent_t e = sync_events[sync_used++];
        cudaEventRecord(e, s);
        return e;
    }
};

#define CU(call)                                                                                           \
    do {                                                                                                   \
        cudaError_t _e = (call);                                                                           \
        if (_e != cudaSuccess)                                                                             \
            return sim->fail(ATTPC_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, \
                             __LINE__);                                                                    \
    } while (0)

namespace {

int next_pow2(int64_t v) {
    int64_t p = 1;
    while (p < v) p <<= 1;
    return (int)p;
}

// 64-bit words of scratch per event for the entry lists that the ordering kernels cannot keep in shared memory: two item
// arrays and two bit-mask / running-count arrays
int64_t scratch_stride(int64_t hash_cap) { return 2 * hash_cap + hash_cap / 32 + 2; }

// `chunk_groups`: groups whose kernels run in one launch (run_groups): sizes the per-event entry lists, the ordering
// scratch and the staged rows -- the big buffers (16 B x hash_cap per event each).
int ensure_work_buffers(AttpcSim* sim, int64_t launch_events, int32_t ranks, int64_t chunk_groups) {
    const int64_t n_groups = (launch_events + sim->group_events - 1) / sim->group_events;
    if (sim->group_point_cap == 0) sim->group_point_cap = (int64_t)sim->group_events * 1024;
    const int64_t pts = n_groups * sim->group_point_cap;
    sim->ranks = ranks;
    for (auto& ls : sim->slot) {
        CU(ls.px.reserve(pts));
        CU(ls.py.reserve(pts));
        CU(ls.pt.reserve(pts));
        CU(ls.pq.reserve(pts));
        CU(ls.pev.reserve(pts));
        CU(ls.prank.reserve(pts));
        CU(ls.pj.reserve(pts));
        CU(ls.group_count.reserve(n_groups));
        CU(ls.pcnt.reserve(launch_events * ranks));
        CU(ls.counters.reserve(1));
        CU(ls.counters_host.reserve(1));
    }
    sim->max_units = (int32_t)(sim->group_events + sim->group_point_cap / sim->unit_points + 1);
    int64_t units = sim->max_units;
    if (sim->P.long_diffusion > 0.0) {
        // first guess 256 points per event, each spread over long_buckets; grown on overflow (overflow_sub)
        if (sim->sub_cap == 0) sim->sub_cap = (int64_t)sim->group_events * 256 * std::min(sim->long_buckets, 16);
        const int64_t subs = std::min<int64_t>(n_groups, SUB_CHUNK_GROUPS) * sim->sub_cap;
        CU(sim->geom.reserve(subs * GEOM_DOUBLES));
        CU(sim->rec.reserve(subs * REC_WORDS));
        CU(sim->nsub.reserve(pts));
        CU(sim->sub_cnt.reserve(launch_events * ranks));
        CU(sim->sub_start.reserve(launch_events * ranks));
        CU(sim->sub_total.reserve(SUB_CHUNK_GROUPS));
        sim->sub_max_units = (int32_t)(sim->group_events + sim->sub_cap / sim->unit_points + 1);
        units = std::max<int64_t>(units, sim->sub_max_units);
    } else {
        CU(sim->geom.reserve(pts * GEOM_DOUBLES));
        CU(sim->rec.reserve(pts * REC_WORDS));
    }
    CU(sim->unit_event.reserve(n_groups * units));
    CU(sim->unit_first.reserve(n_groups * units));
    CU(sim->unit_count.reserve(n_groups * units));
    CU(sim->unit_order.reserve(n_groups * units));
    CU(sim->n_units.reserve(n_groups));
    CU(sim->pstart.reserve(launch_events * ranks));
    CU(sim->n_entries.reserve(launch_events));
    CU(sim->mode.reserve(launch_events));
    // tables and sort scratch for one chunk of groups (run_groups)
    int64_t table_groups = std::min<int64_t>(n_groups, std::max<int64_t>(1, chunk_groups));
    if (sim->P.long_diffusion > 0.0) table_groups = std::min<int64_t>(table_groups, SUB_CHUNK_GROUPS);  // run_groups' chunks
    CU(sim->hash.reserve(table_groups * sim->group_events * sim->hash_cap));
    CU(sim->sort_items.reserve(table_groups * sim->group_events * scratch_stride(sim->hash_cap)));
    CU(sim->staged.reserve(table_groups * sim->group_events * sim->hash_cap));
    sim->big_list_events = std::max<int64_t>(sim->big_list_events, table_groups * sim->group_events);
    CU(sim->big_list.reserve(2 * sim->big_list_events + 4));
    CU(sim->csr_total.reserve(3));  // cloud rows, electron counts >= 2^32, Spyral rows
    CU(sim->csr_host.reserve(3));
    CU(sim->chunk_totals.reserve(2 * (n_groups + 1)));
    return ATTPC_OK;
}

PointBuf point_buf(AttpcSim* sim, int which) {
    AttpcSim::LaunchSlot& ls = sim->slot[which];
    PointBuf pb;
    pb.x = ls.px.p;
    pb.y = ls.py.p;
    pb.t = ls.pt.p;
    pb.q = ls.pq.p;
    pb.ev = ls.pev.p;
    pb.rank = ls.prank.p;
    pb.j = ls.pj.p;
    pb.count = ls.group_count.p;
    pb.cnt = ls.pcnt.p;
    pb.start = sim->pstart.p;
    pb.geom = sim->geom.p;
    pb.rec = sim->rec.p;
    pb.unit_event = sim->unit_event.p;
    pb.unit_first = sim->unit_first.p;
    pb.unit_count = sim->unit_count.p;
    pb.unit_order = sim->unit_order.p;
    pb.n_units = sim->n_units.p;
    pb.max_units = sim->max_units;
    pb.unit_points = sim->unit_points;
    pb.group_cap = sim->group_point_cap;
    pb.group_events = sim->group_events;
    pb.ranks = sim->ranks;
    return pb;
}

// The sub-points of the chunk whose first group is g0 (longitudinal diffusion), as the point_scan and deposit kernels
// read points: records from sim->rec / sim->geom, lists counted in sub_cnt, groups numbered from 0 inside the chunk.
PointBuf sub_buf(AttpcSim* sim, int which, int64_t g0) {
    PointBuf sb = point_buf(sim, which);
    sb.cnt = sim->sub_cnt.p;
    sb.start = sim->sub_start.p;
    sb.max_units = sim->sub_max_units;
    sb.unit_event += g0 * sb.max_units;
    sb.unit_first += g0 * sb.max_units;
    sb.unit_count += g0 * sb.max_units;
    sb.unit_order += g0 * sb.max_units;
    sb.n_units += g0;
    sb.group_cap = sim->sub_cap;
    return sb;
}

template <bool RECORD>
int launch_tracks(AttpcSim* sim, const TrackBatch& tb, int64_t n_tracks, int which, cudaStream_t stream) {
    // The kernel is latency bound (FP64 dependency chains): spread the tracks over all SMs first, then add warps per
    // SM up to the one-CTA-per-SM limit the register file allows.  Lanes pull further tracks from a global cursor.
    const int64_t lanes_per_sm = (n_tracks + sim->sm_count - 1) / sim->sm_count;
    const int warps = (int)std::max<int64_t>(1, std::min<int64_t>(sim->track_warps_max, (lanes_per_sm + 31) / 32));
    const int threads = warps * 32;
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((n_tracks + threads - 1) / threads, sim->sm_count));
    PointBuf pb = point_buf(sim, which);
    Counters* ctr = sim->slot[which].counters.p;
    const size_t slot_bytes = (size_t)warps * TRACK_SLOT_BYTES_PER_WARP;
    if (sim->tables_in_smem) {
        auto kern = track_kernel<true, RECORD>;
        CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)(sim->track_warps_max * TRACK_SLOT_BYTES_PER_WARP + sim->table_smem_bytes)));
        kern<<<blocks, threads, slot_bytes + sim->table_smem_bytes, stream>>>(sim->P, tb, pb, ctr);
    } else {
        auto kern = track_kernel<false, RECORD>;
        CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)((TRACK_THREADS / 32) * TRACK_SLOT_BYTES_PER_WARP)));
        kern<<<blocks, threads, slot_bytes, stream>>>(sim->P, tb, pb, ctr);
    }
    sim->launches += 1;
    CU(cudaGetLastError());
    return ATTPC_OK;
}

struct SpyralPass {  // what run_groups needs to add the Spyral passes of a chunk (null: none)
    bool typed;
};
SpyralArgs spyral_args(AttpcSim* sim, int64_t first, int64_t n_events, bool typed, bool keep_all, const Counters* ctr);
int launch_spyral(AttpcSim* sim, const SpyralArgs& sa);

// deposit + finalize of every group of one launch; the track/replay kernel has already filled the point buffers.
// One entry per chunk of groups whose rows can be copied to the host as soon as `done` has fired.
struct ChunkFence {
    cudaEvent_t done;
    int64_t last_event;  // events [.., last_event) of the launch are final after this chunk
    int slot;            // index into sim->chunk_totals (running CSR total after the chunk)
};

int run_groups(AttpcSim* sim, int64_t launch_events, FinalizeArgs fa, int which,
               std::vector<std::pair<cudaEvent_t, cudaEvent_t>>& ord_marks,
               std::vector<std::pair<cudaEvent_t, cudaEvent_t>>& dep_marks,
               std::vector<std::pair<cudaEvent_t, cudaEvent_t>>& fin_marks, int groups_per_chunk,
               std::vector<ChunkFence>* fences, const SpyralPass* spyral, int64_t launch_first_event) {
    PointBuf pb = point_buf(sim, which);
    Counters* ctr = sim->slot[which].counters.p;
    const int64_t n_groups = (launch_events + sim->group_events - 1) / sim->group_events;
    fa.sort_items = sim->sort_items.p;
    fa.scratch_stride = scratch_stride(sim->hash_cap);
    fa.staged = sim->staged.p;
    fa.csr_total = sim->csr_total.p;
    // The second tier is persistent CTAs with 197 KB of shared memory.  Alone on the GPU they pay (device-resident
    // calls).  Beside the kernels of other engines and chunks (calls that copy to the host, pipelined) every one of
    // them, even with an empty queue, waits for an SM whose deposit CTAs have drained and holds up the stream behind
    // it: measured 2.25 -> 1.69 M events/s end to end (a two-per-SM, 98 KB variant: 2.25 -> 2.10 M, 0.54 -> 0.44 M
    // for 12C(a,a')3a).  Such calls order the lists beyond order_kernel's 8192 entries in global scratch (the third tier:
    // persistent CTAs again, but without dynamic shared memory - they fit beside anything and keep the whole L1).
    const bool use_big = fences == nullptr;
    unsigned* qbase = sim->big_list.p + 2 * sim->big_list_events;  // {big count, big cursor, far count, far cursor}
    fa.big = {use_big ? sim->big_list.p : nullptr, qbase, qbase + 1};
    fa.far = {sim->big_list.p + sim->big_list_events, qbase + 2, qbase + 3};
    auto big_kernel = order_queue_kernel<FIN_BIG_THREADS, FIN_BIG_ITEMS, 1>;
    auto far_kernel = order_queue_kernel<FIN_THREADS, 0, 2>;
    CU(cudaFuncSetAttribute(big_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FIN_BIG_SMEM_BYTES));
    CU(cudaFuncSetAttribute(order_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FIN_SMEM_BYTES));
    // Groups are processed in chunks: every kernel is launched once per chunk with one grid row per group (the deposit
    // kernel's persistent CTAs walk the chunk's groups in turn), so the ramp-up and tail of a launch are paid once per
    // chunk.  When rows go to the host a chunk is what is copied while the next chunk computes; otherwise it is as many
    // groups as the tables are sized for.
    const bool split = sim->P.long_diffusion > 0.0;
    int64_t gpc = std::max<int64_t>(1, fences ? groups_per_chunk : sim->chunk_groups);
    if (split) gpc = std::min<int64_t>(gpc, SUB_CHUNK_GROUPS);
    for (int64_t g0 = 0; g0 < n_groups; g0 += gpc) {
        const int64_t ng = std::min<int64_t>(gpc, n_groups - g0);
        GroupView gv;
        gv.first_slot = (int32_t)(g0 * sim->group_events);
        gv.n_events = (int32_t)std::min<int64_t>(ng * sim->group_events, launch_events - gv.first_slot);
        gv.group = (int32_t)g0;
        gv.hash_cap = sim->hash_cap;
        gv.tables = sim->hash.p;
        gv.n_entries = sim->n_entries.p;
        gv.mode = sim->mode.p;
        gv.exact_mesh = (fa.flags & ATTPC_EXACT_MESH) ? 1 : 0;
        gv.group_events = sim->group_events;
        gv.chunk_e0 = 0;
        gv.spill_keys = sim->spill_keys;
        cudaEvent_t d0 = sim->mark();
        const dim3 point_grid((unsigned)std::max<int64_t>(1, sim->sm_count * 4 / ng), (unsigned)ng);
        point_scan_kernel<<<(unsigned)ng, 1024, 0, sim->stream>>>(pb, gv, ctr);
        if (!split) {
            point_order_kernel<<<point_grid, 256, 0, sim->stream>>>(sim->P, pb, gv, ctr);
        } else {  // points -> one sub-point per time bucket of their window, then units over sub-points
            PointBuf sb = sub_buf(sim, which, g0);
            GroupView gvs = gv;
            gvs.group = 0;
            CU(cudaMemsetAsync(sim->sub_total.p, 0, (size_t)ng * sizeof(unsigned long long), sim->stream));
            sub_count_kernel<<<point_grid, 256, 0, sim->stream>>>(sim->P, pb, gv, ctr, sim->nsub.p);
            sub_scan_kernel<<<point_grid, 256, 0, sim->stream>>>(pb, sb, gv, ctr, sim->nsub.p, sim->sub_total.p);
            point_scan_kernel<<<(unsigned)ng, 1024, 0, sim->stream>>>(sb, gvs, ctr);
            sub_point_kernel<<<point_grid, 256, 0, sim->stream>>>(sim->P, pb, sb, gv, ctr, sim->nsub.p);
            sim->launches += 3;
        }
        CU(cudaMemsetAsync(sim->n_entries.p + gv.first_slot, 0, (size_t)gv.n_events * sizeof(unsigned), sim->stream));
        cudaEvent_t k0 = sim->mark();
        CU(cudaMemsetAsync(sim->deposit_cursor.p, 0, sizeof(unsigned), sim->stream));
        if (!split) {
            deposit_kernel<<<(unsigned)sim->deposit_ctas, DEPOSIT_THREADS, DEPOSIT_SMEM_BYTES, sim->stream>>>(
                sim->P, pb, gv, (int)ng, sim->deposit_cursor.p, ctr);
        } else {
            GroupView gvs = gv;
            gvs.group = 0;
            deposit_kernel<<<(unsigned)sim->deposit_ctas, DEPOSIT_THREADS, DEPOSIT_SMEM_BYTES, sim->stream>>>(
                sim->P, sub_buf(sim, which, g0), gvs, (int)ng, sim->deposit_cursor.p, ctr);
        }
        cudaEvent_t d1 = sim->mark();
        CU(cudaMemsetAsync(qbase, 0, 4 * sizeof(unsigned), sim->stream));
        order_kernel<<<(unsigned)gv.n_events, FIN_THREADS, FIN_SMEM_BYTES, sim->stream>>>(sim->P, fa, gv, ctr);
        far_kernel<<<(unsigned)(2 * sim->sm_count), FIN_THREADS, 0, sim->stream>>>(sim->P, fa, gv, ctr, fa.far);
        if (use_big)
            big_kernel<<<(unsigned)sim->sm_count, FIN_BIG_THREADS, FIN_BIG_SMEM_BYTES, sim->stream>>>(sim->P, fa, gv, ctr, fa.big);
        offsets_kernel<<<1, 1024, 0, sim->stream>>>(fa, gv, ctr);
        emit_kernel<<<(unsigned)gv.n_events, EMIT_THREADS, 0, sim->stream>>>(sim->P, fa, gv, ctr);
        sim->launches += use_big ? 8 : 7;
        if (spyral) {  // replayed uniforms have 53 bits: the Spyral passes read the float64 cloud instead (parity tests)
            int rc = launch_spyral(sim, spyral_args(sim, launch_first_event + gv.first_slot, gv.n_events, spyral->typed, false, ctr));
            if (rc) return rc;
        }
        cudaEvent_t f1 = sim->mark();
        ord_marks.push_back({d0, k0});
        dep_marks.push_back({k0, d1});
        fin_marks.push_back({d1, f1});
        if (fences) {
            const int slot = (int)fences->size();
            if (2 * slot + 1 < (int)sim->chunk_totals.n) {
                publish_total_kernel<<<1, 1, 0, sim->stream>>>(sim->csr_total.p, sim->chunk_totals.p + 2 * slot);
                sim->launches += 1;
                fences->push_back({sim->fence(sim->stream), gv.first_slot + (int64_t)gv.n_events, slot});
            }
        }
    }
    CU(cudaGetLastError());
    return ATTPC_OK;
}

float sum_ms(const std::vector<std::pair<cudaEvent_t, cudaEvent_t>>& marks) {
    float total = 0.f;
    for (auto& m : marks) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, m.first, m.second) == cudaSuccess) total += ms;
    }
    return total;
}

// The Spyral rows of a call: float64 rows, or (`typed`, ATTPC_SPYRAL_COLUMNS) the typed columns.
SpyralSink spyral_sink(AttpcSim* sim, bool typed) {
    if (typed)
        return {nullptr, nullptr, sim->rcol_pad.d(), sim->rcol_tbq.d(), sim->rcol_elo.d(), sim->rcol_ehi.d(),
                sim->rcol_label.d()};
    return {sim->rows.d(), sim->row_labels.d(), nullptr, nullptr, nullptr, nullptr, nullptr};
}

SpyralArgs spyral_args(AttpcSim* sim, int64_t first, int64_t n_events, bool typed, bool keep_all, const Counters* ctr) {
    SpyralArgs sa;
    memset(&sa, 0, sizeof sa);
    sa.offsets = sim->offsets_dev.p;
    sa.cloud = sim->cloud.d();
    sa.labels = sim->labels.d();
    sa.n_events = n_events;
    sa.first = first;
    sa.total = sim->csr_total.p + 2;
    sa.scratch_rows = sim->row_sort_keys.n / 2;
    sa.ctr = ctr;
    sa.cloud_cap = std::min<int64_t>(sim->labels.dev.n / sim->labels.row_bytes, sa.scratch_rows);
    sa.kept = sim->row_kept.p;
    sa.row_offsets = sim->row_offsets_dev.p;
    sa.sink = spyral_sink(sim, typed);
    sa.sort_keys = sim->row_sort_keys.p;
    sa.sort_idx = sim->row_sort_idx.p;
    sa.keep_all = keep_all ? 1 : 0;
    return sa;
}

// detector/response.py:35-57 + detector/writer.py:61-112, 232-238 for events first .. first + n_events - 1 of the cloud
// in device memory: amplitude / threshold count, running row offsets, rows in z order.
int launch_spyral(AttpcSim* sim, const SpyralArgs& sa) {
    if (sa.n_events <= 0) return ATTPC_OK;
    const size_t smem = (size_t)SPYRAL_SMEM_ITEMS * (sizeof(uint64_t) + sizeof(uint32_t));
    CU(cudaFuncSetAttribute(spyral_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    spyral_count_kernel<<<(unsigned)sa.n_events, 256, 0, sim->stream>>>(sim->P, sa);
    spyral_scan_kernel<<<1, 1024, 0, sim->stream>>>(sa);
    spyral_rows_kernel<<<(unsigned)sa.n_events, 256, smem, sim->stream>>>(sim->P, sa);
    sim->launches += 3;
    CU(cudaGetLastError());
    return ATTPC_OK;
}

struct LaunchPlan {
    // production
    const double* momenta_dev = nullptr;
    const double* vertices_dev = nullptr;
    int32_t n_nuclei = 0;
    const int32_t* track_nucleus = nullptr;
    const int32_t* track_species = nullptr;
    int32_t n_tracks_per_event = 0;
    uint64_t seed = 0;
    int64_t first_event = 0;
    // replay
    const ReplayBatch* replay = nullptr;
    const int32_t* label_of_event_rank_dev = nullptr;
    ReplayUniforms uniforms{nullptr, nullptr, nullptr};
};

// What one call writes and returns, derived from its flags once.
struct OutputPlan {
    bool copy_host = false;
    bool use_columns = false, use_q32 = false, use_packed = false;
    bool spy_cols = false, spy_rows = false, spy = false, spy_fused = false;
    bool copy_cloud = false, want_cloud = false;
    struct Use {
        RowSink* sink;
        bool to_host;  // copied to its pinned mirror; otherwise it stays on the device
    };
    std::vector<Use> cloud_rows;   // the sinks the call writes, indexed by cloud row, in the order they are copied
    std::vector<Use> spyral_rows;  // ... indexed by Spyral row
};

OutputPlan plan_outputs(AttpcSim* sim, const LaunchPlan& plan, uint32_t flags) {
    OutputPlan op;
    op.copy_host = !(flags & ATTPC_SKIP_HOST_COPY);
    op.use_columns = op.copy_host && (flags & ATTPC_COLUMNS);
    op.use_q32 = op.use_columns && (flags & ATTPC_COLUMNS32) && !sim->q32_off;
    // packed columns: pad ids and track ranks share 16 bits, the library's own 16-bit wiggle, masked time buckets
    op.use_packed = op.use_columns && (flags & ATTPC_COLUMNS_PACKED) && !plan.replay && !(flags & ATTPC_KEEP_ALL_TB) &&
                    sim->P.n_pads <= (1 << 14) && plan.n_tracks_per_event <= 4;
    op.spy_cols = (flags & ATTPC_SPYRAL_COLUMNS) != 0;               // Spyral rows as typed columns
    op.spy_rows = (flags & ATTPC_SPYRAL_ROWS) != 0 && !op.spy_cols;  // ... as float64 [M, 8]
    op.spy = op.spy_cols || op.spy_rows;
    op.copy_cloud = op.copy_host && !op.use_columns && !((flags & ATTPC_SKIP_CLOUD_COPY) && op.spy);
    // the float64 rows on the device: the product of a device-resident call, the input of the Spyral passes
    // (replayed 53-bit uniforms and unmasked time buckets: separate passes over the float64 cloud)
    op.spy_fused = op.spy && !plan.replay && !(flags & ATTPC_KEEP_ALL_TB);
    // nobody reads the float64 rows when the call returns typed columns, or only the Spyral rows, to the host
    const bool cloud_unread = op.copy_host && (op.use_columns || ((flags & ATTPC_SKIP_CLOUD_COPY) && op.spy));
    op.want_cloud = !cloud_unread || (op.spy && !op.spy_fused);
    if (op.want_cloud) op.cloud_rows = {{&sim->cloud, op.copy_cloud}, {&sim->labels, op.copy_cloud}};
    if (op.use_columns) {
        op.cloud_rows.push_back({&sim->col_pad, true});
        if (op.use_packed) op.cloud_rows.push_back({&sim->col_wig, true});
        else op.cloud_rows.push_back({&sim->col_tbq, true});
        if (op.use_q32) op.cloud_rows.push_back({&sim->col_q32, true});
        else op.cloud_rows.push_back({&sim->col_q, true});
        if (!op.use_packed) op.cloud_rows.push_back({&sim->col_label, true});
    }
    const bool h = op.copy_host;
    if (op.spy_rows) op.spyral_rows = {{&sim->rows, h}, {&sim->row_labels, h}};
    if (op.spy_cols)
        op.spyral_rows = {{&sim->rcol_pad, h}, {&sim->rcol_tbq, h}, {&sim->rcol_elo, h}, {&sim->rcol_ehi, h},
                          {&sim->rcol_label, h}};
    return op;
}

// Room for n_events events and `rows` cloud rows in the outputs of `op`.  `keep`: the rows written so far survive, on
// the device and on the host (regrowth after an output overflow).  The pinned mirrors are sized like the device
// arrays: pinning is slow, so they are (re)allocated only when those grow.
int reserve_outputs(AttpcSim* sim, const OutputPlan& op, int64_t n_events, int64_t rows, bool keep) {
    cudaStream_t s = sim->stream;
    CU(sim->offsets_dev.reserve(n_events + 1, keep, s));
    CU(sim->kept.reserve(n_events + 1, keep, s));
    if (op.copy_host) CU(sim->offsets_host.reserve(sim->offsets_dev.n, keep));
    if (op.use_packed) {
        CU(sim->tbc_dev.reserve((n_events + 1) * NUM_TB, keep, s));
        CU(sim->tbc_host.reserve(sim->tbc_dev.n, keep));
    }
    if (op.use_q32) {
        CU(sim->big_rows_dev.reserve(ATTPC_BIG_CAP));
        CU(sim->big_q_dev.reserve(ATTPC_BIG_CAP));
    }
    if (op.spy) {
        CU(sim->row_kept.reserve(n_events + 1));
        CU(sim->row_offsets_dev.reserve(n_events + 1));
        if (op.copy_host) CU(sim->row_offsets_host.reserve(n_events + 1, keep));
        CU(sim->row_sort_keys.reserve(rows * 2));  // scratch of the Spyral passes: nothing to keep
        CU(sim->row_sort_idx.reserve(rows * 2));
    }
    for (const auto* list : {&op.cloud_rows, &op.spyral_rows})
        for (const OutputPlan::Use& u : *list) {
            CU(u.sink->reserve(rows, keep, s));
            if (u.to_host) CU(u.sink->reserve_host(rows, keep));
        }
    sim->out_rows = std::max(sim->out_rows, rows);
    return ATTPC_OK;
}

// How far the host copies have got: events of the current launch whose offsets are final there, cloud rows and
// Spyral rows of the call.
struct CopyMark {
    int64_t events;
    unsigned long long cloud, spyral;
};

// Enqueues on the copy stream what became final between `from` and `to` in the launch whose first event is b0.
int copy_outputs(AttpcSim* sim, const OutputPlan& op, int64_t b0, const CopyMark& from, const CopyMark& to) {
    cudaStream_t C = sim->stream_c;
    const int64_t first_off = (b0 + from.events == 0) ? 0 : b0 + from.events + 1;  // the entry before is there already
    const int64_t end_off = b0 + to.events + 1;
    if (end_off > first_off) {
        CU(cudaMemcpyAsync(sim->offsets_host.p + first_off, sim->offsets_dev.p + first_off,
                           (size_t)(end_off - first_off) * sizeof(int64_t), cudaMemcpyDeviceToHost, C));
        if (op.spy)
            CU(cudaMemcpyAsync(sim->row_offsets_host.p + first_off, sim->row_offsets_dev.p + first_off,
                               (size_t)(end_off - first_off) * sizeof(int64_t), cudaMemcpyDeviceToHost, C));
    }
    if (op.use_packed && to.events > from.events)
        CU(cudaMemcpyAsync(sim->tbc_host.p + (b0 + from.events) * NUM_TB, sim->tbc_dev.p + (b0 + from.events) * NUM_TB,
                           (size_t)(to.events - from.events) * NUM_TB * sizeof(uint16_t), cudaMemcpyDeviceToHost, C));
    const int64_t r_new = (int64_t)(to.spyral - from.spyral);
    for (const OutputPlan::Use& u : op.spyral_rows)
        if (u.to_host && r_new > 0) CU(u.sink->copy_to_host((int64_t)from.spyral, r_new, C));
    const int64_t n_new = (int64_t)(to.cloud - from.cloud);
    for (const OutputPlan::Use& u : op.cloud_rows)
        if (u.to_host && n_new > 0) CU(u.sink->copy_to_host((int64_t)from.cloud, n_new, C));
    return ATTPC_OK;
}

// The finalize kernels' arguments for the launch whose first event is b0.
FinalizeArgs finalize_args(AttpcSim* sim, const LaunchPlan& plan, const OutputPlan& op, uint32_t flags, int64_t b0) {
    FinalizeArgs fa;
    memset(&fa, 0, sizeof fa);
    fa.seed = plan.seed;
    fa.first_event = plan.first_event + b0;
    fa.flags = flags;
    fa.kept = sim->kept.p + b0;
    fa.offsets = sim->offsets_dev.p + b0;
    fa.cloud = op.want_cloud ? sim->cloud.d() : nullptr;  // typed columns only: the float64 rows are not written
    fa.labels = op.want_cloud ? sim->labels.d() : nullptr;
    fa.out_cap = sim->out_rows;
    if (op.use_columns) {
        fa.col_pad = sim->col_pad.d();
        if (op.use_packed) {
            fa.col_wiggle = sim->col_wig.d();
            fa.tb_counts = sim->tbc_dev.p + b0 * NUM_TB;
            fa.rank_shift = 14;
        } else {
            fa.col_tb_q16 = sim->col_tbq.d();
            fa.col_label = sim->col_label.d();
        }
        if (op.use_q32) {
            fa.col_electrons32 = sim->col_q32.d();
            fa.big_rows = sim->big_rows_dev.p;
            fa.big_electrons = sim->big_q_dev.p;
            fa.big_count = sim->csr_total.p + 1;
            fa.big_cap = sim->big_cap;
        } else {
            fa.col_electrons = sim->col_q.d();
        }
    }
    if (op.spy_fused) {
        fa.spyral = true;
        fa.row_kept = sim->row_kept.p + b0;
        fa.row_offsets = sim->row_offsets_dev.p + b0;
        fa.rsink = spyral_sink(sim, op.spy_cols);
    }
    fa.replay = plan.uniforms;
    if (fa.replay.offsets) fa.replay.offsets += b0;
    fa.n_tracks_per_event = plan.n_tracks_per_event;
    if (plan.replay) {
        fa.label_of_event_rank = plan.label_of_event_rank_dev;
    } else {
        for (int t = 0; t < plan.n_tracks_per_event; ++t) fa.label_of_rank[t] = plan.track_nucleus[t];
    }
    return fa;
}

// Grows what a launch overflowed before it is redone.  The output rows of earlier launches are kept, on the device
// and on the host.
int grow_buffers(AttpcSim* sim, const Counters& now, const OutputPlan& op, int64_t n_events, int64_t work_events,
                 int32_t ranks, int64_t table_groups) {
    CU(cudaStreamSynchronize(sim->stream_t));  // the next launch's track kernel may be using buffers we are about to free
    CU(cudaStreamSynchronize(sim->stream_c));
    if (now.overflow_sub) {  // (overflow_points is raised with it: the point lists themselves were complete)
        if (sim->sub_cap >= (1LL << 30)) return sim->fail(ATTPC_E_CAPACITY, "a group needs > 2^30 sub-points");
        sim->sub_cap *= 2;
        sim->geom.release(); sim->rec.release();
        sim->unit_event.release(); sim->unit_first.release(); sim->unit_count.release();
        sim->unit_order.release();
    } else if (now.overflow_points) {
        sim->group_point_cap *= 2;
        for (auto& s2 : sim->slot) s2.release_points();
        sim->geom.release(); sim->rec.release();
        sim->unit_event.release(); sim->unit_first.release(); sim->unit_count.release();
        sim->unit_order.release();
    }
    if (now.overflow_hash) {
        if (sim->hash_cap >= (1 << 20)) return sim->fail(ATTPC_E_CAPACITY, "event needs > 2^20 hash slots");
        sim->hash_cap *= 2;
        sim->hash.release();
        sim->sort_items.release();
        sim->staged.release();
    }
    if (now.overflow_out) {
        const int64_t rows = std::max<int64_t>(sim->out_rows * 2, (int64_t)sim->csr_host.p[0] + (1 << 20));
        const int rc = reserve_outputs(sim, op, n_events, rows, true);
        if (rc) return rc;
    }
    return ensure_work_buffers(sim, work_events, ranks, table_groups);
}

void add_counters(Counters& totals, const Counters& now) {
    totals.traj_points += now.traj_points;
    totals.active_points += now.active_points;
    totals.primary_electrons += now.primary_electrons;
    totals.deposits += now.deposits;
    totals.keys += now.keys;
    totals.probes += now.probes;
    totals.flushes += now.flushes;
    totals.rk_steps += now.rk_steps;
    totals.rk_rejects += now.rk_rejects;
    totals.max_track_passes = std::max(totals.max_track_passes, now.max_track_passes);
}

// The counters of a finished call and where its outputs are: `done` holds its events, cloud rows and Spyral rows,
// n_big its electron counts >= 2^32.
int publish_result(AttpcSim* sim, const OutputPlan& op, const Counters& totals, int retries, const CopyMark& done,
                   unsigned long long n_big, AttpcResult* res) {
    res->n_points = (int64_t)done.cloud;
    res->offsets_dev = sim->offsets_dev.p;
    if (op.want_cloud) {
        res->cloud_dev = sim->cloud.d();
        res->labels_dev = sim->labels.d();
    }
    res->n_trajectory_points = (int64_t)totals.traj_points;
    res->n_active_points = (int64_t)totals.active_points;
    res->n_primary_electrons = (int64_t)totals.primary_electrons;
    res->n_deposits = (int64_t)totals.deposits;
    res->n_keys = (int64_t)totals.keys;
    res->n_hash_probes = (int64_t)totals.probes;
    res->n_table_flushes = (int64_t)totals.flushes;
    res->n_rk_steps = (int64_t)totals.rk_steps;
    res->n_rk_rejects = (int64_t)totals.rk_rejects;
    res->max_track_passes = (int64_t)totals.max_track_passes;
    res->n_retries = retries;
    if (op.spy) res->n_rows = (int64_t)done.spyral;
    if (!op.copy_host) return ATTPC_OK;
    if (done.events == 0) {  // no launch copied the leading offsets
        const int rc = copy_outputs(sim, op, 0, CopyMark{0, 0, 0}, CopyMark{0, 0, 0});
        if (rc) return rc;
    }
    cudaStream_t C = sim->stream_c;
    res->offsets = sim->offsets_host.p;
    if (op.copy_cloud) {
        res->cloud = sim->cloud.h();
        res->labels = sim->labels.h();
    }
    if (op.use_columns) {
        res->col_pad = sim->col_pad.h();
        if (op.use_packed) {
            res->col_wiggle = sim->col_wig.h();
            res->tb_counts = sim->tbc_host.p;
            res->pad_rank_shift = 14;
        } else {
            res->col_tb_q16 = sim->col_tbq.h();
            res->col_label = sim->col_label.h();
        }
        if (!op.use_q32) {
            res->col_electrons = sim->col_q.h();
        } else {
            res->col_electrons32 = sim->col_q32.h();
            res->n_big = (int64_t)n_big;
            if (n_big > 0) {
                CU(sim->big_rows_host.reserve((int64_t)n_big));
                CU(sim->big_q_host.reserve((int64_t)n_big));
                CU(cudaMemcpyAsync(sim->big_rows_host.p, sim->big_rows_dev.p, (size_t)n_big * sizeof(int64_t),
                                   cudaMemcpyDeviceToHost, C));
                CU(cudaMemcpyAsync(sim->big_q_host.p, sim->big_q_dev.p, (size_t)n_big * sizeof(int64_t),
                                   cudaMemcpyDeviceToHost, C));
                res->big_rows = sim->big_rows_host.p;
                res->big_electrons = sim->big_q_host.p;
            }
        }
    }
    if (op.spy) {
        res->row_offsets = sim->row_offsets_host.p;
        if (op.spy_rows) {
            res->rows = sim->rows.h();
            res->row_labels = sim->row_labels.h();
        } else {
            res->row_col_pad = sim->rcol_pad.h();
            res->row_col_tb_q16 = sim->rcol_tbq.h();
            res->row_col_e_lo = sim->rcol_elo.h();
            res->row_col_e_hi = sim->rcol_ehi.h();
            res->row_col_label = sim->rcol_label.h();
        }
    }
    return ATTPC_OK;
}

// Shared driver of attpc_simulate / attpc_simulate_dev / attpc_simulate_replay.
//
// Three streams: T runs the (latency-bound, few-warp) track kernel of launch i+1 while G runs the deposit and
// finalize kernels of launch i, and C copies the finished rows of launch i-1 to the host.  After every launch the
// host reads that launch's counters; a capacity overflow grows the buffer in question and redoes the launch.
int run_batch(AttpcSim* sim, const LaunchPlan& plan, int64_t n_events, uint32_t flags, AttpcResult* res,
              float ms_h2d) {
    memset(res, 0, sizeof *res);
    sim->events_used = 0;
    sim->sync_used = 0;
    sim->launches = 0;
    res->n_events = n_events;
    res->ms_h2d = ms_h2d;
    const OutputPlan op = plan_outputs(sim, plan, flags);
    int rc = reserve_outputs(sim, op, n_events,
                             std::max<int64_t>(sim->out_rows, std::max<int64_t>(n_events * 2048, 1 << 20)), false);
    if (rc) return rc;
    // big launches: the latency-bound track kernel wants many tracks in flight.  When rows go to the host they are
    // copied in chunks of a few groups while the following groups are still being computed.
    const int64_t launch_cap = plan.replay ? std::max<int64_t>(n_events, 1) : sim->launch_events;
    const int groups_per_chunk =
        std::max<int>(1, (int)((sim->copy_launch_events + sim->group_events - 1) / sim->group_events));
    const int32_t ranks = std::max<int32_t>(1, plan.n_tracks_per_event);
    // a call that copies its rows to the host works in chunks of a few groups: its engine needs an eighth of the memory
    const int64_t table_groups = op.copy_host ? groups_per_chunk : sim->chunk_groups;
    const int64_t work_events = std::min<int64_t>(std::max<int64_t>(n_events, 1), launch_cap);
    rc = ensure_work_buffers(sim, work_events, ranks, table_groups);
    if (rc) return rc;
    const SpyralPass spyral_pass{op.spy_cols};
    cudaStream_t G = sim->stream, T = sim->stream_t, C = sim->stream_c;
    CU(cudaMemsetAsync(sim->csr_total.p, 0, 3 * sizeof(unsigned long long), G));
    if (op.spy) CU(cudaMemsetAsync(sim->row_offsets_dev.p, 0, sizeof(int64_t), G));
    CU(cudaMemsetAsync(sim->offsets_dev.p, 0, sizeof(int64_t), G));
    cudaEvent_t t_begin = sim->mark(G);
    CU(cudaStreamWaitEvent(T, t_begin, 0));
    CU(cudaStreamWaitEvent(C, t_begin, 0));

    // Launch boundaries.  When rows go to the host the first launch is one group: its (latency-bound) track kernel
    // and its group kernels finish early, so the copy engine -- the bottleneck of such a call -- starts ~1 ms sooner,
    // while the big second track kernel runs beside the first launch's group kernels.
    std::vector<int64_t> launch_begin;
    {
        int64_t at = 0;
        if (op.copy_host && !plan.replay && n_events > 2 * (int64_t)sim->group_events && launch_cap > sim->group_events) {
            launch_begin.push_back(0);
            at = sim->group_events;
        }
        for (; at < n_events; at += launch_cap) launch_begin.push_back(at);
        launch_begin.push_back(std::max<int64_t>(n_events, 0));
    }
    const int64_t n_launch = n_events > 0 ? (int64_t)launch_begin.size() - 1 : 0;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> trk_marks(n_launch), ord_marks, dep_marks, fin_marks, copy_marks;
    std::vector<cudaEvent_t> track_done(n_launch);
    Counters totals;
    memset(&totals, 0, sizeof totals);
    unsigned long long csr_before = 0;  // rows emitted by the launches completed so far
    unsigned long long big_before = 0;  // ... and electron counts >= 2^32 among them
    unsigned long long rows_before = 0; // ... and Spyral rows
    int retries = 0;
    int64_t next_track = 0;  // launches whose track kernel is enqueued

    auto enqueue_track = [&](int64_t i) -> int {
        const int which = (int)(i & 1);
        AttpcSim::LaunchSlot& ls = sim->slot[which];
        const int64_t b0 = launch_begin[i], nb = launch_begin[i + 1] - b0;
        const int64_t n_groups = (nb + sim->group_events - 1) / sim->group_events;
        CU(cudaMemsetAsync(ls.counters.p, 0, sizeof(Counters), T));
        CU(cudaMemsetAsync(ls.group_count.p, 0, (size_t)n_groups * sizeof(unsigned), T));
        CU(cudaMemsetAsync(ls.pcnt.p, 0, (size_t)nb * ranks * sizeof(unsigned), T));
        cudaEvent_t k0 = sim->mark(T);
        if (plan.replay) {
            const ReplayBatch& rb = *plan.replay;
            if (rb.n_rows > 0) {
                const int blocks = (int)((rb.n_rows + 255) / 256);
                replay_kernel<<<blocks, 256, 0, T>>>(sim->P, rb, point_buf(sim, which), ls.counters.p);
                sim->launches += 1;
                CU(cudaGetLastError());
            }
        } else {
            TrackBatch tb;
            memset(&tb, 0, sizeof tb);
            tb.momenta = plan.momenta_dev + b0 * plan.n_nuclei * 4;
            tb.vertices = plan.vertices_dev + b0 * 3;
            tb.n_events = nb;
            tb.n_nuclei = plan.n_nuclei;
            tb.n_tracks_per_event = plan.n_tracks_per_event;
            for (int t = 0; t < plan.n_tracks_per_event; ++t) {
                tb.nucleus[t] = plan.track_nucleus[t];
                tb.species[t] = plan.track_species[t];
            }
            tb.seed = plan.seed;
            tb.first_event = plan.first_event + b0;
            const int64_t n_trk = nb * plan.n_tracks_per_event;
            if (n_trk >= 4 * (int64_t)sim->sm_count * 32) {  // enough tracks for the order to matter
                const int ctas = (int)((n_trk + PLAN_THREADS - 1) / PLAN_THREADS);
                CU(sim->plan_cls.reserve(n_trk));
                CU(sim->plan_counts.reserve((int64_t)ctas * PLAN_CLASSES));
                CU(sim->plan_order.reserve(n_trk));
                track_plan_count_kernel<<<ctas, PLAN_THREADS, 0, T>>>(sim->P, tb, sim->plan_cls.p, sim->plan_counts.p);
                track_plan_scan_kernel<<<1, 1024, 0, T>>>(sim->plan_counts.p, ctas * PLAN_CLASSES);
                track_plan_scatter_kernel<<<ctas, PLAN_THREADS, 0, T>>>(sim->plan_cls.p, sim->plan_counts.p, n_trk,
                                                                        sim->plan_order.p);
                sim->launches += 3;
                tb.order = sim->plan_order.p;
            }
            int r = launch_tracks<false>(sim, tb, n_trk, which, T);
            if (r) return r;
        }
        cudaEvent_t k1 = sim->mark(T);
        trk_marks[i] = {k0, k1};
        track_done[i] = k1;
        return ATTPC_OK;
    };

    for (int64_t i = 0; i < n_launch;) {
        const int which = (int)(i & 1);
        AttpcSim::LaunchSlot& ls = sim->slot[which];
        const int64_t b0 = launch_begin[i], nb = launch_begin[i + 1] - b0;
        while (next_track <= i) {
            rc = enqueue_track(next_track++);
            if (rc) return rc;
        }
        const FinalizeArgs fa = finalize_args(sim, plan, op, flags, b0);
        CU(cudaStreamWaitEvent(G, track_done[i], 0));
        const size_t dep_before = dep_marks.size(), fin_before = fin_marks.size(), copy_before = copy_marks.size();
        const size_t ord_before = ord_marks.size();
        std::vector<ChunkFence> fences;
        rc = run_groups(sim, nb, fa, which, ord_marks, dep_marks, fin_marks, groups_per_chunk,
                        op.copy_host ? &fences : nullptr, op.spy && !op.spy_fused ? &spyral_pass : nullptr, b0);
        if (rc) return rc;
        publish_kernel<<<1, 1, 0, G>>>(ls.counters.p, sim->csr_total.p, ls.counters_host.p, sim->csr_host.p);
        sim->launches += 1;
        cudaEvent_t groups_done = sim->fence(G);
        if (next_track <= i + 1 && i + 1 < n_launch) {  // overlaps with the groups just enqueued
            rc = enqueue_track(next_track++);
            if (rc) return rc;
        }
        // rows of finished chunks go home while the later groups (and the next launch's tracks) compute
        CopyMark copied{0, csr_before, rows_before};  // events of this launch, rows of the call, on the host
        auto copy_rows = [&](const CopyMark& upto) -> int {
            cudaEvent_t c0 = sim->mark(C);
            const int r = copy_outputs(sim, op, b0, copied, upto);
            if (r) return r;
            copy_marks.push_back({c0, sim->mark(C)});
            copied = upto;
            return ATTPC_OK;
        };
        for (const ChunkFence& cf : fences) {
            CU(cudaEventSynchronize(cf.done));
            const unsigned long long upto = sim->chunk_totals.p[2 * cf.slot];
            if ((int64_t)upto > sim->out_rows) break;  // output overflow: the launch will be redone below
            CU(cudaStreamWaitEvent(C, cf.done, 0));
            rc = copy_rows(CopyMark{cf.last_event, upto, sim->chunk_totals.p[2 * cf.slot + 1]});
            if (rc) return rc;
        }
        CU(cudaEventSynchronize(groups_done));
        const Counters now = *ls.counters_host.p;
        if (now.replay_miss) return sim->fail(ATTPC_E_BADARG, "replay uniforms do not cover every (event, key)");
        if (now.overflow_charge)
            return sim->fail(ATTPC_E_CAPACITY, "a (pad, time bucket) charge exceeded 2^48 electrons");
        if (now.overflow_points || now.overflow_hash || now.overflow_out) {
            ord_marks.resize(ord_before);
            dep_marks.resize(dep_before);
            fin_marks.resize(fin_before);
            copy_marks.resize(copy_before);
            if (++retries > 24) return sim->fail(ATTPC_E_CAPACITY, "buffers still too small after 24 retries");
            rc = grow_buffers(sim, now, op, n_events, work_events, ranks, table_groups);
            if (rc) return rc;
            sim->csr_host.p[0] = csr_before;  // forget the rows (and the big-count exceptions) of the failed attempt
            sim->csr_host.p[1] = big_before;
            sim->csr_host.p[2] = rows_before;
            CU(cudaMemcpyAsync(sim->csr_total.p, sim->csr_host.p, 3 * sizeof(unsigned long long),
                               cudaMemcpyHostToDevice, G));
            CU(cudaStreamSynchronize(G));
            next_track = i;  // redo this launch (and the one that was running ahead)
            continue;
        }
        add_counters(totals, now);
        const unsigned long long csr_after = sim->csr_host.p[0], rows_after = sim->csr_host.p[2];
        big_before = sim->csr_host.p[1];
        if (op.copy_host && (copied.cloud < csr_after || copied.spyral < rows_after || copied.events < nb)) {  // whatever the chunk copies did not cover
            CU(cudaStreamWaitEvent(C, groups_done, 0));
            rc = copy_rows(CopyMark{nb, csr_after, rows_after});
            if (rc) return rc;
        }
        csr_before = csr_after;
        rows_before = rows_after;
        ++i;
    }
    if (op.use_q32 && (int64_t)big_before > sim->big_cap) {
        // too many exceptions for the list (heavy ions): the full-width column, now and from now on
        sim->q32_off = true;
        CU(cudaStreamSynchronize(T));
        CU(cudaStreamSynchronize(C));
        CU(cudaStreamSynchronize(G));
        return run_batch(sim, plan, n_events, flags, res, ms_h2d);
    }
    rc = publish_result(sim, op, totals, retries, CopyMark{n_events, csr_before, rows_before}, big_before, res);
    if (rc) return rc;
    // close the timeline on G after the other two streams have drained
    CU(cudaStreamWaitEvent(G, sim->fence(T), 0));
    CU(cudaStreamWaitEvent(G, sim->fence(C), 0));
    cudaEvent_t t_end = sim->mark(G);
    CU(cudaStreamSynchronize(G));
    res->ms_tracks = sum_ms(trk_marks);
    res->ms_order = sum_ms(ord_marks);
    res->ms_deposit = sum_ms(dep_marks);
    res->ms_finalize = sum_ms(fin_marks);
    res->ms_d2h = sum_ms(copy_marks);
    cudaEventElapsedTime(&res->ms_total, t_begin, t_end);
    res->ms_total += ms_h2d;
    res->n_kernel_launches = sim->launches;
    res->n_track_launches = (int32_t)trk_marks.size();
    res->n_group_launches = (int32_t)dep_marks.size();
    res->hash_capacity = sim->hash_cap;
    return ATTPC_OK;
}

int check_tracks(AttpcSim* sim, int32_t n_nuclei, const int32_t* track_nucleus, const int32_t* track_species,
                 int32_t n_tracks) {
    if (!track_nucleus || !track_species) return sim->fail(ATTPC_E_BADARG, "null track arrays");
    if (n_tracks <= 0 || n_tracks > MAX_TRACKS_PER_EVENT)
        return sim->fail(ATTPC_E_BADARG, "n_tracks_per_event must be in 1..%d", MAX_TRACKS_PER_EVENT);
    for (int t = 0; t < n_tracks; ++t) {
        if (track_nucleus[t] < 0 || track_nucleus[t] >= n_nuclei)
            return sim->fail(ATTPC_E_BADARG, "track_nucleus[%d]=%d outside 0..%d", t, track_nucleus[t], n_nuclei - 1);
        if (track_species[t] >= sim->P.n_species)
            return sim->fail(ATTPC_E_BADARG, "track_species[%d]=%d outside the %d species of this simulator", t,
                             track_species[t], sim->P.n_species);
    }
    return ATTPC_OK;
}

// attpc_create after its argument checks: streams, constants and tables of a new simulator on the current device.
int init_sim(AttpcSim* sim, const AttpcConfig* cfg, const int16_t* pad_lut, const double* pad_xy, const double* pad_scale,
             int32_t n_pads, const double* response, int32_t n_response, const AttpcSpecies* species, int32_t n_species) {
    CU(cudaStreamCreateWithFlags(&sim->stream, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&sim->stream_t, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&sim->stream_c, cudaStreamNonBlocking));
    int sm = 0;
    CU(cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, sim->device));
    sim->sm_count = sm > 0 ? sm : 148;
    CU(cudaFuncSetAttribute(deposit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DEPOSIT_SMEM_BYTES));
    int deposit_per_sm = 0;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&deposit_per_sm, deposit_kernel, DEPOSIT_THREADS,
                                                     DEPOSIT_SMEM_BYTES));
    sim->deposit_ctas = std::max(1, deposit_per_sm) * sim->sm_count;
    CU(sim->deposit_cursor.reserve(1));

    SimParams& P = sim->P;
    P.length = cfg->length;
    P.dv = cfg->drift_velocity;
    P.mm_edge = (double)cfg->micromegas_edge;
    P.win_edge = (double)cfg->windows_edge;
    P.diffusion = cfg->diffusion;
    P.long_diffusion = cfg->longitudinal_diffusion;
    if (P.long_diffusion > 0.0) {  // widest window: sigma_L one bucket past the window edge (no point drifts longer)
        const double t = P.win_edge + 1.0;
        const double sl = std::sqrt(2.0 * P.long_diffusion * P.dv * t / cfg->efield) / P.dv;
        if (!(sl < 1.0e6))
            return sim->fail(ATTPC_E_BADARG, "attpc_create: longitudinal diffusion needs efield > 0 (sigma_L = %g)", sl);
        sim->long_buckets = (int32_t)std::floor(6.0 * sl) + 2;
    }
    P.efield = cfg->efield;
    P.fano = cfg->fano_factor;
    P.ev_per_w = 1.0e6 / cfg->w_value;
    P.B = cfg->bfield * -1.0;
    P.E = cfg->efield * -1.0;
    P.gain = cfg->mpgd_gain;
    P.grid_low = cfg->grid_low_mm;
    P.grid_high = cfg->grid_high_mm;
    P.lut_origin = cfg->lut_origin_mm;
    P.lut_n = cfg->lut_n;
    P.adc_threshold = cfg->adc_threshold;
    P.rtol = cfg->ode_rtol > 0 ? cfg->ode_rtol : 1e-6;
    P.atol = cfg->ode_atol > 0 ? cfg->ode_atol : 1e-10;
    P.freeze_ke = cfg->freeze_ke_mev;
    P.lm = n_species ? species[0].lm : 0;
    P.e_min = n_species ? species[0].e_min : 0;
    P.n_oct = n_species ? species[0].n_oct : 0;
    P.n_nodes = P.n_oct * (1 << P.lm) + 1;
    P.n_species = n_species;
    P.n_pads = n_pads;
    P.n_response = n_response;
    if (cfg->max_events_per_launch > 0) sim->launch_events = cfg->max_events_per_launch;
    if (cfg->copy_events_per_launch > 0) sim->copy_launch_events = cfg->copy_events_per_launch;  // events per launch when rows go to the host
    if (cfg->hash_capacity > 0) sim->hash_cap = next_pow2(cfg->hash_capacity);
    if (cfg->unit_points > 0) sim->unit_points = std::min<int32_t>(cfg->unit_points, UNIT_POINTS);
    if (cfg->table_spill_keys > 0) sim->spill_keys = std::min<int32_t>(cfg->table_spill_keys, SMEM_SPILL_AT);
    sim->group_events = std::min(sim->group_events, sim->launch_events);
    if (const char* env = getenv("ATTPC_CHUNK_GROUPS")) sim->chunk_groups = std::max(1, atoi(env));  // tuning aid
    if (const char* env = getenv("ATTPC_BIG_CAP")) sim->big_cap = std::min<int64_t>(ATTPC_BIG_CAP, std::max(0, atoi(env)));  // tests

    const int64_t lut_cells = (int64_t)cfg->lut_n * cfg->lut_n;
    CU(sim->lut.reserve(lut_cells));
    CU(cudaMemcpy(sim->lut.p, pad_lut, (size_t)lut_cells * sizeof(int16_t), cudaMemcpyHostToDevice));
    CU(sim->pad_xy.reserve((int64_t)n_pads * 2));
    CU(cudaMemcpy(sim->pad_xy.p, pad_xy, (size_t)n_pads * 2 * sizeof(double), cudaMemcpyHostToDevice));
    CU(sim->pad_scale.reserve(n_pads));
    CU(cudaMemcpy(sim->pad_scale.p, pad_scale, (size_t)n_pads * sizeof(double), cudaMemcpyHostToDevice));
    CU(sim->response.reserve(n_response));
    CU(cudaMemcpy(sim->response.p, response, (size_t)n_response * sizeof(double), cudaMemcpyHostToDevice));
    {
        std::vector<double> sorted(response, response + n_response);
        std::sort(sorted.begin(), sorted.end(), [](double a, double b) { return a > b; });
        std::vector<double> prefix(n_response + 1, 0.0);
        for (int i = 0; i < n_response; ++i) prefix[i + 1] = prefix[i] + sorted[i];
        CU(sim->resp_sorted.reserve(n_response));
        CU(cudaMemcpy(sim->resp_sorted.p, sorted.data(), (size_t)n_response * sizeof(double), cudaMemcpyHostToDevice));
        CU(sim->resp_prefix.reserve(n_response + 1));
        CU(cudaMemcpy(sim->resp_prefix.p, prefix.data(), (size_t)(n_response + 1) * sizeof(double),
                       cudaMemcpyHostToDevice));
        P.resp_max = sorted[0];
        // smallest electron count that passes the ADC threshold (detector/writer.py:232): amp = min(r_max e, 4095) is
        // monotone in e, so the comparison can be made on the integer charge
        {
            const double thr = cfg->adc_threshold;
            long long keep = 0;
            if (!(thr < 4095.0)) {
                keep = INT64_MAX;
            } else if (thr >= 0.0 && sorted[0] > 0.0) {
                keep = std::max<long long>(0, (long long)std::floor(thr / sorted[0]) - 2);
                while (!(std::fmin(sorted[0] * (double)keep, 4095.0) > thr)) ++keep;
            } else if (thr >= 0.0) {
                keep = INT64_MAX;  // a null response never passes a non-negative threshold
            }
            P.e_keep_min = keep;
        }
    }
    {
        // deceleration tables: dE/dx [MeV/(g/cm^2)] * MEV_2_JOULE * density * 100 / m_kg / c  (detector/solver.py:64-76)
        std::vector<double> scaled((size_t)n_species * P.n_nodes);
        for (int s = 0; s < n_species; ++s) {
            if (!species[s].dedx || !(species[s].mass > 0.0))
                return sim->fail(ATTPC_E_BADARG, "species %d: null table or non-positive mass", s);
            const double mass_kg = species[s].mass * MEV_2_KG;
            const double scale = MEV_2_JOULE * cfg->gas_density * 100.0 / mass_kg / C_LIGHT;
            for (int i = 0; i < P.n_nodes; ++i) scaled[(size_t)s * P.n_nodes + i] = species[s].dedx[i] * scale;
            P.sp[s].mass = species[s].mass;
            P.sp[s].qm_c = (double)species[s].z * E_CHARGE / mass_kg / C_LIGHT;
            P.sp[s].z = species[s].z;
            P.sp[s].table = s * P.n_nodes;
            // terminal drift energy: first table node where the drag reaches the field acceleration |q E / (m c)|
            {
                const double field = std::fabs(P.sp[s].qm_c * P.E);
                const double* t = &scaled[(size_t)s * P.n_nodes];
                const int per_oct = 1 << P.lm;
                double ke_eq = 0.0;
                if (field > 0.0) {
                    const double ke0 = std::ldexp(1.0, P.e_min);
                    if (t[0] >= field) {  // below the table: drag = t[0] sqrt(ke / ke0)
                        ke_eq = t[0] > 0.0 ? ke0 * (field / t[0]) * (field / t[0]) : 0.0;
                    } else {
                        for (int i = 1; i < P.n_nodes; ++i) {
                            if (t[i] >= field) {
                                auto node = [&](int j) {
                                    return std::ldexp(1.0 + (double)(j % per_oct) / per_oct, P.e_min + j / per_oct);
                                };
                                const double f = (field - t[i - 1]) / (t[i] - t[i - 1]);
                                ke_eq = node(i - 1) + f * (node(i) - node(i - 1));
                                break;
                            }
                        }
                    }
                }
                P.sp[s].ke_eq = ke_eq;
            }
        }
        CU(sim->tables.reserve(std::max<int64_t>(1, (int64_t)scaled.size())));
        if (!scaled.empty())
            CU(cudaMemcpy(sim->tables.p, scaled.data(), scaled.size() * sizeof(double), cudaMemcpyHostToDevice));
        // time [ns] to slow down from node i to node 0: integral of d(gamma beta) / deceleration (trapezoids); only the
        // launch order of the tracks depends on it
        std::vector<double> stop((size_t)n_species * P.n_nodes, 0.0);
        for (int s = 0; s < n_species; ++s) {
            const int per_oct = 1 << P.lm;
            auto node = [&](int j) { return std::ldexp(1.0 + (double)(j % per_oct) / per_oct, P.e_min + j / per_oct); };
            auto gb = [&](double ke) { const double g = ke / species[s].mass + 1.0; return std::sqrt(g * g - 1.0); };
            const double* a = &scaled[(size_t)s * P.n_nodes];
            double* out = &stop[(size_t)s * P.n_nodes];
            for (int i = 1; i < P.n_nodes; ++i) {
                const double mean = 0.5 * (a[i] + a[i - 1]);
                out[i] = out[i - 1] + (mean > 0.0 ? (gb(node(i)) - gb(node(i - 1))) / mean * 1e9 : 0.0);
            }
        }
        CU(sim->stop_ns.reserve(std::max<int64_t>(1, (int64_t)stop.size())));
        if (!stop.empty())
            CU(cudaMemcpy(sim->stop_ns.p, stop.data(), stop.size() * sizeof(double), cudaMemcpyHostToDevice));
        sim->table_smem_bytes = scaled.size() * sizeof(double);
        // the tables share the SM's 227 KB with the step slots of the warps: many species -> fewer warps per CTA;
        // below four warps the tables stay in global memory (L1/L2) instead
        const int64_t room = 227 * 1024 - (int64_t)sim->table_smem_bytes;
        const int fit = (int)std::min<int64_t>(TRACK_THREADS / 32, room / (int64_t)TRACK_SLOT_BYTES_PER_WARP);
        sim->tables_in_smem = fit >= 4;
        sim->track_warps_max = sim->tables_in_smem ? fit : TRACK_THREADS / 32;
    }
    {
        // constant mesh weights pdf * step^2 of detector/transporter.py:217-246 in exact arithmetic (sigma cancels):
        // (36 / 81) / (2 pi) * exp(-(a_i^2 + a_j^2) / 2), a_i = -3 + 6 i / 9, rounded once from extended precision
        const long double pi_l = 3.14159265358979323846264338327950288L;
        for (int i = 0; i < MESH_N; ++i)
            for (int j = 0; j < MESH_N; ++j) {
                const long double ai = -3.0L + 6.0L * i / 9.0L, aj = -3.0L + 6.0L * j / 9.0L;
                P.mesh_w[i * MESH_N + j] = (double)((2.0L / (9.0L * pi_l)) * expl(-(ai * ai + aj * aj) / 2.0L));
            }
        // the distinct values of the table (the mesh is symmetric): what the per-point exactness test multiplies
        P.n_mesh_w_unique = 0;
        for (int k = 0; k < MESH_N * MESH_N; ++k) {
            bool seen = false;
            for (int u = 0; u < P.n_mesh_w_unique; ++u) seen = seen || P.mesh_w_unique[u] == P.mesh_w[k];
            if (!seen) P.mesh_w_unique[P.n_mesh_w_unique++] = P.mesh_w[k];
        }
    }
    P.lut = sim->lut.p;
    P.tables = sim->tables.p;
    P.stop_ns = sim->stop_ns.p;
    P.pad_xy = sim->pad_xy.p;
    P.pad_scale = sim->pad_scale.p;
    P.response = sim->response.p;
    P.resp_sorted = sim->resp_sorted.p;
    P.resp_prefix = sim->resp_prefix.p;
    return ATTPC_OK;
}

}  // namespace

// ------------------------------------------------------------------------------------------------------- C ABI
extern "C" {

int attpc_abi_version(void) { return ATTPC_ABI_VERSION; }

int attpc_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return ATTPC_E_CUDA;
    return n;
}

const char* attpc_last_error(const AttpcSim* sim) { return sim ? sim->error.c_str() : g_create_error.c_str(); }

void attpc_destroy(AttpcSim* sim) {
    if (!sim) return;
    cudaSetDevice(sim->device);
    delete sim;
}

int attpc_create(const AttpcConfig* cfg, const int16_t* pad_lut, const double* pad_xy, const double* pad_scale,
                 int32_t n_pads, const double* response, int32_t n_response, const AttpcSpecies* species,
                 int32_t n_species, int32_t device, AttpcSim** out) {
    if (!cfg || !pad_lut || !pad_xy || !pad_scale || !response || (!species && n_species > 0) || !out) {
        g_create_error = "attpc_create: null argument";
        return ATTPC_E_BADARG;
    }
    if (n_species < 0 || n_species > MAX_SPECIES || n_pads < 1 || n_response < 1 || cfg->lut_n < 1) {
        g_create_error = "attpc_create: n_species must be 0..8, n_pads/n_response/lut_n positive";
        return ATTPC_E_BADARG;
    }
    for (int s = 1; s < n_species; ++s)
        if (species[s].lm != species[0].lm || species[s].e_min != species[0].e_min ||
            species[s].n_oct != species[0].n_oct) {
            g_create_error = "attpc_create: all species tables must share one grid (lm, e_min, n_oct)";
            return ATTPC_E_BADARG;
        }
    if (cfg->windows_edge == cfg->micromegas_edge || !(cfg->drift_velocity > 0.0) || !(cfg->w_value > 0.0)) {
        g_create_error = "attpc_create: windows_edge == micromegas_edge, drift_velocity <= 0 or w_value <= 0";
        return ATTPC_E_BADARG;
    }
    // a point drifts for up to windows_edge time buckets, and the 28-bit table key holds 13 bits of time bucket: a
    // wider window would lose the points beyond bucket 8191 without a word (ATTPC_KEEP_ALL_TB keeps them otherwise)
    if (cfg->windows_edge > 8191) {
        g_create_error = "attpc_create: windows_edge must be <= 8191 (time buckets are kept in 13 bits)";
        return ATTPC_E_BADARG;
    }
    if (!(cfg->longitudinal_diffusion >= 0.0) || !std::isfinite(cfg->longitudinal_diffusion)) {
        g_create_error = "attpc_create: longitudinal_diffusion must be finite and >= 0";
        return ATTPC_E_BADARG;
    }
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) {
        g_create_error = std::string("cudaSetDevice: ") + cudaGetErrorString(e);
        return ATTPC_E_CUDA;
    }
    AttpcSim* sim = new AttpcSim();
    sim->device = device;
    sim->cfg = *cfg;
    const int rc = init_sim(sim, cfg, pad_lut, pad_xy, pad_scale, n_pads, response, n_response, species, n_species);
    if (rc) {
        g_create_error = sim->error;
        delete sim;
        return rc;
    }
    *out = sim;
    return ATTPC_OK;
}

int attpc_simulate_dev(AttpcSim* sim, const double* momenta_dev, const double* vertices_dev, int64_t n_events,
                       int32_t n_nuclei, const int32_t* track_nucleus, const int32_t* track_species,
                       int32_t n_tracks_per_event, uint64_t seed, int64_t first_event, uint32_t flags,
                       AttpcResult* result) {
    if (!sim) return ATTPC_E_BADARG;
    if (!result || n_events < 0 || n_nuclei <= 0 || (n_events > 0 && (!momenta_dev || !vertices_dev)))
        return sim->fail(ATTPC_E_BADARG, "attpc_simulate: bad arguments");
    int rc = check_tracks(sim, n_nuclei, track_nucleus, track_species, n_tracks_per_event);
    if (rc) return rc;
    CU(cudaSetDevice(sim->device));
    LaunchPlan plan;
    plan.momenta_dev = momenta_dev;
    plan.vertices_dev = vertices_dev;
    plan.n_nuclei = n_nuclei;
    plan.track_nucleus = track_nucleus;
    plan.track_species = track_species;
    plan.n_tracks_per_event = n_tracks_per_event;
    plan.seed = seed;
    plan.first_event = first_event;
    rc = run_batch(sim, plan, n_events, flags, result, 0.f);
    if (rc == ATTPC_OK) {
        int charged = 0;
        for (int t = 0; t < n_tracks_per_event; ++t) charged += track_species[t] >= 0;
        result->n_tracks = n_events * charged;
    }
    return rc;
}

int attpc_simulate(AttpcSim* sim, const double* momenta, const double* vertices, int64_t n_events, int32_t n_nuclei,
                   const int32_t* track_nucleus, const int32_t* track_species, int32_t n_tracks_per_event,
                   uint64_t seed, int64_t first_event, uint32_t flags, AttpcResult* result) {
    if (!sim) return ATTPC_E_BADARG;
    if (!result || n_events < 0 || n_nuclei <= 0 || (n_events > 0 && (!momenta || !vertices)))
        return sim->fail(ATTPC_E_BADARG, "attpc_simulate: bad arguments");
    CU(cudaSetDevice(sim->device));
    CU(sim->in_momenta.reserve(std::max<int64_t>(1, n_events * n_nuclei * 4)));
    CU(sim->in_vertices.reserve(std::max<int64_t>(1, n_events * 3)));
    sim->events_used = 0;
    cudaEvent_t h0 = sim->mark();
    if (n_events > 0) {
        CU(cudaMemcpyAsync(sim->in_momenta.p, momenta, (size_t)n_events * n_nuclei * 4 * sizeof(double),
                           cudaMemcpyHostToDevice, sim->stream));
        CU(cudaMemcpyAsync(sim->in_vertices.p, vertices, (size_t)n_events * 3 * sizeof(double),
                           cudaMemcpyHostToDevice, sim->stream));
    }
    cudaEvent_t h1 = sim->mark();
    CU(cudaStreamSynchronize(sim->stream));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, h0, h1);
    int rc = attpc_simulate_dev(sim, sim->in_momenta.p, sim->in_vertices.p, n_events, n_nuclei, track_nucleus,
                                track_species, n_tracks_per_event, seed, first_event, flags, result);
    if (rc == ATTPC_OK) {
        result->ms_h2d = ms;
        result->ms_total += ms;
    }
    return rc;
}

int attpc_simulate_replay(AttpcSim* sim, const int64_t* track_offsets, const double* points, const double* normals,
                          const int32_t* track_event, const int32_t* track_rank, const int32_t* track_label,
                          const int32_t* track_species, int64_t n_tracks, int64_t n_events,
                          const AttpcReplay* replay, uint32_t flags, int64_t* electrons_out, AttpcResult* result) {
    if (!sim) return ATTPC_E_BADARG;
    if (!result || n_tracks < 0 || n_events < 0 || !track_offsets ||
        (n_tracks > 0 && (!points || !normals || !track_event || !track_rank || !track_label || !track_species)))
        return sim->fail(ATTPC_E_BADARG, "attpc_simulate_replay: bad arguments");
    CU(cudaSetDevice(sim->device));
    const int64_t n_rows = track_offsets[n_tracks];
    int32_t t_max = 1;
    for (int64_t t = 0; t < n_tracks; ++t) {
        if (track_event[t] < 0 || track_event[t] >= n_events)
            return sim->fail(ATTPC_E_BADARG, "track_event[%lld] outside 0..n_events-1", (long long)t);
        if (track_rank[t] < 0 || track_rank[t] >= MAX_TRACKS_PER_EVENT)
            return sim->fail(ATTPC_E_BADARG, "track_rank[%lld] outside 0..%d", (long long)t, MAX_TRACKS_PER_EVENT - 1);
        if (track_species[t] >= sim->P.n_species)
            return sim->fail(ATTPC_E_BADARG, "track_species[%lld] outside the species of this simulator", (long long)t);
        if (track_offsets[t + 1] < track_offsets[t]) return sim->fail(ATTPC_E_BADARG, "track_offsets not monotone");
        t_max = std::max(t_max, track_rank[t] + 1);
    }
    std::vector<int32_t> label_map((size_t)std::max<int64_t>(1, n_events) * t_max, -1);
    for (int64_t t = 0; t < n_tracks; ++t) label_map[(size_t)track_event[t] * t_max + track_rank[t]] = track_label[t];

    DevArray<int64_t> d_off, d_ukeys, d_uoff;
    DevArray<double> d_rows, d_norm, d_uvals;
    DevArray<int32_t> d_ev, d_rank, d_sp, d_lab;
    DevArray<long long> d_el;
    auto up = [&](auto& arr, const auto* src, int64_t n) -> cudaError_t {
        cudaError_t e = arr.reserve(std::max<int64_t>(1, n));
        if (e != cudaSuccess || n == 0) return e;
        return cudaMemcpyAsync(arr.p, src, (size_t)n * sizeof(*src), cudaMemcpyHostToDevice, sim->stream);
    };
    CU(up(d_off, track_offsets, n_tracks + 1));
    CU(up(d_rows, points, n_rows * 6));
    CU(up(d_norm, normals, n_rows));
    CU(up(d_ev, track_event, n_tracks));
    CU(up(d_rank, track_rank, n_tracks));
    CU(up(d_sp, track_species, n_tracks));
    CU(up(d_lab, label_map.data(), (int64_t)label_map.size()));
    if (electrons_out) CU(d_el.reserve(std::max<int64_t>(1, n_rows)));
    LaunchPlan plan;
    if (replay && replay->u_offsets) {
        const int64_t nu = replay->u_offsets[n_events];
        CU(up(d_uoff, replay->u_offsets, n_events + 1));
        CU(up(d_ukeys, replay->u_keys, nu));
        CU(up(d_uvals, replay->u_vals, nu));
        plan.uniforms = ReplayUniforms{d_uoff.p, d_ukeys.p, d_uvals.p};
    }
    ReplayBatch rb;
    rb.track_offsets = d_off.p;
    rb.rows = d_rows.p;
    rb.normals = d_norm.p;
    rb.track_event = d_ev.p;
    rb.track_rank = d_rank.p;
    rb.track_species = d_sp.p;
    rb.n_tracks = n_tracks;
    rb.n_rows = n_rows;
    rb.electrons_out = electrons_out ? d_el.p : nullptr;
    plan.replay = &rb;
    plan.label_of_event_rank_dev = d_lab.p;
    plan.n_tracks_per_event = t_max;
    const int rc = run_batch(sim, plan, n_events, flags, result, 0.f);
    if (rc) return rc;
    if (electrons_out && n_rows > 0)
        CU(cudaMemcpy(electrons_out, d_el.p, (size_t)n_rows * sizeof(long long), cudaMemcpyDeviceToHost));
    result->n_tracks = n_tracks;
    return ATTPC_OK;
}

int attpc_trajectories(AttpcSim* sim, const double* momenta, const double* vertices, const int32_t* species,
                       int64_t n_tracks, int32_t stride, int32_t max_points, double* out_points, int32_t* out_counts) {
    if (!sim) return ATTPC_E_BADARG;
    if (n_tracks < 0 || stride < 1 || max_points < 1 || !out_points || !out_counts ||
        (n_tracks > 0 && (!momenta || !vertices || !species)))
        return sim->fail(ATTPC_E_BADARG, "attpc_trajectories: bad arguments");
    if (n_tracks == 0) return ATTPC_OK;
    for (int64_t t = 0; t < n_tracks; ++t)
        if (species[t] >= sim->P.n_species) return sim->fail(ATTPC_E_BADARG, "species[%lld] out of range", (long long)t);
    CU(cudaSetDevice(sim->device));
    int rc = ensure_work_buffers(sim, 1, 1, 1);
    if (rc) return rc;
    DevArray<double> d_m, d_v, d_out;
    DevArray<int32_t> d_sp, d_cnt;
    CU(d_m.reserve(n_tracks * 4));
    CU(d_v.reserve(n_tracks * 3));
    CU(d_sp.reserve(n_tracks));
    CU(d_cnt.reserve(n_tracks));
    CU(d_out.reserve(n_tracks * max_points * 6));
    CU(cudaMemcpyAsync(d_m.p, momenta, (size_t)n_tracks * 4 * sizeof(double), cudaMemcpyHostToDevice, sim->stream));
    CU(cudaMemcpyAsync(d_v.p, vertices, (size_t)n_tracks * 3 * sizeof(double), cudaMemcpyHostToDevice, sim->stream));
    CU(cudaMemcpyAsync(d_sp.p, species, (size_t)n_tracks * sizeof(int32_t), cudaMemcpyHostToDevice, sim->stream));
    CU(cudaMemsetAsync(d_out.p, 0, (size_t)n_tracks * max_points * 6 * sizeof(double), sim->stream));
    CU(cudaMemsetAsync(d_cnt.p, 0, (size_t)n_tracks * sizeof(int32_t), sim->stream));
    CU(cudaMemsetAsync(sim->slot[0].counters.p, 0, sizeof(Counters), sim->stream));
    TrackBatch tb;
    memset(&tb, 0, sizeof tb);
    tb.momenta = d_m.p;
    tb.vertices = d_v.p;
    tb.n_events = n_tracks;
    tb.n_nuclei = 1;
    tb.n_tracks_per_event = 1;
    tb.rec_species = d_sp.p;
    tb.rec_points = d_out.p;
    tb.rec_counts = d_cnt.p;
    tb.rec_stride = stride;
    tb.rec_max = max_points;
    rc = launch_tracks<true>(sim, tb, n_tracks, 0, sim->stream);
    if (rc) return rc;
    CU(cudaMemcpyAsync(out_points, d_out.p, (size_t)n_tracks * max_points * 6 * sizeof(double), cudaMemcpyDeviceToHost,
                       sim->stream));
    CU(cudaMemcpyAsync(out_counts, d_cnt.p, (size_t)n_tracks * sizeof(int32_t), cudaMemcpyDeviceToHost, sim->stream));
    CU(cudaStreamSynchronize(sim->stream));
    return ATTPC_OK;
}

int attpc_convert_to_spyral(AttpcSim* sim, const int64_t* offsets, const double* cloud, const int64_t* labels,
                            int64_t n_events, uint32_t flags, AttpcResult* result) {
    if (!sim) return ATTPC_E_BADARG;
    if (!result || n_events < 0 || !offsets) return sim->fail(ATTPC_E_BADARG, "attpc_convert_to_spyral: bad arguments");
    const int64_t n_points = offsets[n_events];
    if (n_points < 0 || (n_points > 0 && (!cloud || !labels)))
        return sim->fail(ATTPC_E_BADARG, "attpc_convert_to_spyral: bad cloud");
    CU(cudaSetDevice(sim->device));
    memset(result, 0, sizeof *result);
    sim->events_used = 0;
    sim->launches = 0;
    OutputPlan op;  // the cloud comes from the host; the rows go back in one copy once they are counted
    op.spy = op.spy_rows = true;
    op.cloud_rows = {{&sim->cloud, false}, {&sim->labels, false}};
    op.spyral_rows = {{&sim->rows, false}, {&sim->row_labels, false}};
    int rc = reserve_outputs(sim, op, n_events, std::max<int64_t>(1, n_points), false);
    if (rc) return rc;
    CU(cudaMemcpyAsync(sim->offsets_dev.p, offsets, (size_t)(n_events + 1) * sizeof(int64_t), cudaMemcpyHostToDevice,
                       sim->stream));
    if (n_points > 0) {
        CU(cudaMemcpyAsync(sim->cloud.d(), cloud, (size_t)n_points * 3 * sizeof(double), cudaMemcpyHostToDevice,
                           sim->stream));
        CU(cudaMemcpyAsync(sim->labels.d(), labels, (size_t)n_points * sizeof(int64_t), cudaMemcpyHostToDevice,
                           sim->stream));
    }
    result->n_events = n_events;
    result->n_points = n_points;
    CU(sim->csr_total.reserve(3));
    CU(cudaMemsetAsync(sim->csr_total.p + 2, 0, sizeof(unsigned long long), sim->stream));
    CU(cudaMemsetAsync(sim->row_offsets_dev.p, 0, sizeof(int64_t), sim->stream));
    rc = launch_spyral(sim, spyral_args(sim, 0, n_events, false, (flags & ATTPC_ROWS_KEEP_ALL) != 0, nullptr));
    if (rc) return rc;
    CU(sim->row_offsets_host.reserve(n_events + 1));
    CU(cudaMemcpyAsync(sim->row_offsets_host.p, sim->row_offsets_dev.p, (size_t)(n_events + 1) * sizeof(int64_t),
                       cudaMemcpyDeviceToHost, sim->stream));
    CU(cudaStreamSynchronize(sim->stream));
    const int64_t n_rows = sim->row_offsets_host.p[n_events];
    result->n_rows = n_rows;
    result->row_offsets = sim->row_offsets_host.p;
    CU(sim->rows.reserve_host(std::max<int64_t>(1, n_rows), false));
    CU(sim->row_labels.reserve_host(std::max<int64_t>(1, n_rows), false));
    if (n_rows > 0) {
        CU(sim->rows.copy_to_host(0, n_rows, sim->stream));
        CU(sim->row_labels.copy_to_host(0, n_rows, sim->stream));
    }
    CU(cudaStreamSynchronize(sim->stream));
    result->rows = sim->rows.h();
    result->row_labels = sim->row_labels.h();
    result->n_kernel_launches = sim->launches;
    return ATTPC_OK;
}

int attpc_read_device(AttpcSim* sim, const void* dev, void* host, int64_t n_bytes) {
    if (!sim) return ATTPC_E_BADARG;
    if (n_bytes < 0 || (n_bytes > 0 && (!dev || !host))) return sim->fail(ATTPC_E_BADARG, "attpc_read_device: bad arguments");
    if (n_bytes == 0) return ATTPC_OK;
    CU(cudaSetDevice(sim->device));
    CU(cudaStreamSynchronize(sim->stream));
    CU(cudaMemcpy(host, dev, (size_t)n_bytes, cudaMemcpyDeviceToHost));
    return ATTPC_OK;
}

int attpc_lookup_pads(AttpcSim* sim, const double* xy, int64_t n, int32_t* pads_out) {
    if (!sim) return ATTPC_E_BADARG;
    if (n < 0 || (n > 0 && (!xy || !pads_out))) return sim->fail(ATTPC_E_BADARG, "attpc_lookup_pads: bad arguments");
    if (n == 0) return ATTPC_OK;
    CU(cudaSetDevice(sim->device));
    DevArray<double> d_xy;
    DevArray<int32_t> d_out;
    CU(d_xy.reserve(n * 2));
    CU(d_out.reserve(n));
    CU(cudaMemcpyAsync(d_xy.p, xy, (size_t)n * 2 * sizeof(double), cudaMemcpyHostToDevice, sim->stream));
    lookup_kernel<<<(unsigned)((n + 255) / 256), 256, 0, sim->stream>>>(sim->P, d_xy.p, n, d_out.p);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(pads_out, d_out.p, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, sim->stream));
    CU(cudaStreamSynchronize(sim->stream));
    return ATTPC_OK;
}

}  // extern "C"
