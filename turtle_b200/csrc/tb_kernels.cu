/*
 * tb_kernels.cu -- sm_100a kernels and the batched C ABI of turtle-b200.
 *
 * Hot path: turtle_stepper_step (ref: src/turtle/stepper.c:780-875) for millions
 * of independent rays. Design (DESIGN.md has the full story):
 *
 *  - one ray per lane, persistent CTAs sized to the SM count, rays pulled from a
 *    global cursor; finished lanes are refilled with a warp ballot/popc
 *    compaction so that heavy-tailed rays do not idle their warp;
 *  - the unit of lockstep work is the geometry SAMPLE, not the step: each loop
 *    iteration evaluates exactly one stepper_sample (geodetic transform ->
 *    projection -> 2x2 gather) for every lane, then a branch-light update of a
 *    three-state machine {INIT, TENTATIVE, BISECT}. The 23-iteration boundary
 *    bisection of one lane therefore costs its warp nothing extra;
 *  - DEM tiles are int16/uint16 grids resident in HBM, rows south first with a
 *    32-byte aligned pitch; the flattened geometry travels as a __grid_constant__
 *    kernel parameter (constant bank), map descriptors and the tile table sit in
 *    global memory behind the read-only cache;
 *  - FP64 throughout, compiled with -fmad=false: see tb_core.cuh.
 *
 * No tensor cores: the path is FP64-pipe / issue bound (DESIGN.md roofline).
 */
#include <cuda_runtime.h>
#include <cuda_pipeline.h>
#include <cub/device/device_radix_sort.cuh>

#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <float.h>

#include <algorithm>
#include <map>
#include <mutex>
#include <new>
#include <vector>

#include "tb_host.hpp"
#include "tb_io.hpp"
#include "turtle_b200.h"

#define FN(f) ((turtle_function_t *)(f))
static const char * BATCH_CU = "turtle_b200/csrc/tb_kernels.cu";

#define CUDA_TRY(fn, call)                                                         \
        do {                                                                       \
                cudaError_t err_ = (call);                                         \
                if (err_ != cudaSuccess)                                           \
                        return tbh::raise(FN(fn), TURTLE_RETURN_LIBRARY_ERROR,     \
                            BATCH_CU, __LINE__, "CUDA error: %s (%s)",             \
                            cudaGetErrorString(err_), #call);                      \
        } while (0)

/* ======================================================================== */
/* Device code                                                               */
/* ======================================================================== */

namespace {

enum { MODE_IDLE = 0, MODE_INIT = 1, MODE_TENT = 2, MODE_BISECT = 3,
       MODE_REBUILD = 4, /* runs the three transforms of a stale Jacobian that is about to be read */
       MODE_WAIT = 6, /* holds a queue ticket whose ray has not arrived on the device yet */
       MODE_DONE = 7  /* trace: the record is complete in shared memory, to be written out */ };

struct TraceArgs {
        unsigned long long n;
        const unsigned * order; /* queue position -> ray index, or NULL (identity) */
        const double * position;
        const double * direction;
        turtle_trace_result * results;
        unsigned long long * cursor; /* [0] next ray, [1] steps, [2] samples */
        double altitude_min, altitude_max, length_max;
        int max_steps;
        /* streaming (host-pointer calls, see trace_streamed): rays [0, *watermark) have
         * arrived; chunk_done[k] counts the finished rays of chunk k = ray >> chunk_shift.
         * NULL: everything is resident, nothing is counted. */
        int chunk_shift;
        const unsigned long long * watermark;
        unsigned * chunk_done;
        unsigned * chunk_flags; /* host-mapped: chunk k is complete (set by the kernel) */
        /* medium changes of every ray (turtle_stepper_trace_crossings), or NULL */
        turtle_trace_crossing * crossings;
        int max_crossings;
};

/* Device tables of a fan (fan_upload): ray r belongs to station s = r / per_station and starts
 * at its origin; direction of ray (i, j) from the host's sines / cosines of the angles,
 * az[i] = { sin az, cos az }, el[j] = { cos el, sin el }, and the station's East / North / Up
 * vectors (ecef.c:136-178). */
struct FanTables {
        const double2 * az;
        const double2 * el;
        const double * station; /* [n_station][12]: origin, East, North, Up */
        unsigned long long naz, bundle, per_station;
        unsigned long long ray0; /* first ray of this launch */
};

/* Compact input / output (turtle_stepper_trace_fan / _fields): a kernel parameter of its
 * own, of the COMPACT kernels only -- the mere presence of these members in TraceArgs
 * costs every trace kernel four registers. */
struct CompactArgs {
        FanTables fan; /* fan input (turtle_stepper_trace_fan[s]; TraceArgs::position == NULL) */
        /* field outputs (turtle_trace_fields: device arrays, any NULL), when use_fields */
        turtle_trace_fields fields;
        int use_fields;
};

struct NoCompactArgs {
        int unused;
};

/* How the trace kernel of a uniform stack gathers its nodes (turtle_plan_gather_set):
 * GATHER_GLOBAL four 16-bit loads, GATHER_PACKED one 8-byte load from the cell-packed copy
 * of the tiles, GATHER_WINDOW a window of one tile staged in shared memory. */
enum { GATHER_GLOBAL = 0, GATHER_PACKED = 1, GATHER_WINDOW = 2 };
enum { WINDOW_NODES = 64 }; /* nodes per side of the window: 8 kB of shared memory per CTA */

/* The window of a GATHER_WINDOW kernel: WINDOW_NODES x WINDOW_NODES nodes of ONE tile,
 * first node (x0, y0); x0 is a multiple of 8 nodes (16-byte aligned rows for the bulk
 * copies). */
struct WindowArgs {
        const uint16_t * tile; /* row-major nodes of the tile, as in its TileRec */
        int x0, y0, pitch;
        unsigned long long * hits; /* [0] samples served by the window, [1] all samples */
};

/* Third kernel parameter by variant (never both: the compact kernels gather globally). */
template <bool COMPACT, int GATHER = GATHER_GLOBAL> struct ExtraOf {
        typedef NoCompactArgs type;
};
template <> struct ExtraOf<true, GATHER_GLOBAL> {
        typedef CompactArgs type;
};
template <> struct ExtraOf<false, GATHER_WINDOW> {
        typedef WindowArgs type;
};

#define STREAM_ABORT (~0ull)
#define STREAM_TIMEOUT_NS 20000000000ull /* a lane never waits longer for its ray */

__device__ __forceinline__ unsigned long long global_ns()
{
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        return t;
}

/* Streamed calls: a record must be visible before it is counted for its chunk. The fence
 * that guarantees it stalls the whole warp, so counts are deferred: a lane remembers what
 * it owes (chunk in the high bits, number of rays in the low 8) and the warp settles its
 * debts with ONE fence -- every 1024 iterations, when it runs dry, or when a lane would owe
 * to two chunks. The records are stored by other lanes of the warp than the one that owes
 * (warp-cooperative write-out below): every lane fences its own stores, the warp
 * synchronises, then the owners count. Warp uniform. */
__device__ __forceinline__ void settle_done(const TraceArgs & A, int & owed)
{
        if (__any_sync(0xffffffffu, owed >= 0)) {
                __threadfence();
                __syncwarp();
                if (owed >= 0) {
                        const unsigned k = (unsigned)(owed >> 8), add = (unsigned)(owed & 0xff);
                        const unsigned before = atomicAdd(A.chunk_done + k, add);
                        /* the count that completes a chunk tells the host, which drains
                         * the chunks in the order they complete */
                        const unsigned long long first = (unsigned long long)k << A.chunk_shift;
                        const unsigned long long rest = A.n - first;
                        const unsigned size = (rest >> A.chunk_shift) ? (1u << A.chunk_shift) :
                                                                        (unsigned)rest;
                        if (before + add == size) {
                                __threadfence_system();
                                *(volatile unsigned *)(A.chunk_flags + k) = 1u;
                        }
                }
                owed = -1;
        }
}

__device__ __forceinline__ bool finite3(const double v[3])
{
        return isfinite(v[0]) && isfinite(v[1]) && isfinite(v[2]);
}

/* Per-lane ray state of the trace kernel, kept in SHARED memory (structure of arrays,
 * one column per thread: conflict free). Nothing of it is needed while a sample is
 * being evaluated, so parking it here instead of in registers leaves the register
 * file to the FP64 code of the sample: no spills at 6 CTAs per SM. */
enum { F_POS = 0, F_DIR = 3, F_ALT = 6, F_ELEV0, F_ELEV1, F_DS, F_DS0, F_DS1,
       F_LEN, F_TOTAL = F_LEN + TURTLE_TRACE_MEDIA,
       N_F_BASE,                  /* rows of a trace without the local approximation */
       F_LASTPOS = N_F_BASE,      /* + stepper->last.position (local approximation only) */
       N_F_LLA = F_LASTPOS + 3,
       F_LAT = N_F_LLA, F_LON,    /* + published latitude, longitude (step_batch only) */
       N_F = F_LON + 1 };
enum { I_IDX0 = 0, I_IDX1, I_MEDIUM0, I_NSTEPS, I_NCHANGES, I_HASH, I_RAYLO, I_RAYHI,
       N_I_BASE,
       I_PEND = N_I_BASE, /* + local approximation: transforms whose Jacobian is stale */
       I_RB_MASK,         /*   ... of which the ones being rebuilt now (MODE_REBUILD) */
       I_RESUME, I_RB_AXIS, N_I };

/* Only the rows a kernel uses are allocated: the shared memory a CTA does not take is
 * L1 cache for the DEM gathers (17 + 4 kB per CTA for a trace without the local
 * approximation: 6 CTAs per SM leave ~120 kB of L1 instead of 60 kB). */
template <int NF, int NI> struct LaneStoreT {
        double f[NF][128];
        int i[NI][128];
};
typedef LaneStoreT<N_F, N_I> LaneStore;

__device__ __forceinline__ void compiler_fence() { asm volatile("" ::: "memory"); }

/* Row k of this lane's column of `store`, a LaneStoreT<NF, NI> (rows beyond the allocation
 * are only named in code that is compiled out). */
#define SF(k) store.f[((k) < NF) ? (k) : 0][tid]
#define SI(k) store.i[((k) < NI) ? (k) : 0][tid]

/* ---- pieces of the lane-store stepper that the trace, horizon, voxel and walk kernels share ---- */

/* Start ray r at pos, dir in this lane's column: every ray starts from a reset stepper
 * (turtle_stepper_reset, stepper.c:647-651). Returns MODE_INIT, or MODE_DONE for a ray that
 * is never traced: an empty INVALID record (position as given), written out with the others. */
template <bool LLA, int NF, int NI>
__device__ __forceinline__ int ray_start(const tb::Geometry & G, const tb::LlaShared & V,
    LaneStoreT<NF, NI> & store, const unsigned tid, unsigned long long r, const double pos[3],
    const double dir[3])
{
        SF(F_POS) = pos[0];
        SF(F_POS + 1) = pos[1];
        SF(F_POS + 2) = pos[2];
        SF(F_DIR) = dir[0];
        SF(F_DIR + 1) = dir[1];
        SF(F_DIR + 2) = dir[2];
#pragma unroll
        for (int m = 0; m < TURTLE_TRACE_MEDIA; m++)
                SF(F_LEN + m) = 0.;
        SF(F_TOTAL) = 0.;
        SI(I_NSTEPS) = 0;
        SI(I_NCHANGES) = 0;
        SI(I_RAYLO) = (int)(unsigned)(r & 0xffffffffull);
        SI(I_RAYHI) = (int)(unsigned)(r >> 32);
        if (LLA) {
                SI(I_PEND) = 0;
                SF(F_LASTPOS) = SF(F_LASTPOS + 1) = SF(F_LASTPOS + 2) = DBL_MAX;
                tb::lla_reset(G, V);
        }
        if (!finite3(pos) || !finite3(dir)) {
                SF(F_ALT) = 0.;
                SI(I_IDX0) = -1;
                SI(I_IDX1) = -1;
                SI(I_HASH) = 0;
                SI(I_MEDIUM0) = TURTLE_TRACE_INVALID;
                return MODE_DONE;
        }
        return MODE_INIT;
}

/* 8-byte field k < 12 of the 96-byte record of the finished lane t of this warp (MODE_DONE).
 * Lane k stores field k: the twelve fields of a record go side by side, three full sectors
 * in one request instead of twelve partial ones from one lane -- what makes the stores into
 * a PEER's memory (multi-GPU, DESIGN.md section 7) cheap on NVLink, where every request is
 * a packet. */
template <int NF, int NI>
__device__ __forceinline__ unsigned long long record_field(const LaneStoreT<NF, NI> & store,
    unsigned t, unsigned k)
{
        if (k < 9u) {
                const int row = (k < 3u) ? (int)(F_POS + k) :
                    ((k == 3u) ? (int)F_ALT : ((k < 8u) ? (int)(F_LEN + k - 4u) : (int)F_TOTAL));
                return (unsigned long long)__double_as_longlong(store.f[row][t]);
        }
        const int lo = (k == 9u) ? I_NSTEPS : ((k == 10u) ? I_IDX0 : I_HASH);
        const int hi = (k == 9u) ? I_MEDIUM0 : ((k == 10u) ? I_IDX1 : I_NCHANGES);
        return ((unsigned long long)(unsigned)store.i[hi][t] << 32) | (unsigned long long)(unsigned)store.i[lo][t];
}

/* Why a trace stops after a step (or the initial query) that settled on `last`, `total`
 * metres and `n_steps` steps from its start (the limits of its turtle_trace_rule), or -1:
 * it goes on. */
template <class Args>
__device__ __forceinline__ int stop_status(const Args & A, const tb::Sample & last, double total,
    int n_steps)
{
        int status = -1;
        if (last.idx0 < 0)
                status = TURTLE_TRACE_DOMAIN;
        else if (!(last.alt < A.altitude_max) || !(last.alt > A.altitude_min))
                status = TURTLE_TRACE_ALTITUDE;
        else if (total >= A.length_max)
                status = TURTLE_TRACE_LENGTH;
        else if (n_steps >= A.max_steps)
                status = TURTLE_TRACE_STEPS;
        return status;
}

/* The state update of a lane after its sample S (stepper.c:822-863): MODE_INIT's initial
 * query, MODE_TENT's tentative step, MODE_BISECT's bisection of a medium change. S is
 * published to the lane store when it becomes stepper->last. Returns true when a step (or
 * the initial query) settled, with `last` = stepper->last and `ds` = the step's length;
 * medium0 is the medium the step started in. HASH: MODE_INIT starts the FNV-1a hash of
 * the media in I_HASH (a trace record; the horizon kernel uses that row otherwise). SHAPE_STACK: `moved` is the sampled position
 * (lane_sample). */
template <bool LLA, int SHAPE, bool HASH, int NF, int NI>
__device__ __forceinline__ bool lane_advance(LaneStoreT<NF, NI> & store, const unsigned tid,
    int & mode, const tb::Sample & S, const double moved[3], const int medium0, double & ds,
    tb::Sample & last)
{
        bool settle = false;  /* a step (or the initial query) completed */
        bool publish = false; /* S becomes stepper->last */
        if (mode == MODE_INIT) {
                publish = true;
                if (HASH) SI(I_HASH) = (int)((2166136261u ^ (unsigned)(S.idx0 + 1)) * 16777619u);
                settle = true;
        } else if (mode == MODE_TENT) {
                /* position += direction * ds, stepper.c:824 */
                if (SHAPE == tb::SHAPE_STACK) {
                        SF(F_POS) = moved[0];
                        SF(F_POS + 1) = moved[1];
                        SF(F_POS + 2) = moved[2];
                } else {
                        SF(F_POS) += SF(F_DIR) * ds;
                        SF(F_POS + 1) += SF(F_DIR + 1) * ds;
                        SF(F_POS + 2) += SF(F_DIR + 2) * ds;
                }
                publish = true;
                if (S.idx0 != medium0) { /* stepper.c:832-838 */
                        SF(F_DS0) = -ds;
                        SF(F_DS1) = 0.;
                        mode = MODE_BISECT;
                        settle = !(0. - (-ds) > 1E-08);
                } else {
                        settle = true;
                }
        } else {
                double ds0 = SF(F_DS0), ds1 = SF(F_DS1);
                const double ds2 = 0.5 * (ds0 + ds1);
                if (S.idx0 == medium0) { /* stepper.c:848-859 */
                        ds0 = ds2;
                        SF(F_DS0) = ds0;
                } else {
                        ds1 = ds2;
                        SF(F_DS1) = ds1;
                        publish = true;
                        if (LLA) { /* last.position = position2 */
                                SF(F_LASTPOS) = SF(F_POS) + SF(F_DIR) * ds2;
                                SF(F_LASTPOS + 1) = SF(F_POS + 1) + SF(F_DIR + 1) * ds2;
                                SF(F_LASTPOS + 2) = SF(F_POS + 2) + SF(F_DIR + 2) * ds2;
                        }
                }
                if (!(ds1 - ds0 > 1E-08)) { /* stepper.c:861-863 */
                        ds += ds1;
                        SF(F_POS) += SF(F_DIR) * ds1;
                        SF(F_POS + 1) += SF(F_DIR + 1) * ds1;
                        SF(F_POS + 2) += SF(F_DIR + 2) * ds1;
                        settle = true;
                }
        }
        if (publish) { /* latitude and longitude are not part of a trace result */
                SF(F_ALT) = S.alt;
                SF(F_ELEV0) = S.elev0;
                SF(F_ELEV1) = S.elev1;
                SI(I_IDX0) = S.idx0;
                SI(I_IDX1) = S.idx1;
        }
        if (!settle) return false;
        last.lat = last.lon = 0.;
        last.alt = publish ? S.alt : SF(F_ALT);
        last.elev0 = publish ? S.elev0 : SF(F_ELEV0);
        last.elev1 = publish ? S.elev1 : SF(F_ELEV1);
        last.idx0 = publish ? S.idx0 : SI(I_IDX0);
        last.idx1 = publish ? S.idx1 : SI(I_IDX1);
        return true;
}

/* Add the counters of this warp's lanes to a call's: [1] steps, [2] samples, [4] Jacobian
 * columns (local approximation only). */
template <bool LLA>
__device__ __forceinline__ void flush_counters(unsigned long long * cursor, unsigned lane,
    unsigned steps, unsigned samples, unsigned rebuilds)
{
        unsigned long long steps64 = steps, samples64 = samples, rebuilds64 = rebuilds;
        for (int o = 16; o > 0; o >>= 1) {
                steps64 += __shfl_down_sync(0xffffffffu, steps64, o);
                samples64 += __shfl_down_sync(0xffffffffu, samples64, o);
                if (LLA) rebuilds64 += __shfl_down_sync(0xffffffffu, rebuilds64, o);
        }
        if (lane == 0u) {
                atomicAdd(cursor + 1, steps64);
                atomicAdd(cursor + 2, samples64);
                if (LLA) atomicAdd(cursor + 4, rebuilds64);
        }
}

/* Compact input / output of the trace kernel (COMPACT variants only: the kernels of
 * turtle_stepper_trace_fan / _fields; the others do not carry this code). */

/* Origin and direction of ray r of a fan: the products and sums of
 * turtle_ecef_from_horizontal (ecef.c:170-177) on the host's sines / cosines of the two
 * angles and the frame of the ray's station, read once per ray. */
__device__ __forceinline__ void fan_ray(const CompactArgs & A, unsigned long long r, double pos[3],
    double dir[3])
{
        const FanTables & T = A.fan;
        const unsigned long long per_band = T.naz * T.bundle;
        const unsigned long long rs = r + T.ray0;
        const unsigned long long s = rs / T.per_station;
        const unsigned long long rr = rs - s * T.per_station;
        const unsigned long long band = rr / per_band;
        const unsigned long long rem = rr - band * per_band;
        const unsigned long long i = rem / T.bundle;
        const unsigned long long j = band * T.bundle + (rem - i * T.bundle);
        const double2 az = __ldg(T.az + i);
        const double2 el = __ldg(T.el + j);
        const double r0 = el.x * az.x, r1 = el.x * az.y, r2 = el.y;
        const double * f = T.station + 12ull * s;
#pragma unroll
        for (int c = 0; c < 3; c++) {
                pos[c] = __ldg(f + c);
                dir[c] = r0 * __ldg(f + 3 + c) + r1 * __ldg(f + 6 + c) + r2 * __ldg(f + 9 + c);
        }
}

__device__ __forceinline__ void fan_ray(const NoCompactArgs &, unsigned long long, double *, double *) {}
__device__ __forceinline__ void store_fields(const NoCompactArgs &, const double *, const int *) {}
__device__ __forceinline__ bool wants_fields(const NoCompactArgs &) { return false; }
__device__ __forceinline__ bool wants_fields(const WindowArgs &) { return false; }
__device__ __forceinline__ void fan_ray(const WindowArgs &, unsigned long long, double *, double *) {}
__device__ __forceinline__ void store_fields(const WindowArgs &, const double *, const int *) {}

/* Nodes of a cell from the shared-memory window when the cell lies in it, else from
 * global memory (tb::NodesGlobal). */
struct NodesWindow {
        const uint16_t * window;
        const uint16_t * tile;
        int x0, y0;
        mutable unsigned hits;
        __device__ __forceinline__ void fetch(const uint16_t * nodes, int pitch, int ix, int iy,
            uint16_t r[4]) const
        {
                const unsigned dx = (unsigned)(ix - x0), dy = (unsigned)(iy - y0);
                if ((nodes == tile) && (dx < WINDOW_NODES - 1u) && (dy < WINDOW_NODES - 1u)) {
                        const uint16_t * w = window + dy * WINDOW_NODES + dx;
                        r[0] = w[0];
                        r[1] = w[1];
                        r[2] = w[WINDOW_NODES];
                        r[3] = w[WINDOW_NODES + 1];
                        hits++;
                } else {
                        tb::NodesGlobal().fetch(nodes, pitch, ix, iy, r);
                }
        }
};

/* Stage the window: one bulk copy (cp.async.bulk, the TMA engine's 1-D form) per row,
 * all completing on ONE mbarrier that every thread of the CTA then waits on. */
__device__ __forceinline__ void window_load(uint16_t * window, unsigned long long * barrier,
    const WindowArgs & W)
{
        const unsigned bar = (unsigned)__cvta_generic_to_shared(barrier);
        if (threadIdx.x == 0) {
                asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
                asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncthreads();
        if (threadIdx.x == 0) {
                const unsigned row_bytes = WINDOW_NODES * (unsigned)sizeof(uint16_t);
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar),
                    "r"(row_bytes * WINDOW_NODES)
                    : "memory");
                for (int r = 0; r < WINDOW_NODES; r++) {
                        const unsigned dst = (unsigned)__cvta_generic_to_shared(window + r * WINDOW_NODES);
                        const uint16_t * src = W.tile + (size_t)(W.y0 + r) * (size_t)W.pitch + W.x0;
                        asm volatile(
                            "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes "
                            "[%0], [%1], %2, [%3];" ::"r"(dst),
                            "l"(src), "r"(row_bytes), "r"(bar)
                            : "memory");
                }
        }
        unsigned done = 0u;
        while (!done) {
                asm volatile("{\n.reg .pred p;\n"
                             "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n"
                             "selp.u32 %0, 1, 0, p;\n}"
                             : "=r"(done)
                             : "r"(bar)
                             : "memory");
        }
}

__device__ __forceinline__ void window_setup(NodesWindow & from, uint16_t * window,
    unsigned long long * barrier, const WindowArgs & W)
{
        window_load(window, barrier, W);
        from.tile = W.tile;
        from.x0 = W.x0;
        from.y0 = W.y0;
}
template <class Other>
__device__ __forceinline__ void window_setup(NodesWindow &, uint16_t *, unsigned long long *,
    const Other &)
{
}
__device__ __forceinline__ bool wants_fields(const CompactArgs & C) { return C.use_fields != 0; }

/* The columns of a finished ray the caller asked for (turtle_trace_fields), from the
 * rows of the lane store: f = &store.f[0][tid], i = &store.i[0][tid], 128 apart. */
__device__ __forceinline__ void store_fields(const CompactArgs & A, const double * f, const int * i)
{
        const unsigned long long ray = ((unsigned long long)(unsigned)i[I_RAYHI * 128] << 32) |
            (unsigned long long)(unsigned)i[I_RAYLO * 128];
#pragma unroll
        for (int m = 0; m < TURTLE_TRACE_MEDIA; m++)
                if (A.fields.length[m] != NULL) A.fields.length[m][ray] = f[(F_LEN + m) * 128];
        if (A.fields.total != NULL) A.fields.total[ray] = f[F_TOTAL * 128];
        if (A.fields.altitude != NULL) A.fields.altitude[ray] = f[F_ALT * 128];
        if (A.fields.position != NULL) {
                A.fields.position[3 * ray] = f[F_POS * 128];
                A.fields.position[3 * ray + 1] = f[(F_POS + 1) * 128];
                A.fields.position[3 * ray + 2] = f[(F_POS + 2) * 128];
        }
        if (A.fields.n_steps != NULL) A.fields.n_steps[ray] = i[I_NSTEPS * 128];
        if (A.fields.status != NULL) A.fields.status[ray] = i[I_MEDIUM0 * 128];
        if (A.fields.index != NULL) {
                A.fields.index[2 * ray] = i[I_IDX0 * 128];
                A.fields.index[2 * ray + 1] = i[I_IDX1 * 128];
        }
        if (A.fields.medium_hash != NULL) A.fields.medium_hash[ray] = (uint32_t)i[I_HASH * 128];
        if (A.fields.n_changes != NULL) A.fields.n_changes[ray] = i[I_NCHANGES * 128];
}

/* The persistent ray-tracing kernel. MINB = CTAs of 128 threads per SM the register
 * allocation is bounded for (occupancy vs registers is a measured trade, DESIGN.md). */
template <bool LLA, bool PROJ, int MINB, int SHAPE = tb::SHAPE_GENERIC, bool STREAM = false,
    bool COMPACT = false, int GATHER = GATHER_GLOBAL>
__global__ void __launch_bounds__(128, MINB)
    trace_kernel(const __grid_constant__ tb::Geometry G, const TraceArgs A,
        const typename ExtraOf<COMPACT, GATHER>::type C)
{
        constexpr int NF = LLA ? N_F_LLA : N_F_BASE, NI = LLA ? N_I : N_I_BASE;
        __shared__ LaneStoreT<NF, NI> store;
        const unsigned tid = threadIdx.x;
        const unsigned lane = tid & 31u;
        const unsigned FULL = 0xffffffffu;

        int mode = MODE_IDLE;
        /* local approximation: G.lla_rows columns of per-lane state in DYNAMIC shared memory
         * (sized by the transforms the geometry uses, tb::LlaView) */
        extern __shared__ double lla_store[];
        const tb::LlaShared V = { lla_store + tid };
        /* (GATHER_WINDOW: the DEM window of this CTA, staged once by the bulk copy engine) */
        __shared__ __align__(128) uint16_t window[(GATHER == GATHER_WINDOW) ? WINDOW_NODES * WINDOW_NODES : 8];
        __shared__ unsigned long long window_barrier;
        NodesWindow from_window = { window, NULL, 0, 0, 0u };
        window_setup(from_window, window, &window_barrier, C);
        unsigned my_steps = 0u, my_samples = 0u, my_rebuilds = 0u;
        constexpr bool LLA_COUNT = LLA;
        bool exhausted = false;
        bool pending_wait = false; /* warp uniform: some lane holds a ticket */
        int owed = -1;             /* chunk whose completion count this lane still owes */
        unsigned iteration = 0u;
        unsigned long long t_wait = 0ull; /* STREAM: when this lane took its ticket */
        unsigned long long w_seen = 0ull; /* STREAM: the watermark as this lane saw it last */

        for (;;) {
                if (STREAM && ((++iteration & 1023u) == 0u)) settle_done(A, owed);
                /* ---- write out finished rays, one 96-byte record per instruction -------
                 * A finished lane has left its record in shared memory (MODE_DONE). */
                unsigned done_mask = __ballot_sync(FULL, mode == MODE_DONE);
                if (COMPACT && (done_mask != 0u) && wants_fields(C) && (mode == MODE_DONE))
                        store_fields(C, &store.f[0][tid], &store.i[0][tid]); /* field arrays */
                if (done_mask != 0u) __syncwarp(); /* the records are read across lanes */
                const bool wrote = done_mask != 0u;
                while (done_mask != 0u) {
                        const unsigned src = (unsigned)__ffs((int)done_mask) - 1u;
                        done_mask &= done_mask - 1u;
                        const unsigned t = (tid & ~31u) + src;
                        const unsigned long long ray =
                            ((unsigned long long)(unsigned)store.i[I_RAYHI][t] << 32) |
                            (unsigned long long)(unsigned)store.i[I_RAYLO][t];
                        if ((lane < 12u) && (!COMPACT || (A.results != NULL)))
                                reinterpret_cast<unsigned long long *>(A.results + ray)[lane] =
                                    record_field(store, t, lane);
                        if (STREAM) {
                                const int chunk = (int)(ray >> A.chunk_shift);
                                const int o = __shfl_sync(FULL, owed, (int)src);
                                if ((o >= 0) && (((o >> 8) != chunk) || ((o & 0xff) == 0xff)))
                                        settle_done(A, owed);
                                if (lane == src) owed = (owed >= 0) ? owed + 1 : ((chunk << 8) | 1);
                        }
                        if (lane == src) mode = MODE_IDLE;
                }
                if (wrote) __syncwarp(); /* ... before their columns are refilled */
                /* ---- refill idle lanes from the global ray queue ----------
                 * An idle lane takes a ticket q (one atomicAdd per warp, ballot / popc
                 * ranks) and WAITs until ray q is on the device: at once when the whole
                 * batch is resident, else when the copy stream has moved the watermark
                 * past q -- the other lanes of the warp keep stepping meanwhile. */
                const unsigned idle = __ballot_sync(FULL, mode == MODE_IDLE);
                if ((idle != 0u) || (STREAM && pending_wait)) {
                        if ((idle != 0u) && !exhausted) {
                                const int need = __popc(idle);
                                unsigned long long base = 0ull;
                                if (lane == 0u)
                                        base = atomicAdd(A.cursor, (unsigned long long)need);
                                base = __shfl_sync(FULL, base, 0);
                                if (mode == MODE_IDLE) {
                                        const unsigned rank = __popc(idle & ((1u << lane) - 1u));
                                        const unsigned long long q = base + rank;
                                        if (q < A.n) {
                                                SI(I_RAYLO) = (int)(unsigned)(q & 0xffffffffull);
                                                SI(I_RAYHI) = (int)(unsigned)(q >> 32);
                                                mode = MODE_WAIT;
                                                if (STREAM) t_wait = global_ns();
                                        }
                                }
                                if (base + (unsigned long long)need >= A.n) exhausted = true;
                        }
                        if (mode == MODE_WAIT) {
                                const unsigned long long q =
                                    ((unsigned long long)(unsigned)SI(I_RAYHI) << 32) |
                                    (unsigned long long)(unsigned)SI(I_RAYLO);
                                bool arrived = true;
                                if (STREAM) {
                                        /* (the watermark only moves forward: it is read
                                         * again only when what this lane saw last does not
                                         * cover its ticket -- never, once a fan's tables or
                                         * the last chunk are in) */
                                        if (q >= w_seen)
                                                w_seen = *(const volatile unsigned long long *)A.watermark;
                                        const unsigned long long w = w_seen;
                                        arrived = q < w;
                                        if (w == STREAM_ABORT) {
                                                mode = MODE_IDLE; /* the host gave up */
                                        } else if (!arrived &&
                                            (global_ns() - t_wait > STREAM_TIMEOUT_NS)) {
                                                /* the copies never came (a fault on the host
                                                 * side): give the GPU back and flag it */
                                                A.cursor[3] = 1ull;
                                                mode = MODE_IDLE;
                                        }
                                }
                                if (arrived && (mode == MODE_WAIT)) {
                                        /* acquire: the ray was written before the watermark
                                         * moved past it; no load below may be satisfied
                                         * before the watermark load above */
                                        if (STREAM) __threadfence();
                                        const unsigned long long r =
                                            (A.order != NULL) ? A.order[q] : q;
                                        double pos[3], dir[3];
                                        if (COMPACT && (A.position == NULL)) {
                                                fan_ray(C, r, pos, dir);
                                        } else {
                                                /* (L2 loads: a streamed ray has just been written
                                                 * by a copy engine, L1 must not serve an older line) */
                                                const double * p = A.position + 3ull * r;
                                                const double * d = A.direction + 3ull * r;
#pragma unroll
                                                for (int c = 0; c < 3; c++) {
                                                        pos[c] = __ldcg(p + c);
                                                        dir[c] = __ldcg(d + c);
                                                }
                                        }
                                        mode = ray_start<LLA>(G, V, store, tid, r, pos, dir);
                                }
                        }
                        if (STREAM) {
                                const unsigned waiting = __ballot_sync(FULL, mode == MODE_WAIT);
                                const unsigned resting = __ballot_sync(FULL, mode == MODE_IDLE);
                                pending_wait = waiting != 0u;
                                if ((waiting | resting) == FULL) { /* no lane has a ray */
                                        settle_done(A, owed);
                                        if (waiting != 0u)
                                                __nanosleep(500);
                                        else if (exhausted)
                                                break;
                                        continue;
                                }
                        } else if (__all_sync(FULL, mode == MODE_IDLE)) {
                                if (exhausted) break; /* (a resident ray never waits) */
                                continue;
                        }
                }
                if ((mode == MODE_IDLE) || (mode == MODE_WAIT) || (mode == MODE_DONE)) continue;

                /* ---- exactly one ECEF -> geodetic transform per lane and iteration:
                 * the one of a geometry sample, or -- local approximation on -- one of
                 * the three finite-difference transforms of a Jacobian (stepper.c:144-162)
                 * that went stale when its reference point moved and that the coming
                 * sample is about to apply (in range & stale; lazily: a Jacobian nobody reads
                 * is never built, see tb::get_geographic). Running the rebuild as
                 * iterations of its own keeps the lanes of a warp on equal work. */
                tb::Sample S;
                /* SHAPE_STACK leaves registers free: the sampled position stays in them, it
                 * IS the new position of a tentative step (same expression, same bits) */
                double moved[3] = { 0., 0., 0. };
                if (SHAPE == tb::SHAPE_STACK) {
                        /* one layer, one uniform geodetic stack: no list walk */
                        double p[3] = { SF(F_POS), SF(F_POS + 1), SF(F_POS + 2) };
                        if (mode != MODE_INIT) {
                                const double step = (mode == MODE_TENT) ?
                                    SF(F_DS) : 0.5 * (SF(F_DS0) + SF(F_DS1));
                                p[0] += SF(F_DIR) * step;
                                p[1] += SF(F_DIR + 1) * step;
                                p[2] += SF(F_DIR + 2) * step;
                        }
                        if (GATHER == GATHER_PACKED)
                                tb::sample_single_stack(tb::NodesPacked(), G, p, S);
                        else if (GATHER == GATHER_WINDOW)
                                tb::sample_single_stack(from_window, G, p, S);
                        else
                                tb::sample_single_stack(tb::NodesGlobal(), G, p, S);
                        moved[0] = p[0];
                        moved[1] = p[1];
                        moved[2] = p[2];
                } else {
                        double p[3];
                        int rb_t = 0, rb_axis = 0;
                        bool heavy = true;
                        unsigned in_range = 0u; /* LLA: transforms whose reference is in range */
                        if (!LLA || (mode != MODE_REBUILD)) {
                                double step = 0.; /* MODE_INIT: sample the start position */
                                if (mode == MODE_TENT) /* stepper.c:824 */
                                        step = SF(F_DS);
                                else if (mode == MODE_BISECT) /* stepper.c:840-844 */
                                        step = 0.5 * (SF(F_DS0) + SF(F_DS1));
                                p[0] = SF(F_POS);
                                p[1] = SF(F_POS + 1);
                                p[2] = SF(F_POS + 2);
                                if (mode != MODE_INIT) {
                                        p[0] += SF(F_DIR) * step;
                                        p[1] += SF(F_DIR + 1) * step;
                                        p[2] += SF(F_DIR + 2) * step;
                                }
                                if (LLA) { /* the range tests of this sample, ONCE */
                                        in_range = tb::lla_range_mask(G, V, p);
                                        const unsigned due = in_range & (unsigned)SI(I_PEND);
                                        if (due != 0u) {
                                                SI(I_RESUME) = mode;
                                                SI(I_RB_MASK) = (int)due;
                                                SI(I_RB_AXIS) = 0;
                                                mode = MODE_REBUILD;
                                        }
                                }
                        }
                        if (LLA && (mode == MODE_REBUILD)) {
                                rb_t = __ffs(SI(I_RB_MASK)) - 1;
                                rb_axis = SI(I_RB_AXIS);
                                const int row0 = G.lla_row[rb_t];
                                p[0] = tb::lla_at(V, row0);
                                p[1] = tb::lla_at(V, row0 + 1);
                                p[2] = tb::lla_at(V, row0 + 2);
                                if (rb_axis == 0) p[0] += 10.;
                                else if (rb_axis == 1) p[1] += 10.;
                                else p[2] += 10.;
                        } else if (LLA) {
                                heavy = !((in_range >> G.lla_first) & 1u);
                        }
                        double pre[3] = { 0., 0., 0. };
                        if (heavy) tb::geodetic_with_geoid(G, p, pre);
                        if (LLA && (mode == MODE_REBUILD)) {
                                tb::rebuild_column<PROJ>(G, V, rb_t, rb_axis, pre);
                                if (LLA_COUNT) my_rebuilds++;
                                if (rb_axis == 2) {
                                        SI(I_RB_MASK) &= ~(1 << rb_t);
                                        SI(I_PEND) &= ~(1 << rb_t);
                                        SI(I_RB_AXIS) = 0;
                                        if (SI(I_RB_MASK) == 0) mode = SI(I_RESUME);
                                } else {
                                        SI(I_RB_AXIS) = rb_axis + 1;
                                }
                                continue;
                        }
                        double last_pos[3] = { 0., 0., 0. };
                        unsigned stale = 0u;
                        if (LLA) {
                                last_pos[0] = SF(F_LASTPOS);
                                last_pos[1] = SF(F_LASTPOS + 1);
                                last_pos[2] = SF(F_LASTPOS + 2);
                                stale = (unsigned)SI(I_PEND);
                        }
                        tb::sample_geometry<LLA, PROJ, true>(G, V, stale, last_pos,
                            mode != MODE_BISECT, p, S, heavy ? pre : NULL, in_range);
                        if (LLA) {
                                SI(I_PEND) = (int)stale;
                                if (mode != MODE_BISECT) {
                                        SF(F_LASTPOS) = last_pos[0];
                                        SF(F_LASTPOS + 1) = last_pos[1];
                                        SF(F_LASTPOS + 2) = last_pos[2];
                                }
                        }
                }
                compiler_fence(); /* keep the state loads below out of the sample code */
                my_samples++;

                /* ---- state update (lane_advance) ---- */
                const int medium0 = SI(I_MEDIUM0);
                double ds = SF(F_DS);
                tb::Sample last; /* stepper->last: this sample, or the one published before */
                if (!lane_advance<LLA, SHAPE, true>(store, tid, mode, S, moved, medium0, ds, last)) continue;
                double total = SF(F_TOTAL);
                int n_steps = SI(I_NSTEPS);
                if (mode != MODE_INIT) {
                        /* example-stepper.c:136-139: length by STARTING medium */
                        const int m = (medium0 < TURTLE_TRACE_MEDIA - 1) ? medium0 :
                                                                           TURTLE_TRACE_MEDIA - 1;
                        store.f[F_LEN + m][tid] += ds;
                        total += ds;
                        SF(F_TOTAL) = total;
                        n_steps++;
                        SI(I_NSTEPS) = n_steps;
                        my_steps++;
                        if (last.idx0 != medium0) {
                                const int k = SI(I_NCHANGES);
                                if ((A.crossings != NULL) && (k < A.max_crossings)) {
                                        const unsigned long long ray =
                                            ((unsigned long long)(unsigned)SI(I_RAYHI) << 32) |
                                            (unsigned long long)(unsigned)SI(I_RAYLO);
                                        turtle_trace_crossing * c = A.crossings +
                                            ray * (unsigned long long)A.max_crossings + k;
                                        c->length = total;
                                        c->medium_from = medium0;
                                        c->medium_to = last.idx0;
                                }
                                SI(I_NCHANGES) += 1;
                                SI(I_HASH) = (int)(((unsigned)SI(I_HASH) ^
                                                       (unsigned)(last.idx0 + 1)) * 16777619u);
                        }
                }

                const int status = stop_status(A, last, total, n_steps);
                if (status >= 0) {
                        /* position, altitude, lengths, counters, index and hash are in the
                         * lane store already; the status takes the row of `medium0` */
                        SI(I_MEDIUM0) = status;
                        mode = MODE_DONE;
                } else {
                        SI(I_MEDIUM0) = last.idx0;
                        SF(F_DS) = tb::step_length(G, last); /* stepper.c:798-813 */
                        mode = MODE_TENT;
                }
        }

        /* ([3] is the time-out flag of a streamed call, [5] the window's hits) */
        flush_counters<LLA>(A.cursor, lane, my_steps, my_samples, my_rebuilds);
        if (GATHER == GATHER_WINDOW) {
                unsigned long long hits64 = from_window.hits;
                for (int o = 16; o > 0; o >>= 1) hits64 += __shfl_down_sync(FULL, hits64, o);
                if (lane == 0u) atomicAdd(A.cursor + 5, hits64);
        }
}

/* ---- horizon search (turtle_stepper_horizon) -------------------------------------------- */

/* Arguments of the horizon kernel. A kernel of its own rather than a variant of trace_kernel:
 * members added to TraceArgs cost every trace kernel registers (see CompactArgs). */
struct HorizonArgs {
        const double2 * az; /* { sin az, cos az } per azimuth, taken on the host (fan_upload) */
        /* station[12 s ...]: origin, East, North, Up of station s (fan_upload) */
        const double * station;
        unsigned long long n;         /* work items: n_station x n_azimuth */
        unsigned long long n_azimuth; /* item a is azimuth a % n_azimuth of station a / n_azimuth */
        double elevation_min, elevation_max, tolerance;
        double altitude_min, altitude_max, length_max;
        int max_steps;
        turtle_horizon * results;
        /* [0] next azimuth, [1] steps, [2] samples, [4] Jacobian columns, [6] probes */
        unsigned long long * cursor;
};

/* Rows of the lane store that a probe uses differently from a traced ray. */
enum { F_PROBE = F_LEN,          /* elevation of the probe, degrees */
       I_OUTCOME = I_HASH,       /* HORIZON_OBSTRUCTED, or the trace status of a clear probe */
       I_STATION = I_NCHANGES }; /* medium of the station: the probe's first sample */
enum { HORIZON_OBSTRUCTED = -1, HORIZON_ROUNDS_MAX = 64 };

/* K-ary search for the horizon, one azimuth per warp at a time. Each round the 32 lanes
 * trace 32 probe rays with the sample-granular state machine of trace_kernel (the same
 * samples, steps and bits as a traced ray: a probe is a prefix of the trace of its ray),
 * ending a probe at its first step into a medium >= 0 other than the station's. When the
 * round's last probe has ended, a ballot narrows the bracket to [highest obstructed probe,
 * next probe above it]. Round 0 probes both ends of the window and 30 points between
 * them, every later round 32 points inside the bracket (33 x narrower). Lanes whose probe
 * has ended wait for the slowest probe of the round: the azimuth's record counts the loop
 * iterations it took (n_iterations) so that the cost of that wait can be measured. */
template <bool LLA, bool PROJ, int MINB, int SHAPE>
__global__ void __launch_bounds__(128, MINB)
    horizon_kernel(const __grid_constant__ tb::Geometry G, const HorizonArgs A)
{
        constexpr int NF = LLA ? N_F_LLA : N_F_BASE, NI = LLA ? N_I : N_I_BASE;
        __shared__ LaneStoreT<NF, NI> store;
        __shared__ turtle_horizon record[4]; /* one per warp: the azimuth being searched */
        __shared__ double frame[4][12];      /* ... and the frame of its station */
        const unsigned tid = threadIdx.x;
        const unsigned lane = tid & 31u;
        const unsigned FULL = 0xffffffffu;
        turtle_horizon & R = record[tid >> 5];
        const double * F = frame[tid >> 5];
        extern __shared__ double lla_store[];
        const tb::LlaShared V = { lla_store + tid };
        unsigned my_steps = 0u, my_samples = 0u, my_rebuilds = 0u, my_probes = 0u;
        int mode = MODE_DONE;
        bool active = false; /* warp uniform: R holds an azimuth being searched */
        unsigned long long azimuth = 0ull;
        int round = 0;
        double2 sc = make_double2(0., 0.);

        for (;;) {
                if (__all_sync(FULL, mode == MODE_DONE)) {
                        /* ---- the round is over: narrow the bracket (warp uniform) ---- */
                        bool finished = true;
                        if (active) {
                                const int outcome = SI(I_OUTCOME);
                                const unsigned obstructed =
                                    __ballot_sync(FULL, outcome == HORIZON_OBSTRUCTED);
                                const bool invalid =
                                    __any_sync(FULL, outcome == TURTLE_TRACE_INVALID);
                                const double lo = R.elevation[0], hi = R.elevation[1];
                                __syncwarp();
                                int status = TURTLE_HORIZON_FOUND;
                                int low_end = -1, high_end = -1; /* lanes now holding the ends */
                                if (invalid) {
                                        status = TURTLE_HORIZON_INVALID;
                                } else if (round == 0) {
                                        if (!(obstructed & 1u)) {
                                                status = TURTLE_HORIZON_BELOW;
                                                high_end = 0;
                                        } else if (obstructed >> 31) {
                                                status = TURTLE_HORIZON_ABOVE;
                                                low_end = 31;
                                        } else {
                                                low_end = 31 - __clz((int)obstructed);
                                                high_end = low_end + 1;
                                        }
                                } else if (obstructed == 0u) {
                                        high_end = 0;
                                } else {
                                        low_end = 31 - __clz((int)obstructed);
                                        if (low_end < 31) high_end = low_end + 1;
                                }
                                if ((int)lane == low_end) {
                                        R.elevation[0] = SF(F_PROBE);
                                        for (int c = 0; c < 3; c++) R.direction[0][c] = SF(F_DIR + c);
                                        R.length = SF(F_TOTAL);
                                        R.medium[1] = SI(I_IDX0);
                                }
                                if ((int)lane == high_end) {
                                        R.elevation[1] = SF(F_PROBE);
                                        for (int c = 0; c < 3; c++) R.direction[1][c] = SF(F_DIR + c);
                                        R.clear_status = SI(I_OUTCOME);
                                }
                                if (lane == 0u) {
                                        if (round == 0) R.medium[0] = SI(I_STATION);
                                        R.status = status;
                                        R.n_probes += 32;
                                }
                                __syncwarp();
                                round++;
                                /* the search ends at the tolerance, or when the probes can no
                                 * longer split the bracket (it is a few doubles wide) */
                                finished = (status != TURTLE_HORIZON_FOUND) ||
                                    !(R.elevation[1] - R.elevation[0] > A.tolerance) ||
                                    ((R.elevation[0] == lo) && (R.elevation[1] == hi)) ||
                                    (round >= HORIZON_ROUNDS_MAX);
                                if (finished) {
                                        /* the 96-byte record, twelve lanes side by side */
                                        if (lane < 12u)
                                                reinterpret_cast<unsigned long long *>(A.results + azimuth)[lane] =
                                                    reinterpret_cast<const unsigned long long *>(&R)[lane];
                                        __syncwarp();
                                }
                        }
                        if (finished) { /* ---- next azimuth: one atomicAdd per warp ---- */
                                unsigned long long a = 0ull;
                                if (lane == 0u) a = atomicAdd(A.cursor, 1ull);
                                azimuth = __shfl_sync(FULL, a, 0);
                                if (azimuth >= A.n) break;
                                active = true;
                                round = 0;
                                const unsigned long long s = azimuth / A.n_azimuth;
                                sc = __ldg(A.az + (azimuth - s * A.n_azimuth));
                                if (lane < 12u) frame[tid >> 5][lane] = __ldg(A.station + 12ull * s + lane);
                                if (lane == 0u) {
                                        const double nan = __longlong_as_double(0x7ff8000000000000ll);
                                        R.elevation[0] = R.elevation[1] = R.length = nan;
                                        for (int c = 0; c < 3; c++)
                                                R.direction[0][c] = R.direction[1][c] = nan;
                                        R.medium[0] = R.medium[1] = -1;
                                        R.status = TURTLE_HORIZON_INVALID;
                                        R.clear_status = -1;
                                        R.n_probes = 0;
                                        R.n_iterations = 0;
                                }
                                __syncwarp();
                        }
                        /* ---- the probes of this round, one per lane ---- */
                        double el;
                        if (round == 0) {
                                el = (lane == 31u) ? A.elevation_max :
                                    A.elevation_min + (A.elevation_max - A.elevation_min) *
                                                          ((double)lane / 31.);
                        } else {
                                const double lo = R.elevation[0], hi = R.elevation[1];
                                el = lo + (hi - lo) * ((double)(lane + 1u) / 33.);
                        }
                        /* turtle_ecef_from_horizontal (ecef.c:160-178) on the host's sine and
                         * cosine of the azimuth and the device's of the elevation */
                        double s_el, c_el;
                        sincos(el * M_PI / 180., &s_el, &c_el);
                        const double r0 = c_el * sc.x, r1 = c_el * sc.y, r2 = s_el;
                        double dir[3];
                        for (int c = 0; c < 3; c++) {
                                SF(F_POS + c) = F[c];
                                dir[c] = r0 * F[3 + c] + r1 * F[6 + c] + r2 * F[9 + c];
                                SF(F_DIR + c) = dir[c];
                        }
                        SF(F_PROBE) = el;
                        SF(F_TOTAL) = 0.;
                        SI(I_NSTEPS) = 0;
                        SI(I_IDX0) = -1;
                        mode = MODE_INIT;
                        if (LLA) { /* a reset stepper (stepper.c:647-651) */
                                SI(I_PEND) = 0;
                                SF(F_LASTPOS) = SF(F_LASTPOS + 1) = SF(F_LASTPOS + 2) = DBL_MAX;
                                tb::lla_reset(G, V);
                        }
                        const double origin[3] = { F[0], F[1], F[2] };
                        if (!finite3(origin) || !finite3(dir)) {
                                SI(I_OUTCOME) = TURTLE_TRACE_INVALID;
                                SI(I_STATION) = -1;
                                mode = MODE_DONE;
                        }
                        if (lane == 0u) my_probes += 32u;
                        continue;
                }
                if (lane == 0u) R.n_iterations++;
                if (mode == MODE_DONE) continue;

                /* ---- one sample per lane: as in trace_kernel ---- */
                tb::Sample S;
                double moved[3] = { 0., 0., 0. };
                if (SHAPE == tb::SHAPE_STACK) {
                        double p[3] = { SF(F_POS), SF(F_POS + 1), SF(F_POS + 2) };
                        if (mode != MODE_INIT) {
                                const double step = (mode == MODE_TENT) ?
                                    SF(F_DS) : 0.5 * (SF(F_DS0) + SF(F_DS1));
                                p[0] += SF(F_DIR) * step;
                                p[1] += SF(F_DIR + 1) * step;
                                p[2] += SF(F_DIR + 2) * step;
                        }
                        tb::sample_single_stack(tb::NodesGlobal(), G, p, S);
                        moved[0] = p[0];
                        moved[1] = p[1];
                        moved[2] = p[2];
                } else {
                        double p[3];
                        int rb_t = 0, rb_axis = 0;
                        bool heavy = true;
                        unsigned in_range = 0u;
                        if (!LLA || (mode != MODE_REBUILD)) {
                                double step = 0.;
                                if (mode == MODE_TENT)
                                        step = SF(F_DS);
                                else if (mode == MODE_BISECT)
                                        step = 0.5 * (SF(F_DS0) + SF(F_DS1));
                                p[0] = SF(F_POS);
                                p[1] = SF(F_POS + 1);
                                p[2] = SF(F_POS + 2);
                                if (mode != MODE_INIT) {
                                        p[0] += SF(F_DIR) * step;
                                        p[1] += SF(F_DIR + 1) * step;
                                        p[2] += SF(F_DIR + 2) * step;
                                }
                                if (LLA) {
                                        in_range = tb::lla_range_mask(G, V, p);
                                        const unsigned due = in_range & (unsigned)SI(I_PEND);
                                        if (due != 0u) {
                                                SI(I_RESUME) = mode;
                                                SI(I_RB_MASK) = (int)due;
                                                SI(I_RB_AXIS) = 0;
                                                mode = MODE_REBUILD;
                                        }
                                }
                        }
                        if (LLA && (mode == MODE_REBUILD)) {
                                rb_t = __ffs(SI(I_RB_MASK)) - 1;
                                rb_axis = SI(I_RB_AXIS);
                                const int row0 = G.lla_row[rb_t];
                                p[0] = tb::lla_at(V, row0);
                                p[1] = tb::lla_at(V, row0 + 1);
                                p[2] = tb::lla_at(V, row0 + 2);
                                if (rb_axis == 0) p[0] += 10.;
                                else if (rb_axis == 1) p[1] += 10.;
                                else p[2] += 10.;
                        } else if (LLA) {
                                heavy = !((in_range >> G.lla_first) & 1u);
                        }
                        double pre[3] = { 0., 0., 0. };
                        if (heavy) tb::geodetic_with_geoid(G, p, pre);
                        if (LLA && (mode == MODE_REBUILD)) {
                                tb::rebuild_column<PROJ>(G, V, rb_t, rb_axis, pre);
                                my_rebuilds++;
                                if (rb_axis == 2) {
                                        SI(I_RB_MASK) &= ~(1 << rb_t);
                                        SI(I_PEND) &= ~(1 << rb_t);
                                        SI(I_RB_AXIS) = 0;
                                        if (SI(I_RB_MASK) == 0) mode = SI(I_RESUME);
                                } else {
                                        SI(I_RB_AXIS) = rb_axis + 1;
                                }
                                continue;
                        }
                        double last_pos[3] = { 0., 0., 0. };
                        unsigned stale = 0u;
                        if (LLA) {
                                last_pos[0] = SF(F_LASTPOS);
                                last_pos[1] = SF(F_LASTPOS + 1);
                                last_pos[2] = SF(F_LASTPOS + 2);
                                stale = (unsigned)SI(I_PEND);
                        }
                        tb::sample_geometry<LLA, PROJ, true>(G, V, stale, last_pos,
                            mode != MODE_BISECT, p, S, heavy ? pre : NULL, in_range);
                        if (LLA) {
                                SI(I_PEND) = (int)stale;
                                if (mode != MODE_BISECT) {
                                        SF(F_LASTPOS) = last_pos[0];
                                        SF(F_LASTPOS + 1) = last_pos[1];
                                        SF(F_LASTPOS + 2) = last_pos[2];
                                }
                        }
                }
                compiler_fence();
                my_samples++;

                /* ---- state update (lane_advance) ---- */
                const int medium0 = SI(I_MEDIUM0);
                double ds = SF(F_DS);
                tb::Sample last; /* stepper->last: this sample, or the one published before */
                if (!lane_advance<LLA, SHAPE, false>(store, tid, mode, S, moved, medium0, ds, last)) continue;
                double total = SF(F_TOTAL);
                int n_steps = SI(I_NSTEPS);
                int outcome = TURTLE_TRACE_INVALID + 1; /* none yet */
                if (mode == MODE_INIT) {
                        SI(I_STATION) = last.idx0;
                        if (last.idx0 < 0) outcome = TURTLE_TRACE_INVALID; /* station without data */
                } else {
                        total += ds;
                        SF(F_TOTAL) = total;
                        n_steps++;
                        SI(I_NSTEPS) = n_steps;
                        my_steps++;
                        /* the only new stop condition: the first step into another medium
                         * that is not "outside of the data" (that one ends the trace) */
                        if ((last.idx0 != medium0) && (last.idx0 >= 0))
                                outcome = HORIZON_OBSTRUCTED;
                }
                if (outcome > TURTLE_TRACE_INVALID) {
                        const int status = stop_status(A, last, total, n_steps);
                        if (status >= 0) outcome = status;
                }
                if (outcome <= TURTLE_TRACE_INVALID) {
                        SI(I_OUTCOME) = outcome;
                        mode = MODE_DONE;
                } else {
                        SI(I_MEDIUM0) = last.idx0;
                        SF(F_DS) = tb::step_length(G, last);
                        mode = MODE_TENT;
                }
        }

        flush_counters<LLA>(A.cursor, lane, my_steps, my_samples, my_rebuilds);
        if (lane == 0u) atomicAdd(A.cursor + 6, (unsigned long long)my_probes);
}

/* ---- rock length per cell of a voxel grid (turtle_stepper_trace_voxels) --------------------- */

/* Arguments of the voxel kernel: a kernel of its own, like the horizon kernel (members added to
 * TraceArgs cost every trace kernel registers). */
struct VoxelArgs {
        unsigned long long n;
        const double * position; /* [n][3] with `direction`, or NULL: the rays of `fan` */
        const double * direction;
        CompactArgs fan;         /* fan tables (fan_upload), when position == NULL */
        turtle_trace_result * results; /* or NULL */
        turtle_voxel_entry * entries;  /* [n][capacity], or NULL when capacity == 0 */
        int32_t * count;
        int capacity;
        unsigned media;
        double altitude_min, altitude_max, length_max;
        int max_steps;
        unsigned long long * cursor; /* [0] next ray, [1] steps, [2] samples, [4] Jacobian columns */
        double frame[12];            /* origin, East, North, Up of the grid (fan_upload's frame) */
        double corner[3], size[3];
        int cells[3];
        /* the opacity form (turtle_voxel_opacity): each pointer or NULL */
        const double * density;  /* [cells] */
        double * opacity;        /* [n] */
        double * outside;        /* [n] */
        const double * weight;   /* [n] */
        double * gradient;       /* [cells], added to */
};

/* Per-ray rows of the voxel walk, next to the lane store: the ray in grid coordinates, the
 * path lengths where its line enters and leaves the grid, and the open entry; the opacity form
 * adds its running sums and the ray's weight. */
enum { VF_U0 = 0, VF_V = 3, VF_TIN = 6, VF_TOUT, VF_OPEN, N_VF,
       VF_OPACITY = N_VF, VF_OUTSIDE, VF_WEIGHT, N_VF_OPACITY };
enum { VI_CELL = 0, VI_MEDIUM, VI_COUNT, N_VI };

/* Path length at which the ray line u0 + s v meets plane k of axis a of the grid. */
__device__ __forceinline__ double voxel_plane(const VoxelArgs & A, int a, int k, double u0, double v)
{
        return (A.corner[a] + (double)k * A.size[a] - u0) / v;
}

/* Close the open entry of a lane: store it if it fits, count it. The opacity form consumes it
 * instead: density x length into the lane's opacity, weight x length into the cell's gradient. */
template <bool OPACITY, int NVF>
__device__ __forceinline__ void voxel_close(const VoxelArgs & A, unsigned long long ray, int cell,
    int medium, double length, int & count, double (&vf)[NVF][128], unsigned tid)
{
        if (cell < 0) return;
        if constexpr (OPACITY) {
                if (A.density != NULL)
                        vf[VF_OPACITY][tid] = __dadd_rn(vf[VF_OPACITY][tid],
                            __dmul_rn(__ldg(A.density + cell), length));
                if (A.gradient != NULL)
                        atomicAdd(A.gradient + cell, __dmul_rn(vf[VF_WEIGHT][tid], length));
        } else if (count < A.capacity) {
                turtle_voxel_entry * e = A.entries + ray * (unsigned long long)A.capacity + count;
                e->length = length;
                e->voxel = cell;
                e->medium = medium;
        }
        count++;
}

/* trace_kernel's rays (same samples, steps and bits, same queue and settle point), where the
 * length of every step that starts in a selected medium is split over the cells of the grid
 * by a 3-D DDA along the ray line, with cell planes at absolute path lengths. OPACITY: the
 * entries are consumed where they close (voxel_close) and the parts of the selected steps
 * outside the grid are summed; the ray ends with its opacity and outside instead of a count. */
template <bool LLA, bool PROJ, int MINB, int SHAPE, bool OPACITY>
__global__ void __launch_bounds__(128, MINB)
    voxel_kernel(const __grid_constant__ tb::Geometry G, const __grid_constant__ VoxelArgs A)
{
        constexpr int NF = LLA ? N_F_LLA : N_F_BASE, NI = LLA ? N_I : N_I_BASE;
        __shared__ LaneStoreT<NF, NI> store;
        __shared__ double vf[OPACITY ? N_VF_OPACITY : N_VF][128];
        __shared__ int vi[N_VI][128];
        const unsigned tid = threadIdx.x;
        const unsigned lane = tid & 31u;
        const unsigned FULL = 0xffffffffu;
        extern __shared__ double lla_store[];
        const tb::LlaShared V = { lla_store + tid };
        unsigned my_steps = 0u, my_samples = 0u, my_rebuilds = 0u;
        int mode = MODE_IDLE;
        bool exhausted = false;

        for (;;) {
                /* ---- write out finished records (record_field) ---- */
                unsigned done_mask = __ballot_sync(FULL, mode == MODE_DONE);
                if (done_mask != 0u) __syncwarp();
                const bool wrote = done_mask != 0u;
                while (done_mask != 0u) {
                        const unsigned src = (unsigned)__ffs((int)done_mask) - 1u;
                        done_mask &= done_mask - 1u;
                        const unsigned t = (tid & ~31u) + src;
                        const unsigned long long ray =
                            ((unsigned long long)(unsigned)store.i[I_RAYHI][t] << 32) |
                            (unsigned long long)(unsigned)store.i[I_RAYLO][t];
                        if ((lane < 12u) && (A.results != NULL))
                                reinterpret_cast<unsigned long long *>(A.results + ray)[lane] =
                                    record_field(store, t, lane);
                        if (lane == src) {
                                if constexpr (OPACITY) {
                                        if (A.opacity != NULL) A.opacity[ray] = vf[VF_OPACITY][tid];
                                        if (A.outside != NULL) A.outside[ray] = vf[VF_OUTSIDE][tid];
                                } else {
                                        A.count[ray] = vi[VI_COUNT][tid];
                                }
                                mode = MODE_IDLE;
                        }
                }
                if (wrote) __syncwarp();
                /* ---- refill idle lanes from the ray queue (every ray is resident) ---- */
                const unsigned idle = __ballot_sync(FULL, mode == MODE_IDLE);
                if (idle != 0u) {
                        if (!exhausted) {
                                const int need = __popc(idle);
                                unsigned long long base = 0ull;
                                if (lane == 0u) base = atomicAdd(A.cursor, (unsigned long long)need);
                                base = __shfl_sync(FULL, base, 0);
                                if (mode == MODE_IDLE) {
                                        const unsigned long long r =
                                            base + __popc(idle & ((1u << lane) - 1u));
                                        if (r < A.n) {
                                                double pos[3], dir[3];
                                                if (A.position == NULL) {
                                                        fan_ray(A.fan, r, pos, dir);
                                                } else {
#pragma unroll
                                                        for (int c = 0; c < 3; c++) {
                                                                pos[c] = __ldg(A.position + 3ull * r + c);
                                                                dir[c] = __ldg(A.direction + 3ull * r + c);
                                                        }
                                                }
                                                mode = ray_start<LLA>(G, V, store, tid, r, pos, dir);
                                                vi[VI_CELL][tid] = -1;
                                                vi[VI_COUNT][tid] = 0;
                                                if constexpr (OPACITY) {
                                                        vf[VF_OPACITY][tid] = 0.;
                                                        vf[VF_OUTSIDE][tid] = 0.;
                                                        vf[VF_WEIGHT][tid] = (A.gradient != NULL) ?
                                                            __ldg(A.weight + r) : 0.;
                                                }
                                                /* the ray in grid coordinates, and where its line
                                                 * enters and leaves the grid (+inf: never) */
                                                double t_in = -DBL_MAX, t_out = DBL_MAX;
                                                for (int a = 0; a < 3; a++) {
                                                        const double * e = A.frame + 3 + 3 * a;
                                                        const double u0 = e[0] * (pos[0] - A.frame[0]) +
                                                            e[1] * (pos[1] - A.frame[1]) + e[2] * (pos[2] - A.frame[2]);
                                                        const double v = e[0] * dir[0] + e[1] * dir[1] + e[2] * dir[2];
                                                        vf[VF_U0 + a][tid] = u0;
                                                        vf[VF_V + a][tid] = v;
                                                        if (v != 0.) {
                                                                const double t0 = voxel_plane(A, a, 0, u0, v);
                                                                const double t1 = voxel_plane(A, a, A.cells[a], u0, v);
                                                                t_in = fmax(t_in, fmin(t0, t1));
                                                                t_out = fmin(t_out, fmax(t0, t1));
                                                        } else {
                                                                const double i = floor((u0 - A.corner[a]) / A.size[a]);
                                                                if (!((i >= 0.) && (i < (double)A.cells[a]))) t_in = DBL_MAX;
                                                        }
                                                }
                                                vf[VF_TIN][tid] = t_in;
                                                vf[VF_TOUT][tid] = t_out;
                                        }
                                }
                                if (base + (unsigned long long)need >= A.n) exhausted = true;
                        }
                        if (__all_sync(FULL, mode == MODE_IDLE)) {
                                if (exhausted) break;
                                continue;
                        }
                }
                if ((mode == MODE_IDLE) || (mode == MODE_DONE)) continue;

                /* ---- one sample per lane: as in trace_kernel ---- */
                tb::Sample S;
                double moved[3] = { 0., 0., 0. };
                if (SHAPE == tb::SHAPE_STACK) {
                        double p[3] = { SF(F_POS), SF(F_POS + 1), SF(F_POS + 2) };
                        if (mode != MODE_INIT) {
                                const double step = (mode == MODE_TENT) ?
                                    SF(F_DS) : 0.5 * (SF(F_DS0) + SF(F_DS1));
                                p[0] += SF(F_DIR) * step;
                                p[1] += SF(F_DIR + 1) * step;
                                p[2] += SF(F_DIR + 2) * step;
                        }
                        tb::sample_single_stack(tb::NodesGlobal(), G, p, S);
                        moved[0] = p[0];
                        moved[1] = p[1];
                        moved[2] = p[2];
                } else {
                        double p[3];
                        int rb_t = 0, rb_axis = 0;
                        bool heavy = true;
                        unsigned in_range = 0u;
                        if (!LLA || (mode != MODE_REBUILD)) {
                                double step = 0.;
                                if (mode == MODE_TENT)
                                        step = SF(F_DS);
                                else if (mode == MODE_BISECT)
                                        step = 0.5 * (SF(F_DS0) + SF(F_DS1));
                                p[0] = SF(F_POS);
                                p[1] = SF(F_POS + 1);
                                p[2] = SF(F_POS + 2);
                                if (mode != MODE_INIT) {
                                        p[0] += SF(F_DIR) * step;
                                        p[1] += SF(F_DIR + 1) * step;
                                        p[2] += SF(F_DIR + 2) * step;
                                }
                                if (LLA) {
                                        in_range = tb::lla_range_mask(G, V, p);
                                        const unsigned due = in_range & (unsigned)SI(I_PEND);
                                        if (due != 0u) {
                                                SI(I_RESUME) = mode;
                                                SI(I_RB_MASK) = (int)due;
                                                SI(I_RB_AXIS) = 0;
                                                mode = MODE_REBUILD;
                                        }
                                }
                        }
                        if (LLA && (mode == MODE_REBUILD)) {
                                rb_t = __ffs(SI(I_RB_MASK)) - 1;
                                rb_axis = SI(I_RB_AXIS);
                                const int row0 = G.lla_row[rb_t];
                                p[0] = tb::lla_at(V, row0);
                                p[1] = tb::lla_at(V, row0 + 1);
                                p[2] = tb::lla_at(V, row0 + 2);
                                if (rb_axis == 0) p[0] += 10.;
                                else if (rb_axis == 1) p[1] += 10.;
                                else p[2] += 10.;
                        } else if (LLA) {
                                heavy = !((in_range >> G.lla_first) & 1u);
                        }
                        double pre[3] = { 0., 0., 0. };
                        if (heavy) tb::geodetic_with_geoid(G, p, pre);
                        if (LLA && (mode == MODE_REBUILD)) {
                                tb::rebuild_column<PROJ>(G, V, rb_t, rb_axis, pre);
                                my_rebuilds++;
                                if (rb_axis == 2) {
                                        SI(I_RB_MASK) &= ~(1 << rb_t);
                                        SI(I_PEND) &= ~(1 << rb_t);
                                        SI(I_RB_AXIS) = 0;
                                        if (SI(I_RB_MASK) == 0) mode = SI(I_RESUME);
                                } else {
                                        SI(I_RB_AXIS) = rb_axis + 1;
                                }
                                continue;
                        }
                        double last_pos[3] = { 0., 0., 0. };
                        unsigned stale = 0u;
                        if (LLA) {
                                last_pos[0] = SF(F_LASTPOS);
                                last_pos[1] = SF(F_LASTPOS + 1);
                                last_pos[2] = SF(F_LASTPOS + 2);
                                stale = (unsigned)SI(I_PEND);
                        }
                        tb::sample_geometry<LLA, PROJ, true>(G, V, stale, last_pos,
                            mode != MODE_BISECT, p, S, heavy ? pre : NULL, in_range);
                        if (LLA) {
                                SI(I_PEND) = (int)stale;
                                if (mode != MODE_BISECT) {
                                        SF(F_LASTPOS) = last_pos[0];
                                        SF(F_LASTPOS + 1) = last_pos[1];
                                        SF(F_LASTPOS + 2) = last_pos[2];
                                }
                        }
                }
                compiler_fence();
                my_samples++;

                /* ---- state update (lane_advance) ---- */
                const int medium0 = SI(I_MEDIUM0);
                double ds = SF(F_DS);
                tb::Sample last; /* stepper->last: this sample, or the one published before */
                if (!lane_advance<LLA, SHAPE, true>(store, tid, mode, S, moved, medium0, ds, last)) continue;
                double total = SF(F_TOTAL);
                int n_steps = SI(I_NSTEPS);
                const unsigned long long ray =
                    ((unsigned long long)(unsigned)SI(I_RAYHI) << 32) | (unsigned long long)(unsigned)SI(I_RAYLO);
                if (mode != MODE_INIT) {
                        const int m = (medium0 < TURTLE_TRACE_MEDIA - 1) ? medium0 :
                                                                           TURTLE_TRACE_MEDIA - 1;
                        store.f[F_LEN + m][tid] += ds;
                        const double s0 = total; /* the step covers [s0, total] of the ray line */
                        total += ds;
                        SF(F_TOTAL) = total;
                        n_steps++;
                        SI(I_NSTEPS) = n_steps;
                        my_steps++;
                        if (last.idx0 != medium0) {
                                SI(I_NCHANGES) += 1;
                                SI(I_HASH) = (int)(((unsigned)SI(I_HASH) ^
                                                       (unsigned)(last.idx0 + 1)) * 16777619u);
                        }
                        /* ---- the step's segment through the grid ---- */
                        double s = fmax(s0, vf[VF_TIN][tid]);
                        const double s_end = fmin(total, vf[VF_TOUT][tid]);
                        if constexpr (OPACITY) {
                                /* the parts of a selected step before and after the box, or
                                 * all of it when it misses the box */
                                if (((unsigned)medium0 < 32u) && ((A.media >> medium0) & 1u))
                                        vf[VF_OUTSIDE][tid] = __dadd_rn(vf[VF_OUTSIDE][tid], (s < s_end) ?
                                            __dadd_rn(__dsub_rn(s, s0), __dsub_rn(total, s_end)) : ds);
                        }
                        if (((unsigned)medium0 < 32u) && ((A.media >> medium0) & 1u) && (s < s_end)) {
                                int i[3];
                                double next[3];
                                for (int a = 0; a < 3; a++) {
                                        const double u0 = vf[VF_U0 + a][tid], v = vf[VF_V + a][tid];
                                        const int n = A.cells[a];
                                        /* the cell just after s, with the plane crossings as
                                         * the truth: a first guess from the position, then
                                         * moved until t(i) <= s < t(i + 1) (v > 0), or
                                         * t(i + 1) <= s < t(i) (v < 0) */
                                        const double g = floor((u0 + s * v - A.corner[a]) / A.size[a]);
                                        int k = (g < 0.) ? 0 : ((g > (double)(n - 1)) ? n - 1 : (int)g);
                                        if (v > 0.) {
                                                while ((k + 1 < n) && (voxel_plane(A, a, k + 1, u0, v) <= s)) k++;
                                                while ((k > 0) && (voxel_plane(A, a, k, u0, v) > s)) k--;
                                                next[a] = voxel_plane(A, a, k + 1, u0, v);
                                        } else if (v < 0.) {
                                                while ((k > 0) && (voxel_plane(A, a, k, u0, v) <= s)) k--;
                                                while ((k + 1 < n) && (voxel_plane(A, a, k + 1, u0, v) > s)) k++;
                                                next[a] = voxel_plane(A, a, k, u0, v);
                                        } else {
                                                next[a] = DBL_MAX;
                                        }
                                        i[a] = k;
                                }
                                int open_cell = vi[VI_CELL][tid], open_medium = vi[VI_MEDIUM][tid];
                                int count = vi[VI_COUNT][tid];
                                double open_length = vf[VF_OPEN][tid];
                                for (;;) {
                                        const double t = fmin(next[0], fmin(next[1], next[2]));
                                        const double e = fmin(t, s_end);
                                        if (e > s) {
                                                const int cell = i[0] + A.cells[0] * (i[1] + A.cells[1] * i[2]);
                                                if ((cell == open_cell) && (medium0 == open_medium)) {
                                                        open_length += e - s;
                                                } else {
                                                        voxel_close<OPACITY>(A, ray, open_cell, open_medium,
                                                            open_length, count, vf, tid);
                                                        open_cell = cell;
                                                        open_medium = medium0;
                                                        open_length = e - s;
                                                }
                                                s = e;
                                        }
                                        if (!(t < s_end)) break;
                                        /* every axis whose plane comes now: one cell on */
                                        bool out = false;
                                        for (int a = 0; a < 3; a++) {
                                                if (next[a] != t) continue;
                                                const double u0 = vf[VF_U0 + a][tid], v = vf[VF_V + a][tid];
                                                i[a] += (v > 0.) ? 1 : -1;
                                                if ((i[a] < 0) || (i[a] >= A.cells[a])) out = true;
                                                else next[a] = voxel_plane(A, a, (v > 0.) ? i[a] + 1 : i[a], u0, v);
                                        }
                                        if (out) break;
                                }
                                vi[VI_CELL][tid] = open_cell;
                                vi[VI_MEDIUM][tid] = open_medium;
                                vi[VI_COUNT][tid] = count;
                                vf[VF_OPEN][tid] = open_length;
                        }
                }

                const int status = stop_status(A, last, total, n_steps);
                if (status >= 0) {
                        SI(I_MEDIUM0) = status;
                        int count = vi[VI_COUNT][tid];
                        voxel_close<OPACITY>(A, ray, vi[VI_CELL][tid], vi[VI_MEDIUM][tid], vf[VF_OPEN][tid],
                            count, vf, tid);
                        vi[VI_COUNT][tid] = count;
                        mode = MODE_DONE;
                } else {
                        SI(I_MEDIUM0) = last.idx0;
                        SF(F_DS) = tb::step_length(G, last);
                        mode = MODE_TENT;
                }
        }

        flush_counters<LLA>(A.cursor, lane, my_steps, my_samples, my_rebuilds);
}

/* Longest-expected-first scheduling: the number of steps of a ray grows as it runs
 * closer to the horizontal (it stays near the ground), and the kernel time is bounded
 * below by the LATEST-starting long ray. Key = |sin(elevation)| w.r.t. the geocentric
 * vertical at the origin; rays are handed out by increasing key. */
__global__ void schedule_key_kernel(unsigned long long n, const double * __restrict__ position,
    const double * __restrict__ direction, unsigned * __restrict__ keys,
    unsigned * __restrict__ index)
{
        const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
        for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
             i < n; i += stride) {
                const double px = position[3 * i], py = position[3 * i + 1], pz = position[3 * i + 2];
                const double dx = direction[3 * i], dy = direction[3 * i + 1], dz = direction[3 * i + 2];
                const double pp = px * px + py * py + pz * pz;
                const double dd = dx * dx + dy * dy + dz * dz;
                float k = 1.f;
                if ((pp > 0.) && (dd > 0.))
                        k = (float)(fabs(px * dx + py * dy + pz * dz) * rsqrt(pp * dd));
                if (!(k >= 0.f)) k = 1.f; /* NaN: the kernel flags the ray anyway */
                if (k > 1.f) k = 1.f;
                keys[i] = __float_as_uint(k); /* non negative floats sort as integers */
                index[i] = (unsigned)i;
        }
}

/* Device-side particle states of turtle_stepper_step_batch: what `struct turtle_stepper`
 * remembers for ONE track between two calls, FIELD-MAJOR -- field f of particle i at
 * states[f * stride + i] -- so that the lanes of a warp (consecutive particles) read and
 * write whole sectors. Fields: last position (3), lat / lon / alt / elev0 / elev1 (5), the
 * two indices packed in one slot (1), the stale-Jacobian mask of the local approximation
 * (1), then the G.lla_rows rows of the local approximations themselves (tb::LlaView with
 * this very stride: the core functions use them IN PLACE -- a step usually only reads the
 * reference point to find that it is out of range; the Jacobian is touched when it is
 * applied or rebuilt). */
enum { PS_LASTPOS = 0, PS_LAT = 3, PS_LON, PS_ALT, PS_ELEV0, PS_ELEV1, PS_INDEX, PS_STALE,
       PS_FIELDS };

struct StepArgs {
        unsigned long long n;
        double * states; /* or NULL */
        unsigned long long stride;
        double * position;
        const double * direction; /* or NULL: query mode */
        double * latitude;
        double * longitude;
        double * altitude;
        double * elevation;
        double * step;
        int * index;
        unsigned long long * counters; /* [1] steps */
        int n_steps; /* MULTI: steps per particle in this launch; outputs are [n_steps][n] */
};

/* One turtle_stepper_step per particle (ref: stepper.c:780-875), with the SAME
 * sample-granular scheduling as the trace kernel: persistent lanes pull particles from
 * a queue; every loop iteration evaluates one stepper_sample per lane (start sample
 * unless the particle's cached last sample is at its position, tentative end, bisection
 * mid-points) or one column of a stale Jacobian that the coming sample will read; a
 * particle that is done writes its outputs and state and its lane is refilled.
 * Step-granular lockstep (one thread = one whole step) would make every warp pay the
 * 23-sample bisection of its unluckiest lane on most steps. */
/* The local approximations of a particle: a column of the device states (STATES) or, when
 * every particle starts from a reset stepper, of the kernel's shared scratch. */
template <bool STATES> struct WalkView {
        typedef tb::LlaShared type;
};
template <> struct WalkView<true> {
        typedef tb::LlaGlobal type;
};
__device__ __forceinline__ void view_of_particle(tb::LlaGlobal & V, double * base, size_t stride)
{
        V.base = base;
        V.stride = stride;
}
__device__ __forceinline__ void view_of_particle(tb::LlaShared &, double *, size_t) {}

/* MULTI = turtle_stepper_walk_batch: n_steps successive turtle_stepper_step calls per
 * particle in ONE launch, direction[j][i] for step j of particle i. The particle's state is
 * loaded once, lives in the lane store (and, local approximation on, in shared columns) for
 * all its steps and is stored once: per step only the direction comes in and the outputs go
 * out -- where the one-step call moves the whole state both ways every step and is bound by
 * that traffic. */
template <bool LLA, bool PROJ, bool STATES, bool MULTI = false>
__global__ void __launch_bounds__(128, 5)
    walk_kernel(const __grid_constant__ tb::Geometry G, const StepArgs A)
{
        constexpr int NF = N_F, NI = N_I;
        __shared__ LaneStore store;
        extern __shared__ double lla_store[]; /* LLA: scratch (no states), or the state (MULTI) */
        const unsigned tid = threadIdx.x;
        const unsigned lane = tid & 31u;
        const unsigned FULL = 0xffffffffu;

        int mode = MODE_IDLE;
        typename WalkView<STATES && !MULTI>::type V;
        V.base = lla_store + tid;
        const bool with_states = STATES && (!MULTI || (A.states != NULL));
        unsigned my_steps = 0u, my_samples = 0u, my_rebuilds = 0u;
        bool exhausted = false;
        bool carry = false; /* MULTI: the next step of this particle starts on its cached sample */

        for (;;) {
                bool started = carry; /* the start sample is available in the lane store */
                carry = false;
                bool finish = false;
                double step_out = 0.;
                const unsigned idle = __ballot_sync(FULL, mode == MODE_IDLE);
                if (idle != 0u) {
                        if (!exhausted) {
                                const int need = __popc(idle);
                                unsigned long long base = 0ull;
                                if (lane == 0u)
                                        base = atomicAdd(A.counters, (unsigned long long)need);
                                base = __shfl_sync(FULL, base, 0);
                                if (mode == MODE_IDLE) {
                                        const unsigned long long r =
                                            base + __popc(idle & ((1u << lane) - 1u));
                                        if (r < A.n) {
                                                SI(I_RAYLO) = (int)(unsigned)(r & 0xffffffffull);
                                                SI(I_RAYHI) = (int)(unsigned)(r >> 32);
                                                const double pos[3] = { A.position[3 * r],
                                                        A.position[3 * r + 1], A.position[3 * r + 2] };
                                                SF(F_POS) = pos[0];
                                                SF(F_POS + 1) = pos[1];
                                                SF(F_POS + 2) = pos[2];
                                                if (A.direction != NULL) {
                                                        SF(F_DIR) = A.direction[3 * r];
                                                        SF(F_DIR + 1) = A.direction[3 * r + 1];
                                                        SF(F_DIR + 2) = A.direction[3 * r + 2];
                                                }
                                                double lp[3] = { DBL_MAX, DBL_MAX, DBL_MAX };
                                                SI(I_PEND) = 0;
                                                if (MULTI) SI(I_NSTEPS) = 0;
                                                if (with_states) {
                                                        const double * ps = A.states + r;
                                                        lp[0] = ps[(PS_LASTPOS + 0) * A.stride];
                                                        lp[1] = ps[(PS_LASTPOS + 1) * A.stride];
                                                        lp[2] = ps[(PS_LASTPOS + 2) * A.stride];
                                                        if (LLA) {
                                                                view_of_particle(V,
                                                                    A.states + PS_FIELDS * A.stride + r,
                                                                    A.stride);
                                                                SI(I_PEND) = __double2loint(
                                                                    ps[PS_STALE * A.stride]);
                                                                if (MULTI) {
                                                                        /* the state moves in, once:
                                                                         * asynchronous copies, one
                                                                         * latency for all the rows */
                                                                        for (int row = 0; row < G.lla_rows; row++)
                                                                                __pipeline_memcpy_async(
                                                                                    &lla_store[row * 128 + tid],
                                                                                    &ps[(PS_FIELDS + row) * A.stride], 8);
                                                                        __pipeline_commit();
                                                                        __pipeline_wait_prior(0);
                                                                }
                                                        }
                                                } else if (LLA) {
                                                        tb::lla_reset(G, V);
                                                }
                                                SF(F_LASTPOS) = lp[0];
                                                SF(F_LASTPOS + 1) = lp[1];
                                                SF(F_LASTPOS + 2) = lp[2];
                                                mode = MODE_INIT;
                                                /* stepper.c:708-710: exact cache test */
                                                if (with_states && (pos[0] == lp[0]) && (pos[1] == lp[1]) &&
                                                    (pos[2] == lp[2])) {
                                                        const double * ps = A.states + r;
                                                        SF(F_LAT) = ps[PS_LAT * A.stride];
                                                        SF(F_LON) = ps[PS_LON * A.stride];
                                                        SF(F_ALT) = ps[PS_ALT * A.stride];
                                                        SF(F_ELEV0) = ps[PS_ELEV0 * A.stride];
                                                        SF(F_ELEV1) = ps[PS_ELEV1 * A.stride];
                                                        const double packed = ps[PS_INDEX * A.stride];
                                                        SI(I_IDX0) = __double2loint(packed);
                                                        SI(I_IDX1) = __double2hiint(packed);
                                                        started = true;
                                                }
                                        }
                                }
                                if (base + (unsigned long long)need >= A.n) exhausted = true;
                        }
                        if (__all_sync(FULL, mode == MODE_IDLE)) {
                                if (exhausted) break;
                                continue;
                        }
                }
                if (mode == MODE_IDLE) continue;

                /* the start sample is known (stepper.c:791-821): the step is over (outside of
                 * the layers, query mode) or its length is */
                auto start_known = [&]() {
                        tb::Sample last;
                        last.lat = last.lon = 0.;
                        last.alt = SF(F_ALT);
                        last.elev0 = SF(F_ELEV0);
                        last.elev1 = SF(F_ELEV1);
                        last.idx0 = SI(I_IDX0);
                        last.idx1 = SI(I_IDX1);
                        if (last.idx0 < 0) {
                                finish = true;
                                step_out = 0.;
                        } else {
                                const double ds = tb::step_length(G, last);
                                if (A.direction == NULL) {
                                        finish = true;
                                        step_out = ds;
                                } else {
                                        SI(I_MEDIUM0) = last.idx0;
                                        SF(F_DS) = ds;
                                        mode = MODE_TENT;
                                }
                        }
                };
                /* a particle that comes with the sample at its position (the usual case of a
                 * walk: the last step ended there) goes on to its tentative sample in this
                 * very iteration */
                if (started && (mode == MODE_INIT)) {
                        start_known();
                        if (!finish) started = false;
                }

                /* the position of the coming sample (none: idle lane, finished step,
                 * Jacobian column) */
                double p[3] = { 0., 0., 0. };
                unsigned in_range = 0u; /* LLA: transforms whose reference is in range */
                const bool sampling = !started;
                bool cached = false;  /* the tentative sample is the published one */
                if (sampling && (!LLA || (mode != MODE_REBUILD))) {
                        double step = 0.;
                        if (mode == MODE_TENT)
                                step = SF(F_DS);
                        else if (mode == MODE_BISECT)
                                step = 0.5 * (SF(F_DS0) + SF(F_DS1));
                        p[0] = SF(F_POS);
                        p[1] = SF(F_POS + 1);
                        p[2] = SF(F_POS + 2);
                        if (mode != MODE_INIT) {
                                p[0] += SF(F_DIR) * step;
                                p[1] += SF(F_DIR + 1) * step;
                                p[2] += SF(F_DIR + 2) * step;
                        }
                        /* stepper.c:708-710: a step that does not move the particle (direction
                         * 0 0 0) ends on the last sampled position, whose sample is the cached
                         * one -- nothing is evaluated, no reference point moves */
                        cached = (mode == MODE_TENT) && (p[0] == SF(F_LASTPOS)) &&
                            (p[1] == SF(F_LASTPOS + 1)) && (p[2] == SF(F_LASTPOS + 2));
                        if (LLA && !cached) { /* the range tests of this sample, ONCE; a stale
                                               * Jacobian about to be read is rebuilt first */
                                in_range = tb::lla_range_mask(G, V, p);
                                const unsigned due = in_range & (unsigned)SI(I_PEND);
                                if (due != 0u) {
                                        SI(I_RESUME) = mode;
                                        SI(I_RB_MASK) = (int)due;
                                        SI(I_RB_AXIS) = 0;
                                        mode = MODE_REBUILD;
                                }
                        }
                }
                if (!started) {
                        /* ---- one ECEF -> geodetic transform ------------------------- */
                        tb::Sample S;
                        if (cached) {
                                S.lat = SF(F_LAT);
                                S.lon = SF(F_LON);
                                S.alt = SF(F_ALT);
                                S.elev0 = SF(F_ELEV0);
                                S.elev1 = SF(F_ELEV1);
                                S.idx0 = SI(I_IDX0);
                                S.idx1 = SI(I_IDX1);
                        } else {
                                int rb_t = 0, rb_axis = 0;
                                bool heavy = true;
                                if (LLA && (mode == MODE_REBUILD)) {
                                        rb_t = __ffs(SI(I_RB_MASK)) - 1;
                                        rb_axis = SI(I_RB_AXIS);
                                        const int row0 = G.lla_row[rb_t];
                                        p[0] = tb::lla_at(V, row0);
                                        p[1] = tb::lla_at(V, row0 + 1);
                                        p[2] = tb::lla_at(V, row0 + 2);
                                        if (rb_axis == 0) p[0] += 10.;
                                        else if (rb_axis == 1) p[1] += 10.;
                                        else p[2] += 10.;
                                } else if (LLA) {
                                        heavy = !((in_range >> G.lla_first) & 1u);
                                }
                                double pre[3] = { 0., 0., 0. };
                                if (heavy) tb::geodetic_with_geoid(G, p, pre);
                                if (LLA && (mode == MODE_REBUILD)) {
                                        tb::rebuild_column<PROJ>(G, V, rb_t, rb_axis, pre);
                                        my_rebuilds++;
                                        if (rb_axis == 2) {
                                                SI(I_RB_MASK) &= ~(1 << rb_t);
                                                SI(I_PEND) &= ~(1 << rb_t);
                                                SI(I_RB_AXIS) = 0;
                                                if (SI(I_RB_MASK) == 0) mode = SI(I_RESUME);
                                        } else {
                                                SI(I_RB_AXIS) = rb_axis + 1;
                                        }
                                        continue;
                                }
                                double last_pos[3] = { SF(F_LASTPOS), SF(F_LASTPOS + 1),
                                        SF(F_LASTPOS + 2) };
                                unsigned stale = LLA ? (unsigned)SI(I_PEND) : 0u;
                                tb::sample_geometry<LLA, PROJ, true>(G, V, stale, last_pos,
                                    mode != MODE_BISECT, p, S, heavy ? pre : NULL, in_range);
                                if (LLA) SI(I_PEND) = (int)stale;
                                if (mode != MODE_BISECT) {
                                        SF(F_LASTPOS) = last_pos[0];
                                        SF(F_LASTPOS + 1) = last_pos[1];
                                        SF(F_LASTPOS + 2) = last_pos[2];
                                }
                        }
                        compiler_fence();
                        my_samples++;

                        bool publish = false;
                        const int medium0 = SI(I_MEDIUM0);
                        double ds = SF(F_DS);
                        if (mode == MODE_INIT) {
                                publish = true;
                                started = true;
                        } else if (mode == MODE_TENT) {
                                SF(F_POS) += SF(F_DIR) * ds;
                                SF(F_POS + 1) += SF(F_DIR + 1) * ds;
                                SF(F_POS + 2) += SF(F_DIR + 2) * ds;
                                publish = true;
                                if (S.idx0 != medium0) {
                                        SF(F_DS0) = -ds;
                                        SF(F_DS1) = 0.;
                                        mode = MODE_BISECT;
                                        finish = !(0. - (-ds) > 1E-08);
                                } else {
                                        finish = true;
                                }
                                step_out = ds;
                        } else {
                                double ds0 = SF(F_DS0), ds1 = SF(F_DS1);
                                const double ds2 = 0.5 * (ds0 + ds1);
                                if (S.idx0 == medium0) {
                                        ds0 = ds2;
                                        SF(F_DS0) = ds0;
                                } else {
                                        ds1 = ds2;
                                        SF(F_DS1) = ds1;
                                        publish = true;
                                        SF(F_LASTPOS) = SF(F_POS) + SF(F_DIR) * ds2;
                                        SF(F_LASTPOS + 1) = SF(F_POS + 1) + SF(F_DIR + 1) * ds2;
                                        SF(F_LASTPOS + 2) = SF(F_POS + 2) + SF(F_DIR + 2) * ds2;
                                }
                                if (!(ds1 - ds0 > 1E-08)) {
                                        ds += ds1;
                                        SF(F_POS) += SF(F_DIR) * ds1;
                                        SF(F_POS + 1) += SF(F_DIR + 1) * ds1;
                                        SF(F_POS + 2) += SF(F_DIR + 2) * ds1;
                                        finish = true;
                                        step_out = ds;
                                }
                        }
                        if (publish) {
                                SF(F_LAT) = S.lat;
                                SF(F_LON) = S.lon;
                                SF(F_ALT) = S.alt;
                                SF(F_ELEV0) = S.elev0;
                                SF(F_ELEV1) = S.elev1;
                                SI(I_IDX0) = S.idx0;
                                SI(I_IDX1) = S.idx1;
                        }
                        if (finish) my_steps++;
                }

                if (started && !finish && (mode == MODE_INIT)) start_known();
                if (!finish) continue;

                /* ---- outputs of a finished step; state of a finished particle (a Jacobian
                 * that is still stale stays so: the mask is part of the state) ------------ */
                const unsigned long long r = ((unsigned long long)(unsigned)SI(I_RAYHI) << 32) |
                    (unsigned long long)(unsigned)SI(I_RAYLO);
                const int idx0 = SI(I_IDX0);
                const int j = MULTI ? SI(I_NSTEPS) : 0;
                const unsigned long long o = MULTI ? (unsigned long long)j * A.n + r : r;
                if (A.latitude != NULL) A.latitude[o] = SF(F_LAT);
                if (A.longitude != NULL) A.longitude[o] = SF(F_LON);
                if (A.altitude != NULL) A.altitude[o] = SF(F_ALT);
                if (A.elevation != NULL) { /* stepper.c:765-772 */
                        A.elevation[2 * o] = (idx0 >= 0) ? SF(F_ELEV0) : 0.;
                        A.elevation[2 * o + 1] = (idx0 >= 0) ? SF(F_ELEV1) : 0.;
                }
                if (A.step != NULL) A.step[o] = step_out;
                if (A.index != NULL) {
                        A.index[2 * o] = idx0;
                        A.index[2 * o + 1] = SI(I_IDX1);
                }
                if (MULTI && (j + 1 < A.n_steps)) {
                        /* the next turtle_stepper_step of this particle: its direction comes
                         * in; the sample at its position is the cached one when the position
                         * is the last sampled one (stepper.c:708-710) */
                        const double * d = A.direction + 3ull * ((unsigned long long)(j + 1) * A.n + r);
                        SI(I_NSTEPS) = j + 1;
                        SF(F_DIR) = d[0];
                        SF(F_DIR + 1) = d[1];
                        SF(F_DIR + 2) = d[2];
                        carry = (SF(F_POS) == SF(F_LASTPOS)) && (SF(F_POS + 1) == SF(F_LASTPOS + 1)) &&
                            (SF(F_POS + 2) == SF(F_LASTPOS + 2));
                        mode = MODE_INIT;
                        continue;
                }
                if (A.direction != NULL) {
                        A.position[3 * r] = SF(F_POS);
                        A.position[3 * r + 1] = SF(F_POS + 1);
                        A.position[3 * r + 2] = SF(F_POS + 2);
                }
                if (with_states) {
                        double * ps = A.states + r;
                        ps[(PS_LASTPOS + 0) * A.stride] = SF(F_LASTPOS);
                        ps[(PS_LASTPOS + 1) * A.stride] = SF(F_LASTPOS + 1);
                        ps[(PS_LASTPOS + 2) * A.stride] = SF(F_LASTPOS + 2);
                        ps[PS_LAT * A.stride] = SF(F_LAT);
                        ps[PS_LON * A.stride] = SF(F_LON);
                        ps[PS_ALT * A.stride] = SF(F_ALT);
                        ps[PS_ELEV0 * A.stride] = SF(F_ELEV0);
                        ps[PS_ELEV1 * A.stride] = SF(F_ELEV1);
                        ps[PS_INDEX * A.stride] = __hiloint2double(SI(I_IDX1), idx0);
                        if (LLA) {
                                ps[PS_STALE * A.stride] = __hiloint2double(0, SI(I_PEND));
                                if (MULTI) /* ... and out, once */
#pragma unroll 4
                                        for (int row = 0; row < G.lla_rows; row++)
                                                ps[(PS_FIELDS + row) * A.stride] =
                                                    lla_store[row * 128 + tid];
                        }
                }
                mode = MODE_IDLE;
        }
        flush_counters<LLA>(A.counters, lane, my_steps, my_samples, my_rebuilds);
}

#undef SF
#undef SI

/* turtle_stepper_reset for every particle (stepper.c:602-615): last position and every
 * reference point at DBL_MAX; the last sample is cleared, no Jacobian is stale. */
__global__ void states_reset_kernel(const __grid_constant__ tb::Geometry G, double * states,
    unsigned long long stride, unsigned long long n)
{
        const unsigned long long step = (unsigned long long)gridDim.x * blockDim.x;
        for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
             i < n; i += step) {
                double * ps = states + i;
                for (int k = 0; k < 3; k++) ps[(PS_LASTPOS + k) * stride] = DBL_MAX;
                for (int k = PS_LAT; k < PS_INDEX; k++) ps[k * stride] = 0.;
                ps[PS_INDEX * stride] = __hiloint2double(-1, -1);
                ps[PS_STALE * stride] = __hiloint2double(0, 0);
                const tb::LlaGlobal V = { states + PS_FIELDS * stride + i, (size_t)stride };
                tb::lla_reset(G, V);
        }
}

/* ref: turtle_stepper_position, stepper.c:877-931 */
__global__ void position_kernel(const __grid_constant__ tb::Geometry G,
    unsigned long long n, const double * latitude, const double * longitude,
    const double * height, int layer_index, double * position, int * data_index)
{
        const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
        const tb::LayerDesc layer = G.layers[layer_index];
        for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
             i < n; i += stride) {
                const double la = latitude[i], lo = longitude[i];
                int found = -1;
                for (int k = 0; k < layer.n; k++) {
                        const tb::MetaDesc & meta = G.metas[layer.first + k];
                        const tb::DataDesc & d = G.data[meta.data];
                        double z = 0.;
                        int inside;
                        if (d.kind == tb::DATA_FLAT) {
                                inside = 1;
                        } else if (d.kind == tb::DATA_STACK) {
                                inside = tb::stack_elevation(G, G.stacks[d.ref], la, lo, z);
                        } else if (G.transforms[d.transform].type != tb::PROJ_GEODETIC) {
                                double x, y;
                                tb::project(G.transforms[d.transform], la, lo, x, y);
                                inside = tb::map_elevation(G.maps[d.ref], x, y, z);
                        } else {
                                inside = tb::map_elevation(G.maps[d.ref], lo, la, z);
                        }
                        if (!inside) continue;
                        z += meta.offset;
                        if (G.geoid >= 0) {
                                const double l360 = (lo >= 0) ? lo : lo + 360.;
                                double undulation;
                                if (tb::map_elevation(G.maps[G.geoid], l360, la, undulation))
                                        z += undulation;
                        }
                        double ecef[3];
                        tb::ecef_from_geodetic(la, lo, z + height[i], ecef);
                        position[3 * i] = ecef[0];
                        position[3 * i + 1] = ecef[1];
                        position[3 * i + 2] = ecef[2];
                        found = k;
                        break;
                }
                if (data_index != NULL) data_index[i] = found;
        }
}

/* Ground elevation of one layer at the nodes of a grid (turtle_map_resample): node ->
 * inverse projection -> the layer's first data that holds the point (the elevation rule
 * of stepper.c:266-324, without the geoid). */
__global__ void __launch_bounds__(256) resample_kernel(const __grid_constant__ tb::Geometry G,
    const tb::ProjDesc P, int nx, int ny, double x0, double dx, double y0, double dy,
    int layer_index, double * __restrict__ z_out, int * __restrict__ inside_out)
{
        const size_t total = (size_t)nx * (size_t)ny;
        const size_t stride = (size_t)gridDim.x * blockDim.x;
        const tb::LayerDesc layer = G.layers[layer_index];
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
                const int iy = (int)(i / (size_t)nx);
                const int ix = (int)(i - (size_t)iy * nx);
                const double x = x0 + ix * dx, y = y0 + iy * dy; /* map.c:219-220 */
                double la = y, lo = x;
                if (P.type != tb::PROJ_GEODETIC) tb::unproject(P, x, y, la, lo);
                int found = 0;
                double z = 0.;
                for (int k = 0; (k < layer.n) && !found; k++) {
                        const tb::MetaDesc & meta = G.metas[layer.first + k];
                        const tb::DataDesc & d = G.data[meta.data];
                        if (d.kind == tb::DATA_FLAT) {
                                found = 1;
                                z = 0.;
                        } else if (d.kind == tb::DATA_STACK) {
                                found = tb::stack_elevation(G, G.stacks[d.ref], la, lo, z);
                        } else if (G.transforms[d.transform].type != tb::PROJ_GEODETIC) {
                                double mx, my;
                                tb::project(G.transforms[d.transform], la, lo, mx, my);
                                found = tb::map_elevation(G.maps[d.ref], mx, my, z);
                        } else {
                                found = tb::map_elevation(G.maps[d.ref], lo, la, z);
                        }
                        if (found) z += meta.offset;
                }
                z_out[i] = z;
                inside_out[i] = found;
        }
}

/* ---- frame transform kernels (ref: ecef.c) -------------------------------- */

__global__ void __launch_bounds__(256) to_geodetic_kernel(unsigned long long n,
    const double * __restrict__ ecef, double * __restrict__ latitude,
    double * __restrict__ longitude, double * __restrict__ altitude)
{
        const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
        for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
             i < n; i += stride) {
                const double r[3] = { ecef[3 * i], ecef[3 * i + 1], ecef[3 * i + 2] };
                double la, lo, al;
                tb::ecef_to_geodetic(r, la, lo, al);
                if (latitude != NULL) latitude[i] = la;
                if (longitude != NULL) longitude[i] = lo;
                if (altitude != NULL) altitude[i] = al;
        }
}

__global__ void __launch_bounds__(256) from_geodetic_kernel(unsigned long long n,
    const double * __restrict__ latitude, const double * __restrict__ longitude,
    const double * __restrict__ elevation, double * __restrict__ ecef)
{
        const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
        for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
             i < n; i += stride) {
                double r[3];
                tb::ecef_from_geodetic(latitude[i], longitude[i], elevation[i], r);
                ecef[3 * i] = r[0];
                ecef[3 * i + 1] = r[1];
                ecef[3 * i + 2] = r[2];
        }
}

__global__ void __launch_bounds__(256) from_horizontal_kernel(unsigned long long n,
    const double * __restrict__ latitude, const double * __restrict__ longitude,
    const double * __restrict__ azimuth, const double * __restrict__ elevation,
    double * __restrict__ direction)
{
        const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
        for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
             i < n; i += stride) {
                double r[3];
                tb::ecef_from_horizontal(latitude[i], longitude[i], azimuth[i], elevation[i], r);
                direction[3 * i] = r[0];
                direction[3 * i + 1] = r[1];
                direction[3 * i + 2] = r[2];
        }
}

/* ---- projections (ref: projection.c:192-233; SURVEY.md 8f N3) ------------------- */

__global__ void __launch_bounds__(256) projection_kernel(const tb::ProjDesc P, int inverse,
    unsigned long long n, const double * __restrict__ a, const double * __restrict__ b,
    double * __restrict__ c, double * __restrict__ d)
{
        const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
        for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
             i < n; i += stride) {
                double u, v;
                if (inverse)
                        tb::unproject(P, a[i], b[i], u, v);
                else
                        tb::project(P, a[i], b[i], u, v);
                c[i] = u;
                d[i] = v;
        }
}

/* ---- elevation kernels (ref: map.c:229-277) -------------------------------- */

template <class Fetch>
__global__ void __launch_bounds__(256) map_elevation_kernel(const tb::MapDesc M,
    unsigned long long n, const double * __restrict__ x, const double * __restrict__ y,
    double * __restrict__ z, int * __restrict__ inside)
{
        const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
        for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
             i < n; i += stride) {
                double zi;
                const int in = tb::map_elevation(Fetch(), M, x[i], y[i], zi);
                if (in) z[i] = zi;
                if (inside != NULL) inside[i] = in;
        }
}

/* ref: turtle_map_gradient, map.c:280-378 */
__global__ void __launch_bounds__(256) map_gradient_kernel(const tb::MapDesc M,
    unsigned long long n, const double * __restrict__ x, const double * __restrict__ y,
    double * __restrict__ gx, double * __restrict__ gy, int * __restrict__ inside)
{
        const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
        for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
             i < n; i += stride) {
                double a = gx[i], b = gy[i];
                const int in = tb::map_gradient(M, x[i], y[i], a, b);
                if (in) {
                        gx[i] = a;
                        gy[i] = b;
                }
                if (inside != NULL) inside[i] = in;
        }
}

/* ref: turtle_stack_gradient, stack.c:364-388, and turtle_stack_elevation, stack.c:338-361,
 * on a stack of a plan (the resident tile table): outside -> 0 (stack.c:349-355,376-380) */
__global__ void __launch_bounds__(256) stack_query_kernel(const __grid_constant__ tb::Geometry G,
    int stack, int gradient, unsigned long long n, const double * __restrict__ latitude,
    const double * __restrict__ longitude, double * __restrict__ a, double * __restrict__ b,
    int * __restrict__ inside)
{
        const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
        for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
             i < n; i += stride) {
                double u = 0., v = 0.;
                int in;
                if (gradient)
                        in = tb::stack_gradient(G, G.stacks[stack], latitude[i], longitude[i], u, v);
                else
                        in = tb::stack_elevation(G, G.stacks[stack], latitude[i], longitude[i], u);
                if (!in) u = v = 0.;
                a[i] = u;
                if (gradient) b[i] = v;
                if (inside != NULL) inside[i] = in;
        }
}

/* ECEF -> geodetic -> (projection) -> bilinear, fused: 24 B in, up to 36 B out
 * per point, nothing intermediate in HBM. */
template <class Fetch>
__global__ void __launch_bounds__(256) map_elevation_ecef_kernel(const tb::MapDesc M,
    const tb::ProjDesc P, unsigned long long n, const double * __restrict__ ecef,
    double * __restrict__ latitude, double * __restrict__ longitude,
    double * __restrict__ altitude, double * __restrict__ z, int * __restrict__ inside)
{
        const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
        for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
             i < n; i += stride) {
                const double r[3] = { ecef[3 * i], ecef[3 * i + 1], ecef[3 * i + 2] };
                double la, lo, al;
                tb::ecef_to_geodetic(r, la, lo, al);
                double mx = lo, my = la;
                if (P.type != tb::PROJ_GEODETIC) tb::project(P, la, lo, mx, my);
                double zi;
                const int in = tb::map_elevation(Fetch(), M, mx, my, zi);
                if (latitude != NULL) latitude[i] = la;
                if (longitude != NULL) longitude[i] = lo;
                if (altitude != NULL) altitude[i] = al;
                if (in) z[i] = zi;
                if (inside != NULL) inside[i] = in;
        }
}

/* Device-side tile ingestion: `raw` holds the nodes of one tile in FILE order (row 0 is
 * the northernmost when north_first, samples big-endian when big_endian); they are
 * written to the tile pool rows south first, native endian, `pitch` nodes per row: a pure
 * HBM stream of 2 + 2 bytes per node, coalesced on both sides. */
__global__ void __launch_bounds__(256) ingest_kernel(uint16_t * __restrict__ dst, int pitch,
    const uint16_t * __restrict__ raw, int nx, int ny, int big_endian, int north_first)
{
        const size_t total = (size_t)nx * (size_t)ny;
        const size_t stride = (size_t)gridDim.x * blockDim.x;
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
                const int iy = (int)(i / (size_t)nx);
                const int ix = (int)(i - (size_t)iy * nx);
                uint16_t v = raw[i];
                if (big_endian) v = (uint16_t)((v << 8) | (v >> 8));
                const int oy = north_first ? ny - 1 - iy : iy;
                dst[(size_t)oy * pitch + ix] = v;
        }
}

/* The cell-packed copy of a grid (tb::NodesPacked): cell (ix, iy) = { z00, z10, z01, z11 } in
 * ONE 8-byte word, same pitch as the grid; the last column / row of cells repeat the edge
 * (never addressed: a query on the closed upper edge uses the cell before, map.c:256-265). */
__global__ void __launch_bounds__(256) pack_cells_kernel(uint2 * __restrict__ cells,
    const uint16_t * __restrict__ nodes, int pitch, int nx, int ny)
{
        const size_t total = (size_t)pitch * (size_t)ny;
        const size_t stride = (size_t)gridDim.x * blockDim.x;
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
                const int iy = (int)(i / (size_t)pitch);
                const int ix = (int)(i - (size_t)iy * pitch);
                const int jx = (ix + 1 < nx) ? ix + 1 : ((ix < nx) ? ix : nx - 1);
                const int kx = (ix < nx) ? ix : nx - 1;
                const int jy = (iy + 1 < ny) ? iy + 1 : iy;
                const unsigned z00 = nodes[(size_t)iy * pitch + kx], z10 = nodes[(size_t)iy * pitch + jx];
                const unsigned z01 = nodes[(size_t)jy * pitch + kx], z11 = nodes[(size_t)jy * pitch + jx];
                cells[i] = make_uint2(z00 | (z10 << 16), z01 | (z11 << 16));
        }
}

/* ---- self test of tb::divide against the compiler's IEEE division ---------------- */

__device__ __forceinline__ unsigned long long mix64(unsigned long long x)
{
        x += 0x9E3779B97F4A7C15ull;
        x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
        x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
        return x ^ (x >> 31);
}

/* Random operands: full 52-bit significands, binary exponents in [lo, hi]. */
__device__ __forceinline__ double random_double(unsigned long long k, int lo, int hi)
{
        const unsigned long long r = mix64(k);
        const int e = lo + (int)((r >> 52) % (unsigned)(hi - lo + 1));
        const unsigned long long bits = ((unsigned long long)(1023 + e) << 52) |
            (r & 0xFFFFFFFFFFFFFull) | ((mix64(k ^ 0x5bd1e995ull) & 1ull) << 63);
        return __longlong_as_double((long long)bits);
}

__global__ void divide_selftest_kernel(unsigned long long n, unsigned long long seed,
    unsigned long long * mismatches)
{
        const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
        unsigned long long bad = 0ull;
        for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
             i < n; i += stride) {
                const double a = random_double(seed + 2ull * i, -60, 60);
                const double b = fabs(random_double(seed + 2ull * i + 1ull, -60, 60));
                const tb::Divisor d = tb::make_divisor(b);
                const double q1 = tb::divide(a, d);
                const double q2 = a / b;
                if (__double_as_longlong(q1) != __double_as_longlong(q2)) bad++;
                /* a second numerator against the same divisor, and exact cases */
                const double a2 = a * 0.75 + 1.0;
                if (__double_as_longlong(tb::divide(a2, d)) != __double_as_longlong(a2 / b)) bad++;
                if (tb::divide(0., d) != 0. || tb::divide(b, d) != 1.) bad++;
                const int k = (int)(mix64(i) & 0xffff) - 32768;
                if (tb::int_to_double(k) != (double)k) bad++;
                /* tb::sqrt_in_range against the library's sqrt over its whole range */
                const double sq = fabs(random_double(seed + 2ull * i + 7ull, -960, 1020));
                if (__double_as_longlong(tb::sqrt_in_range(sq)) != __double_as_longlong(sqrt(sq)))
                        bad++;
                const double sq1 = 0.25 + 0.75 * fabs(random_double(seed + 2ull * i + 9ull, -1, -1));
                if (__double_as_longlong(tb::sqrt_in_range(sq1)) != __double_as_longlong(sqrt(sq1)))
                        bad++;
                /* divisors with a correctly rounded reciprocal (tb::known_divisor): the
                 * random one, pi (degrees) and the usual grid pitches */
                const double fixed[6] = { b, M_PI, 1. / 3600., 1. / 1200., 10., 1. / 3. };
                const double c = fixed[i % 6ull];
                const tb::Divisor kd = tb::known_divisor(c, 1. / c);
                if (__double_as_longlong(tb::divide(a, kd)) != __double_as_longlong(a / c)) bad++;
                if (__double_as_longlong(tb::divide(a2, kd)) != __double_as_longlong(a2 / c)) bad++;
        }
        if (bad) atomicAdd(mismatches, bad);
}

/* ---- FP64 FMA peak (roofline denominator of the stepper) --------------------- */

__global__ void __launch_bounds__(256) dfma_kernel(double * out, int iterations)
{
        double a0 = threadIdx.x * 1e-9, a1 = a0 + 1., a2 = a0 + 2., a3 = a0 + 3.;
        double a4 = a0 + 4., a5 = a0 + 5., a6 = a0 + 6., a7 = a0 + 7.;
        const double b = 1.0000001, c = 1e-7;
        for (int i = 0; i < iterations; i++) {
                a0 = fma(a0, b, c); a1 = fma(a1, b, c); a2 = fma(a2, b, c); a3 = fma(a3, b, c);
                a4 = fma(a4, b, c); a5 = fma(a5, b, c); a6 = fma(a6, b, c); a7 = fma(a7, b, c);
        }
        out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] =
            a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

} /* namespace */

/* ======================================================================== */
/* Host side: plans, residency, launches                                     */
/* ======================================================================== */

namespace {
const int N_SLOTS = 3;              /* host-pointer pipeline depth */
const int DEV_SLOTS = 8;            /* device-pointer calls that may be in flight per plan */
const int ALL_SLOTS = N_SLOTS + DEV_SLOTS;
const int HOST_SLICES = DEV_SLOTS;  /* counter blocks of the slices of a host-pointer fan, after
                                     * the ALL_SLOTS blocks */
const int CTR = 8;                  /* counters per launch: [0] queue cursor, [1] steps,
                                     * [2] samples, [3] stream time-out, [4] Jacobian columns */
const size_t CHUNK_RAYS = 1u << 20; /* rays per pipeline chunk (one kernel per chunk) */
const int STREAM_CHUNK_SHIFT = 18;  /* rays per copy of a streamed call: 256 Ki */
const size_t STREAM_CHUNK_RAYS = (size_t)1 << STREAM_CHUNK_SHIFT;
const int N_DRAINS = 4;             /* result streams of a streamed call */
const size_t STREAM_MAX_RAYS = (size_t)1 << 25; /* rays per round of a streamed call */
}

struct turtle_plan {
        int device;
        int sm_count;
        int ctas_per_sm, threads;
        tb::Geometry G; /* device pointers */
        void * pool;    /* every tile of the plan, one allocation */
        tb::MapDesc * d_maps;
        tb::TileRec * d_tiles;
        size_t bytes;
        turtle_residency_report report;
        std::vector<struct turtle_stack *> pinned;
        unsigned long long * d_counters; /* ALL_SLOTS + HOST_SLICES blocks of CTR counters */
        int dev_slot;                    /* block of the latest device-pointer call */
        /* per device slot: recorded on the caller's stream after the last operation of the
         * call that holds the slot (NULL until the slot is first used), and the number of
         * the device-pointer call that took it */
        cudaEvent_t slot_done[DEV_SLOTS];
        unsigned long long slot_call[DEV_SLOTS];
        unsigned long long dev_calls;
        turtle_plan_counters counters;
        /* ray scheduling (turtle_plan_schedule_set) */
        int schedule;
        int specialise; /* turtle_plan_specialise_set */
        int pipeline_mode; /* turtle_plan_pipeline_set */
        unsigned * d_sched[ALL_SLOTS]; /* per slot: keys, index, keys', order */
        void * d_sched_tmp[ALL_SLOTS];
        size_t sched_rays[ALL_SLOTS], sched_tmp_bytes[ALL_SLOTS];
        /* host-pointer pipeline */
        cudaStream_t stream[N_SLOTS];
        cudaEvent_t ev0[N_SLOTS], ev1[N_SLOTS];
        double * d_in[N_SLOTS];
        turtle_trace_result * d_out[N_SLOTS];
        size_t slot_rays;
        /* streamed host-pointer calls (trace_streamed) */
        double * d_all_in;
        turtle_trace_result * d_all_out;
        size_t all_rays, all_records;
        unsigned long long * d_stream_state; /* watermark + per-chunk counters */
        unsigned long long * h_marks;        /* pinned: the watermark values to copy */
        unsigned * h_flags;                  /* pinned + mapped: chunk completion flags */
        size_t stream_chunks;
        cudaEvent_t ev_reset;
        cudaStream_t drain[N_DRAINS]; /* result streams */
        /* fan tables (turtle_stepper_trace_fan[s], _horizon[s]), per slot: pinned host copy +
         * device copy of the angles' sines / cosines and the stations' frames (fan_upload) */
        double2 * h_fan[ALL_SLOTS];
        double2 * d_fan[ALL_SLOTS];
        size_t fan_entries[ALL_SLOTS]; /* double2 entries allocated */
        /* device staging of the field arrays of a host-pointer call */
        void * d_field_pool;
        size_t field_pool_bytes;
        /* node gathers of the single-stack trace kernel (turtle_plan_gather_set) */
        int gather;
        std::vector<tb::TileRec> h_tiles; /* the tile table as uploaded */
        std::vector<tb::MapDesc> h_maps;  /* ... and the descriptors it refers to */
        void * packed_pool;               /* cell-packed copies of the tiles */
        tb::TileRec * d_tiles_packed;     /* tile table whose `nodes` are the packed copies */
        WindowArgs window;
};

struct turtle_states {
        struct turtle_plan * plan;
        int device;        /* the plan's: destroying the states does not need the plan */
        size_t n;
        double * d_states; /* PS_FIELDS + G.lla_rows field rows of `stride` particles */
        size_t stride;
};

static int round_up(int x, int m) { return (x + m - 1) / m * m; }

static enum turtle_return require_device(turtle_function_t * fn, int device)
{
        int count = 0;
        cudaError_t err = cudaGetDeviceCount(&count);
        if ((err != cudaSuccess) || (count == 0)) {
                cudaGetLastError();
                return tbh::raise(fn, TURTLE_RETURN_LIBRARY_ERROR, BATCH_CU, __LINE__,
                    "no CUDA device: the batched path has no CPU fallback (%s)",
                    (err != cudaSuccess) ? cudaGetErrorString(err) : "0 devices");
        }
        if ((device < 0) || (device >= count))
                return tbh::raise(fn, TURTLE_RETURN_DOMAIN_ERROR, BATCH_CU, __LINE__,
                    "invalid device %d (have %d)", device, count);
        return TURTLE_RETURN_SUCCESS;
}

extern "C" int turtle_b200_device_count(void)
{
        int count = 0;
        if (cudaGetDeviceCount(&count) != cudaSuccess) {
                cudaGetLastError();
                return 0;
        }
        return count;
}

extern "C" const char * turtle_b200_version(void) { return "turtle-b200 0.1 (sm_100a)"; }

/* Device self test: tb::divide (shared reciprocal, tb_core.cuh) against `a / b` on
 * 2 * n random operand pairs; returns the number of results that differ in any bit
 * (must be 0), or -1 without a device. */
extern "C" long long turtle_b200_selftest_division(size_t n, uint64_t seed)
{
        if (turtle_b200_device_count() == 0) return -1;
        unsigned long long * d_bad = NULL;
        unsigned long long bad = 0ull;
        if (cudaMalloc((void **)&d_bad, sizeof(bad)) != cudaSuccess) return -1;
        cudaMemset(d_bad, 0x0, sizeof(bad));
        divide_selftest_kernel<<<148 * 8, 256>>>(n, seed, d_bad);
        cudaMemcpy(&bad, d_bad, sizeof(bad), cudaMemcpyDeviceToHost);
        cudaFree(d_bad);
        return (cudaGetLastError() == cudaSuccess) ? (long long)bad : -1;
}

/* Copy a host grid into the device pool with a padded pitch. */
static cudaError_t upload_nodes(uint16_t * dst, int pitch, const struct turtle_map * map)
{
        return cudaMemcpy2D(dst, (size_t)pitch * sizeof(uint16_t), map->nodes.data(),
            (size_t)map->nx * sizeof(uint16_t), (size_t)map->nx * sizeof(uint16_t),
            (size_t)map->ny, cudaMemcpyHostToDevice);
}

static size_t padded_nodes(const struct turtle_map * map, int * pitch)
{
        /* rows start on a 32-byte sector; one spare row keeps the +pitch gather
         * of the closed upper edge inside the allocation */
        *pitch = round_up(map->nx, 16);
        return (size_t)*pitch * (size_t)(map->ny + 1);
}

static enum turtle_return check_rule(turtle_function_t * fn, const struct turtle_trace_rule * rule);

static size_t padded_shape(int nx, int ny, int * pitch)
{
        *pitch = round_up(nx, 16);
        return (size_t)*pitch * (size_t)(ny + 1);
}

static double wall_ms()
{
        struct timespec t;
        clock_gettime(CLOCK_MONOTONIC, &t);
        return 1e3 * (double)t.tv_sec + 1e-6 * (double)t.tv_nsec;
}

/* One tile that is not on the host: file -> nodes in file order -> device -> ingest_kernel. */
static enum turtle_return ingest_tile(turtle_function_t * fn, const std::string & path,
    const tb::MapDesc & want, uint16_t * dst, int pitch, uint16_t ** scratch,
    size_t * scratch_nodes, turtle_residency_report * report)
{
        tbio::Header h;
        tbio::RawLayout layout;
        tbio::Error err;
        std::vector<uint16_t> raw;
        const double t0 = wall_ms();
        if (tbio::read_map(path.c_str(), h, layout, raw, err) != 0)
                return tbh::raise(fn, err.code, err.file, __LINE__, "%s", err.message.c_str());
        if ((h.nx != want.nx) || (h.ny != want.ny))
                return tbh::raise(fn, TURTLE_RETURN_BAD_FORMAT, BATCH_CU, __LINE__,
                    "tile `%s' changed since the stack was created", path.c_str());
        const double t1 = wall_ms();
        if (*scratch_nodes < raw.size()) {
                cudaFree(*scratch);
                *scratch = NULL;
                *scratch_nodes = 0;
                CUDA_TRY(fn, cudaMalloc((void **)scratch, raw.size() * sizeof(uint16_t)));
                *scratch_nodes = raw.size();
        }
        CUDA_TRY(fn, cudaMemcpy(*scratch, raw.data(), raw.size() * sizeof(uint16_t),
                         cudaMemcpyHostToDevice));
        const int blocks = (int)std::min<size_t>((raw.size() + 255) / 256, 148 * 16);
        ingest_kernel<<<blocks, 256>>>(dst, pitch, *scratch, h.nx, h.ny, layout.big_endian,
            layout.north_first);
        CUDA_TRY(fn, cudaGetLastError());
        CUDA_TRY(fn, cudaDeviceSynchronize()); /* the scratch buffer is reused */
        report->read_ms += t1 - t0;
        report->upload_ms += wall_ms() - t1;
        report->tiles_ingested++;
        return TURTLE_RETURN_SUCCESS;
}

static enum turtle_return freeze_plan(turtle_function_t * fn, struct turtle_stepper * stepper,
    int device, const struct turtle_residency * region, struct turtle_plan ** plan_)
{
        *plan_ = NULL;
        enum turtle_return rc = require_device(fn, device);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        if (stepper->layers.empty() || stepper->layers[0].empty())
                return tbh::raise(fn, TURTLE_RETURN_DOMAIN_ERROR, BATCH_CU, __LINE__,
                    "empty geometry");
        /* a flattening of its own: tiles that are not on the host stay on disk until they
         * are ingested below, and the region leaves tiles out */
        tb_flat_geometry F;
        rc = tbh::flatten_into(stepper, F, fn, 0, region);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;

        CUDA_TRY(fn, cudaSetDevice(device));
        struct turtle_plan * plan = new (std::nothrow) turtle_plan();
        if (plan == NULL)
                return tbh::raise(fn, TURTLE_RETURN_MEMORY_ERROR, BATCH_CU, __LINE__,
                    "could not allocate memory");
        memset(&plan->counters, 0x0, sizeof(plan->counters));
        memset(&plan->report, 0x0, sizeof(plan->report));
        plan->device = device;
        plan->pool = NULL;
        plan->d_maps = NULL;
        plan->d_tiles = NULL;
        plan->d_counters = NULL;
        plan->dev_slot = N_SLOTS;
        for (int s = 0; s < DEV_SLOTS; s++) {
                plan->slot_done[s] = NULL;
                plan->slot_call[s] = 0;
        }
        plan->dev_calls = 0;
        plan->schedule = 0;
        plan->specialise = 1;
        plan->pipeline_mode = 0;
        for (int s = 0; s < ALL_SLOTS; s++) {
                plan->d_sched[s] = NULL;
                plan->d_sched_tmp[s] = NULL;
                plan->sched_rays[s] = 0;
                plan->sched_tmp_bytes[s] = 0;
        }
        plan->slot_rays = 0;
        for (int s = 0; s < N_SLOTS; s++) {
                plan->stream[s] = NULL;
                plan->d_in[s] = NULL;
                plan->d_out[s] = NULL;
        }
        plan->d_all_in = NULL;
        plan->d_all_out = NULL;
        plan->all_rays = 0;
        plan->all_records = 0;
        plan->d_stream_state = NULL;
        plan->h_marks = NULL;
        plan->h_flags = NULL;
        plan->stream_chunks = 0;
        plan->ev_reset = NULL;
        for (int j = 0; j < 4; j++) plan->drain[j] = NULL;
        for (int k = 0; k < ALL_SLOTS; k++) {
                plan->h_fan[k] = NULL;
                plan->d_fan[k] = NULL;
                plan->fan_entries[k] = 0;
        }
        plan->d_field_pool = NULL;
        plan->field_pool_bytes = 0;
        plan->gather = GATHER_GLOBAL;
        plan->packed_pool = NULL;
        plan->d_tiles_packed = NULL;
        memset(&plan->window, 0x0, sizeof plan->window);
        cudaDeviceProp prop;
        cudaGetDeviceProperties(&prop, device);
        plan->sm_count = prop.multiProcessorCount;
        plan->ctas_per_sm = 0;
        plan->threads = 0;

        /* residency plan: one pool for all grids, identical maps stored once */
        const size_t n_maps = F.maps.size();
        std::vector<size_t> offset(n_maps, 0);
        std::vector<int> pitch(n_maps, 0);
        std::vector<size_t> owner(n_maps, 0); /* first descriptor of the same grid */
        std::map<const struct turtle_map *, size_t> first;
        size_t total = 0;
        for (size_t i = 0; i < n_maps; i++) {
                owner[i] = i;
                if (F.src[i] != NULL) {
                        std::map<const struct turtle_map *, size_t>::iterator it =
                            first.find(F.src[i]);
                        if (it != first.end()) {
                                owner[i] = it->second;
                                offset[i] = offset[it->second];
                                pitch[i] = pitch[it->second];
                                continue;
                        }
                        first[F.src[i]] = i;
                }
                offset[i] = total;
                total += (padded_shape(F.maps[i].nx, F.maps[i].ny, &pitch[i]) + 127) / 128 * 128;
        }
        const size_t pool_bytes = std::max<size_t>(total, 128) * sizeof(uint16_t);
        size_t limit = (region != NULL) ? region->memory_limit : 0;
        if (limit == 0) {
                size_t free_bytes = 0, total_bytes = 0;
                if (cudaMemGetInfo(&free_bytes, &total_bytes) == cudaSuccess) limit = free_bytes;
        }
        if ((limit > 0) && (pool_bytes > limit)) {
                delete plan;
                return tbh::raise(fn, TURTLE_RETURN_MEMORY_ERROR, BATCH_CU, __LINE__,
                    "the residency plan needs %zu bytes of device memory for %zu grids, "
                    "%zu are allowed: restrict the region (turtle_stepper_freeze_region)",
                    pool_bytes, n_maps, limit);
        }
        cudaError_t err = cudaMalloc(&plan->pool, pool_bytes);
        if (err == cudaSuccess) err = cudaMemset(plan->pool, 0x0, pool_bytes);
        std::vector<tb::MapDesc> maps = F.maps;
        uint16_t * scratch = NULL;
        size_t scratch_nodes = 0;
        for (size_t i = 0; (i < n_maps) && (err == cudaSuccess); i++) {
                uint16_t * dst = (uint16_t *)plan->pool + offset[i];
                maps[i].nodes = dst;
                maps[i].pitch = pitch[i];
                if (owner[i] != i) continue;
                if (F.src[i] != NULL) {
                        const double t0 = wall_ms();
                        err = upload_nodes(dst, pitch[i], F.src[i]);
                        plan->report.upload_ms += wall_ms() - t0;
                } else {
                        rc = ingest_tile(fn, F.file[i], F.maps[i], dst, pitch[i], &scratch,
                            &scratch_nodes, &plan->report);
                        if (rc != TURTLE_RETURN_SUCCESS) {
                                cudaFree(scratch);
                                turtle_plan_destroy(&plan);
                                return rc;
                        }
                }
        }
        cudaFree(scratch);
        const size_t maps_bytes = std::max<size_t>(n_maps, 1) * sizeof(tb::MapDesc);
        const size_t tiles_bytes = std::max<size_t>(F.tiles.size(), 1) * sizeof(tb::TileRec);
        /* device copies of the tile records: device node pointers and padded pitch */
        std::vector<tb::TileRec> tiles = F.tiles;
        for (size_t i = 0; i < tiles.size(); i++)
                if (tiles[i].map >= 0) {
                        tiles[i].nodes = maps[tiles[i].map].nodes;
                        plan->report.tiles_resident++;
                }
        plan->report.tiles_skipped = F.skipped;
        if (err == cudaSuccess) err = cudaMalloc((void **)&plan->d_maps, maps_bytes);
        if ((err == cudaSuccess) && n_maps)
                err = cudaMemcpy(plan->d_maps, maps.data(), n_maps * sizeof(tb::MapDesc),
                    cudaMemcpyHostToDevice);
        if (err == cudaSuccess) err = cudaMalloc((void **)&plan->d_tiles, tiles_bytes);
        if ((err == cudaSuccess) && !tiles.empty())
                err = cudaMemcpy(plan->d_tiles, tiles.data(), tiles.size() * sizeof(tb::TileRec),
                    cudaMemcpyHostToDevice);
        if (err == cudaSuccess)
                err = cudaMalloc((void **)&plan->d_counters,
                    (ALL_SLOTS + HOST_SLICES) * CTR * sizeof(unsigned long long));
        if (err != cudaSuccess) {
                turtle_plan_destroy(&plan);
                return tbh::raise(fn, TURTLE_RETURN_LIBRARY_ERROR, BATCH_CU, __LINE__,
                    "CUDA error while uploading the geometry: %s", cudaGetErrorString(err));
        }
        plan->h_tiles = tiles;
        plan->h_maps = maps;
        plan->G = F.G;
        plan->G.maps = plan->d_maps;
        plan->G.tiles = plan->d_tiles;
        for (int k = 0; k < plan->G.n_stacks; k++) { /* the device pitch is padded */
                tb::StackDesc & S = plan->G.stacks[k];
                for (int c = 0; c < S.nlat * S.nlon; c++) {
                        const int id = tiles[S.tile0 + c].map;
                        if (id >= 0) {
                                S.pitch = maps[id].pitch;
                                break;
                        }
                }
        }
        plan->bytes = pool_bytes + maps_bytes + tiles_bytes;
        plan->report.bytes = plan->bytes;
        *plan_ = plan;
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_stepper_freeze(
    struct turtle_stepper * stepper, int device, struct turtle_plan ** plan_)
{
        return freeze_plan(FN(&turtle_stepper_freeze), stepper, device, NULL, plan_);
}

extern "C" enum turtle_return turtle_stepper_freeze_region(struct turtle_stepper * stepper,
    int device, const struct turtle_residency * region, struct turtle_plan ** plan_)
{
        return freeze_plan(FN(&turtle_stepper_freeze_region), stepper, device, region, plan_);
}

extern "C" void turtle_plan_residency_get(
    const struct turtle_plan * plan, struct turtle_residency_report * report)
{
        *report = plan->report;
}

/* Bounding box of the ground tracks of the rays (turtle_b200.h). Host code: it runs
 * once per batch, before the plan exists. */
extern "C" enum turtle_return turtle_residency_from_rays(size_t n, const double * position,
    const double * direction, const struct turtle_trace_rule * rule, double step,
    double margin, struct turtle_residency * region)
{
        enum turtle_return rc = check_rule(FN(&turtle_residency_from_rays), rule);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        if (!(step > 0.)) step = 1000.;
        double la0 = DBL_MAX, la1 = -DBL_MAX, lo0 = DBL_MAX, lo1 = -DBL_MAX;
        bool open_longitude = false;
        const double radius = TB_WGS84_A + rule->altitude_max;
        for (size_t i = 0; i < n; i++) {
                const double * p = position + 3 * i;
                const double * d = direction + 3 * i;
                const double dd = d[0] * d[0] + d[1] * d[1] + d[2] * d[2];
                if (!(dd > 0.) || !isfinite(dd) || !isfinite(p[0] + p[1] + p[2])) continue;
                /* path length at which the ray is above altitude_max for certain: the
                 * geocentric radius of a point at altitude h is at most a + h */
                const double pd = p[0] * d[0] + p[1] * d[1] + p[2] * d[2];
                const double pp = p[0] * p[0] + p[1] * p[1] + p[2] * p[2];
                const double disc = pd * pd - dd * (pp - radius * radius);
                double reach = (disc > 0.) ? (-pd + sqrt(disc)) / dd * sqrt(dd) : 0.;
                if (!(reach > 0.)) reach = 0.;
                if (reach > rule->length_max) reach = rule->length_max;
                const double norm = sqrt(dd);
                const int pieces = (int)std::min(1e6, ceil(reach / step)) + 1;
                double previous = 0.;
                for (int k = 0; k <= pieces; k++) {
                        const double t = reach * k / pieces / norm;
                        const double q[3] = { p[0] + d[0] * t, p[1] + d[1] * t, p[2] + d[2] * t };
                        double la, lo, al;
                        tb::ecef_to_geodetic(q, la, lo, al);
                        if ((q[0] == 0.) && (q[1] == 0.)) open_longitude = true;
                        if ((k > 0) && (fabs(lo - previous) > 180.)) open_longitude = true;
                        previous = lo;
                        la0 = std::min(la0, la);
                        la1 = std::max(la1, la);
                        lo0 = std::min(lo0, lo);
                        lo1 = std::max(lo1, lo);
                }
        }
        region->memory_limit = 0;
        if (la0 > la1) { /* no valid ray: an empty box */
                region->latitude_min = region->longitude_min = DBL_MAX;
                region->latitude_max = region->longitude_max = -DBL_MAX;
                return TURTLE_RETURN_SUCCESS;
        }
        region->latitude_min = la0 - margin;
        region->latitude_max = la1 + margin;
        region->longitude_min = open_longitude ? NAN : lo0 - margin;
        region->longitude_max = open_longitude ? NAN : lo1 + margin;
        return TURTLE_RETURN_SUCCESS;
}

extern "C" void turtle_plan_destroy(struct turtle_plan ** plan_)
{
        if ((plan_ == NULL) || (*plan_ == NULL)) return;
        struct turtle_plan * plan = *plan_;
        cudaSetDevice(plan->device);
        for (int s = 0; s < N_SLOTS; s++) {
                if (plan->stream[s] != NULL) {
                        cudaStreamSynchronize(plan->stream[s]);
                        cudaEventDestroy(plan->ev0[s]);
                        cudaEventDestroy(plan->ev1[s]);
                        cudaStreamDestroy(plan->stream[s]);
                }
                cudaFree(plan->d_in[s]);
                cudaFree(plan->d_out[s]);
        }
        for (int s = 0; s < ALL_SLOTS; s++) {
                cudaFree(plan->d_sched[s]);
                cudaFree(plan->d_sched_tmp[s]);
        }
        for (int s = 0; s < DEV_SLOTS; s++)
                if (plan->slot_done[s] != NULL) cudaEventDestroy(plan->slot_done[s]);
        cudaFree(plan->d_all_in);
        cudaFree(plan->d_all_out);
        cudaFree(plan->d_field_pool);
        cudaFree(plan->packed_pool);
        cudaFree(plan->d_tiles_packed);
        for (int k = 0; k < ALL_SLOTS; k++) {
                if (plan->h_fan[k] != NULL) cudaFreeHost(plan->h_fan[k]);
                cudaFree(plan->d_fan[k]);
        }
        cudaFree(plan->d_stream_state);
        if (plan->h_marks != NULL) cudaFreeHost(plan->h_marks);
        if (plan->h_flags != NULL) cudaFreeHost(plan->h_flags);
        if (plan->ev_reset != NULL) cudaEventDestroy(plan->ev_reset);
        for (int j = 0; j < N_DRAINS; j++)
                if (plan->drain[j] != NULL) cudaStreamDestroy(plan->drain[j]);
        cudaFree(plan->pool);
        cudaFree(plan->d_maps);
        cudaFree(plan->d_tiles);
        cudaFree(plan->d_counters);
        delete plan;
        *plan_ = NULL;
}

extern "C" int turtle_plan_device(const struct turtle_plan * plan) { return plan->device; }
extern "C" size_t turtle_plan_bytes(const struct turtle_plan * plan) { return plan->bytes; }

extern "C" void turtle_plan_counters_get(
    const struct turtle_plan * plan, struct turtle_plan_counters * counters)
{
        *counters = plan->counters;
}

extern "C" void turtle_plan_launch_set(struct turtle_plan * plan, int ctas_per_sm, int threads)
{
        plan->ctas_per_sm = ctas_per_sm;
        plan->threads = threads;
}

extern "C" void turtle_plan_schedule_set(struct turtle_plan * plan, int mode)
{
        plan->schedule = mode;
}

extern "C" void turtle_plan_specialise_set(struct turtle_plan * plan, int enable)
{
        plan->specialise = enable;
}

extern "C" void turtle_plan_pipeline_set(struct turtle_plan * plan, int mode)
{
        plan->pipeline_mode = mode;
}

/* How the single-stack trace kernel gathers its nodes (turtle_b200.h). */
extern "C" enum turtle_return turtle_plan_gather_set(struct turtle_plan * plan, int mode,
    double latitude, double longitude)
{
        turtle_function_t * fn = FN(&turtle_plan_gather_set);
        if ((mode < GATHER_GLOBAL) || (mode > GATHER_WINDOW))
                return tbh::raise(fn, TURTLE_RETURN_DOMAIN_ERROR, BATCH_CU, __LINE__,
                    "invalid gather mode %d", mode);
        if (mode == GATHER_GLOBAL) {
                plan->gather = mode;
                return TURTLE_RETURN_SUCCESS;
        }
        if (tb::geometry_shape(plan->G) != tb::SHAPE_STACK)
                return tbh::raise(fn, TURTLE_RETURN_DOMAIN_ERROR, BATCH_CU, __LINE__,
                    "packed / windowed gathers are for a geometry of one uniform stack");
        CUDA_TRY(fn, cudaSetDevice(plan->device));
        const tb::StackDesc & S = plan->G.stacks[0];
        if ((mode == GATHER_PACKED) && (plan->d_tiles_packed == NULL)) {
                /* a second, cell-packed copy of every tile: 4 x the bytes of the first */
                const size_t per_tile = ((size_t)S.pitch * S.ny * sizeof(uint2) + 255) / 256 * 256;
                size_t n_tiles = 0;
                for (size_t i = 0; i < plan->h_tiles.size(); i++)
                        if (plan->h_tiles[i].map >= 0) n_tiles++;
                CUDA_TRY(fn, cudaMalloc(&plan->packed_pool, std::max<size_t>(per_tile * n_tiles, 256)));
                std::vector<tb::TileRec> packed = plan->h_tiles;
                size_t at = 0;
                for (size_t i = 0; i < packed.size(); i++) {
                        if (packed[i].map < 0) continue;
                        uint2 * dst = (uint2 *)((char *)plan->packed_pool + at);
                        pack_cells_kernel<<<plan->sm_count * 8, 256>>>(dst, packed[i].nodes, S.pitch,
                            S.nx, S.ny);
                        packed[i].nodes = (const uint16_t *)dst;
                        at += per_tile;
                }
                CUDA_TRY(fn, cudaGetLastError());
                CUDA_TRY(fn, cudaMalloc((void **)&plan->d_tiles_packed,
                                 std::max<size_t>(packed.size(), 1) * sizeof(tb::TileRec)));
                CUDA_TRY(fn, cudaMemcpy(plan->d_tiles_packed, packed.data(),
                                 packed.size() * sizeof(tb::TileRec), cudaMemcpyHostToDevice));
                CUDA_TRY(fn, cudaDeviceSynchronize());
                plan->bytes += per_tile * n_tiles;
        }
        if (mode == GATHER_WINDOW) {
                /* the window: WINDOW_NODES^2 nodes of the tile that holds (latitude,
                 * longitude), centred there as far as the tile allows */
                const int cx = (int)floor((longitude - S.lon0) / S.dlon);
                const int cy = (int)floor((latitude - S.lat0) / S.dlat);
                if ((cx < 0) || (cx >= S.nlon) || (cy < 0) || (cy >= S.nlat) ||
                    (plan->h_tiles[S.tile0 + cy * S.nlon + cx].map < 0) ||
                    (S.nx < WINDOW_NODES) || (S.ny < WINDOW_NODES))
                        return tbh::raise(fn, TURTLE_RETURN_DOMAIN_ERROR, BATCH_CU, __LINE__,
                            "no tile under the centre of the window");
                const tb::TileRec & t = plan->h_tiles[S.tile0 + cy * S.nlon + cx];
                int x0 = (int)((longitude - t.x0) / S.dx) - WINDOW_NODES / 2;
                int y0 = (int)((latitude - t.y0) / S.dy) - WINDOW_NODES / 2;
                x0 = std::max(0, std::min(x0, S.nx - WINDOW_NODES)) / 8 * 8;
                y0 = std::max(0, std::min(y0, S.ny - WINDOW_NODES));
                plan->window.tile = t.nodes;
                plan->window.x0 = x0;
                plan->window.y0 = y0;
                plan->window.pitch = S.pitch;
        }
        plan->gather = mode;
        return TURTLE_RETURN_SUCCESS;
}

/* A staging buffer of a plan: device memory, or pinned host memory allocated with
 * cudaHostAlloc(`host_flags`) when host_flags >= 0. */
struct Staging {
        void ** p;
        size_t bytes;
        int host_flags = -1;
};

/* Grow-only staging: while `*have` (in the caller's unit) is below `need`, the buffers are
 * freed and allocated again at their `bytes`. `*have` becomes `need` once all of them are
 * allocated, and stays 0 after a failure so that the next call tries again. */
template <size_t K>
static cudaError_t grow(size_t * have, size_t need, const Staging (&buffers)[K])
{
        if (*have >= need) return cudaSuccess;
        *have = 0;
        for (const Staging & b : buffers) {
                if (b.host_flags < 0)
                        cudaFree(*b.p);
                else if (*b.p != NULL)
                        cudaFreeHost(*b.p);
                *b.p = NULL;
        }
        for (const Staging & b : buffers) {
                const cudaError_t err = (b.host_flags < 0) ? cudaMalloc(b.p, b.bytes) :
                                                             cudaHostAlloc(b.p, b.bytes, b.host_flags);
                if (err != cudaSuccess) return err;
        }
        *have = need;
        return cudaSuccess;
}

/* Small RAII helper for the host-pointer wrappers of the simple kernels. */
namespace {
struct DeviceBuffers {
        std::vector<void *> ptrs;
        ~DeviceBuffers()
        {
                for (size_t i = 0; i < ptrs.size(); i++) cudaFree(ptrs[i]);
        }
        /* allocate `bytes` and optionally copy from host; NULL host + copy_in=false = output */
        cudaError_t get(void ** dev, const void * host, size_t bytes, bool copy_in)
        {
                *dev = NULL;
                cudaError_t err = cudaMalloc(dev, std::max<size_t>(bytes, 8));
                if (err != cudaSuccess) return err;
                ptrs.push_back(*dev);
                if (copy_in && (host != NULL) && bytes)
                        err = cudaMemcpy(*dev, host, bytes, cudaMemcpyHostToDevice);
                return err;
        }
};
}

/* Build the queue order of a launch (longest-expected-first) in plan->d_sched. */
static cudaError_t schedule_rays(struct turtle_plan * plan, int slot, size_t n,
    const double * d_position, const double * d_direction, cudaStream_t stream,
    const unsigned ** order)
{
        *order = NULL;
        if ((plan->schedule == 0) || (n < 2) || (n > 0x7fffffffull)) return cudaSuccess;
        cudaError_t err = cudaSuccess;
        if (plan->sched_rays[slot] < n) {
                size_t tmp = 0;
                err = cub::DeviceRadixSort::SortPairs(NULL, tmp, (const unsigned *)NULL,
                    (unsigned *)NULL, (const unsigned *)NULL, (unsigned *)NULL, (int)n, 0, 31,
                    stream);
                if (err == cudaSuccess)
                        err = grow(&plan->sched_rays[slot], n,
                            { { (void **)&plan->d_sched[slot], 4 * n * sizeof(unsigned) },
                                { &plan->d_sched_tmp[slot], tmp } });
                if (err != cudaSuccess) return err;
                plan->sched_tmp_bytes[slot] = tmp;
        }
        unsigned * keys = plan->d_sched[slot];
        unsigned * index = keys + plan->sched_rays[slot];
        unsigned * keys_out = index + plan->sched_rays[slot];
        unsigned * sorted = keys_out + plan->sched_rays[slot];
        const int blocks = (int)std::min<size_t>((n + 255) / 256, (size_t)plan->sm_count * 16);
        schedule_key_kernel<<<blocks, 256, 0, stream>>>(n, d_position, d_direction, keys, index);
        plan->counters.launches++;
        err = cudaGetLastError();
        if (err != cudaSuccess) return err;
        size_t tmp = plan->sched_tmp_bytes[slot];
        err = cub::DeviceRadixSort::SortPairs(plan->d_sched_tmp[slot], tmp, keys, keys_out, index, sorted,
            (int)n, 0, 31, stream);
        plan->counters.launches += 4; /* radix sort passes (library kernels) */
        *order = sorted;
        return err;
}

/* Dynamic shared memory of a kernel of the local approximation: G.lla_rows columns of
 * 128 doubles (tb::LlaView). */
static size_t lla_bytes(const struct turtle_plan * plan)
{
        return (plan->G.range > 0.) ? (size_t)plan->G.lla_rows * 128 * sizeof(double) : 0;
}

/* The kernel variant of a plan's geometry: the local approximation (range > 0), any
 * projected map (else the projection code is compiled out), and the single-stack
 * specialisation (turtle_plan_specialise_set). */
struct Variant {
        bool lla, proj, stack_shape;
};
static Variant variant_of(const struct turtle_plan * plan)
{
        Variant v;
        v.lla = plan->G.range > 0.;
        v.proj = false;
        for (int t = 0; t < plan->G.n_transforms; t++)
                if (plan->G.transforms[t].type != tb::PROJ_GEODETIC) v.proj = true;
        v.stack_shape = plan->specialise && (tb::geometry_shape(plan->G) == tb::SHAPE_STACK);
        return v;
}

template <bool LLA_, bool PROJ_, int SHAPE_, int MINB_> struct VariantOf {
        static const bool LLA = LLA_, PROJ = PROJ_;
        static const int SHAPE = SHAPE_, MINB = MINB_;
};

/* f(VariantOf<LLA, PROJ, SHAPE, MINB>()) for the variant `v`, at the default residency of its
 * kernels: 4 CTAs per SM with the local approximation (trace_grid), else 6. */
template <class F> static auto with_variant(const Variant & v, F && f)
{
        if (v.stack_shape) return f(VariantOf<false, false, tb::SHAPE_STACK, 6>());
        if (v.lla && v.proj) return f(VariantOf<true, true, tb::SHAPE_GENERIC, 4>());
        if (v.lla) return f(VariantOf<true, false, tb::SHAPE_GENERIC, 4>());
        if (v.proj) return f(VariantOf<false, true, tb::SHAPE_GENERIC, 6>());
        return f(VariantOf<false, false, tb::SHAPE_GENERIC, 6>());
}

/* Grid of the persistent kernel: a multiple of the SM count. With the local approximation
 * the lane store of a CTA grows by the state of the transforms the geometry uses, and the
 * CTAs per SM are what fits the 227 kB of shared memory (4 for one projected transform). */
static int trace_grid(const struct turtle_plan * plan, size_t n, int * blocks, int * threads)
{
        *threads = (plan->threads > 0) ? round_up(plan->threads, 32) : 128;
        if (*threads > 128) *threads = 128; /* __launch_bounds__(128, .) */
        int per_sm = (plan->ctas_per_sm > 0) ? plan->ctas_per_sm : 6;
        if (plan->G.range > 0.) {
                const size_t cta = sizeof(LaneStoreT<N_F_LLA, N_I>) + lla_bytes(plan) + 1024;
                const int fit = (int)((227 * 1024) / cta);
                if (per_sm > fit) per_sm = (fit > 0) ? fit : 1;
                if (per_sm > 4) per_sm = 4; /* the register budget these kernels are built for */
        }
        long long want = (long long)plan->sm_count * per_sm;
        const long long need = (long long)((n + *threads - 1) / *threads);
        if (need < want) want = (need > 0) ? need : 1;
        *blocks = (int)want;
        return per_sm;
}

static enum turtle_return check_rule(turtle_function_t * fn, const struct turtle_trace_rule * rule)
{
        if ((rule == NULL) || !(rule->max_steps > 0) || isnan(rule->altitude_max) ||
            isnan(rule->altitude_min) || isnan(rule->length_max))
                return tbh::raise(fn, TURTLE_RETURN_DOMAIN_ERROR, BATCH_CU, __LINE__,
                    "invalid trace rule");
        return TURTLE_RETURN_SUCCESS;
}

/* Launch one instance of the trace kernel. The shared-memory carve-out is asked to be
 * just what the resident CTAs need: whatever they leave of the 256 kB is L1 for the DEM
 * gathers (the default heuristic takes the next larger configuration). */
template <bool LLA, bool PROJ, int MINB, int SHAPE, bool STREAM = false, bool COMPACT = false,
    int GATHER = GATHER_GLOBAL>
static void trace_start(const struct turtle_plan * plan, int per_sm, int blocks, int threads,
    cudaStream_t stream, const TraceArgs & A, const typename ExtraOf<COMPACT, GATHER>::type & C)
{
        void (*kernel)(const tb::Geometry, const TraceArgs,
            const typename ExtraOf<COMPACT, GATHER>::type) =
            trace_kernel<LLA, PROJ, MINB, SHAPE, STREAM, COMPACT, GATHER>;
        const size_t dynamic = LLA ? lla_bytes(plan) : 0;
        static int carveout_of[16] = { 0 };
        static size_t dynamic_of[16] = { 0 };
        const int key = per_sm & 15;
        if ((carveout_of[key] == 0) || (dynamic_of[key] != dynamic)) {
                cudaFuncAttributes attr;
                if (cudaFuncGetAttributes(&attr, kernel) == cudaSuccess) {
                        const size_t need = (size_t)per_sm * (attr.sharedSizeBytes + dynamic + 1024);
                        int percent = (int)((need * 100 + 228 * 1024 - 1) / (228 * 1024));
                        if (percent > 100) percent = 100;
                        carveout_of[key] = percent + 1;
                } else {
                        carveout_of[key] = 101;
                }
                dynamic_of[key] = dynamic;
                cudaGetLastError();
        }
        if (dynamic > 0)
                cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                    (int)dynamic);
        cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
            carveout_of[key] - 1);
        if (GATHER == GATHER_PACKED) { /* the tile table of the cell-packed copies */
                tb::Geometry G = plan->G;
                G.tiles = plan->d_tiles_packed;
                kernel<<<blocks, threads, dynamic, stream>>>(G, A, C);
                return;
        }
        kernel<<<blocks, threads, dynamic, stream>>>(plan->G, A, C);
}

/* Device-pointer calls are asynchronous: up to DEV_SLOTS of them may be in flight on a
 * plan (on different streams -- how a caller backfills the tail of one batch with the
 * head of the next). Each takes a slot of the ring -- counter block (the queue cursor of its
 * kernel), schedule buffers, fan / azimuth tables -- that no call in flight holds: the first
 * one after the latest slot whose event (release_device_slot) has completed, so that calls
 * made one after the other go round the ring. Calls may complete in any order (a long call
 * on one stream, short ones on another): when every slot is held, the host waits for the
 * call that took its slot first. The slot is *slot on return, and the caller must release
 * it on its stream once it has queued the call's last operation, also when that failed. */
static cudaError_t next_device_slot(struct turtle_plan * plan, int * slot)
{
        int s = -1, oldest = -1;
        for (int k = 1; (k <= DEV_SLOTS) && (s < 0); k++) {
                const int t = (plan->dev_slot - N_SLOTS + k) % DEV_SLOTS;
                if (plan->slot_done[t] == NULL) {
                        const cudaError_t err = cudaEventCreateWithFlags(&plan->slot_done[t],
                            cudaEventDisableTiming);
                        if (err != cudaSuccess) return err;
                        s = t;
                        break;
                }
                const cudaError_t q = cudaEventQuery(plan->slot_done[t]);
                if (q == cudaSuccess) {
                        s = t;
                } else if (q == cudaErrorNotReady) {
                        cudaGetLastError(); /* still in flight: not an error of this call */
                        if ((oldest < 0) || (plan->slot_call[t] < plan->slot_call[oldest]))
                                oldest = t;
                } else {
                        return q;
                }
        }
        if (s < 0) {
                const cudaError_t err = cudaEventSynchronize(plan->slot_done[oldest]);
                if (err != cudaSuccess) return err;
                s = oldest;
        }
        plan->slot_call[s] = ++plan->dev_calls;
        plan->dev_slot = N_SLOTS + s;
        *slot = N_SLOTS + s;
        return cudaSuccess;
}

/* The slot is free again once `stream` has done what is queued on it so far. `err`: the
 * status of the call, returned unless it is a success. */
static cudaError_t release_device_slot(struct turtle_plan * plan, int slot, cudaStream_t stream,
    cudaError_t err)
{
        const cudaError_t rec = cudaEventRecord(plan->slot_done[slot - N_SLOTS], stream);
        return (err != cudaSuccess) ? err : rec;
}

/* The frame of a device-pointer call: on the plan's device, the counters reset to a call of
 * `rays` rays (unless `reset` is false: a walk keeps them), a slot of the ring taken,
 * body(slot) queued on `stream`, and the slot released with the body's status. */
template <class Body>
static enum turtle_return device_call(turtle_function_t * fn, struct turtle_plan * plan,
    bool reset, size_t rays, cudaStream_t stream, Body && body)
{
        CUDA_TRY(fn, cudaSetDevice(plan->device));
        if (reset) {
                memset(&plan->counters, 0x0, sizeof(plan->counters));
                plan->counters.rays = rays;
        }
        int slot;
        CUDA_TRY(fn, next_device_slot(plan, &slot));
        CUDA_TRY(fn, release_device_slot(plan, slot, stream, body(slot)));
        return TURTLE_RETURN_SUCCESS;
}

/* Device state of a streamed call: [0] watermark, then one counter per chunk. */
struct StreamState {
        int chunk_shift;
        const unsigned long long * watermark;
        unsigned * chunk_done;
        unsigned * chunk_flags;
};

/* What one launch reads and writes: DEVICE memory throughout. */
struct DeviceIo {
        const double * position;  /* with `direction`, or both NULL: a fan */
        const double * direction;
        const FanTables * fan;
        struct turtle_trace_result * results; /* or NULL */
        const struct turtle_trace_fields * fields; /* or NULL */
};

static cudaError_t launch_trace(struct turtle_plan * plan, int slot, size_t n,
    const DeviceIo & io, const struct turtle_trace_rule * rule,
    unsigned long long * d_counters, cudaStream_t stream, const StreamState * streamed = NULL,
    turtle_trace_crossing * d_crossings = NULL, int max_crossings = 0)
{
        cudaError_t err = cudaMemsetAsync(d_counters, 0x0, CTR * sizeof(unsigned long long), stream);
        if (err != cudaSuccess) return err;
        TraceArgs A;
        memset(&A, 0x0, sizeof A);
        A.n = n;
        A.chunk_shift = (streamed != NULL) ? streamed->chunk_shift : 0;
        A.watermark = (streamed != NULL) ? streamed->watermark : NULL;
        A.chunk_done = (streamed != NULL) ? streamed->chunk_done : NULL;
        A.chunk_flags = (streamed != NULL) ? streamed->chunk_flags : NULL;
        A.crossings = d_crossings;
        A.max_crossings = max_crossings;
        A.order = NULL;
        if ((streamed == NULL) && (io.fan == NULL))
                err = schedule_rays(plan, slot, n, io.position, io.direction, stream, &A.order);
        if (err != cudaSuccess) return err;
        A.position = io.position;
        A.direction = io.direction;
        CompactArgs C;
        memset(&C, 0x0, sizeof C);
        const NoCompactArgs none = { 0 };
        if (io.fan != NULL) {
                A.position = A.direction = NULL;
                C.fan = *io.fan;
        }
        A.results = io.results;
        C.use_fields = (io.fields != NULL);
        if (io.fields != NULL) C.fields = *io.fields;
        A.cursor = d_counters;
        A.altitude_min = rule->altitude_min;
        A.altitude_max = rule->altitude_max;
        A.length_max = rule->length_max;
        A.max_steps = rule->max_steps;
        int blocks, threads;
        const int per_sm = trace_grid(plan, n, &blocks, &threads);
        const Variant v = variant_of(plan);
        const bool compact = (io.fan != NULL) || (io.fields != NULL);
        /* the register budget of a resident kernel without the local approximation follows the
         * requested residency (in units of 128 threads) */
        const int minb = per_sm * threads / 128;
        if (compact || (streamed != NULL) || v.lla) {
                /* fan input and / or field outputs (the COMPACT kernels), streamed calls (the
                 * kernels waiting for their rays) and the local approximation: the default
                 * residency of the variant */
                const int sm6 = (per_sm < 6) ? per_sm : 6;
                if (blocks > plan->sm_count * sm6) blocks = plan->sm_count * sm6;
                with_variant(v, [&](auto V) {
                        typedef decltype(V) K;
                        if (compact && (streamed != NULL))
                                trace_start<K::LLA, K::PROJ, K::MINB, K::SHAPE, true, true>(
                                    plan, sm6, blocks, threads, stream, A, C);
                        else if (compact)
                                trace_start<K::LLA, K::PROJ, K::MINB, K::SHAPE, false, true>(
                                    plan, sm6, blocks, threads, stream, A, C);
                        else if (streamed != NULL)
                                trace_start<K::LLA, K::PROJ, K::MINB, K::SHAPE, true>(
                                    plan, sm6, blocks, threads, stream, A, none);
                        else
                                trace_start<K::LLA, K::PROJ, K::MINB, K::SHAPE>(
                                    plan, sm6, blocks, threads, stream, A, none);
                });
        } else if (v.stack_shape) {
                if ((minb <= 6) && (plan->gather == GATHER_PACKED))
                        trace_start<false, false, 6, tb::SHAPE_STACK, false, false, GATHER_PACKED>(
                            plan, per_sm, blocks, threads, stream, A, none);
                else if ((minb <= 6) && (plan->gather == GATHER_WINDOW)) {
                        WindowArgs W = plan->window;
                        W.hits = d_counters;
                        trace_start<false, false, 6, tb::SHAPE_STACK, false, false, GATHER_WINDOW>(
                            plan, per_sm, blocks, threads, stream, A, W);
                } else if (minb <= 6)
                        trace_start<false, false, 6, tb::SHAPE_STACK>(plan, per_sm, blocks, threads, stream, A, none);
                else
                        trace_start<false, false, 8, tb::SHAPE_STACK>(plan, per_sm, blocks, threads, stream, A, none);
        } else if (minb <= 4) {
                if (v.proj)
                        trace_start<false, true, 4, tb::SHAPE_GENERIC>(plan, per_sm, blocks, threads, stream, A, none);
                else
                        trace_start<false, false, 4, tb::SHAPE_GENERIC>(plan, per_sm, blocks, threads, stream, A, none);
        } else if (minb == 5) {
                if (v.proj)
                        trace_start<false, true, 5, tb::SHAPE_GENERIC>(plan, per_sm, blocks, threads, stream, A, none);
                else
                        trace_start<false, false, 5, tb::SHAPE_GENERIC>(plan, per_sm, blocks, threads, stream, A, none);
        } else if (minb <= 7) {
                if (v.proj)
                        trace_start<false, true, 6, tb::SHAPE_GENERIC>(plan, per_sm, blocks, threads, stream, A, none);
                else
                        trace_start<false, false, 6, tb::SHAPE_GENERIC>(plan, per_sm, blocks, threads, stream, A, none);
        } else if (v.proj) {
                trace_start<false, true, 8, tb::SHAPE_GENERIC>(plan, per_sm, blocks, threads, stream, A, none);
        } else {
                trace_start<false, false, 8, tb::SHAPE_GENERIC>(plan, per_sm, blocks, threads, stream, A, none);
        }
        plan->counters.launches++;
        return cudaGetLastError();
}

extern "C" enum turtle_return turtle_stepper_trace_batch_device(
    struct turtle_plan * plan, size_t n, const double * position,
    const double * direction, const struct turtle_trace_rule * rule,
    struct turtle_trace_result * results, void * stream)
{
        turtle_function_t * fn = FN(&turtle_stepper_trace_batch_device);
        enum turtle_return rc = check_rule(fn, rule);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        if (n == 0) return TURTLE_RETURN_SUCCESS;
        const DeviceIo io = { position, direction, NULL, results, NULL };
        return device_call(fn, plan, true, n, (cudaStream_t)stream, [&](int slot) {
                return launch_trace(plan, slot, n, io, rule, plan->d_counters + CTR * slot,
                    (cudaStream_t)stream);
        });
}

extern "C" enum turtle_return turtle_stepper_trace_crossings_device(
    struct turtle_plan * plan, size_t n, const double * position,
    const double * direction, const struct turtle_trace_rule * rule,
    struct turtle_trace_result * results, struct turtle_trace_crossing * crossings,
    int max_crossings, void * stream)
{
        turtle_function_t * fn = FN(&turtle_stepper_trace_crossings_device);
        enum turtle_return rc = check_rule(fn, rule);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        if ((max_crossings < 0) || ((max_crossings > 0) && (crossings == NULL)))
                return tbh::raise(fn, TURTLE_RETURN_DOMAIN_ERROR, BATCH_CU, __LINE__,
                    "invalid crossings buffer");
        if (n == 0) return TURTLE_RETURN_SUCCESS;
        const DeviceIo io = { position, direction, NULL, results, NULL };
        return device_call(fn, plan, true, n, (cudaStream_t)stream, [&](int slot) {
                return launch_trace(plan, slot, n, io, rule, plan->d_counters + CTR * slot,
                    (cudaStream_t)stream, NULL, (max_crossings > 0) ? crossings : NULL,
                    max_crossings);
        });
}

/* Lazily create the streams and staging buffers of the host-pointer pipeline. */
static cudaError_t plan_pipeline(struct turtle_plan * plan, size_t rays)
{
        cudaError_t err = cudaSuccess;
        for (int s = 0; (s < N_SLOTS) && (err == cudaSuccess); s++) {
                if (plan->stream[s] == NULL) {
                        err = cudaStreamCreateWithFlags(&plan->stream[s], cudaStreamNonBlocking);
                        if (err == cudaSuccess) err = cudaEventCreate(&plan->ev0[s]);
                        if (err == cudaSuccess) err = cudaEventCreate(&plan->ev1[s]);
                }
        }
        if (err != cudaSuccess) return err;
        Staging buffers[2 * N_SLOTS];
        for (int s = 0; s < N_SLOTS; s++) {
                buffers[2 * s] = { (void **)&plan->d_in[s], rays * 6 * sizeof(double) };
                buffers[2 * s + 1] = { (void **)&plan->d_out[s], rays * sizeof(turtle_trace_result) };
        }
        return grow(&plan->slot_rays, rays, buffers);
}

/* Adds the steps, samples and rebuilds of the k <= HOST_SLICES counter blocks from block
 * `first`, whose launches are over, to `to`; c (or NULL): every counter summed over the k
 * blocks. */
static cudaError_t add_counters(const struct turtle_plan * plan, int first, int k,
    turtle_plan_counters & to, unsigned long long * c = NULL)
{
        unsigned long long blocks[HOST_SLICES][CTR], sum[CTR] = { 0 };
        const cudaError_t err = cudaMemcpy(blocks, plan->d_counters + CTR * first,
            k * sizeof blocks[0], cudaMemcpyDeviceToHost);
        if (err != cudaSuccess) return err;
        for (int b = 0; b < k; b++)
                for (int j = 0; j < CTR; j++) sum[j] += blocks[b][j];
        to.steps += sum[1];
        to.samples += sum[2];
        to.rebuilds += sum[4];
        if (c != NULL) memcpy(c, sum, sizeof sum);
        return cudaSuccess;
}

/* The step / sample counters of the launch that used counter block `slot`, once it is over. */
static void read_counters(struct turtle_plan * plan, int slot)
{
        turtle_plan_counters read = plan->counters;
        read.steps = read.samples = read.rebuilds = 0;
        unsigned long long c[CTR];
        if (add_counters(plan, slot, 1, read, c) != cudaSuccess) return;
        read.window_hits = c[5];
        if (c[6] != 0ull) read.rays = c[6]; /* the probes of a horizon search */
        plan->counters = read;
}

extern "C" void turtle_plan_counters_sync(struct turtle_plan * plan)
{
        /* device-pointer calls: the caller has synchronised its stream */
        cudaSetDevice(plan->device);
        read_counters(plan, plan->dev_slot);
}

/* ---- fans and field arrays ------------------------------------------------------------- */

static enum turtle_return check_fan(turtle_function_t * fn, const struct turtle_fan * fan,
    size_t * n, size_t * bundle)
{
        if ((fan == NULL) || ((fan->n_azimuth > 0) && (fan->azimuth == NULL)) ||
            ((fan->n_elevation > 0) && (fan->elevation == NULL)))
                return tbh::raise(fn, TURTLE_RETURN_BAD_ADDRESS, BATCH_CU, __LINE__,
                    "missing fan angles");
        *bundle = (fan->bundle > 0) ? fan->bundle : 1;
        if ((fan->n_elevation % *bundle) != 0)
                return tbh::raise(fn, TURTLE_RETURN_DOMAIN_ERROR, BATCH_CU, __LINE__,
                    "the number of elevations of a fan (%zu) must be a multiple of its bundle (%zu)",
                    fan->n_elevation, *bundle);
        *n = fan->n_azimuth * fan->n_elevation;
        return TURTLE_RETURN_SUCCESS;
}

static enum turtle_return check_fans(turtle_function_t * fn, const struct turtle_fans * fans,
    size_t * n, size_t * bundle)
{
        if ((fans == NULL) || ((fans->n_azimuth > 0) && (fans->azimuth == NULL)) ||
            ((fans->n_elevation > 0) && (fans->elevation == NULL)))
                return tbh::raise(fn, TURTLE_RETURN_BAD_ADDRESS, BATCH_CU, __LINE__,
                    "missing fan angles");
        if ((fans->n_station > 0) && ((fans->latitude == NULL) || (fans->longitude == NULL) ||
                                         (fans->position == NULL)))
                return tbh::raise(fn, TURTLE_RETURN_BAD_ADDRESS, BATCH_CU, __LINE__,
                    "missing station latitudes, longitudes or positions");
        *bundle = (fans->bundle > 0) ? fans->bundle : 1;
        if ((fans->n_elevation % *bundle) != 0)
                return tbh::raise(fn, TURTLE_RETURN_DOMAIN_ERROR, BATCH_CU, __LINE__,
                    "the number of elevations of a fan (%zu) must be a multiple of its bundle (%zu)",
                    fans->n_elevation, *bundle);
        *n = fans->n_station * fans->n_azimuth * fans->n_elevation;
        return TURTLE_RETURN_SUCCESS;
}

/* A fan as the one-station case of struct turtle_fans. */
static struct turtle_fans one_station(const struct turtle_fan * fan)
{
        struct turtle_fans fans;
        fans.n_station = 1;
        fans.latitude = &fan->latitude;
        fans.longitude = &fan->longitude;
        fans.position = fan->position;
        fans.n_azimuth = fan->n_azimuth;
        fans.n_elevation = fan->n_elevation;
        fans.azimuth = fan->azimuth;
        fans.elevation = fan->elevation;
        fans.bundle = fan->bundle;
        return fans;
}

/* The East / North / Up vectors at (latitude, longitude) (compute_enu, ecef.c:136-158):
 * f[3..5], f[6..8], f[9..11]. */
static void enu_frame(double latitude, double longitude, double f[12])
{
        const double lambda = longitude * M_PI / 180.;
        const double phi = latitude * M_PI / 180.;
        const double sl = sin(lambda), cl = cos(lambda), sp = sin(phi), cp = cos(phi);
        const double e[3] = { -sl, cl, 0. }, nn[3] = { -cl * sp, -sl * sp, cp };
        const double u[3] = { cl * cp, sl * cp, sp };
        for (int c = 0; c < 3; c++) {
                f[3 + c] = e[c];
                f[6 + c] = nn[c];
                f[9 + c] = u[c];
        }
}

/* Sines and cosines of the angles of the fans, taken on the host by the calls of
 * turtle_ecef_from_horizontal (ecef.c:139-144,170-173), then the origin and the East / North
 * / Up frame of every station (enu_frame), 12 doubles each; ONE table per slot, queued for
 * upload on `stream`. */
static cudaError_t fan_upload(struct turtle_plan * plan, int slot, const struct turtle_fans * fans,
    size_t bundle, size_t ray0, cudaStream_t stream, FanTables * T)
{
        const size_t angles = fans->n_azimuth + fans->n_elevation;
        const size_t entries = angles + 6 * fans->n_station; /* in double2 */
        const cudaError_t err = grow(&plan->fan_entries[slot], entries,
            { { (void **)&plan->h_fan[slot], entries * sizeof(double2), cudaHostAllocDefault },
                { (void **)&plan->d_fan[slot], entries * sizeof(double2) } });
        if (err != cudaSuccess) return err;
        double2 * h = plan->h_fan[slot];
        for (size_t i = 0; i < fans->n_azimuth; i++) {
                const double az = fans->azimuth[i] * M_PI / 180.;
                h[i].x = sin(az);
                h[i].y = cos(az);
        }
        for (size_t j = 0; j < fans->n_elevation; j++) {
                const double el = fans->elevation[j] * M_PI / 180.;
                h[fans->n_azimuth + j].x = cos(el);
                h[fans->n_azimuth + j].y = sin(el);
        }
        double * station = (double *)(h + angles);
        for (size_t s = 0; s < fans->n_station; s++) {
                double * f = station + 12 * s;
                enu_frame(fans->latitude[s], fans->longitude[s], f);
                for (int c = 0; c < 3; c++) f[c] = fans->position[3 * s + c];
        }
        T->az = plan->d_fan[slot];
        T->el = plan->d_fan[slot] + fans->n_azimuth;
        T->station = (const double *)(plan->d_fan[slot] + angles);
        T->naz = fans->n_azimuth;
        T->bundle = bundle;
        T->per_station = fans->n_azimuth * fans->n_elevation;
        T->ray0 = ray0;
        return cudaMemcpyAsync(plan->d_fan[slot], h, entries * sizeof(double2),
            cudaMemcpyHostToDevice, stream);
}

/* The field arrays of a call, one after the other. */
struct FieldSpec {
        size_t offset; /* of the array's pointer in struct turtle_trace_fields */
        size_t bytes;  /* per ray */
};

static int field_specs(const struct turtle_trace_fields * f, FieldSpec specs[12])
{
        int k = 0;
#define FIELD(member, size)                                                          \
        if (f->member != NULL) {                                                     \
                specs[k].offset = (size_t)((const char *)&f->member - (const char *)f); \
                specs[k].bytes = (size);                                             \
                k++;                                                                 \
        }
        FIELD(length[0], 8) FIELD(length[1], 8) FIELD(length[2], 8) FIELD(length[3], 8)
        FIELD(total, 8) FIELD(altitude, 8) FIELD(position, 24) FIELD(n_steps, 4)
        FIELD(status, 4) FIELD(index, 8) FIELD(medium_hash, 4) FIELD(n_changes, 4)
#undef FIELD
        return k;
}

/* The array of `spec` in `f`, and setting it (the members are pointers of several types). */
static char * field_array(const struct turtle_trace_fields & f, const FieldSpec & spec)
{
        char * p;
        memcpy(&p, (const char *)&f + spec.offset, sizeof p);
        return p;
}
static void set_field_array(struct turtle_trace_fields & f, const FieldSpec & spec, char * p)
{
        memcpy((char *)&f + spec.offset, &p, sizeof p);
}

/* The arrays of `f` from ray `first` on. */
static struct turtle_trace_fields offset_fields(struct turtle_trace_fields f, size_t first)
{
        FieldSpec specs[12];
        const int k = field_specs(&f, specs);
        for (int i = 0; i < k; i++)
                set_field_array(f, specs[i], field_array(f, specs[i]) + first * specs[i].bytes);
        return f;
}

/* Device staging of the field arrays of a host-pointer call of n rays, carved from the plan's
 * field pool, each on a 256-byte boundary: *d_fields has an array where `fields` (or NULL) has
 * one, *n_fields of them. */
static cudaError_t stage_fields(struct turtle_plan * plan, size_t n,
    const struct turtle_trace_fields * fields, struct turtle_trace_fields * d_fields, int * n_fields)
{
        memset(d_fields, 0x0, sizeof *d_fields);
        FieldSpec specs[12];
        *n_fields = (fields != NULL) ? field_specs(fields, specs) : 0;
        size_t need = 0;
        for (int k = 0; k < *n_fields; k++) need += (n * specs[k].bytes + 255) / 256 * 256;
        const cudaError_t err = grow(&plan->field_pool_bytes, need, { { &plan->d_field_pool, need } });
        if (err != cudaSuccess) return err;
        size_t at = 0;
        for (int k = 0; k < *n_fields; k++) {
                set_field_array(*d_fields, specs[k], (char *)plan->d_field_pool + at);
                at += (n * specs[k].bytes + 255) / 256 * 256;
        }
        return cudaSuccess;
}

/* Queue on `stream` the copy of rays [first, first + m) of a host-pointer call from the plan's
 * staging (plan->d_all_out, the fields of stage_fields) to the caller's `results` and `fields`
 * (either NULL). */
static cudaError_t copy_out(const struct turtle_plan * plan, size_t first, size_t m,
    struct turtle_trace_result * results, const struct turtle_trace_fields * fields,
    const struct turtle_trace_fields & d_fields, cudaStream_t stream)
{
        cudaError_t err = cudaSuccess;
        if (results != NULL)
                err = cudaMemcpyAsync(results + first, plan->d_all_out + first,
                    m * sizeof(turtle_trace_result), cudaMemcpyDeviceToHost, stream);
        if (fields == NULL) return err;
        FieldSpec specs[12];
        const int k = field_specs(fields, specs);
        const struct turtle_trace_fields dst = offset_fields(*fields, first);
        const struct turtle_trace_fields src = offset_fields(d_fields, first);
        for (int f = 0; (f < k) && (err == cudaSuccess); f++)
                err = cudaMemcpyAsync(field_array(dst, specs[f]), field_array(src, specs[f]),
                    m * specs[f].bytes, cudaMemcpyDeviceToHost, stream);
        return err;
}

/* Host-pointer call, streamed: ONE persistent trace kernel over all the rays while the
 * copy engines feed and drain it.
 *   stream 1 (H2D): for each chunk, positions and directions, then the new watermark
 *                   (an 8-byte copy, ordered after the data of the chunk);
 *   stream 0      : the trace kernel -- a lane that holds ticket q waits until the
 *                   watermark has passed q (MODE_WAIT), and every finished ray is counted
 *                   for its chunk after a __threadfence;
 *   drain streams : the lane that counts the last ray of a chunk raises the chunk's flag in
 *                   mapped host memory; the calling thread watches the flags and queues the
 *                   copy of each chunk's records and / or field slices as it completes.
 * Compared with one kernel per chunk there is a single kernel tail instead of one per
 * chunk, and no lane ever idles between chunks. The call adds its counts to the plan's
 * counters. */
static enum turtle_return trace_streamed(turtle_function_t * fn, struct turtle_plan * plan,
    size_t n, const double * position, const double * direction,
    const struct turtle_trace_rule * rule, struct turtle_trace_result * results,
    const struct turtle_trace_fields * fields)
{
        const size_t chunk = STREAM_CHUNK_RAYS;
        const size_t n_chunks = (n + chunk - 1) / chunk;
        CUDA_TRY(fn, plan_pipeline(plan, 1)); /* the three streams and their events */
        if (plan->ev_reset == NULL) CUDA_TRY(fn, cudaEventCreate(&plan->ev_reset));
        CUDA_TRY(fn, grow(&plan->all_rays, n,
                         { { (void **)&plan->d_all_in, (n * 6 + 32) * sizeof(double) } }));
        if (results != NULL)
                CUDA_TRY(fn, grow(&plan->all_records, n,
                                 { { (void **)&plan->d_all_out, n * sizeof(turtle_trace_result) } }));
        struct turtle_trace_fields d_fields;
        int n_fields;
        CUDA_TRY(fn, stage_fields(plan, n, fields, &d_fields, &n_fields));
        CUDA_TRY(fn, grow(&plan->stream_chunks, n_chunks,
                         { { (void **)&plan->d_stream_state, (n_chunks + 2) * sizeof(unsigned long long) },
                             { (void **)&plan->h_marks, (n_chunks + 1) * sizeof(unsigned long long),
                                 cudaHostAllocDefault },
                             { (void **)&plan->h_flags, n_chunks * sizeof(unsigned), cudaHostAllocMapped } }));
        cudaStream_t compute = plan->stream[0], h2d = plan->stream[1];
        for (int j = 0; j < N_DRAINS; j++)
                if (plan->drain[j] == NULL)
                        CUDA_TRY(fn, cudaStreamCreateWithFlags(&plan->drain[j], cudaStreamNonBlocking));
        /* both arrays start on a 256-byte boundary and a chunk is a multiple of 128 bytes:
         * no cache line holds rays of two chunks */
        double * d_pos = plan->d_all_in;
        double * d_dir = plan->d_all_in + (3 * n + 31) / 32 * 32;
        StreamState st;
        st.chunk_shift = STREAM_CHUNK_SHIFT;
        st.watermark = plan->d_stream_state;
        st.chunk_done = (unsigned *)(plan->d_stream_state + 1);
        CUDA_TRY(fn, cudaHostGetDevicePointer((void **)&st.chunk_flags, plan->h_flags, 0));
        for (size_t k = 0; k < n_chunks; k++) plan->h_flags[k] = 0u;

        /* reset the stream state; queue the copies in; THEN start the kernel, which waits
         * for its rays. (This order also holds when kernel launches are made synchronous --
         * a profiler, CUDA_LAUNCH_BLOCKING --: the copies are already on their way.) */
        CUDA_TRY(fn, cudaMemsetAsync(plan->d_stream_state, 0x0,
                         (n_chunks + 2) * sizeof(unsigned long long), compute));
        CUDA_TRY(fn, cudaEventRecord(plan->ev_reset, compute));
        CUDA_TRY(fn, cudaStreamWaitEvent(h2d, plan->ev_reset, 0));
        cudaError_t err = cudaSuccess;
        for (size_t k = 0; (k < n_chunks) && (err == cudaSuccess); k++) {
                const size_t i0 = k * chunk;
                const size_t m = std::min(chunk, n - i0);
                plan->h_marks[k] = i0 + m;
                err = cudaMemcpyAsync(d_pos + 3 * i0, position + 3 * i0, m * 3 * sizeof(double),
                    cudaMemcpyHostToDevice, h2d);
                if (err == cudaSuccess)
                        err = cudaMemcpyAsync(d_dir + 3 * i0, direction + 3 * i0,
                            m * 3 * sizeof(double), cudaMemcpyHostToDevice, h2d);
                if (err == cudaSuccess)
                        err = cudaMemcpyAsync(plan->d_stream_state, &plan->h_marks[k],
                            sizeof(unsigned long long), cudaMemcpyHostToDevice, h2d);
        }
        if (err != cudaSuccess) { /* nothing waits yet */
                cudaDeviceSynchronize();
                return tbh::raise(fn, TURTLE_RETURN_LIBRARY_ERROR, BATCH_CU, __LINE__,
                    "CUDA error in the streamed trace: %s", cudaGetErrorString(err));
        }
        CUDA_TRY(fn, cudaEventRecord(plan->ev0[0], compute));
        const DeviceIo io = { d_pos, d_dir, NULL, (results != NULL) ? plan->d_all_out : NULL,
                (n_fields > 0) ? &d_fields : NULL };
        err = launch_trace(plan, 0, n, io, rule, plan->d_counters, compute, &st);
        if (err == cudaSuccess) err = cudaEventRecord(plan->ev1[0], compute);
        /* Drain the chunks in the order they COMPLETE (a chunk waits for its longest ray:
         * the first chunks of a batch sorted longest-first complete late): the thread that
         * counts the last ray of a chunk raises its flag in mapped host memory, this thread
         * watches the flags and queues the copies, round robin on N_DRAINS streams. */
        std::vector<char> drained(n_chunks, 0);
        size_t remaining = n_chunks;
        bool kernel_over = false;
        while ((remaining > 0) && (err == cudaSuccess)) {
                bool progress = false;
                for (size_t k = 0; (k < n_chunks) && (err == cudaSuccess); k++) {
                        if (drained[k]) continue;
                        if (!kernel_over && (*(volatile unsigned *)(plan->h_flags + k) == 0u))
                                continue;
                        const size_t i0 = k * chunk;
                        err = copy_out(plan, i0, std::min(chunk, n - i0), results, fields, d_fields,
                            plan->drain[(n_chunks - remaining) % N_DRAINS]);
                        drained[k] = 1;
                        remaining--;
                        progress = true;
                }
                if (!progress && !kernel_over) {
                        /* a finished kernel has completed every chunk (or timed out, which
                         * is reported below): whatever is left is copied at once */
                        const cudaError_t q = cudaStreamQuery(compute);
                        if (q == cudaSuccess)
                                kernel_over = true;
                        else if (q != cudaErrorNotReady)
                                err = q;
                }
        }
        if (err != cudaSuccess) { /* wake every waiting lane up, drain, then report */
                plan->h_marks[n_chunks] = STREAM_ABORT;
                cudaStreamSynchronize(h2d);
                cudaMemcpyAsync(plan->d_stream_state, &plan->h_marks[n_chunks],
                    sizeof(unsigned long long), cudaMemcpyHostToDevice, h2d);
                cudaDeviceSynchronize();
                return tbh::raise(fn, TURTLE_RETURN_LIBRARY_ERROR, BATCH_CU, __LINE__,
                    "CUDA error in the streamed trace: %s", cudaGetErrorString(err));
        }
        CUDA_TRY(fn, cudaStreamSynchronize(h2d));
        CUDA_TRY(fn, cudaStreamSynchronize(compute));
        for (int j = 0; j < N_DRAINS; j++) CUDA_TRY(fn, cudaStreamSynchronize(plan->drain[j]));
        float ms = 0.f;
        cudaEventElapsedTime(&ms, plan->ev0[0], plan->ev1[0]);
        unsigned long long c[CTR];
        CUDA_TRY(fn, add_counters(plan, 0, 1, plan->counters, c));
        plan->counters.rays += n;
        plan->counters.kernel_ms += ms;
        plan->counters.launches += 1;
        if (c[3] != 0ull)
                return tbh::raise(fn, TURTLE_RETURN_LIBRARY_ERROR, BATCH_CU, __LINE__,
                    "the streamed trace timed out waiting for its rays to reach the device");
        return TURTLE_RETURN_SUCCESS;
}

/* A host-pointer call in rounds of at most STREAM_MAX_RAYS rays, which bounds the device
 * staging of a call whatever the size of the batch. The caller has reset the counters. */
static enum turtle_return trace_rounds(turtle_function_t * fn, struct turtle_plan * plan,
    size_t n, const double * position, const double * direction,
    const struct turtle_trace_rule * rule, struct turtle_trace_result * results,
    const struct turtle_trace_fields * fields)
{
        size_t round_rays = STREAM_MAX_RAYS;
        if (getenv("TURTLE_B200_STREAM_MAX_RAYS") != NULL) { /* tests: small rounds */
                const long long v = atoll(getenv("TURTLE_B200_STREAM_MAX_RAYS"));
                if (v >= (long long)STREAM_CHUNK_RAYS) round_rays = (size_t)v;
        }
        for (size_t first = 0; first < n; first += round_rays) {
                const struct turtle_trace_fields part =
                    (fields != NULL) ? offset_fields(*fields, first) : turtle_trace_fields();
                const enum turtle_return rc = trace_streamed(fn, plan, std::min(round_rays, n - first),
                    position + 3 * first, direction + 3 * first, rule,
                    (results != NULL) ? results + first : NULL, (fields != NULL) ? &part : NULL);
                if (rc != TURTLE_RETURN_SUCCESS) return rc;
        }
        return TURTLE_RETURN_SUCCESS;
}

/* Host-pointer fan: nothing per ray goes in, so there is nothing to stream IN -- the fan is
 * cut in up to 8 slices of consecutive rays (in ray order: station by station, the lowest
 * elevation bands, i.e. the longest rays, first; a slice is made of whole bands and may
 * begin within a station), each a RESIDENT compact kernel followed by the copy of its records / field
 * slices to the host, alternating on two streams: the copy of a slice runs under the
 * kernel of the next, and the SMs that the tail of one slice leaves idle are taken by the
 * head of the next (concurrent launches on one plan). Only the copy
 * of the last slice is exposed. (The streamed kernel -- chunk flags, fences, a lane-side
 * watermark -- does the same at 5 % more kernel time; it stays the path of calls that
 * must stream rays in.) The call adds its counts to the plan's counters, which the caller
 * has reset. */
static enum turtle_return trace_fan_sliced(turtle_function_t * fn, struct turtle_plan * plan,
    size_t n, const struct turtle_fans * fan, size_t bundle, const struct turtle_trace_rule * rule,
    struct turtle_trace_result * results, const struct turtle_trace_fields * fields)
{
        CUDA_TRY(fn, cudaSetDevice(plan->device));
        CUDA_TRY(fn, plan_pipeline(plan, 1)); /* the streams and their events */
        if (results != NULL)
                CUDA_TRY(fn, grow(&plan->all_records, n,
                                 { { (void **)&plan->d_all_out, n * sizeof(turtle_trace_result) } }));
        struct turtle_trace_fields d_fields;
        int n_fields;
        CUDA_TRY(fn, stage_fields(plan, n, fields, &d_fields, &n_fields));
        /* slices: whole bands of the fan (bundle x n_azimuth rays), about 2 Mi rays each */
        const size_t band = std::max<size_t>(bundle * fan->n_azimuth, 1);
        size_t slice_rays = (size_t)1 << 21;
        if (getenv("TURTLE_B200_FAN_SLICE_RAYS") != NULL) { /* tests: several small slices */
                const long long v = atoll(getenv("TURTLE_B200_FAN_SLICE_RAYS"));
                if (v > 0) slice_rays = (size_t)v;
        }
        size_t n_slices = std::min<size_t>(DEV_SLOTS, std::max<size_t>(1, n / slice_rays));
        size_t per_slice = (n / band + n_slices - 1) / n_slices * band;
        if (per_slice == 0) per_slice = n;
        n_slices = (n + per_slice - 1) / per_slice;
        cudaStream_t lanes[2] = { plan->stream[0], plan->stream[1] };
        FanTables tables;
        CUDA_TRY(fn, fan_upload(plan, 0, fan, bundle, 0, lanes[0], &tables));
        CUDA_TRY(fn, cudaEventRecord(plan->ev0[0], lanes[0]));
        CUDA_TRY(fn, cudaStreamWaitEvent(lanes[1], plan->ev0[0], 0));
        /* a host-pointer call: counter blocks of its own, none of the device-pointer ring */
        unsigned long long * d_counters = plan->d_counters + CTR * ALL_SLOTS;
        for (size_t k = 0; k < n_slices; k++) {
                const size_t first = k * per_slice;
                const size_t m = std::min(per_slice, n - first);
                cudaStream_t st = lanes[k & 1];
                FanTables slice = tables;
                slice.ray0 = first;
                const struct turtle_trace_fields slice_fields = offset_fields(d_fields, first);
                const DeviceIo io = { NULL, NULL, &slice,
                        (results != NULL) ? plan->d_all_out + first : NULL,
                        (n_fields > 0) ? &slice_fields : NULL };
                CUDA_TRY(fn, launch_trace(plan, 0, m, io, rule, d_counters + CTR * k, st));
                CUDA_TRY(fn, copy_out(plan, first, m, results, fields, d_fields, st));
        }
        CUDA_TRY(fn, cudaEventRecord(plan->ev1[0], lanes[0]));
        CUDA_TRY(fn, cudaEventRecord(plan->ev1[1], lanes[1]));
        CUDA_TRY(fn, cudaStreamSynchronize(lanes[0]));
        CUDA_TRY(fn, cudaStreamSynchronize(lanes[1]));
        float ms = 0.f, ms1 = 0.f; /* kernels + copies of both streams */
        cudaEventElapsedTime(&ms, plan->ev0[0], plan->ev1[0]);
        cudaEventElapsedTime(&ms1, plan->ev0[0], plan->ev1[1]);
        if (ms1 > ms) ms = ms1;
        CUDA_TRY(fn, add_counters(plan, ALL_SLOTS, (int)n_slices, plan->counters));
        plan->counters.rays = n;
        plan->counters.kernel_ms = ms;
        return TURTLE_RETURN_SUCCESS;
}

/* A device and a plan, for entry points that check their arguments before either is used. */
static enum turtle_return check_plan(turtle_function_t * fn, const struct turtle_plan * plan)
{
        const enum turtle_return rc = require_device(fn, (plan != NULL) ? plan->device : 0);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        if (plan == NULL)
                return tbh::raise(fn, TURTLE_RETURN_BAD_ADDRESS, BATCH_CU, __LINE__, "missing plan");
        return TURTLE_RETURN_SUCCESS;
}

/* The n > 0 rays of checked fans, device-pointer results: ONE launch, asynchronous. */
static enum turtle_return trace_fans_device(turtle_function_t * fn, struct turtle_plan * plan,
    const struct turtle_fans * fans, size_t n, size_t bundle, const struct turtle_trace_rule * rule,
    struct turtle_trace_result * results, const struct turtle_trace_fields * fields, void * stream)
{
        return device_call(fn, plan, true, n, (cudaStream_t)stream, [&](int slot) {
                FanTables tables;
                cudaError_t err = fan_upload(plan, slot, fans, bundle, 0, (cudaStream_t)stream, &tables);
                const DeviceIo io = { NULL, NULL, &tables, results, fields };
                if (err == cudaSuccess)
                        err = launch_trace(plan, slot, n, io, rule, plan->d_counters + CTR * slot,
                            (cudaStream_t)stream);
                return err;
        });
}

extern "C" enum turtle_return turtle_stepper_trace_fan(struct turtle_plan * plan,
    const struct turtle_fan * fan, const struct turtle_trace_rule * rule,
    struct turtle_trace_result * results, const struct turtle_trace_fields * fields)
{
        turtle_function_t * fn = FN(&turtle_stepper_trace_fan);
        enum turtle_return rc = check_rule(fn, rule);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        size_t n, bundle;
        rc = check_fan(fn, fan, &n, &bundle);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        memset(&plan->counters, 0x0, sizeof(plan->counters));
        if (n == 0) return TURTLE_RETURN_SUCCESS;
        const struct turtle_fans fans = one_station(fan);
        return trace_fan_sliced(fn, plan, n, &fans, bundle, rule, results, fields);
}

extern "C" enum turtle_return turtle_stepper_trace_fan_device(struct turtle_plan * plan,
    const struct turtle_fan * fan, const struct turtle_trace_rule * rule,
    struct turtle_trace_result * results, const struct turtle_trace_fields * fields,
    void * stream)
{
        turtle_function_t * fn = FN(&turtle_stepper_trace_fan_device);
        enum turtle_return rc = check_rule(fn, rule);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        size_t n, bundle;
        rc = check_fan(fn, fan, &n, &bundle);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        if (n == 0) return TURTLE_RETURN_SUCCESS;
        const struct turtle_fans fans = one_station(fan);
        return trace_fans_device(fn, plan, &fans, n, bundle, rule, results, fields, stream);
}

extern "C" enum turtle_return turtle_stepper_trace_fans(struct turtle_plan * plan,
    const struct turtle_fans * fans, const struct turtle_trace_rule * rule,
    struct turtle_trace_result * results, const struct turtle_trace_fields * fields)
{
        turtle_function_t * fn = FN(&turtle_stepper_trace_fans);
        enum turtle_return rc = check_rule(fn, rule);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        size_t n, bundle;
        rc = check_fans(fn, fans, &n, &bundle);
        if ((rc != TURTLE_RETURN_SUCCESS) || (n == 0)) return rc;
        rc = check_plan(fn, plan);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        memset(&plan->counters, 0x0, sizeof(plan->counters));
        return trace_fan_sliced(fn, plan, n, fans, bundle, rule, results, fields);
}

extern "C" enum turtle_return turtle_stepper_trace_fans_device(struct turtle_plan * plan,
    const struct turtle_fans * fans, const struct turtle_trace_rule * rule,
    struct turtle_trace_result * results, const struct turtle_trace_fields * fields,
    void * stream)
{
        turtle_function_t * fn = FN(&turtle_stepper_trace_fans_device);
        enum turtle_return rc = check_rule(fn, rule);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        size_t n, bundle;
        rc = check_fans(fn, fans, &n, &bundle);
        if ((rc != TURTLE_RETURN_SUCCESS) || (n == 0)) return rc;
        rc = check_plan(fn, plan);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        return trace_fans_device(fn, plan, fans, n, bundle, rule, results, fields, stream);
}

extern "C" enum turtle_return turtle_stepper_trace_fields(struct turtle_plan * plan, size_t n,
    const double * position, const double * direction, const struct turtle_trace_rule * rule,
    const struct turtle_trace_fields * fields)
{
        turtle_function_t * fn = FN(&turtle_stepper_trace_fields);
        enum turtle_return rc = check_rule(fn, rule);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        memset(&plan->counters, 0x0, sizeof(plan->counters));
        if (n == 0) return TURTLE_RETURN_SUCCESS;
        CUDA_TRY(fn, cudaSetDevice(plan->device));
        return trace_rounds(fn, plan, n, position, direction, rule, NULL, fields);
}

extern "C" enum turtle_return turtle_stepper_trace_fields_device(struct turtle_plan * plan,
    size_t n, const double * position, const double * direction,
    const struct turtle_trace_rule * rule, const struct turtle_trace_fields * fields,
    void * stream)
{
        turtle_function_t * fn = FN(&turtle_stepper_trace_fields_device);
        enum turtle_return rc = check_rule(fn, rule);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        if (n == 0) return TURTLE_RETURN_SUCCESS;
        const DeviceIo io = { position, direction, NULL, NULL, fields };
        return device_call(fn, plan, true, n, (cudaStream_t)stream, [&](int slot) {
                return launch_trace(plan, slot, n, io, rule, plan->d_counters + CTR * slot,
                    (cudaStream_t)stream);
        });
}

/* ---- the horizon of a station ---------------------------------------------------------- */

/* Arguments first (no plan, no device needed), then the device, then the plan. */
static enum turtle_return check_horizon(turtle_function_t * fn, const struct turtle_plan * plan,
    size_t n_station, const double * latitude, const double * longitude, const double * position,
    size_t n_azimuth, const double * azimuth, double elevation_min, double elevation_max,
    double tolerance, const struct turtle_trace_rule * rule, const struct turtle_horizon * results)
{
        if ((n_station > 0) && ((latitude == NULL) || (longitude == NULL) || (position == NULL) ||
                                   ((n_azimuth > 0) && ((azimuth == NULL) || (results == NULL)))))
                return tbh::raise(fn, TURTLE_RETURN_BAD_ADDRESS, BATCH_CU, __LINE__,
                    "missing station position, azimuths or results");
        if (!(tolerance > 0.))
                return tbh::raise(fn, TURTLE_RETURN_DOMAIN_ERROR, BATCH_CU, __LINE__,
                    "invalid tolerance %g (must be > 0)", tolerance);
        if (!(elevation_min >= -90.) || !(elevation_max <= 90.) || !(elevation_min < elevation_max))
                return tbh::raise(fn, TURTLE_RETURN_DOMAIN_ERROR, BATCH_CU, __LINE__,
                    "invalid elevation window [%g, %g] (must be an interval of [-90, 90])",
                    elevation_min, elevation_max);
        enum turtle_return rc = check_rule(fn, rule);
        if ((rc != TURTLE_RETURN_SUCCESS) || (n_station * n_azimuth == 0)) return rc;
        return check_plan(fn, plan);
}

/* Queue the search on `stream`: azimuth and station tables (fan_upload), counters, kernel;
 * with the counter block and tables of `slot`. One work item per station and azimuth. */
static cudaError_t launch_horizon(struct turtle_plan * plan, int slot, size_t n_station,
    const double * latitude, const double * longitude, const double * position, size_t n_azimuth,
    const double * azimuth, double elevation_min, double elevation_max, double tolerance,
    const struct turtle_trace_rule * rule, struct turtle_horizon * results, cudaStream_t stream)
{
        unsigned long long * d_counters = plan->d_counters + CTR * slot;
        struct turtle_fans fans;
        memset(&fans, 0x0, sizeof fans);
        fans.n_station = n_station;
        fans.latitude = latitude;
        fans.longitude = longitude;
        fans.position = position;
        fans.n_azimuth = n_azimuth;
        fans.azimuth = azimuth;
        FanTables T;
        cudaError_t err = fan_upload(plan, slot, &fans, 1, 0, stream, &T);
        if (err == cudaSuccess)
                err = cudaMemsetAsync(d_counters, 0x0, CTR * sizeof(unsigned long long), stream);
        if (err != cudaSuccess) return err;
        const size_t items = n_station * n_azimuth;
        HorizonArgs A;
        memset(&A, 0x0, sizeof A);
        A.az = T.az;
        A.station = T.station;
        A.n = items;
        A.n_azimuth = n_azimuth;
        A.elevation_min = elevation_min;
        A.elevation_max = elevation_max;
        A.tolerance = tolerance;
        A.altitude_min = rule->altitude_min;
        A.altitude_max = rule->altitude_max;
        A.length_max = rule->length_max;
        A.max_steps = rule->max_steps;
        A.results = results;
        A.cursor = d_counters;
        /* one azimuth per warp: the grid of the trace kernels, without the warps that would
         * find no azimuth */
        int blocks, threads;
        const int per_sm = trace_grid(plan, 0, &blocks, &threads);
        const size_t warps = (size_t)threads / 32;
        blocks = (int)std::min<size_t>((size_t)plan->sm_count * per_sm, (items + warps - 1) / warps);
        const Variant v = variant_of(plan);
        void (*kernel)(const tb::Geometry, const HorizonArgs) = with_variant(v, [](auto V) {
                typedef decltype(V) K;
                return horizon_kernel<K::LLA, K::PROJ, K::MINB, K::SHAPE>;
        });
        const size_t dynamic = v.lla ? lla_bytes(plan) : 0;
        if (dynamic > 0)
                cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dynamic);
        kernel<<<blocks, threads, dynamic, stream>>>(plan->G, A);
        plan->counters.launches++;
        return cudaGetLastError();
}

/* Checked arguments, items > 0: device-pointer results, asynchronous. */
static enum turtle_return horizons_device(turtle_function_t * fn, struct turtle_plan * plan,
    size_t n_station, const double * latitude, const double * longitude, const double * position,
    size_t n_azimuth, const double * azimuth, double elevation_min, double elevation_max,
    double tolerance, const struct turtle_trace_rule * rule, struct turtle_horizon * results,
    void * stream)
{
        /* the counters report the probes, read back by turtle_plan_counters_sync */
        return device_call(fn, plan, true, 0, (cudaStream_t)stream, [&](int slot) {
                return launch_horizon(plan, slot, n_station, latitude, longitude, position,
                    n_azimuth, azimuth, elevation_min, elevation_max, tolerance, rule, results,
                    (cudaStream_t)stream);
        });
}

/* Checked arguments, items > 0: host-pointer results. */
static enum turtle_return horizons_host(turtle_function_t * fn, struct turtle_plan * plan,
    size_t n_station, const double * latitude, const double * longitude, const double * position,
    size_t n_azimuth, const double * azimuth, double elevation_min, double elevation_max,
    double tolerance, const struct turtle_trace_rule * rule, struct turtle_horizon * results)
{
        CUDA_TRY(fn, cudaSetDevice(plan->device));
        DeviceBuffers buf;
        struct turtle_horizon * d_results;
        const size_t bytes = n_station * n_azimuth * sizeof(*d_results);
        CUDA_TRY(fn, buf.get((void **)&d_results, NULL, bytes, false));
        /* a host-pointer call: the counter block and tables of the host pipeline's slot 0 */
        memset(&plan->counters, 0x0, sizeof(plan->counters));
        CUDA_TRY(fn, launch_horizon(plan, 0, n_station, latitude, longitude, position, n_azimuth,
                         azimuth, elevation_min, elevation_max, tolerance, rule, d_results, NULL));
        CUDA_TRY(fn, cudaMemcpy(results, d_results, bytes, cudaMemcpyDeviceToHost));
        read_counters(plan, 0);
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_stepper_horizon_device(struct turtle_plan * plan,
    double latitude, double longitude, const double position[3], size_t n_azimuth,
    const double * azimuth, double elevation_min, double elevation_max, double tolerance,
    const struct turtle_trace_rule * rule, struct turtle_horizon * results, void * stream)
{
        turtle_function_t * fn = FN(&turtle_stepper_horizon_device);
        enum turtle_return rc = check_horizon(fn, plan, 1, &latitude, &longitude, position,
            n_azimuth, azimuth, elevation_min, elevation_max, tolerance, rule, results);
        if ((rc != TURTLE_RETURN_SUCCESS) || (n_azimuth == 0)) return rc;
        return horizons_device(fn, plan, 1, &latitude, &longitude, position, n_azimuth, azimuth,
            elevation_min, elevation_max, tolerance, rule, results, stream);
}

extern "C" enum turtle_return turtle_stepper_horizon(struct turtle_plan * plan,
    double latitude, double longitude, const double position[3], size_t n_azimuth,
    const double * azimuth, double elevation_min, double elevation_max, double tolerance,
    const struct turtle_trace_rule * rule, struct turtle_horizon * results)
{
        turtle_function_t * fn = FN(&turtle_stepper_horizon);
        enum turtle_return rc = check_horizon(fn, plan, 1, &latitude, &longitude, position,
            n_azimuth, azimuth, elevation_min, elevation_max, tolerance, rule, results);
        if ((rc != TURTLE_RETURN_SUCCESS) || (n_azimuth == 0)) return rc;
        return horizons_host(fn, plan, 1, &latitude, &longitude, position, n_azimuth, azimuth,
            elevation_min, elevation_max, tolerance, rule, results);
}

extern "C" enum turtle_return turtle_stepper_horizons_device(struct turtle_plan * plan,
    size_t n_station, const double * latitude, const double * longitude, const double * position,
    size_t n_azimuth, const double * azimuth, double elevation_min, double elevation_max,
    double tolerance, const struct turtle_trace_rule * rule, struct turtle_horizon * results,
    void * stream)
{
        turtle_function_t * fn = FN(&turtle_stepper_horizons_device);
        enum turtle_return rc = check_horizon(fn, plan, n_station, latitude, longitude, position,
            n_azimuth, azimuth, elevation_min, elevation_max, tolerance, rule, results);
        if ((rc != TURTLE_RETURN_SUCCESS) || (n_station * n_azimuth == 0)) return rc;
        return horizons_device(fn, plan, n_station, latitude, longitude, position, n_azimuth,
            azimuth, elevation_min, elevation_max, tolerance, rule, results, stream);
}

extern "C" enum turtle_return turtle_stepper_horizons(struct turtle_plan * plan,
    size_t n_station, const double * latitude, const double * longitude, const double * position,
    size_t n_azimuth, const double * azimuth, double elevation_min, double elevation_max,
    double tolerance, const struct turtle_trace_rule * rule, struct turtle_horizon * results)
{
        turtle_function_t * fn = FN(&turtle_stepper_horizons);
        enum turtle_return rc = check_horizon(fn, plan, n_station, latitude, longitude, position,
            n_azimuth, azimuth, elevation_min, elevation_max, tolerance, rule, results);
        if ((rc != TURTLE_RETURN_SUCCESS) || (n_station * n_azimuth == 0)) return rc;
        return horizons_host(fn, plan, n_station, latitude, longitude, position, n_azimuth,
            azimuth, elevation_min, elevation_max, tolerance, rule, results);
}
extern "C" enum turtle_return turtle_stepper_trace_batch(
    struct turtle_plan * plan, size_t n, const double * position,
    const double * direction, const struct turtle_trace_rule * rule,
    struct turtle_trace_result * results)
{
        enum turtle_return rc = check_rule(FN(&turtle_stepper_trace_batch), rule);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        memset(&plan->counters, 0x0, sizeof(plan->counters));
        if (n == 0) return TURTLE_RETURN_SUCCESS;
        CUDA_TRY(&turtle_stepper_trace_batch, cudaSetDevice(plan->device));
        /* more than one chunk, caller's ray order: stream the batch through one kernel --
         * in rounds of at most STREAM_MAX_RAYS rays, which bounds the device staging of a
         * call (144 bytes per ray) to 4.6 GB whatever the size of the batch */
        if ((plan->schedule == 0) && (plan->pipeline_mode != 1) && (n > STREAM_CHUNK_RAYS))
                return trace_rounds(FN(&turtle_stepper_trace_batch), plan, n, position, direction,
                    rule, results, NULL);
        const size_t chunk = std::min(n, CHUNK_RAYS);
        CUDA_TRY(&turtle_stepper_trace_batch, plan_pipeline(plan, chunk));

        /* chunked 3-deep pipeline: H2D(c+1) | kernel(c) | D2H(c-1) on 3 streams */
        const size_t n_chunks = (n + chunk - 1) / chunk;
        double kernel_ms = 0.;
        for (size_t c = 0; c < n_chunks + N_SLOTS; c++) {
                const int s = (int)(c % N_SLOTS);
                if (c >= N_SLOTS) { /* drain the slot before reusing it */
                        CUDA_TRY(&turtle_stepper_trace_batch, cudaStreamSynchronize(plan->stream[s]));
                        float ms = 0.f;
                        cudaEventElapsedTime(&ms, plan->ev0[s], plan->ev1[s]);
                        kernel_ms += ms;
                        CUDA_TRY(&turtle_stepper_trace_batch, add_counters(plan, s, 1, plan->counters));
                }
                if (c >= n_chunks) continue;
                const size_t i0 = c * chunk;
                const size_t m = std::min(chunk, n - i0);
                cudaStream_t st = plan->stream[s];
                double * d_pos = plan->d_in[s];
                double * d_dir = plan->d_in[s] + 3 * chunk;
                CUDA_TRY(&turtle_stepper_trace_batch,
                    cudaMemcpyAsync(d_pos, position + 3 * i0, m * 3 * sizeof(double),
                        cudaMemcpyHostToDevice, st));
                CUDA_TRY(&turtle_stepper_trace_batch,
                    cudaMemcpyAsync(d_dir, direction + 3 * i0, m * 3 * sizeof(double),
                        cudaMemcpyHostToDevice, st));
                CUDA_TRY(&turtle_stepper_trace_batch, cudaEventRecord(plan->ev0[s], st));
                const DeviceIo io = { d_pos, d_dir, NULL, plan->d_out[s], NULL };
                CUDA_TRY(&turtle_stepper_trace_batch,
                    launch_trace(plan, s, m, io, rule, plan->d_counters + CTR * s, st));
                CUDA_TRY(&turtle_stepper_trace_batch, cudaEventRecord(plan->ev1[s], st));
                CUDA_TRY(&turtle_stepper_trace_batch,
                    cudaMemcpyAsync(results + i0, plan->d_out[s],
                        m * sizeof(turtle_trace_result), cudaMemcpyDeviceToHost, st));
        }
        plan->counters.rays = n;
        plan->counters.kernel_ms = kernel_ms;
        return TURTLE_RETURN_SUCCESS;
}

/* ---- particle states and single steps ----------------------------------------- */

extern "C" enum turtle_return turtle_states_create(
    struct turtle_plan * plan, size_t n, struct turtle_states ** states_)
{
        *states_ = NULL;
        CUDA_TRY(&turtle_states_create, cudaSetDevice(plan->device));
        struct turtle_states * states = new (std::nothrow) turtle_states();
        if (states == NULL)
                return tbh::raise(FN(&turtle_states_create), TURTLE_RETURN_MEMORY_ERROR,
                    BATCH_CU, __LINE__, "could not allocate memory");
        states->plan = plan;
        states->device = plan->device;
        states->n = n;
        states->d_states = NULL;
        states->stride = (std::max<size_t>(n, 1) + 31) / 32 * 32;
        const size_t rows = PS_FIELDS + ((plan->G.range > 0.) ? plan->G.lla_rows : 0);
        cudaError_t err = cudaMalloc((void **)&states->d_states,
            states->stride * rows * sizeof(double));
        if (err != cudaSuccess) {
                delete states;
                return tbh::raise(FN(&turtle_states_create), TURTLE_RETURN_MEMORY_ERROR,
                    BATCH_CU, __LINE__, "could not allocate %zu particle states: %s", n,
                    cudaGetErrorString(err));
        }
        *states_ = states;
        return turtle_states_reset(states);
}

extern "C" void turtle_states_destroy(struct turtle_states ** states)
{
        if ((states == NULL) || (*states == NULL)) return;
        cudaSetDevice((*states)->device);
        cudaFree((*states)->d_states);
        delete *states;
        *states = NULL;
}

extern "C" size_t turtle_states_bytes_per_particle(const struct turtle_states * states)
{
        const tb::Geometry & G = states->plan->G;
        return (PS_FIELDS + ((G.range > 0.) ? G.lla_rows : 0)) * sizeof(double);
}

extern "C" enum turtle_return turtle_states_reset(struct turtle_states * states)
{
        CUDA_TRY(&turtle_states_reset, cudaSetDevice(states->plan->device));
        if (states->n == 0) return TURTLE_RETURN_SUCCESS;
        const int blocks = (int)std::min<size_t>((states->n + 255) / 256,
            (size_t)states->plan->sm_count * 8);
        tb::Geometry G = states->plan->G;
        if (!(G.range > 0.)) G.n_transforms = 0; /* no local approximation rows */
        states_reset_kernel<<<blocks, 256>>>(G, states->d_states, states->stride, states->n);
        states->plan->counters.launches++;
        CUDA_TRY(&turtle_states_reset, cudaGetLastError());
        CUDA_TRY(&turtle_states_reset, cudaDeviceSynchronize());
        return TURTLE_RETURN_SUCCESS;
}

/* The states, if any, of a call of n particles on `plan`. */
static enum turtle_return check_states(turtle_function_t * fn, const struct turtle_plan * plan,
    const struct turtle_states * states, size_t n)
{
        if ((states != NULL) && ((states->plan != plan) || (states->n < n)))
                return tbh::raise(fn, TURTLE_RETURN_DOMAIN_ERROR, BATCH_CU, __LINE__,
                    "states do not match the plan or are too few");
        return TURTLE_RETURN_SUCCESS;
}

/* Queue the walk kernel on `stream` with the counter block of `slot`: n particles, n_steps
 * turtle_stepper_step each (1: the step_batch calls, states used in place; > 1:
 * turtle_stepper_walk_batch, state resident in the lane store for the whole launch). */
static cudaError_t launch_walk(struct turtle_plan * plan, int slot, struct turtle_states * states,
    size_t n, int n_steps, bool multi, double * position, const double * direction,
    double * latitude, double * longitude, double * altitude, double * elevation, double * step,
    int * index, cudaStream_t stream)
{
        StepArgs A;
        A.n = n;
        A.states = (states != NULL) ? states->d_states : NULL;
        A.stride = (states != NULL) ? states->stride : 0;
        A.position = position;
        A.direction = direction;
        A.latitude = latitude;
        A.longitude = longitude;
        A.altitude = altitude;
        A.elevation = elevation;
        A.step = step;
        A.index = index;
        A.n_steps = n_steps;
        A.counters = plan->d_counters + CTR * slot;
        const int threads = 128;
        int blocks = (int)std::min<size_t>((n + threads - 1) / threads,
            (size_t)plan->sm_count * 5);
        cudaError_t err = cudaMemsetAsync(A.counters, 0x0, CTR * sizeof(unsigned long long), stream);
        if (err != cudaSuccess) return err;
        Variant v = variant_of(plan);
        v.stack_shape = false; /* no walk kernel for the stack shape: the generic ones */
        void (*kernel)(const tb::Geometry, const StepArgs) = with_variant(v, [&](auto V) {
                typedef decltype(V) K;
                return multi ? walk_kernel<K::LLA, K::PROJ, true, true> :
                    (states != NULL) ? walk_kernel<K::LLA, K::PROJ, true> :
                                       walk_kernel<K::LLA, K::PROJ, false>;
        });
        /* the local approximations live in the device states (one step), else in dynamic
         * shared memory (no states: every particle starts from a reset stepper; several
         * steps: the state moves in and out once) */
        const size_t dynamic = (v.lla && (multi || (states == NULL))) ? lla_bytes(plan) : 0;
        /* the CTAs per SM get the carve-out they need and no more: the rest is L1 for the
         * DEM gathers (as for the trace kernel) */
        cudaFuncAttributes attr;
        if (cudaFuncGetAttributes(&attr, kernel) == cudaSuccess) {
                const size_t cta = attr.sharedSizeBytes + dynamic + 1024;
                int per_sm = (int)((227 * 1024) / cta);
                if (per_sm > 5) per_sm = 5;
                if (per_sm < 1) per_sm = 1;
                blocks = (int)std::min<size_t>((size_t)blocks, (size_t)plan->sm_count * per_sm);
                int percent = (int)((per_sm * cta * 100 + 228 * 1024 - 1) / (228 * 1024));
                if (percent > 100) percent = 100;
                cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, percent);
        }
        if (dynamic > 0)
                cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                    (int)dynamic);
        cudaGetLastError();
        kernel<<<blocks, threads, dynamic, stream>>>(plan->G, A);
        plan->counters.launches++;
        plan->counters.rays = n;
        plan->counters.steps = (direction != NULL) ? n * (size_t)n_steps : 0;
        return cudaGetLastError();
}

extern "C" enum turtle_return turtle_stepper_step_batch_device(
    struct turtle_plan * plan, struct turtle_states * states, size_t n,
    double * position, const double * direction, double * latitude,
    double * longitude, double * altitude, double * elevation, double * step,
    int * index, void * stream)
{
        turtle_function_t * fn = FN(&turtle_stepper_step_batch_device);
        const enum turtle_return rc = check_states(fn, plan, states, n);
        if ((rc != TURTLE_RETURN_SUCCESS) || (n == 0)) return rc;
        /* the counters of a walk are not reset: launch_walk sets its rays and steps */
        return device_call(fn, plan, false, 0, (cudaStream_t)stream, [&](int slot) {
                return launch_walk(plan, slot, states, n, 1, false, position, direction, latitude,
                    longitude, altitude, elevation, step, index, (cudaStream_t)stream);
        });
}

/* n_steps successive turtle_stepper_step per particle in one launch (turtle_b200.h). */
extern "C" enum turtle_return turtle_stepper_walk_batch_device(struct turtle_plan * plan,
    struct turtle_states * states, size_t n, int n_steps, double * position,
    const double * direction, double * latitude, double * longitude, double * altitude,
    double * elevation, double * step, int * index, void * stream)
{
        turtle_function_t * fn = FN(&turtle_stepper_walk_batch_device);
        if ((n_steps < 1) || (direction == NULL))
                return tbh::raise(fn, TURTLE_RETURN_DOMAIN_ERROR, BATCH_CU, __LINE__,
                    "a walk needs at least one step and its directions");
        const enum turtle_return rc = check_states(fn, plan, states, n);
        if ((rc != TURTLE_RETURN_SUCCESS) || (n == 0)) return rc;
        return device_call(fn, plan, false, 0, (cudaStream_t)stream, [&](int slot) {
                return launch_walk(plan, slot, states, n, n_steps, true, position, direction,
                    latitude, longitude, altitude, elevation, step, index, (cudaStream_t)stream);
        });
}

#define DEV_IN(fn, B, dptr, hptr, bytes)                                           \
        CUDA_TRY(fn, B.get((void **)&(dptr), (hptr), (bytes), true))
#define DEV_OUT(fn, B, dptr, hptr, bytes)                                          \
        do {                                                                       \
                (dptr) = NULL;                                                     \
                if ((hptr) != NULL)                                                \
                        CUDA_TRY(fn, B.get((void **)&(dptr), NULL, (bytes), false)); \
        } while (0)
#define DEV_BACK(fn, hptr, dptr, bytes)                                            \
        do {                                                                       \
                if ((hptr) != NULL)                                                \
                        CUDA_TRY(fn, cudaMemcpy((hptr), (dptr), (bytes),           \
                                         cudaMemcpyDeviceToHost));                 \
        } while (0)

/* Host buffers: one resident launch (the crossings are a diagnostic stream, not the
 * throughput path: no chunking). */
extern "C" enum turtle_return turtle_stepper_trace_crossings(
    struct turtle_plan * plan, size_t n, const double * position,
    const double * direction, const struct turtle_trace_rule * rule,
    struct turtle_trace_result * results, struct turtle_trace_crossing * crossings,
    int max_crossings)
{
        turtle_function_t * fn = FN(&turtle_stepper_trace_crossings);
        enum turtle_return rc = check_rule(fn, rule);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        if ((max_crossings < 0) || ((max_crossings > 0) && (crossings == NULL)))
                return tbh::raise(fn, TURTLE_RETURN_DOMAIN_ERROR, BATCH_CU, __LINE__,
                    "invalid crossings buffer");
        if (n == 0) return TURTLE_RETURN_SUCCESS;
        CUDA_TRY(fn, cudaSetDevice(plan->device));
        DeviceBuffers buf;
        double *d_pos, *d_dir;
        turtle_trace_result * d_res;
        turtle_trace_crossing * d_cross;
        const size_t cross_bytes = n * (size_t)max_crossings * sizeof(turtle_trace_crossing);
        CUDA_TRY(fn, buf.get((void **)&d_pos, position, n * 3 * sizeof(double), true));
        CUDA_TRY(fn, buf.get((void **)&d_dir, direction, n * 3 * sizeof(double), true));
        CUDA_TRY(fn, buf.get((void **)&d_res, NULL, n * sizeof(*d_res), false));
        CUDA_TRY(fn, buf.get((void **)&d_cross, NULL, cross_bytes ? cross_bytes : 16, false));
        CUDA_TRY(fn, cudaMemset(d_cross, 0x0, cross_bytes ? cross_bytes : 16));
        /* the counter block and schedule buffers of the host pipeline's slot 0 */
        memset(&plan->counters, 0x0, sizeof(plan->counters));
        plan->counters.rays = n;
        const DeviceIo io = { d_pos, d_dir, NULL, d_res, NULL };
        CUDA_TRY(fn, launch_trace(plan, 0, n, io, rule, plan->d_counters, NULL, NULL,
                         (max_crossings > 0) ? d_cross : NULL, max_crossings));
        CUDA_TRY(fn, cudaDeviceSynchronize());
        read_counters(plan, 0);
        CUDA_TRY(fn, cudaMemcpy(results, d_res, n * sizeof(*d_res), cudaMemcpyDeviceToHost));
        if (cross_bytes)
                CUDA_TRY(fn, cudaMemcpy(crossings, d_cross, cross_bytes, cudaMemcpyDeviceToHost));
        return TURTLE_RETURN_SUCCESS;
}

/* ---- rock length per cell of a voxel grid ------------------------------------------------ */

/* The cells, frame and media of a grid (its address is checked by the caller). */
static enum turtle_return check_voxel_grid(turtle_function_t * fn,
    const struct turtle_voxel_grid * grid)
{
        const int32_t * c = grid->n;
        if ((c[0] <= 0) || (c[1] <= 0) || (c[2] <= 0) ||
            ((long long)c[0] * (long long)c[1] * (long long)c[2] > (long long)INT32_MAX))
                return tbh::raise(fn, TURTLE_RETURN_DOMAIN_ERROR, BATCH_CU, __LINE__,
                    "invalid voxel grid of %d x %d x %d cells (must be > 0, at most %d in all)",
                    c[0], c[1], c[2], INT32_MAX);
        const double * s = grid->size;
        if (!(isfinite(s[0]) && (s[0] > 0.) && isfinite(s[1]) && (s[1] > 0.) && isfinite(s[2]) &&
                (s[2] > 0.)))
                return tbh::raise(fn, TURTLE_RETURN_DOMAIN_ERROR, BATCH_CU, __LINE__,
                    "invalid voxel size %g x %g x %g m (must be finite and > 0)", s[0], s[1], s[2]);
        if (!(isfinite(grid->latitude) && isfinite(grid->longitude) && isfinite(grid->height) &&
                isfinite(grid->corner[0]) && isfinite(grid->corner[1]) && isfinite(grid->corner[2])))
                return tbh::raise(fn, TURTLE_RETURN_DOMAIN_ERROR, BATCH_CU, __LINE__,
                    "invalid voxel grid origin or corner (must be finite)");
        if (grid->media == 0u)
                return tbh::raise(fn, TURTLE_RETURN_DOMAIN_ERROR, BATCH_CU, __LINE__,
                    "invalid voxel media 0 (select at least one medium)");
        return TURTLE_RETURN_SUCCESS;
}

/* Arguments first (no plan, no device needed). `rays`: the position and direction arrays of
 * the explicit form are needed (n > 0, not a fan). */
static enum turtle_return check_voxels(turtle_function_t * fn, size_t n, bool rays,
    const double * position, const double * direction, const struct turtle_trace_rule * rule,
    const struct turtle_voxel_grid * grid, const struct turtle_voxel_entry * entries,
    int capacity, const int32_t * count)
{
        if (grid == NULL)
                return tbh::raise(fn, TURTLE_RETURN_BAD_ADDRESS, BATCH_CU, __LINE__,
                    "missing voxel grid");
        if ((n > 0) && ((rays && ((position == NULL) || (direction == NULL))) || (count == NULL)))
                return tbh::raise(fn, TURTLE_RETURN_BAD_ADDRESS, BATCH_CU, __LINE__,
                    "missing ray positions, directions or counts");
        if ((capacity > 0) && (entries == NULL))
                return tbh::raise(fn, TURTLE_RETURN_BAD_ADDRESS, BATCH_CU, __LINE__,
                    "missing voxel entries (capacity %d)", capacity);
        if (capacity < 0)
                return tbh::raise(fn, TURTLE_RETURN_DOMAIN_ERROR, BATCH_CU, __LINE__,
                    "invalid voxel capacity %d (must be >= 0)", capacity);
        const enum turtle_return rc = check_voxel_grid(fn, grid);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        return check_rule(fn, rule);
}

/* The same for the opacity form: its arrays instead of entries and counts. */
static enum turtle_return check_opacity(turtle_function_t * fn, size_t n, bool rays,
    const double * position, const double * direction, const struct turtle_trace_rule * rule,
    const struct turtle_voxel_grid * grid, const struct turtle_voxel_opacity * opacity)
{
        if (grid == NULL)
                return tbh::raise(fn, TURTLE_RETURN_BAD_ADDRESS, BATCH_CU, __LINE__,
                    "missing voxel grid");
        if (opacity == NULL)
                return tbh::raise(fn, TURTLE_RETURN_BAD_ADDRESS, BATCH_CU, __LINE__,
                    "missing voxel opacity arrays");
        if ((n > 0) && rays && ((position == NULL) || (direction == NULL)))
                return tbh::raise(fn, TURTLE_RETURN_BAD_ADDRESS, BATCH_CU, __LINE__,
                    "missing ray positions or directions");
        if ((opacity->opacity != NULL) && (opacity->density == NULL))
                return tbh::raise(fn, TURTLE_RETURN_BAD_ADDRESS, BATCH_CU, __LINE__,
                    "missing voxel densities (an opacity needs them)");
        if ((opacity->gradient != NULL) && (opacity->weight == NULL))
                return tbh::raise(fn, TURTLE_RETURN_BAD_ADDRESS, BATCH_CU, __LINE__,
                    "missing ray weights (a gradient needs them)");
        const enum turtle_return rc = check_voxel_grid(fn, grid);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        return check_rule(fn, rule);
}

/* Queue the voxel kernel on `stream` with the counter block of `slot`: the rays of
 * `d_position` / `d_direction` (device memory), or of the fan tables `fan`. `opacity` (device
 * arrays) selects the opacity form, which takes no entries or counts. */
static cudaError_t launch_voxels(struct turtle_plan * plan, int slot, size_t n,
    const double * d_position, const double * d_direction, const FanTables * fan,
    const struct turtle_trace_rule * rule, const struct turtle_voxel_grid * grid,
    struct turtle_trace_result * results, struct turtle_voxel_entry * entries, int capacity,
    int32_t * count, const struct turtle_voxel_opacity * opacity, cudaStream_t stream)
{
        unsigned long long * d_counters = plan->d_counters + CTR * slot;
        cudaError_t err = cudaMemsetAsync(d_counters, 0x0, CTR * sizeof(unsigned long long), stream);
        if (err != cudaSuccess) return err;
        VoxelArgs A;
        memset(&A, 0x0, sizeof A);
        A.n = n;
        A.position = d_position;
        A.direction = d_direction;
        if (fan != NULL) {
                A.position = A.direction = NULL;
                A.fan.fan = *fan;
        }
        A.results = results;
        A.entries = entries;
        A.count = count;
        A.capacity = capacity;
        A.media = grid->media;
        A.altitude_min = rule->altitude_min;
        A.altitude_max = rule->altitude_max;
        A.length_max = rule->length_max;
        A.max_steps = rule->max_steps;
        A.cursor = d_counters;
        turtle_ecef_from_geodetic(grid->latitude, grid->longitude, grid->height, A.frame);
        enu_frame(grid->latitude, grid->longitude, A.frame);
        for (int a = 0; a < 3; a++) {
                A.corner[a] = grid->corner[a];
                A.size[a] = grid->size[a];
                A.cells[a] = grid->n[a];
        }
        if (opacity != NULL) {
                A.density = opacity->density;
                A.opacity = opacity->opacity;
                A.outside = opacity->outside;
                A.weight = opacity->weight;
                A.gradient = opacity->gradient;
        }
        const Variant v = variant_of(plan);
        void (*kernel)(const tb::Geometry, const VoxelArgs) = (opacity != NULL) ?
            with_variant(v, [](auto V) {
                    typedef decltype(V) K;
                    return voxel_kernel<K::LLA, K::PROJ, K::MINB, K::SHAPE, true>;
            }) :
            with_variant(v, [](auto V) {
                    typedef decltype(V) K;
                    return voxel_kernel<K::LLA, K::PROJ, K::MINB, K::SHAPE, false>;
            });
        const size_t dynamic = v.lla ? lla_bytes(plan) : 0;
        if (dynamic > 0)
                cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dynamic);
        /* the grid of the trace kernels, at most the CTAs that fit an SM with the rows of the
         * walk next to the lane store */
        int blocks, threads;
        int per_sm = trace_grid(plan, n, &blocks, &threads);
        int fit = 0;
        err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&fit, kernel, threads, dynamic);
        if (err != cudaSuccess) return err;
        if (per_sm > fit) per_sm = (fit > 0) ? fit : 1;
        blocks = std::min(blocks, plan->sm_count * per_sm);
        kernel<<<blocks, threads, dynamic, stream>>>(plan->G, A);
        plan->counters.launches++;
        return cudaGetLastError();
}

/* Checked arguments, n > 0: host memory, results in place on return. `fans` NULL: the rays of
 * position / direction. `opacity` (host arrays): the opacity form, without entries or counts. */
static enum turtle_return voxels_host(turtle_function_t * fn, struct turtle_plan * plan, size_t n,
    const double * position, const double * direction, const struct turtle_fans * fans,
    size_t bundle, const struct turtle_trace_rule * rule, const struct turtle_voxel_grid * grid,
    struct turtle_trace_result * results, struct turtle_voxel_entry * entries, int capacity,
    int32_t * count, const struct turtle_voxel_opacity * opacity = NULL)
{
        CUDA_TRY(fn, cudaSetDevice(plan->device));
        DeviceBuffers buf;
        double *d_pos = NULL, *d_dir = NULL;
        turtle_trace_result * d_res;
        turtle_voxel_entry * d_entries = NULL;
        int32_t * d_count;
        const size_t entry_bytes = n * (size_t)capacity * sizeof(turtle_voxel_entry);
        if (fans == NULL) {
                DEV_IN(fn, buf, d_pos, position, n * 3 * sizeof(double));
                DEV_IN(fn, buf, d_dir, direction, n * 3 * sizeof(double));
        }
        DEV_OUT(fn, buf, d_res, results, n * sizeof(*d_res));
        /* the caller's slots past each count stay as they are: staged in, copied back whole */
        if (capacity > 0) DEV_IN(fn, buf, d_entries, entries, entry_bytes);
        DEV_OUT(fn, buf, d_count, count, n * sizeof(*d_count));
        /* the opacity form: densities and weights in, the gradient in and back (it is added
         * to), opacity and outside out */
        turtle_voxel_opacity D;
        memset(&D, 0x0, sizeof D);
        const size_t cell_bytes = (size_t)grid->n[0] * (size_t)grid->n[1] * (size_t)grid->n[2] *
            sizeof(double);
        if (opacity != NULL) {
                double *d_density = NULL, *d_weight = NULL, *d_gradient = NULL;
                if (opacity->density != NULL) DEV_IN(fn, buf, d_density, opacity->density, cell_bytes);
                if (opacity->weight != NULL) DEV_IN(fn, buf, d_weight, opacity->weight, n * sizeof(double));
                if (opacity->gradient != NULL) DEV_IN(fn, buf, d_gradient, opacity->gradient, cell_bytes);
                DEV_OUT(fn, buf, D.opacity, opacity->opacity, n * sizeof(double));
                DEV_OUT(fn, buf, D.outside, opacity->outside, n * sizeof(double));
                D.density = d_density;
                D.weight = d_weight;
                D.gradient = d_gradient;
        }
        /* a host-pointer call: the counter block and tables of the host pipeline's slot 0 */
        memset(&plan->counters, 0x0, sizeof(plan->counters));
        plan->counters.rays = n;
        FanTables T;
        if (fans != NULL) CUDA_TRY(fn, fan_upload(plan, 0, fans, bundle, 0, NULL, &T));
        CUDA_TRY(fn, launch_voxels(plan, 0, n, d_pos, d_dir, (fans != NULL) ? &T : NULL, rule,
                         grid, d_res, d_entries, capacity, d_count, (opacity != NULL) ? &D : NULL,
                         NULL));
        CUDA_TRY(fn, cudaDeviceSynchronize());
        read_counters(plan, 0);
        DEV_BACK(fn, results, d_res, n * sizeof(*d_res));
        if (capacity > 0) DEV_BACK(fn, entries, d_entries, entry_bytes);
        DEV_BACK(fn, count, d_count, n * sizeof(*d_count));
        if (opacity != NULL) {
                DEV_BACK(fn, opacity->opacity, D.opacity, n * sizeof(double));
                DEV_BACK(fn, opacity->outside, D.outside, n * sizeof(double));
                DEV_BACK(fn, opacity->gradient, D.gradient, cell_bytes);
        }
        return TURTLE_RETURN_SUCCESS;
}

/* Checked arguments, n > 0: device memory, one launch, asynchronous on `stream`. `opacity`
 * (device arrays): the opacity form. */
static enum turtle_return voxels_device(turtle_function_t * fn, struct turtle_plan * plan, size_t n,
    const double * position, const double * direction, const struct turtle_fans * fans,
    size_t bundle, const struct turtle_trace_rule * rule, const struct turtle_voxel_grid * grid,
    struct turtle_trace_result * results, struct turtle_voxel_entry * entries, int capacity,
    int32_t * count, void * stream, const struct turtle_voxel_opacity * opacity = NULL)
{
        return device_call(fn, plan, true, n, (cudaStream_t)stream, [&](int slot) {
                FanTables T;
                cudaError_t err = cudaSuccess;
                if (fans != NULL) err = fan_upload(plan, slot, fans, bundle, 0, (cudaStream_t)stream, &T);
                if (err == cudaSuccess)
                        err = launch_voxels(plan, slot, n, position, direction,
                            (fans != NULL) ? &T : NULL, rule, grid, results, entries, capacity, count,
                            opacity, (cudaStream_t)stream);
                return err;
        });
}

extern "C" enum turtle_return turtle_stepper_trace_voxels(struct turtle_plan * plan, size_t n,
    const double * position, const double * direction, const struct turtle_trace_rule * rule,
    const struct turtle_voxel_grid * grid, struct turtle_trace_result * results,
    struct turtle_voxel_entry * entries, int capacity, int32_t * count)
{
        turtle_function_t * fn = FN(&turtle_stepper_trace_voxels);
        enum turtle_return rc = check_voxels(fn, n, true, position, direction, rule, grid, entries,
            capacity, count);
        if ((rc != TURTLE_RETURN_SUCCESS) || (n == 0)) return rc;
        rc = check_plan(fn, plan);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        return voxels_host(fn, plan, n, position, direction, NULL, 1, rule, grid, results, entries,
            capacity, count);
}

extern "C" enum turtle_return turtle_stepper_trace_voxels_device(struct turtle_plan * plan,
    size_t n, const double * position, const double * direction,
    const struct turtle_trace_rule * rule, const struct turtle_voxel_grid * grid,
    struct turtle_trace_result * results, struct turtle_voxel_entry * entries, int capacity,
    int32_t * count, void * stream)
{
        turtle_function_t * fn = FN(&turtle_stepper_trace_voxels_device);
        enum turtle_return rc = check_voxels(fn, n, true, position, direction, rule, grid, entries,
            capacity, count);
        if ((rc != TURTLE_RETURN_SUCCESS) || (n == 0)) return rc;
        rc = check_plan(fn, plan);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        return voxels_device(fn, plan, n, position, direction, NULL, 1, rule, grid, results,
            entries, capacity, count, stream);
}

extern "C" enum turtle_return turtle_stepper_trace_fans_voxels(struct turtle_plan * plan,
    const struct turtle_fans * fans, const struct turtle_trace_rule * rule,
    const struct turtle_voxel_grid * grid, struct turtle_trace_result * results,
    struct turtle_voxel_entry * entries, int capacity, int32_t * count)
{
        turtle_function_t * fn = FN(&turtle_stepper_trace_fans_voxels);
        size_t n, bundle;
        enum turtle_return rc = check_fans(fn, fans, &n, &bundle);
        if (rc == TURTLE_RETURN_SUCCESS)
                rc = check_voxels(fn, n, false, NULL, NULL, rule, grid, entries, capacity, count);
        if ((rc != TURTLE_RETURN_SUCCESS) || (n == 0)) return rc;
        rc = check_plan(fn, plan);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        return voxels_host(fn, plan, n, NULL, NULL, fans, bundle, rule, grid, results, entries,
            capacity, count);
}

extern "C" enum turtle_return turtle_stepper_trace_fans_voxels_device(struct turtle_plan * plan,
    const struct turtle_fans * fans, const struct turtle_trace_rule * rule,
    const struct turtle_voxel_grid * grid, struct turtle_trace_result * results,
    struct turtle_voxel_entry * entries, int capacity, int32_t * count, void * stream)
{
        turtle_function_t * fn = FN(&turtle_stepper_trace_fans_voxels_device);
        size_t n, bundle;
        enum turtle_return rc = check_fans(fn, fans, &n, &bundle);
        if (rc == TURTLE_RETURN_SUCCESS)
                rc = check_voxels(fn, n, false, NULL, NULL, rule, grid, entries, capacity, count);
        if ((rc != TURTLE_RETURN_SUCCESS) || (n == 0)) return rc;
        rc = check_plan(fn, plan);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        return voxels_device(fn, plan, n, NULL, NULL, fans, bundle, rule, grid, results, entries,
            capacity, count, stream);
}

/* ---- L rho and L^T w over a voxel grid without storing L ------------------------------------ */

extern "C" enum turtle_return turtle_stepper_trace_opacity(struct turtle_plan * plan, size_t n,
    const double * position, const double * direction, const struct turtle_trace_rule * rule,
    const struct turtle_voxel_grid * grid, const struct turtle_voxel_opacity * opacity,
    struct turtle_trace_result * results)
{
        turtle_function_t * fn = FN(&turtle_stepper_trace_opacity);
        enum turtle_return rc = check_opacity(fn, n, true, position, direction, rule, grid, opacity);
        if ((rc != TURTLE_RETURN_SUCCESS) || (n == 0)) return rc;
        rc = check_plan(fn, plan);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        return voxels_host(fn, plan, n, position, direction, NULL, 1, rule, grid, results, NULL, 0,
            NULL, opacity);
}

extern "C" enum turtle_return turtle_stepper_trace_opacity_device(struct turtle_plan * plan,
    size_t n, const double * position, const double * direction,
    const struct turtle_trace_rule * rule, const struct turtle_voxel_grid * grid,
    const struct turtle_voxel_opacity * opacity, struct turtle_trace_result * results,
    void * stream)
{
        turtle_function_t * fn = FN(&turtle_stepper_trace_opacity_device);
        enum turtle_return rc = check_opacity(fn, n, true, position, direction, rule, grid, opacity);
        if ((rc != TURTLE_RETURN_SUCCESS) || (n == 0)) return rc;
        rc = check_plan(fn, plan);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        return voxels_device(fn, plan, n, position, direction, NULL, 1, rule, grid, results, NULL,
            0, NULL, stream, opacity);
}

extern "C" enum turtle_return turtle_stepper_trace_fans_opacity(struct turtle_plan * plan,
    const struct turtle_fans * fans, const struct turtle_trace_rule * rule,
    const struct turtle_voxel_grid * grid, const struct turtle_voxel_opacity * opacity,
    struct turtle_trace_result * results)
{
        turtle_function_t * fn = FN(&turtle_stepper_trace_fans_opacity);
        size_t n, bundle;
        enum turtle_return rc = check_fans(fn, fans, &n, &bundle);
        if (rc == TURTLE_RETURN_SUCCESS)
                rc = check_opacity(fn, n, false, NULL, NULL, rule, grid, opacity);
        if ((rc != TURTLE_RETURN_SUCCESS) || (n == 0)) return rc;
        rc = check_plan(fn, plan);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        return voxels_host(fn, plan, n, NULL, NULL, fans, bundle, rule, grid, results, NULL, 0,
            NULL, opacity);
}

extern "C" enum turtle_return turtle_stepper_trace_fans_opacity_device(struct turtle_plan * plan,
    const struct turtle_fans * fans, const struct turtle_trace_rule * rule,
    const struct turtle_voxel_grid * grid, const struct turtle_voxel_opacity * opacity,
    struct turtle_trace_result * results, void * stream)
{
        turtle_function_t * fn = FN(&turtle_stepper_trace_fans_opacity_device);
        size_t n, bundle;
        enum turtle_return rc = check_fans(fn, fans, &n, &bundle);
        if (rc == TURTLE_RETURN_SUCCESS)
                rc = check_opacity(fn, n, false, NULL, NULL, rule, grid, opacity);
        if ((rc != TURTLE_RETURN_SUCCESS) || (n == 0)) return rc;
        rc = check_plan(fn, plan);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        return voxels_device(fn, plan, n, NULL, NULL, fans, bundle, rule, grid, results, NULL, 0,
            NULL, stream, opacity);
}

extern "C" enum turtle_return turtle_map_resample(struct turtle_map * map,
    struct turtle_plan * plan, int layer, size_t * outside)
{
        turtle_function_t * fn = FN(&turtle_map_resample);
        if (outside != NULL) *outside = 0;
        if ((layer < 0) || (layer >= plan->G.n_layers))
                return tbh::raise(fn, TURTLE_RETURN_DOMAIN_ERROR, BATCH_CU, __LINE__,
                    "invalid layer index");
        CUDA_TRY(fn, cudaSetDevice(plan->device));
        tb::ProjDesc P;
        tbh::projection_to_desc(&map->projection, &P);
        const size_t n = (size_t)map->nx * map->ny;
        DeviceBuffers buf;
        double * d_z;
        int * d_inside;
        CUDA_TRY(fn, buf.get((void **)&d_z, NULL, n * sizeof(double), false));
        CUDA_TRY(fn, buf.get((void **)&d_inside, NULL, n * sizeof(int), false));
        const int blocks = (int)std::min<size_t>((n + 255) / 256, (size_t)plan->sm_count * 8);
        resample_kernel<<<blocks, 256>>>(plan->G, P, map->nx, map->ny, map->x0, map->dx, map->y0,
            map->dy, layer, d_z, d_inside);
        CUDA_TRY(fn, cudaGetLastError());
        std::vector<double> z(n);
        std::vector<int> inside(n);
        CUDA_TRY(fn, cudaMemcpy(z.data(), d_z, n * sizeof(double), cudaMemcpyDeviceToHost));
        CUDA_TRY(fn, cudaMemcpy(inside.data(), d_inside, n * sizeof(int), cudaMemcpyDeviceToHost));
        size_t missing = 0;
        for (int iy = 0; iy < map->ny; iy++)
                for (int ix = 0; ix < map->nx; ix++) {
                        const size_t i = (size_t)iy * map->nx + ix;
                        if (!inside[i]) {
                                missing++;
                                continue;
                        }
                        const enum turtle_return rc = turtle_map_fill(map, ix, iy, z[i]);
                        if (rc != TURTLE_RETURN_SUCCESS) return rc; /* raised by turtle_map_fill */
                }
        if (outside != NULL) *outside = missing;
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_stepper_step_batch(struct turtle_plan * plan,
    struct turtle_states * states, size_t n, double * position,
    const double * direction, double * latitude, double * longitude,
    double * altitude, double * elevation, double * step, int * index)
{
        if (n == 0) return TURTLE_RETURN_SUCCESS;
        const enum turtle_return rc = check_states(FN(&turtle_stepper_step_batch), plan, states, n);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        CUDA_TRY(&turtle_stepper_step_batch, cudaSetDevice(plan->device));
        DeviceBuffers B;
        double *d_pos, *d_dir = NULL, *d_lat, *d_lon, *d_alt, *d_el, *d_step;
        int * d_idx;
        DEV_IN(&turtle_stepper_step_batch, B, d_pos, position, n * 3 * sizeof(double));
        if (direction != NULL)
                DEV_IN(&turtle_stepper_step_batch, B, d_dir, direction, n * 3 * sizeof(double));
        DEV_OUT(&turtle_stepper_step_batch, B, d_lat, latitude, n * sizeof(double));
        DEV_OUT(&turtle_stepper_step_batch, B, d_lon, longitude, n * sizeof(double));
        DEV_OUT(&turtle_stepper_step_batch, B, d_alt, altitude, n * sizeof(double));
        DEV_OUT(&turtle_stepper_step_batch, B, d_el, elevation, n * 2 * sizeof(double));
        DEV_OUT(&turtle_stepper_step_batch, B, d_step, step, n * sizeof(double));
        DEV_OUT(&turtle_stepper_step_batch, B, d_idx, index, n * 2 * sizeof(int));
        CUDA_TRY(&turtle_stepper_step_batch, launch_walk(plan, 0, states, n, 1, false, d_pos,
                                                 d_dir, d_lat, d_lon, d_alt, d_el, d_step, d_idx, NULL));
        CUDA_TRY(&turtle_stepper_step_batch, cudaDeviceSynchronize());
        if (direction != NULL)
                DEV_BACK(&turtle_stepper_step_batch, position, d_pos, n * 3 * sizeof(double));
        DEV_BACK(&turtle_stepper_step_batch, latitude, d_lat, n * sizeof(double));
        DEV_BACK(&turtle_stepper_step_batch, longitude, d_lon, n * sizeof(double));
        DEV_BACK(&turtle_stepper_step_batch, altitude, d_alt, n * sizeof(double));
        DEV_BACK(&turtle_stepper_step_batch, elevation, d_el, n * 2 * sizeof(double));
        DEV_BACK(&turtle_stepper_step_batch, step, d_step, n * sizeof(double));
        DEV_BACK(&turtle_stepper_step_batch, index, d_idx, n * 2 * sizeof(int));
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_stepper_walk_batch(struct turtle_plan * plan,
    struct turtle_states * states, size_t n, int n_steps, double * position,
    const double * direction, double * latitude, double * longitude, double * altitude,
    double * elevation, double * step, int * index)
{
        turtle_function_t * fn = FN(&turtle_stepper_walk_batch);
        if ((n_steps < 1) || (direction == NULL))
                return tbh::raise(fn, TURTLE_RETURN_DOMAIN_ERROR, BATCH_CU, __LINE__,
                    "a walk needs at least one step and its directions");
        if (n == 0) return TURTLE_RETURN_SUCCESS;
        const enum turtle_return rc = check_states(fn, plan, states, n);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        CUDA_TRY(fn, cudaSetDevice(plan->device));
        const size_t m = n * (size_t)n_steps;
        DeviceBuffers B;
        double *d_pos, *d_dir, *d_lat, *d_lon, *d_alt, *d_el, *d_step;
        int * d_idx;
        DEV_IN(fn, B, d_pos, position, n * 3 * sizeof(double));
        DEV_IN(fn, B, d_dir, direction, m * 3 * sizeof(double));
        DEV_OUT(fn, B, d_lat, latitude, m * sizeof(double));
        DEV_OUT(fn, B, d_lon, longitude, m * sizeof(double));
        DEV_OUT(fn, B, d_alt, altitude, m * sizeof(double));
        DEV_OUT(fn, B, d_el, elevation, m * 2 * sizeof(double));
        DEV_OUT(fn, B, d_step, step, m * sizeof(double));
        DEV_OUT(fn, B, d_idx, index, m * 2 * sizeof(int));
        CUDA_TRY(fn, launch_walk(plan, 0, states, n, n_steps, true, d_pos, d_dir, d_lat, d_lon,
                         d_alt, d_el, d_step, d_idx, NULL));
        CUDA_TRY(fn, cudaDeviceSynchronize());
        DEV_BACK(fn, position, d_pos, n * 3 * sizeof(double));
        DEV_BACK(fn, latitude, d_lat, m * sizeof(double));
        DEV_BACK(fn, longitude, d_lon, m * sizeof(double));
        DEV_BACK(fn, altitude, d_alt, m * sizeof(double));
        DEV_BACK(fn, elevation, d_el, m * 2 * sizeof(double));
        DEV_BACK(fn, step, d_step, m * sizeof(double));
        DEV_BACK(fn, index, d_idx, m * 2 * sizeof(int));
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_stepper_position_batch(struct turtle_plan * plan,
    size_t n, const double * latitude, const double * longitude, const double * height,
    int layer_index, double * position, int * data_index)
{
        if ((layer_index < 0) || (layer_index >= plan->G.n_layers))
                return tbh::raise(FN(&turtle_stepper_position_batch), TURTLE_RETURN_DOMAIN_ERROR,
                    "src/turtle/stepper.c", __LINE__, "no valid data");
        if (n == 0) return TURTLE_RETURN_SUCCESS;
        CUDA_TRY(&turtle_stepper_position_batch, cudaSetDevice(plan->device));
        DeviceBuffers B;
        double *d_lat, *d_lon, *d_h, *d_pos;
        int * d_idx;
        DEV_IN(&turtle_stepper_position_batch, B, d_lat, latitude, n * sizeof(double));
        DEV_IN(&turtle_stepper_position_batch, B, d_lon, longitude, n * sizeof(double));
        DEV_IN(&turtle_stepper_position_batch, B, d_h, height, n * sizeof(double));
        DEV_IN(&turtle_stepper_position_batch, B, d_pos, position, n * 3 * sizeof(double));
        DEV_OUT(&turtle_stepper_position_batch, B, d_idx, data_index, n * sizeof(int));
        const int blocks = (int)std::min<size_t>((n + 127) / 128, (size_t)plan->sm_count * 8);
        position_kernel<<<blocks, 128>>>(plan->G, n, d_lat, d_lon, d_h, layer_index, d_pos, d_idx);
        plan->counters.launches++;
        CUDA_TRY(&turtle_stepper_position_batch, cudaGetLastError());
        CUDA_TRY(&turtle_stepper_position_batch, cudaDeviceSynchronize());
        DEV_BACK(&turtle_stepper_position_batch, position, d_pos, n * 3 * sizeof(double));
        DEV_BACK(&turtle_stepper_position_batch, data_index, d_idx, n * sizeof(int));
        return TURTLE_RETURN_SUCCESS;
}

/* ---- frame transforms ----------------------------------------------------------- */

static int stream_blocks(size_t n, int threads)
{
        int device = 0, sms = 148;
        cudaGetDevice(&device);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
        const size_t want = (n + threads - 1) / threads;
        return (int)std::max<size_t>(1, std::min<size_t>(want, (size_t)sms * 16));
}

static enum turtle_return require_current(turtle_function_t * fn)
{
        int device = 0;
        if (turtle_b200_device_count() == 0)
                return require_device(fn, 0);
        cudaGetDevice(&device);
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_ecef_to_geodetic_batch_device(size_t n,
    const double * ecef, double * latitude, double * longitude, double * altitude,
    void * stream)
{
        enum turtle_return rc = require_current(FN(&turtle_ecef_to_geodetic_batch_device));
        if ((rc != TURTLE_RETURN_SUCCESS) || (n == 0)) return rc;
        to_geodetic_kernel<<<stream_blocks(n, 256), 256, 0, (cudaStream_t)stream>>>(
            n, ecef, latitude, longitude, altitude);
        CUDA_TRY(&turtle_ecef_to_geodetic_batch_device, cudaGetLastError());
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_ecef_to_geodetic_batch(size_t n, const double * ecef,
    double * latitude, double * longitude, double * altitude)
{
        enum turtle_return rc = require_current(FN(&turtle_ecef_to_geodetic_batch));
        if ((rc != TURTLE_RETURN_SUCCESS) || (n == 0)) return rc;
        DeviceBuffers B;
        double *d_ecef, *d_lat, *d_lon, *d_alt;
        DEV_IN(&turtle_ecef_to_geodetic_batch, B, d_ecef, ecef, n * 3 * sizeof(double));
        DEV_OUT(&turtle_ecef_to_geodetic_batch, B, d_lat, latitude, n * sizeof(double));
        DEV_OUT(&turtle_ecef_to_geodetic_batch, B, d_lon, longitude, n * sizeof(double));
        DEV_OUT(&turtle_ecef_to_geodetic_batch, B, d_alt, altitude, n * sizeof(double));
        rc = turtle_ecef_to_geodetic_batch_device(n, d_ecef, d_lat, d_lon, d_alt, NULL);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        CUDA_TRY(&turtle_ecef_to_geodetic_batch, cudaDeviceSynchronize());
        DEV_BACK(&turtle_ecef_to_geodetic_batch, latitude, d_lat, n * sizeof(double));
        DEV_BACK(&turtle_ecef_to_geodetic_batch, longitude, d_lon, n * sizeof(double));
        DEV_BACK(&turtle_ecef_to_geodetic_batch, altitude, d_alt, n * sizeof(double));
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_ecef_from_geodetic_batch_device(size_t n,
    const double * latitude, const double * longitude, const double * elevation,
    double * ecef, void * stream)
{
        enum turtle_return rc = require_current(FN(&turtle_ecef_from_geodetic_batch_device));
        if ((rc != TURTLE_RETURN_SUCCESS) || (n == 0)) return rc;
        from_geodetic_kernel<<<stream_blocks(n, 256), 256, 0, (cudaStream_t)stream>>>(
            n, latitude, longitude, elevation, ecef);
        CUDA_TRY(&turtle_ecef_from_geodetic_batch_device, cudaGetLastError());
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_ecef_from_geodetic_batch(size_t n,
    const double * latitude, const double * longitude, const double * elevation,
    double * ecef)
{
        enum turtle_return rc = require_current(FN(&turtle_ecef_from_geodetic_batch));
        if ((rc != TURTLE_RETURN_SUCCESS) || (n == 0)) return rc;
        DeviceBuffers B;
        double *d_lat, *d_lon, *d_el, *d_ecef;
        DEV_IN(&turtle_ecef_from_geodetic_batch, B, d_lat, latitude, n * sizeof(double));
        DEV_IN(&turtle_ecef_from_geodetic_batch, B, d_lon, longitude, n * sizeof(double));
        DEV_IN(&turtle_ecef_from_geodetic_batch, B, d_el, elevation, n * sizeof(double));
        DEV_OUT(&turtle_ecef_from_geodetic_batch, B, d_ecef, ecef, n * 3 * sizeof(double));
        rc = turtle_ecef_from_geodetic_batch_device(n, d_lat, d_lon, d_el, d_ecef, NULL);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        CUDA_TRY(&turtle_ecef_from_geodetic_batch, cudaDeviceSynchronize());
        DEV_BACK(&turtle_ecef_from_geodetic_batch, ecef, d_ecef, n * 3 * sizeof(double));
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_ecef_from_horizontal_batch_device(size_t n,
    const double * latitude, const double * longitude, const double * azimuth,
    const double * elevation, double * direction, void * stream)
{
        enum turtle_return rc = require_current(FN(&turtle_ecef_from_horizontal_batch_device));
        if ((rc != TURTLE_RETURN_SUCCESS) || (n == 0)) return rc;
        from_horizontal_kernel<<<stream_blocks(n, 256), 256, 0, (cudaStream_t)stream>>>(
            n, latitude, longitude, azimuth, elevation, direction);
        CUDA_TRY(&turtle_ecef_from_horizontal_batch_device, cudaGetLastError());
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_ecef_from_horizontal_batch(size_t n,
    const double * latitude, const double * longitude, const double * azimuth,
    const double * elevation, double * direction)
{
        enum turtle_return rc = require_current(FN(&turtle_ecef_from_horizontal_batch));
        if ((rc != TURTLE_RETURN_SUCCESS) || (n == 0)) return rc;
        DeviceBuffers B;
        double *d_lat, *d_lon, *d_az, *d_el, *d_dir;
        DEV_IN(&turtle_ecef_from_horizontal_batch, B, d_lat, latitude, n * sizeof(double));
        DEV_IN(&turtle_ecef_from_horizontal_batch, B, d_lon, longitude, n * sizeof(double));
        DEV_IN(&turtle_ecef_from_horizontal_batch, B, d_az, azimuth, n * sizeof(double));
        DEV_IN(&turtle_ecef_from_horizontal_batch, B, d_el, elevation, n * sizeof(double));
        DEV_OUT(&turtle_ecef_from_horizontal_batch, B, d_dir, direction, n * 3 * sizeof(double));
        rc = turtle_ecef_from_horizontal_batch_device(n, d_lat, d_lon, d_az, d_el, d_dir, NULL);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        CUDA_TRY(&turtle_ecef_from_horizontal_batch, cudaDeviceSynchronize());
        DEV_BACK(&turtle_ecef_from_horizontal_batch, direction, d_dir, n * 3 * sizeof(double));
        return TURTLE_RETURN_SUCCESS;
}

/* ---- projections ------------------------------------------------------------------- */

static enum turtle_return projection_batch(turtle_function_t * fn,
    const struct turtle_projection * projection, int inverse, size_t n, const double * a,
    const double * b, double * c, double * d, bool on_device, void * stream)
{
        if (projection == NULL)
                return tbh::raise(fn, TURTLE_RETURN_BAD_ADDRESS, "src/turtle/projection.c",
                    __LINE__, "missing projection");
        if (projection->type < 0)
                return tbh::raise(fn, TURTLE_RETURN_BAD_PROJECTION, "src/turtle/projection.c",
                    __LINE__, "invalid projection");
        enum turtle_return rc = require_current(fn);
        if ((rc != TURTLE_RETURN_SUCCESS) || (n == 0)) return rc;
        tb::ProjDesc P;
        tbh::projection_to_desc(projection, &P);
        if (on_device) {
                projection_kernel<<<stream_blocks(n, 256), 256, 0, (cudaStream_t)stream>>>(
                    P, inverse, n, a, b, c, d);
                CUDA_TRY(fn, cudaGetLastError());
                return TURTLE_RETURN_SUCCESS;
        }
        DeviceBuffers B;
        double *d_a, *d_b, *d_c, *d_d;
        DEV_IN(fn, B, d_a, a, n * sizeof(double));
        DEV_IN(fn, B, d_b, b, n * sizeof(double));
        DEV_OUT(fn, B, d_c, c, n * sizeof(double));
        DEV_OUT(fn, B, d_d, d, n * sizeof(double));
        projection_kernel<<<stream_blocks(n, 256), 256>>>(P, inverse, n, d_a, d_b, d_c, d_d);
        CUDA_TRY(fn, cudaGetLastError());
        CUDA_TRY(fn, cudaDeviceSynchronize());
        DEV_BACK(fn, c, d_c, n * sizeof(double));
        DEV_BACK(fn, d, d_d, n * sizeof(double));
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_projection_project_batch(
    const struct turtle_projection * projection, size_t n, const double * latitude,
    const double * longitude, double * x, double * y)
{
        return projection_batch(FN(&turtle_projection_project_batch), projection, 0, n, latitude,
            longitude, x, y, false, NULL);
}

extern "C" enum turtle_return turtle_projection_project_batch_device(
    const struct turtle_projection * projection, size_t n, const double * latitude,
    const double * longitude, double * x, double * y, void * stream)
{
        return projection_batch(FN(&turtle_projection_project_batch_device), projection, 0, n,
            latitude, longitude, x, y, true, stream);
}

extern "C" enum turtle_return turtle_projection_unproject_batch(
    const struct turtle_projection * projection, size_t n, const double * x, const double * y,
    double * latitude, double * longitude)
{
        return projection_batch(FN(&turtle_projection_unproject_batch), projection, 1, n, x, y,
            latitude, longitude, false, NULL);
}

extern "C" enum turtle_return turtle_projection_unproject_batch_device(
    const struct turtle_projection * projection, size_t n, const double * x, const double * y,
    double * latitude, double * longitude, void * stream)
{
        return projection_batch(FN(&turtle_projection_unproject_batch_device), projection, 1, n,
            x, y, latitude, longitude, true, stream);
}

/* ---- map mirrors and elevation queries -------------------------------------------- */

static std::mutex g_mirror_mutex;

extern "C" void tb_map_release_mirrors(struct turtle_map * map)
{
        std::lock_guard<std::mutex> guard(g_mirror_mutex);
        int current = 0;
        bool have = !map->mirrors.empty() && (cudaGetDevice(&current) == cudaSuccess);
        for (size_t i = 0; i < map->mirrors.size(); i++) {
                if (map->mirrors[i].nodes == NULL) continue;
                cudaSetDevice(map->mirrors[i].device);
                cudaFree(map->mirrors[i].nodes);
                cudaFree(map->mirrors[i].packed);
        }
        if (have) cudaSetDevice(current);
        map->mirrors.clear();
}

/* Device descriptor of `map` on the current device (uploads when stale). */
static enum turtle_return map_mirror(turtle_function_t * fn, struct turtle_map * map,
    tb::MapDesc * desc, bool packed_ok = false)
{
        enum turtle_return rc = require_current(fn);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        std::lock_guard<std::mutex> guard(g_mirror_mutex);
        int device = 0;
        CUDA_TRY(fn, cudaGetDevice(&device));
        tb_device_mirror * mirror = NULL;
        for (size_t i = 0; i < map->mirrors.size(); i++)
                if (map->mirrors[i].device == device) mirror = &map->mirrors[i];
        if (mirror == NULL) {
                map->mirrors.push_back(tb_device_mirror());
                mirror = &map->mirrors.back();
                mirror->device = device;
        }
        if (mirror->nodes == NULL) {
                const size_t count = padded_nodes(map, &mirror->pitch);
                CUDA_TRY(fn, cudaMalloc((void **)&mirror->nodes, count * sizeof(uint16_t)));
                CUDA_TRY(fn, cudaMemset(mirror->nodes, 0x0, count * sizeof(uint16_t)));
                mirror->version = 0;
        }
        if (mirror->version != map->version) {
                CUDA_TRY(fn, upload_nodes(mirror->nodes, mirror->pitch, map));
                mirror->version = map->version;
        }
        desc->nodes = mirror->nodes;
        if (packed_ok && (map->gather == 1)) { /* the cell-packed copy: one load per query */
                if (mirror->packed == NULL)
                        CUDA_TRY(fn, cudaMalloc(&mirror->packed,
                                         (size_t)mirror->pitch * map->ny * sizeof(uint2)));
                if (mirror->packed_version != map->version) {
                        pack_cells_kernel<<<148 * 8, 256>>>((uint2 *)mirror->packed, mirror->nodes,
                            mirror->pitch, map->nx, map->ny);
                        CUDA_TRY(fn, cudaGetLastError());
                        CUDA_TRY(fn, cudaDeviceSynchronize());
                        mirror->packed_version = map->version;
                }
                desc->nodes = (const uint16_t *)mirror->packed;
        }
        desc->nx = map->nx;
        desc->ny = map->ny;
        desc->pitch = mirror->pitch;
        desc->kind = map->kind;
        desc->x0 = map->x0;
        desc->y0 = map->y0;
        desc->dx = map->dx;
        desc->dy = map->dy;
        desc->z0 = map->z0;
        desc->dz = map->dz;
        tb::map_desc_finish(*desc);
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_map_elevation_batch_device(struct turtle_map * map,
    size_t n, const double * x, const double * y, double * z, int * inside, void * stream)
{
        tb::MapDesc M;
        enum turtle_return rc = map_mirror(FN(&turtle_map_elevation_batch_device), map, &M, true);
        if ((rc != TURTLE_RETURN_SUCCESS) || (n == 0)) return rc;
        if (map->gather == 1)
                map_elevation_kernel<tb::NodesPacked><<<stream_blocks(n, 256), 256, 0,
                    (cudaStream_t)stream>>>(M, n, x, y, z, inside);
        else
                map_elevation_kernel<tb::NodesGlobal><<<stream_blocks(n, 256), 256, 0,
                    (cudaStream_t)stream>>>(M, n, x, y, z, inside);
        CUDA_TRY(&turtle_map_elevation_batch_device, cudaGetLastError());
        return TURTLE_RETURN_SUCCESS;
}

/* 0: the batched elevation queries of `map` gather from its row-major mirror; 1: from a
 * cell-packed second copy (turtle_b200.h). The gradient kernel always uses the first. */
extern "C" void turtle_map_gather_set(struct turtle_map * map, int mode)
{
        map->gather = (mode == 1) ? 1 : 0;
}

extern "C" enum turtle_return turtle_map_elevation_batch(struct turtle_map * map, size_t n,
    const double * x, const double * y, double * z, int * inside)
{
        enum turtle_return rc = require_current(FN(&turtle_map_elevation_batch));
        if ((rc != TURTLE_RETURN_SUCCESS) || (n == 0)) return rc;
        DeviceBuffers B;
        double *d_x, *d_y, *d_z;
        int * d_in;
        DEV_IN(&turtle_map_elevation_batch, B, d_x, x, n * sizeof(double));
        DEV_IN(&turtle_map_elevation_batch, B, d_y, y, n * sizeof(double));
        DEV_IN(&turtle_map_elevation_batch, B, d_z, z, n * sizeof(double));
        DEV_OUT(&turtle_map_elevation_batch, B, d_in, inside, n * sizeof(int));
        rc = turtle_map_elevation_batch_device(map, n, d_x, d_y, d_z, d_in, NULL);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        CUDA_TRY(&turtle_map_elevation_batch, cudaDeviceSynchronize());
        DEV_BACK(&turtle_map_elevation_batch, z, d_z, n * sizeof(double));
        DEV_BACK(&turtle_map_elevation_batch, inside, d_in, n * sizeof(int));
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_map_gradient_batch_device(struct turtle_map * map,
    size_t n, const double * x, const double * y, double * gx, double * gy, int * inside,
    void * stream)
{
        tb::MapDesc M;
        enum turtle_return rc = map_mirror(FN(&turtle_map_gradient_batch_device), map, &M);
        if ((rc != TURTLE_RETURN_SUCCESS) || (n == 0)) return rc;
        map_gradient_kernel<<<stream_blocks(n, 256), 256, 0, (cudaStream_t)stream>>>(
            M, n, x, y, gx, gy, inside);
        CUDA_TRY(&turtle_map_gradient_batch_device, cudaGetLastError());
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_map_gradient_batch(struct turtle_map * map, size_t n,
    const double * x, const double * y, double * gx, double * gy, int * inside)
{
        enum turtle_return rc = require_current(FN(&turtle_map_gradient_batch));
        if ((rc != TURTLE_RETURN_SUCCESS) || (n == 0)) return rc;
        DeviceBuffers B;
        double *d_x, *d_y, *d_gx, *d_gy;
        int * d_in;
        DEV_IN(&turtle_map_gradient_batch, B, d_x, x, n * sizeof(double));
        DEV_IN(&turtle_map_gradient_batch, B, d_y, y, n * sizeof(double));
        DEV_IN(&turtle_map_gradient_batch, B, d_gx, gx, n * sizeof(double));
        DEV_IN(&turtle_map_gradient_batch, B, d_gy, gy, n * sizeof(double));
        DEV_OUT(&turtle_map_gradient_batch, B, d_in, inside, n * sizeof(int));
        rc = turtle_map_gradient_batch_device(map, n, d_x, d_y, d_gx, d_gy, d_in, NULL);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        CUDA_TRY(&turtle_map_gradient_batch, cudaDeviceSynchronize());
        DEV_BACK(&turtle_map_gradient_batch, gx, d_gx, n * sizeof(double));
        DEV_BACK(&turtle_map_gradient_batch, gy, d_gy, n * sizeof(double));
        DEV_BACK(&turtle_map_gradient_batch, inside, d_in, n * sizeof(int));
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_map_elevation_ecef_batch_device(struct turtle_map * map,
    size_t n, const double * ecef, double * latitude, double * longitude, double * altitude,
    double * z, int * inside, void * stream)
{
        tb::MapDesc M;
        enum turtle_return rc = map_mirror(FN(&turtle_map_elevation_ecef_batch_device), map, &M, true);
        if ((rc != TURTLE_RETURN_SUCCESS) || (n == 0)) return rc;
        tb::ProjDesc P;
        tbh::projection_to_desc(turtle_map_projection(map), &P);
        if (map->gather == 1)
                map_elevation_ecef_kernel<tb::NodesPacked><<<stream_blocks(n, 256), 256, 0,
                    (cudaStream_t)stream>>>(M, P, n, ecef, latitude, longitude, altitude, z, inside);
        else
                map_elevation_ecef_kernel<tb::NodesGlobal><<<stream_blocks(n, 256), 256, 0,
                    (cudaStream_t)stream>>>(M, P, n, ecef, latitude, longitude, altitude, z, inside);
        CUDA_TRY(&turtle_map_elevation_ecef_batch_device, cudaGetLastError());
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_map_elevation_ecef_batch(struct turtle_map * map, size_t n,
    const double * ecef, double * latitude, double * longitude, double * altitude, double * z,
    int * inside)
{
        enum turtle_return rc = require_current(FN(&turtle_map_elevation_ecef_batch));
        if ((rc != TURTLE_RETURN_SUCCESS) || (n == 0)) return rc;
        DeviceBuffers B;
        double *d_ecef, *d_lat, *d_lon, *d_alt, *d_z;
        int * d_in;
        DEV_IN(&turtle_map_elevation_ecef_batch, B, d_ecef, ecef, n * 3 * sizeof(double));
        DEV_OUT(&turtle_map_elevation_ecef_batch, B, d_lat, latitude, n * sizeof(double));
        DEV_OUT(&turtle_map_elevation_ecef_batch, B, d_lon, longitude, n * sizeof(double));
        DEV_OUT(&turtle_map_elevation_ecef_batch, B, d_alt, altitude, n * sizeof(double));
        DEV_IN(&turtle_map_elevation_ecef_batch, B, d_z, z, n * sizeof(double));
        DEV_OUT(&turtle_map_elevation_ecef_batch, B, d_in, inside, n * sizeof(int));
        rc = turtle_map_elevation_ecef_batch_device(
            map, n, d_ecef, d_lat, d_lon, d_alt, d_z, d_in, NULL);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        CUDA_TRY(&turtle_map_elevation_ecef_batch, cudaDeviceSynchronize());
        DEV_BACK(&turtle_map_elevation_ecef_batch, latitude, d_lat, n * sizeof(double));
        DEV_BACK(&turtle_map_elevation_ecef_batch, longitude, d_lon, n * sizeof(double));
        DEV_BACK(&turtle_map_elevation_ecef_batch, altitude, d_alt, n * sizeof(double));
        DEV_BACK(&turtle_map_elevation_ecef_batch, z, d_z, n * sizeof(double));
        DEV_BACK(&turtle_map_elevation_ecef_batch, inside, d_in, n * sizeof(int));
        return TURTLE_RETURN_SUCCESS;
}

/* ---- stack queries on a plan ---------------------------------------------------------- */

static enum turtle_return stack_query(turtle_function_t * fn, struct turtle_plan * plan, int stack,
    int gradient, size_t n, const double * latitude, const double * longitude, double * a,
    double * b, int * inside, bool on_device, void * stream)
{
        if ((stack < 0) || (stack >= plan->G.n_stacks))
                return tbh::raise(fn, TURTLE_RETURN_DOMAIN_ERROR, BATCH_CU, __LINE__,
                    "invalid stack index %d (the plan has %d)", stack, plan->G.n_stacks);
        if (n == 0) return TURTLE_RETURN_SUCCESS;
        CUDA_TRY(fn, cudaSetDevice(plan->device));
        const int blocks = (int)std::min<size_t>((n + 255) / 256, (size_t)plan->sm_count * 16);
        if (on_device) {
                stack_query_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(plan->G, stack, gradient,
                    n, latitude, longitude, a, b, inside);
                plan->counters.launches++;
                CUDA_TRY(fn, cudaGetLastError());
                return TURTLE_RETURN_SUCCESS;
        }
        DeviceBuffers B;
        double *d_lat, *d_lon, *d_a, *d_b = NULL;
        int * d_in;
        DEV_IN(fn, B, d_lat, latitude, n * sizeof(double));
        DEV_IN(fn, B, d_lon, longitude, n * sizeof(double));
        DEV_OUT(fn, B, d_a, a, n * sizeof(double));
        if (gradient) DEV_OUT(fn, B, d_b, b, n * sizeof(double));
        DEV_OUT(fn, B, d_in, inside, n * sizeof(int));
        stack_query_kernel<<<blocks, 256>>>(plan->G, stack, gradient, n, d_lat, d_lon, d_a, d_b, d_in);
        plan->counters.launches++;
        CUDA_TRY(fn, cudaGetLastError());
        CUDA_TRY(fn, cudaDeviceSynchronize());
        DEV_BACK(fn, a, d_a, n * sizeof(double));
        if (gradient) DEV_BACK(fn, b, d_b, n * sizeof(double));
        DEV_BACK(fn, inside, d_in, n * sizeof(int));
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_stack_gradient_batch(struct turtle_plan * plan, int stack,
    size_t n, const double * latitude, const double * longitude, double * glat, double * glon,
    int * inside)
{
        return stack_query(FN(&turtle_stack_gradient_batch), plan, stack, 1, n, latitude, longitude,
            glat, glon, inside, false, NULL);
}

extern "C" enum turtle_return turtle_stack_gradient_batch_device(struct turtle_plan * plan,
    int stack, size_t n, const double * latitude, const double * longitude, double * glat,
    double * glon, int * inside, void * stream)
{
        return stack_query(FN(&turtle_stack_gradient_batch_device), plan, stack, 1, n, latitude,
            longitude, glat, glon, inside, true, stream);
}

extern "C" enum turtle_return turtle_stack_elevation_batch(struct turtle_plan * plan, int stack,
    size_t n, const double * latitude, const double * longitude, double * elevation, int * inside)
{
        return stack_query(FN(&turtle_stack_elevation_batch), plan, stack, 0, n, latitude,
            longitude, elevation, NULL, inside, false, NULL);
}

extern "C" enum turtle_return turtle_stack_elevation_batch_device(struct turtle_plan * plan,
    int stack, size_t n, const double * latitude, const double * longitude, double * elevation,
    int * inside, void * stream)
{
        return stack_query(FN(&turtle_stack_elevation_batch_device), plan, stack, 0, n, latitude,
            longitude, elevation, NULL, inside, true, stream);
}

/* ---- FP64 peak ------------------------------------------------------------------------ */

/* ---- peer memory (result delivery over NVLink, turtle_b200.h) ------------------- */

extern "C" enum turtle_return turtle_b200_peer_alloc(size_t bytes, void ** device_pointer)
{
        *device_pointer = NULL;
        enum turtle_return rc = require_current(FN(&turtle_b200_peer_alloc));
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        CUDA_TRY(&turtle_b200_peer_alloc, cudaMalloc(device_pointer, bytes ? bytes : 1));
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_b200_peer_free(void * device_pointer)
{
        if (device_pointer == NULL) return TURTLE_RETURN_SUCCESS;
        CUDA_TRY(&turtle_b200_peer_free, cudaFree(device_pointer));
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_b200_peer_export(
    void * device_pointer, unsigned char handle[TURTLE_B200_PEER_HANDLE_BYTES])
{
        static_assert(sizeof(cudaIpcMemHandle_t) == TURTLE_B200_PEER_HANDLE_BYTES,
            "CUDA IPC handle size");
        cudaIpcMemHandle_t h;
        CUDA_TRY(&turtle_b200_peer_export, cudaIpcGetMemHandle(&h, device_pointer));
        memcpy(handle, &h, sizeof h);
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_b200_peer_open(
    const unsigned char handle[TURTLE_B200_PEER_HANDLE_BYTES], void ** device_pointer)
{
        *device_pointer = NULL;
        enum turtle_return rc = require_current(FN(&turtle_b200_peer_open));
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        cudaIpcMemHandle_t h;
        memcpy(&h, handle, sizeof h);
        CUDA_TRY(&turtle_b200_peer_open,
            cudaIpcOpenMemHandle(device_pointer, h, cudaIpcMemLazyEnablePeerAccess));
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_b200_peer_close(void * device_pointer)
{
        if (device_pointer == NULL) return TURTLE_RETURN_SUCCESS;
        CUDA_TRY(&turtle_b200_peer_close, cudaIpcCloseMemHandle(device_pointer));
        return TURTLE_RETURN_SUCCESS;
}

extern "C" double turtle_b200_dfma_peak(int repeats)
{
        if (turtle_b200_device_count() == 0) return 0.;
        int device = 0, sms = 148;
        cudaGetDevice(&device);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
        const int blocks = sms * 8, threads = 256, iterations = 1 << 14;
        double * out = NULL;
        if (cudaMalloc((void **)&out, (size_t)blocks * threads * sizeof(double)) != cudaSuccess)
                return 0.;
        cudaEvent_t e0, e1;
        cudaEventCreate(&e0);
        cudaEventCreate(&e1);
        double best = 0.;
        if (repeats < 1) repeats = 1;
        for (int r = 0; r < repeats + 1; r++) {
                cudaEventRecord(e0);
                dfma_kernel<<<blocks, threads>>>(out, iterations);
                cudaEventRecord(e1);
                cudaEventSynchronize(e1);
                float ms = 0.f;
                cudaEventElapsedTime(&ms, e0, e1);
                const double gops = (double)blocks * threads * 8. * iterations / (ms * 1e6);
                if ((r > 0) && (gops > best)) best = gops; /* r = 0 is the warm-up */
        }
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
        cudaFree(out);
        return best;
}

/* Registers and static shared memory of a built kernel, by role (turtle_b200.h). */
extern "C" int turtle_b200_kernel_info(const char * name, int * registers, int * shared_bytes)
{
        const void * f = NULL;
#define ROLE(role, kernel) \
        if (strcmp(name, role) == 0) f = (const void *)(kernel)
        ROLE("trace_stack", (trace_kernel<false, false, 6, tb::SHAPE_STACK, false>));
        ROLE("trace_stack_stream", (trace_kernel<false, false, 6, tb::SHAPE_STACK, true>));
        ROLE("trace_stack_compact", (trace_kernel<false, false, 6, tb::SHAPE_STACK, false, true>));
        ROLE("trace_stack_stream_compact", (trace_kernel<false, false, 6, tb::SHAPE_STACK, true, true>));
        ROLE("trace", (trace_kernel<false, false, 6, tb::SHAPE_GENERIC, false>));
        ROLE("trace_proj", (trace_kernel<false, true, 6, tb::SHAPE_GENERIC, false>));
        ROLE("trace_lla", (trace_kernel<true, false, 4, tb::SHAPE_GENERIC, false>));
        ROLE("trace_lla_proj", (trace_kernel<true, true, 4, tb::SHAPE_GENERIC, false>));
        ROLE("walk", (walk_kernel<false, false, true>));
        ROLE("walk_proj", (walk_kernel<false, true, true>));
        ROLE("walk_lla", (walk_kernel<true, false, true>));
        ROLE("walk_lla_proj", (walk_kernel<true, true, true>));
        ROLE("walk_multi_proj", (walk_kernel<false, true, true, true>));
        ROLE("walk_multi_lla_proj", (walk_kernel<true, true, true, true>));
        ROLE("to_geodetic", to_geodetic_kernel);
        ROLE("map_elevation", map_elevation_kernel<tb::NodesGlobal>);
        ROLE("map_elevation_ecef", map_elevation_ecef_kernel<tb::NodesGlobal>);
        ROLE("map_elevation_packed", map_elevation_kernel<tb::NodesPacked>);
        ROLE("map_elevation_ecef_packed", map_elevation_ecef_kernel<tb::NodesPacked>);
#undef ROLE
        if (f == NULL) return -1;
        cudaFuncAttributes attr;
        if (cudaFuncGetAttributes(&attr, f) != cudaSuccess) {
                cudaGetLastError();
                return -2;
        }
        if (registers != NULL) *registers = attr.numRegs;
        if (shared_bytes != NULL) *shared_bytes = (int)attr.sharedSizeBytes;
        return 0;
}

/* Names of the batched entry points, for the error message format. */
extern "C" const char * tb_batch_function_name(turtle_function_t * caller)
{
#define NAME(function) \
        if (caller == (turtle_function_t *)function) return #function
        NAME(turtle_stepper_freeze);
        NAME(turtle_stepper_trace_batch);
        NAME(turtle_stepper_trace_batch_device);
        NAME(turtle_stepper_step_batch);
        NAME(turtle_stepper_step_batch_device);
        NAME(turtle_stepper_walk_batch);
        NAME(turtle_stepper_walk_batch_device);
        NAME(turtle_stepper_position_batch);
        NAME(turtle_states_create);
        NAME(turtle_states_reset);
        NAME(turtle_ecef_to_geodetic_batch);
        NAME(turtle_ecef_to_geodetic_batch_device);
        NAME(turtle_ecef_from_geodetic_batch);
        NAME(turtle_ecef_from_geodetic_batch_device);
        NAME(turtle_ecef_from_horizontal_batch);
        NAME(turtle_ecef_from_horizontal_batch_device);
        NAME(turtle_map_elevation_batch);
        NAME(turtle_map_elevation_batch_device);
        NAME(turtle_map_elevation_ecef_batch);
        NAME(turtle_map_elevation_ecef_batch_device);
        NAME(turtle_projection_project_batch);
        NAME(turtle_projection_project_batch_device);
        NAME(turtle_projection_unproject_batch);
        NAME(turtle_projection_unproject_batch_device);
        NAME(turtle_map_gradient_batch);
        NAME(turtle_map_gradient_batch_device);
        NAME(turtle_stepper_freeze_region);
        NAME(turtle_map_resample);
        NAME(turtle_residency_from_rays);
        NAME(turtle_stepper_trace_fan);
        NAME(turtle_stepper_trace_fan_device);
        NAME(turtle_stepper_trace_fans);
        NAME(turtle_stepper_trace_fans_device);
        NAME(turtle_stepper_trace_fields);
        NAME(turtle_stepper_trace_fields_device);
        NAME(turtle_plan_gather_set);
        NAME(turtle_stack_gradient_batch);
        NAME(turtle_stack_gradient_batch_device);
        NAME(turtle_stack_elevation_batch);
        NAME(turtle_stack_elevation_batch_device);
        NAME(turtle_stepper_trace_crossings);
        NAME(turtle_stepper_trace_crossings_device);
        NAME(turtle_stepper_horizon);
        NAME(turtle_stepper_horizon_device);
        NAME(turtle_stepper_horizons);
        NAME(turtle_stepper_horizons_device);
        NAME(turtle_stepper_trace_voxels);
        NAME(turtle_stepper_trace_voxels_device);
        NAME(turtle_stepper_trace_fans_voxels);
        NAME(turtle_stepper_trace_fans_voxels_device);
        NAME(turtle_stepper_trace_opacity);
        NAME(turtle_stepper_trace_opacity_device);
        NAME(turtle_stepper_trace_fans_opacity);
        NAME(turtle_stepper_trace_fans_opacity_device);
        NAME(turtle_b200_peer_alloc);
        NAME(turtle_b200_peer_free);
        NAME(turtle_b200_peer_export);
        NAME(turtle_b200_peer_open);
        NAME(turtle_b200_peer_close);
#undef NAME
        return NULL;
}
