/*
 * turtle_b200.h -- batched, GPU-resident entry points added on top of turtle.h.
 *
 * The scalar interface (turtle.h) describes a geometry with turtle_stepper_add_*
 * and steps ONE particle per call (ref: src/turtle/stepper.c:780-875). The entry
 * points below freeze such a geometry into a device-resident plan (DEM tiles in
 * HBM, flattened layer/meta/data/transform tables) and run the same stepping
 * rules for millions of independent rays per call on one B200. There is no CPU
 * fallback: without a CUDA device every function here returns
 * TURTLE_RETURN_LIBRARY_ERROR and raises through the error handler.
 *
 * Conventions
 *  - plain C ABI: pointers + sizes only. `*_batch` takes HOST pointers (staged
 *    through pinned buffers, chunked and overlapped with compute); `*_batch_device`
 *    takes DEVICE pointers valid on the plan's device plus a `cudaStream_t`
 *    passed as `void *` (NULL = legacy default stream) and is asynchronous.
 *  - arrays are AoS like the scalar API: position[n][3], direction[n][3],
 *    elevation[n][2], index[n][2].
 *  - per-element conditions (outside of every map, NaN input ...) are reported in
 *    per-element outputs, never through the error handler. The handler is used
 *    for argument / launch errors only, with the reference's message format
 *    (ref: src/turtle/error.c:108-138).
 */
#ifndef TURTLE_B200_H
#define TURTLE_B200_H

#include <stddef.h>
#include <stdint.h>
#include "turtle.h"

#ifdef __cplusplus
extern "C" {
#endif

/* A geometry frozen on one device. Built from a turtle_stepper, it captures the
 * layers, the geoid and the range / slope / resolution settings at freeze time
 * (ref: the state walked by stepper_sample, src/turtle/stepper.c:703-756). */
struct turtle_plan;

/* Per-particle stepping state kept on the device between turtle_stepper_step_batch
 * calls: what `struct turtle_stepper` keeps for ONE particle in the reference
 * (last sample + local-approximation references, ref: src/turtle/stepper.h:45-58,
 * 93-110). */
struct turtle_states;

/* Number of media with their own path-length accumulator in a trace result;
 * steps started in medium >= TURTLE_TRACE_MEDIA-1 share the last one. */
#define TURTLE_TRACE_MEDIA 4

/* Why a traced ray stopped. */
enum turtle_trace_status {
        TURTLE_TRACE_ALTITUDE = 0, /* altitude left ]altitude_min, altitude_max[ */
        TURTLE_TRACE_DOMAIN = 1,   /* index[0] < 0: no data below/above any more */
        TURTLE_TRACE_LENGTH = 2,   /* travelled >= length_max */
        TURTLE_TRACE_STEPS = 3,    /* did max_steps steps */
        TURTLE_TRACE_INVALID = 4   /* non finite input */
};

/* Stop rule of the canonical ray loop (ref: examples/example-stepper.c:128-140:
 * `while (altitude < altitude_max) turtle_stepper_step(...)`), made total. A ray
 * keeps stepping while index[0] >= 0, altitude_min < altitude < altitude_max,
 * length < length_max and n_steps < max_steps. */
struct turtle_trace_rule {
        double altitude_min;
        double altitude_max;
        double length_max;
        int32_t max_steps;
        int32_t reserved;
};

/* Result record of one ray (96 bytes). `length[m]` sums the steps that STARTED in
 * medium m, i.e. `if (initial_layer == m) length += step`
 * (ref: examples/example-stepper.c:136-139). */
struct turtle_trace_result {
        double position[3]; /* final ECEF position */
        double altitude;    /* final altitude (geoid corrected if a geoid is set) */
        double length[TURTLE_TRACE_MEDIA];
        double total;       /* sum of all step lengths, in stepping order */
        int32_t n_steps;    /* number of turtle_stepper_step equivalents */
        int32_t status;     /* enum turtle_trace_status */
        int32_t index[2];   /* final layer / data index */
        uint32_t medium_hash; /* order dependent hash of the media visited */
        int32_t n_changes;  /* number of steps that ended in another medium */
};

/* Kernel counters of the last trace/step/horizon call on a plan. */
struct turtle_plan_counters {
        uint64_t rays;     /* rays or particles processed */
        uint64_t steps;    /* turtle_stepper_step equivalents */
        uint64_t samples;  /* geometry samples (stepper_sample equivalents) */
        uint64_t launches; /* CUDA kernels launched */
        double kernel_ms;  /* device time of the kernels (CUDA events), host-pointer calls only */
        uint64_t rebuilds; /* local approximation: Jacobian columns evaluated (one ECEF ->
                            * geodetic transform each, like a sample) */
        uint64_t window_hits; /* gather mode 2: samples whose nodes came from shared memory */
};

/* ---- plans ---------------------------------------------------------------- */

/* Threading: a plan carries the streams, staging buffers and counters of the calls made
 * through it, and is used from one host thread at a time. HOST-pointer calls (`*_batch`,
 * `_trace_fan[s]`, `_trace_fields`, `_trace_crossings`, `_horizon[s]`, `_trace_[fans_]voxels`,
 * `_trace_[fans_]opacity`)
 * return when their results are in place: ONE at a time per plan. DEVICE-pointer calls (`*_device`) are asynchronous on the
 * caller's stream: that is how a caller with several batches hides the tail of one (a launch
 * ends when its slowest ray does) behind the head of the next. A device-pointer call is IN
 * FLIGHT from its return until its stream has done all it queued; up to 8 may be in flight on
 * one plan, on streams of the caller's choice, and they may complete in any order. Each holds
 * one of 8 slots of the plan (the queue cursor of its kernel, its schedule buffers and its
 * fan / azimuth / station tables) until it completes; a ninth call waits on the host until the call
 * that took its slot first is over. Host-pointer calls have slots of their own and may be
 * made while device-pointer calls are in flight; those that stage their arrays in device
 * memory of their own (turtle_stepper_step_batch, _walk_batch, _trace_crossings, _horizon[s],
 * _trace_[fans_]voxels, _trace_[fans_]opacity) free it before they return, which waits for the device to be idle. After the caller has
 * synchronised, turtle_plan_counters_sync reports the device-pointer call issued last.
 * Several plans (one per host thread or per device) are independent; they share nothing but
 * read-only tiles of their own. This is the batched form of the reference's rule "one
 * stepper per thread" (include/turtle.h:141-149 of the reference). */

/* Upload every map / tile referenced by `stepper` to `device` and flatten the
 * geometry. Stacks are made fully resident (all tiles of the grid are loaded):
 * this replaces the reference's on-demand tile cache (ref: src/turtle/stack.c:
 * 399-450, src/turtle/client.c:99-188). The stepper and its maps must outlive
 * nothing: the plan owns device copies. */
TURTLE_API enum turtle_return turtle_stepper_freeze(
    struct turtle_stepper * stepper, int device, struct turtle_plan ** plan);

/* ---- residency planning for stacks larger than one GPU -----------------------------
 * A world-scale stack (14 k SRTMGL1 tiles, 370 GB) does not fit 180 GB of HBM and the
 * device has no on-demand cache. The plan is made for a REGION instead: only the tiles
 * whose footprint meets the box become resident; the others answer `outside`, exactly as
 * a missing tile does. NaN bounds are open. turtle_residency_from_rays derives the box
 * from the rays to be traced and their stop rule (see there).
 *
 * Tiles that are not already loaded on the host are INGESTED ON THE DEVICE: their file is
 * read (any of .hgt .png .tif .grd .asc), the nodes are copied in FILE order and a kernel
 * converts byte order and row order straight into the tile pool -- no host-side copy of
 * the stack is ever built (turtle_stepper_freeze does the same). */
struct turtle_residency {
        double latitude_min, latitude_max, longitude_min, longitude_max;
        size_t memory_limit; /* refuse plans above this many bytes of HBM; 0 = what is free */
};
struct turtle_residency_report {
        uint64_t tiles_resident; /* stack tiles uploaded */
        uint64_t tiles_skipped;  /* stack tiles with a file, left out by the region */
        uint64_t tiles_ingested; /* ... of the resident ones, decoded on the device */
        uint64_t bytes;          /* HBM held by the plan */
        double read_ms, upload_ms; /* file reading / parsing, copies + ingest kernels */
};
TURTLE_API enum turtle_return turtle_stepper_freeze_region(
    struct turtle_stepper * stepper, int device, const struct turtle_residency * region,
    struct turtle_plan ** plan);
TURTLE_API void turtle_plan_residency_get(
    const struct turtle_plan * plan, struct turtle_residency_report * report);
/* Geodetic bounding box of the ground tracks of n rays (host arrays [n][3]), each followed
 * until the stop rule must have ended it: min(rule->length_max, the chord to the sphere of
 * radius a + rule->altitude_max), sampled every `step` metres (<= 0: 1000 m), and widened
 * by `margin` degrees. Conservative for rays that stop on leaving the data set. Rays
 * through a pole or across the date line open the longitude bounds (NaN). */
TURTLE_API enum turtle_return turtle_residency_from_rays(size_t n, const double * position,
    const double * direction, const struct turtle_trace_rule * rule, double step,
    double margin, struct turtle_residency * region);
TURTLE_API void turtle_plan_destroy(struct turtle_plan ** plan);
TURTLE_API int turtle_plan_device(const struct turtle_plan * plan);
/* Bytes of HBM held by the plan (tiles + tables). */
TURTLE_API size_t turtle_plan_bytes(const struct turtle_plan * plan);
TURTLE_API void turtle_plan_counters_get(
    const struct turtle_plan * plan, struct turtle_plan_counters * counters);
/* After a `*_device` call and once the caller has synchronised its stream: read
 * the step / sample counters of that launch back from the device. */
TURTLE_API void turtle_plan_counters_sync(struct turtle_plan * plan);
/* Tuning: CTAs per SM and threads per CTA of the persistent kernels (0 = default). */
TURTLE_API void turtle_plan_launch_set(
    struct turtle_plan * plan, int ctas_per_sm, int threads);
/* Ray scheduling of the trace calls. 0: rays are started in the caller's order.
 * 1: longest-expected-first -- rays are started by increasing |sin(elevation)| of their
 * direction (grazing rays take the most steps; a long ray that starts last bounds the
 * kernel time). Results do not depend on the mode, only the time does. */
TURTLE_API void turtle_plan_schedule_set(struct turtle_plan * plan, int mode);
/* Kernel specialisation by geometry shape. 1 (default): a geometry made of one layer with
 * one uniform geodetic stack (no geoid, range 0) runs a kernel with the list walk of
 * stepper_sample (stepper.c:717-743) resolved at compile time. 0: always the generic
 * kernel. Results are byte-identical (tests/test_gpu_trace.py); only the time differs. */
TURTLE_API void turtle_plan_specialise_set(struct turtle_plan * plan, int enable);
/* How the host-pointer call turtle_stepper_trace_batch overlaps its copies with the
 * stepping. 0 (default): streamed -- one persistent kernel over the whole batch, fed and
 * drained by the copy engines in 256 Ki-ray pieces (lanes wait for their ray, finished
 * chunks are copied back as they complete). 1: chunked -- one kernel per 1 Mi-ray chunk on
 * three streams (also used whenever a ray schedule is set). Results are identical. */
TURTLE_API void turtle_plan_pipeline_set(struct turtle_plan * plan, int mode);

/* How the trace kernel of a single uniform stack (the muography case) gathers the four
 * nodes of a sample (ref: the 2 x 2 gather of turtle_map_elevation_, map.c:266-271).
 *   0  four 16-bit loads from the row-major tiles (default);
 *   1  one 8-byte load from a CELL-PACKED second copy of the tiles, built here on the
 *      device: 4 x the tile bytes of HBM for one request and one sector per sample;
 *   2  a 64 x 64-node window of the tile under (latitude, longitude) -- the station of a
 *      fan -- staged in the shared memory of every CTA by the bulk copy engine
 *      (cp.async.bulk + mbarrier); samples outside of it gather as in mode 0.
 * Results are byte-identical in all modes (tests/test_gpu_trace.py); the device-pointer
 * trace calls honour the mode, the streamed / compact ones gather as in mode 0. See
 * DESIGN.md section 3 for what each mode measures. latitude / longitude: mode 2 only. */
TURTLE_API enum turtle_return turtle_plan_gather_set(struct turtle_plan * plan, int mode,
    double latitude, double longitude);

/* ---- whole rays: reset, query, then step until the rule stops the ray ------ */
TURTLE_API enum turtle_return turtle_stepper_trace_batch(
    struct turtle_plan * plan, size_t n, const double * position,
    const double * direction, const struct turtle_trace_rule * rule,
    struct turtle_trace_result * results);
TURTLE_API enum turtle_return turtle_stepper_trace_batch_device(
    struct turtle_plan * plan, size_t n, const double * position,
    const double * direction, const struct turtle_trace_rule * rule,
    struct turtle_trace_result * results, void * stream);

/* ---- compact input / output of whole rays -----------------------------------------------
 * turtle_stepper_trace_batch moves 48 bytes in and 96 bytes out per ray. The canonical
 * caller needs neither: examples/example-stepper.c:102-140 (ref) shoots rays from ONE
 * station, derives each direction from two angles (turtle_ecef_from_horizontal) and keeps
 * ONE number per ray (the rock length). These entry points are that caller, batched.
 *
 * Fields: the columns of struct turtle_trace_result as separate arrays, any of them NULL
 * (not wanted). position is [n][3], index is [n][2], the others are [n]. What a caller
 * does not ask for is neither stored nor copied. */
struct turtle_trace_fields {
        double * length[TURTLE_TRACE_MEDIA];
        double * total;
        double * altitude;
        double * position;
        int32_t * n_steps;
        int32_t * status;
        int32_t * index;
        uint32_t * medium_hash;
        int32_t * n_changes;
};
/* A fan of n_azimuth x n_elevation rays from one origin. The direction of ray (i, j) is
 * turtle_ecef_from_horizontal(latitude, longitude, azimuth[i], elevation[j]) TO THE BIT
 * (ref: src/turtle/ecef.c:160-178): the sines and cosines of the n_azimuth + n_elevation
 * angles are taken on the host, by the very calls of that function, and the device only
 * multiplies and adds in its order. `azimuth` and `elevation` are HOST arrays, in degrees
 * (also for the _device variant: they are the whole input of a call, a few kB).
 * Ray order: ray r is (i, j) with
 *     band = r / (n_azimuth * bundle), i = (r / bundle) % n_azimuth,
 *     j = band * bundle + r % bundle,
 * i.e. bands of `bundle` consecutive elevations, azimuth by azimuth within a band:
 * bundle = 1 is elevation-major (r = j * n_azimuth + i), bundle = n_elevation is
 * azimuth-major (r = i * n_elevation + j), bundle = 32 makes the 32 rays of a warp share
 * one vertical plane. n_elevation must be a multiple of bundle (0 means 1). Listing the
 * lowest elevations first starts the longest rays first. */
struct turtle_fan {
        double latitude, longitude; /* the station: local frame of azimuth / elevation */
        double position[3];         /* ECEF origin of every ray (turtle_stepper_position) */
        size_t n_azimuth, n_elevation;
        const double * azimuth;
        const double * elevation;
        size_t bundle;
};
/* Trace the fan. `results` (n records) and `fields` may each be NULL; both are HOST memory
 * here and DEVICE memory in the _device variant. */
TURTLE_API enum turtle_return turtle_stepper_trace_fan(struct turtle_plan * plan,
    const struct turtle_fan * fan, const struct turtle_trace_rule * rule,
    struct turtle_trace_result * results, const struct turtle_trace_fields * fields);
TURTLE_API enum turtle_return turtle_stepper_trace_fan_device(struct turtle_plan * plan,
    const struct turtle_fan * fan, const struct turtle_trace_rule * rule,
    struct turtle_trace_result * results, const struct turtle_trace_fields * fields,
    void * stream);
/* One angle grid shot from n_station stations in ONE call: site surveys, joint inversions of
 * several telescopes, the shadows of an antenna array. Ray r = s * (n_azimuth * n_elevation)
 * + q, where q is the ray order of struct turtle_fan (bands of `bundle` elevations) and s the
 * station: ray r is, record and fields byte for byte, ray q of turtle_stepper_trace_fan with
 * the fan { latitude[s], longitude[s], position + 3 * s, n_azimuth, n_elevation, azimuth,
 * elevation, bundle }. The frame of every station is taken on the host by the calls of
 * turtle_ecef_from_horizontal, as for one fan. All arrays of the struct are HOST memory, also
 * for the _device variant; `results` and `fields` (n_station * n_azimuth * n_elevation rays)
 * are host memory here and device memory in the _device variant, which is ONE launch. A
 * station without data or with a non-finite latitude or position gives what the one-station
 * call gives for it (TURTLE_TRACE_INVALID rays for a non-finite position); it is not an error
 * of the call. The arguments are checked before the plan or the device is used; n_station = 0
 * or an empty grid does nothing. The plan counters report all the rays. */
struct turtle_fans {
        size_t n_station;
        const double * latitude;    /* [n_station] degrees: local frame of station s */
        const double * longitude;   /* [n_station] degrees */
        const double * position;    /* [n_station][3] ECEF origin of the rays of station s */
        size_t n_azimuth, n_elevation;
        const double * azimuth;     /* degrees, shared by every station */
        const double * elevation;
        size_t bundle;
};
TURTLE_API enum turtle_return turtle_stepper_trace_fans(struct turtle_plan * plan,
    const struct turtle_fans * fans, const struct turtle_trace_rule * rule,
    struct turtle_trace_result * results, const struct turtle_trace_fields * fields);
TURTLE_API enum turtle_return turtle_stepper_trace_fans_device(struct turtle_plan * plan,
    const struct turtle_fans * fans, const struct turtle_trace_rule * rule,
    struct turtle_trace_result * results, const struct turtle_trace_fields * fields,
    void * stream);
/* turtle_stepper_trace_batch with field arrays instead of records. */
TURTLE_API enum turtle_return turtle_stepper_trace_fields(struct turtle_plan * plan, size_t n,
    const double * position, const double * direction, const struct turtle_trace_rule * rule,
    const struct turtle_trace_fields * fields);
TURTLE_API enum turtle_return turtle_stepper_trace_fields_device(struct turtle_plan * plan,
    size_t n, const double * position, const double * direction,
    const struct turtle_trace_rule * rule, const struct turtle_trace_fields * fields,
    void * stream);

/* ---- the horizon of a station ------------------------------------------------------------
 * For each azimuth, the elevation that separates the rays from `position` that enter the
 * ground from the rays that reach open sky: the contour of a muography transmission map and
 * the edge of its open-sky calibration region. The probe at elevation e is the ray with
 * direction turtle_ecef_from_horizontal(latitude, longitude, azimuth, e), traced under `rule`
 * exactly as turtle_stepper_trace_batch traces it (reset stepper, same steps, same bits). It
 * is OBSTRUCTED when one of its steps ends in a medium >= 0 other than the station's -- it
 * stops right there -- and CLEAR when the rule stops it first (leaving the data is clear).
 * The search runs on the device: each round traces 32 probes of one azimuth and narrows the
 * bracket to [highest obstructed probe, next probe above it] until it is at most
 * `tolerance` degrees wide. Every probe made above elevation[1] was clear. Over terrain that
 * is a graph over the sphere, obstruction is monotone in elevation and the bracket holds the
 * horizon; wherever the stepper's resolution breaks that at the sub-centimetre scale, it is
 * still a bracket of the predicate above.
 *
 * The azimuths' sines and cosines are taken on the host, as for a fan; the elevations of the
 * probes are made on the device, with the device's sine and cosine (within an ulp of the
 * host's): the two probe directions are returned so that either end can be re-traced. The
 * ends of a bracket that no probe established (BELOW, ABOVE, INVALID) are NaN, with
 * medium[1] = -1 and clear_status = -1. The arguments are checked before the plan or the
 * device is used: a tolerance <= 0 or a window that is empty, reversed or not within
 * [-90, 90] is TURTLE_RETURN_DOMAIN_ERROR, a missing position, azimuth table or result
 * array TURTLE_RETURN_BAD_ADDRESS. `azimuth` (degrees) is HOST memory in both variants;
 * `results` is host memory for turtle_stepper_horizon and device memory for the
 * asynchronous _device variant. The plan counters report the probes as rays, with their
 * steps and samples. */
enum turtle_horizon_status {
        TURTLE_HORIZON_FOUND = 0,  /* elevation[0] obstructed, elevation[1] clear, width <= tolerance */
        TURTLE_HORIZON_BELOW = 1,  /* the ray at elevation_min is already clear */
        TURTLE_HORIZON_ABOVE = 2,  /* the ray at elevation_max is still obstructed */
        TURTLE_HORIZON_INVALID = 3 /* station or direction not finite, or station without data */
};
struct turtle_horizon {            /* 96 bytes, one per azimuth */
        double elevation[2];       /* [obstructed, clear] bracket, degrees */
        double direction[2][3];    /* the two probe rays that were traced (ECEF, unit) */
        double length;             /* obstructed probe: path length to its first medium change */
        int32_t medium[2];         /* station's medium, medium the obstructed probe enters */
        int32_t status;            /* enum turtle_horizon_status */
        int32_t clear_status;      /* enum turtle_trace_status of the clear probe */
        int32_t n_probes;          /* rays traced for this azimuth */
        int32_t n_iterations;      /* loop iterations of the warp that searched it (the time
                                    * of the search, in samples one after the other) */
};
TURTLE_API enum turtle_return turtle_stepper_horizon(struct turtle_plan * plan,
    double latitude, double longitude, const double position[3], size_t n_azimuth,
    const double * azimuth, double elevation_min, double elevation_max, double tolerance,
    const struct turtle_trace_rule * rule, struct turtle_horizon * results);
TURTLE_API enum turtle_return turtle_stepper_horizon_device(struct turtle_plan * plan,
    double latitude, double longitude, const double position[3], size_t n_azimuth,
    const double * azimuth, double elevation_min, double elevation_max, double tolerance,
    const struct turtle_trace_rule * rule, struct turtle_horizon * results, void * stream);
/* The horizons of n_station stations in ONE call (the horizon of every antenna of an array,
 * a sky-view raster with one station per node): results[s * n_azimuth + i] is, byte for
 * byte, results[i] of turtle_stepper_horizon(plan, latitude[s], longitude[s], position +
 * 3 * s, n_azimuth, azimuth, ...), n_probes and n_iterations included. latitude, longitude
 * ([n_station], degrees), position ([n_station][3]) and azimuth are HOST memory in both
 * variants. A station without data or with non-finite values gives TURTLE_HORIZON_INVALID
 * records, as alone; a missing array is TURTLE_RETURN_BAD_ADDRESS, a bad window or tolerance
 * TURTLE_RETURN_DOMAIN_ERROR, checked before the plan or the device is used; n_station = 0 or
 * n_azimuth = 0 does nothing. The plan counters report the probes of all stations as rays. */
TURTLE_API enum turtle_return turtle_stepper_horizons(struct turtle_plan * plan,
    size_t n_station, const double * latitude, const double * longitude, const double * position,
    size_t n_azimuth, const double * azimuth, double elevation_min, double elevation_max,
    double tolerance, const struct turtle_trace_rule * rule, struct turtle_horizon * results);
TURTLE_API enum turtle_return turtle_stepper_horizons_device(struct turtle_plan * plan,
    size_t n_station, const double * latitude, const double * longitude, const double * position,
    size_t n_azimuth, const double * azimuth, double elevation_min, double elevation_max,
    double tolerance, const struct turtle_trace_rule * rule, struct turtle_horizon * results,
    void * stream);

/* ---- the stream of medium changes along every ray (SURVEY.md section 8f, N4) --------
 * What a Monte-Carlo engine integrates over the steps -- column density, energy loss per
 * medium, entry and exit points of the rock -- needs more than the per-medium totals of
 * struct turtle_trace_result: it needs WHERE along the ray each medium begins. The
 * crossings variant of the trace records, per ray, its first `max_crossings` medium changes
 * (boundary-located by the stepper's bisection, stepper.c:832-864): the path length from
 * the origin at which the new medium begins and the layer indices on both sides (-1 = left
 * the data). results[i].n_changes tells how many the ray had in all; crossings
 * [i * max_crossings + k] is valid for k < min(n_changes, max_crossings). */
struct turtle_trace_crossing {
        double length;
        int32_t medium_from, medium_to;
};
TURTLE_API enum turtle_return turtle_stepper_trace_crossings(
    struct turtle_plan * plan, size_t n, const double * position,
    const double * direction, const struct turtle_trace_rule * rule,
    struct turtle_trace_result * results, struct turtle_trace_crossing * crossings,
    int max_crossings);
TURTLE_API enum turtle_return turtle_stepper_trace_crossings_device(
    struct turtle_plan * plan, size_t n, const double * position,
    const double * direction, const struct turtle_trace_rule * rule,
    struct turtle_trace_result * results, struct turtle_trace_crossing * crossings,
    int max_crossings, void * stream);

/* ---- the length of every ray in every cell of a voxel grid: the matrix of a density
 * inversion ----------------------------------------------------------------------------------
 * A density inversion solves opacity_i = sum_j L_ij rho_j, where rho_j is the density of cell j
 * of a grid around the mountain and L_ij the length of ray i inside cell j AND inside the rock.
 * These calls build L on the device, one sparse row per ray.
 *
 * Rays. Ray i is traced exactly as turtle_stepper_trace_batch (or, for the fans form,
 * turtle_stepper_trace_fans, same ray order and directions) traces it: same steps, same bits.
 * `results` (may be NULL) receives the very records of the plain call.
 * Segments. Step k of a ray covers the path lengths [s_{k-1}, s_k] of the ray line
 * origin + s * direction, where s is the running `total` before and after the step (the
 * doubles turtle_stepper_trace_crossings reports). A step counts when bit medium0 of
 * grid->media is set, medium0 being the medium its start sample was in (the rule of
 * length[m], by true layer index, not folded to TURTLE_TRACE_MEDIA). Its segment is clipped to
 * the cells of the grid.
 * Cells. The grid frame has its origin at turtle_ecef_from_geodetic(latitude, longitude, height)
 * and the East / North / Up vectors of turtle_ecef_from_horizontal at (latitude, longitude).
 * Cell (ix, iy, iz) is the half-open box [corner + i * size, corner + (i + 1) * size) on each
 * axis. Cell planes are met at absolute path lengths along the ray line, so the steps do not
 * move a cell boundary.
 * Entries. The entries of ray i are entries[i * capacity + k], in order along the ray. A new
 * entry starts whenever the cell or the medium changes; consecutive pieces in the same (cell,
 * medium) are summed into one entry, across step boundaries and across stretches in media
 * that are not selected. No entry has length 0: a (cell, medium) pair appears twice in one ray
 * only with something else between its appearances.
 * Count and capacity. count[i] is the number of entries of ray i in all, which may exceed
 * `capacity`; only the first min(count[i], capacity) are written, the slots after them are
 * left untouched. With capacity = 0, `entries` may be NULL and the call only counts: a first
 * pass that sizes an exact buffer. Invalid rays (TURTLE_TRACE_INVALID) and rays without a
 * selected step in the grid have count 0.
 * Checks. The arguments are checked before the plan or the device is used. A missing grid or
 * fans struct, missing positions, directions or counts (n > 0), or entries NULL with
 * capacity > 0 are TURTLE_RETURN_BAD_ADDRESS. capacity < 0, cell counts <= 0 or of more than
 * INT32_MAX cells in all, sizes that are not finite and > 0, a non-finite origin or corner, or
 * media == 0 are TURTLE_RETURN_DOMAIN_ERROR. n = 0 or an empty fan grid does nothing.
 * Memory. turtle_stepper_trace_voxels and _fans_voxels take HOST memory and return when the
 * results are in place (the entries are staged in device memory of their own, freed before
 * the return). The _device variants take DEVICE memory (the fans' arrays stay on the host, as
 * for turtle_stepper_trace_fans_device), are one asynchronous launch on `stream` and hold one
 * of the plan's 8 slots. The plan counters report rays, steps and samples as a trace does. */
struct turtle_voxel_grid {
        double latitude, longitude, height; /* frame origin, turtle_ecef_from_geodetic(...) */
        double corner[3];  /* E, N, U coordinates (m) of the lowest corner of the grid */
        double size[3];    /* cell edges along E, N, U (m), finite and > 0 */
        int32_t n[3];      /* cells along E, N, U, > 0, n[0] * n[1] * n[2] <= INT32_MAX */
        uint32_t media;    /* bit m set: steps that START in medium m are split (m < 32), != 0 */
};
struct turtle_voxel_entry {        /* 16 bytes */
        double length;             /* metres of the ray in this cell and medium */
        int32_t voxel;             /* ix + n[0] * (iy + n[1] * iz) */
        int32_t medium;            /* medium the steps started in */
};
TURTLE_API enum turtle_return turtle_stepper_trace_voxels(struct turtle_plan * plan, size_t n,
    const double * position, const double * direction, const struct turtle_trace_rule * rule,
    const struct turtle_voxel_grid * grid, struct turtle_trace_result * results,
    struct turtle_voxel_entry * entries, int capacity, int32_t * count);
TURTLE_API enum turtle_return turtle_stepper_trace_voxels_device(struct turtle_plan * plan,
    size_t n, const double * position, const double * direction,
    const struct turtle_trace_rule * rule, const struct turtle_voxel_grid * grid,
    struct turtle_trace_result * results, struct turtle_voxel_entry * entries, int capacity,
    int32_t * count, void * stream);
TURTLE_API enum turtle_return turtle_stepper_trace_fans_voxels(struct turtle_plan * plan,
    const struct turtle_fans * fans, const struct turtle_trace_rule * rule,
    const struct turtle_voxel_grid * grid, struct turtle_trace_result * results,
    struct turtle_voxel_entry * entries, int capacity, int32_t * count);
TURTLE_API enum turtle_return turtle_stepper_trace_fans_voxels_device(struct turtle_plan * plan,
    const struct turtle_fans * fans, const struct turtle_trace_rule * rule,
    const struct turtle_voxel_grid * grid, struct turtle_trace_result * results,
    struct turtle_voxel_entry * entries, int capacity, int32_t * count, void * stream);

/* ---- opacity and its gradient over a voxel grid, without storing the matrix ----------------
 * What a solver does with the L of turtle_stepper_trace_voxels is apply it (L rho, the forward
 * model) and its transpose (L^T w, the gradient of a misfit with respect to the densities).
 * These calls do both while they trace, and store no entry.
 *
 * L. Exactly the L of turtle_stepper_trace_voxels / _trace_fans_voxels on the same rays and
 * grid: the row of ray i is its entries (k = 0 .. count[i] - 1, in order along the ray), with
 * their media merged as a CSR matrix sums them.
 * Rays and records. Rays are traced exactly as turtle_stepper_trace_voxels (for the fans form,
 * turtle_stepper_trace_fans_voxels) traces them: same ray order, same steps, same bits.
 * `results` (may be NULL) receives the plain trace's records byte for byte.
 * Forward, exact. opacity[i] is acc = 0; for k in the entries of ray i, in order:
 * acc = acc + density[voxel_k] * length_k, each product and each sum rounded on its own, in that
 * order, with no fused multiply-add, on the very `length` doubles turtle_stepper_trace_voxels
 * stores: bit for bit that loop on the host over its entries. Rays without an entry, and
 * TURTLE_TRACE_INVALID rays, give 0.
 * Outside. outside[i] is the length of the steps in selected media (grid->media) that lies
 * outside the grid's box, summed in stepping order: the column of L for the rock the grid does
 * not cover. A step that meets the box adds its parts before and after the box; a step that
 * misses it adds its length. On a grid that encloses the ray it is exactly 0.
 * Adjoint. Each entry k of ray i adds weight[i] * length_k (one rounded product) to
 * gradient[voxel_k] with a device atomic. The order of the sums across rays is unspecified: the
 * result is the exact sum of those products within (m_j - 1) * eps * sum |p| for the m_j
 * products p of cell j. `gradient` is ADDED TO, never cleared: several calls may add into one
 * array, device calls in flight together included. Zeroing it is the caller's job.
 * Outputs. Each output is optional and needs only its own input: opacity needs density,
 * gradient needs weight; the forward and the adjoint may be asked for in one call. Densities
 * and weights are the caller's data and are not checked: a NaN propagates.
 * Checks. The arguments are checked before the plan or the device is used. The grid is checked
 * as by turtle_stepper_trace_voxels, with the same codes and messages. A missing opacity, grid
 * or fans struct, missing positions or directions (n > 0), opacity without density, or gradient
 * without weight are TURTLE_RETURN_BAD_ADDRESS. n = 0 or an empty fan grid does nothing.
 * Memory. turtle_stepper_trace_opacity and _fans_opacity take HOST memory and return when the
 * results are in place: density and gradient (n[0] * n[1] * n[2] doubles) and the per-ray arrays
 * are staged in device memory of their own, gradient copied in and back, all freed before the
 * return. The _device variants take DEVICE memory (the fans' arrays stay on the host, as for
 * turtle_stepper_trace_fans_device), are one asynchronous launch on `stream` and hold one of
 * the plan's 8 slots. The plan counters report rays, steps and samples as a trace does. */
struct turtle_voxel_opacity {
        const double * density; /* [n[0] * n[1] * n[2]] rho_j (cell index of turtle_voxel_entry), or NULL */
        double * opacity;       /* [n] sum_j L_ij rho_j; needs density; or NULL */
        double * outside;       /* [n] metres of the selected steps given to no cell, or NULL */
        const double * weight;  /* [n] w_i, or NULL */
        double * gradient;      /* [n[0] * n[1] * n[2]] ADDED TO: += sum_i w_i L_ij; needs weight; or NULL */
};
TURTLE_API enum turtle_return turtle_stepper_trace_opacity(struct turtle_plan * plan, size_t n,
    const double * position, const double * direction, const struct turtle_trace_rule * rule,
    const struct turtle_voxel_grid * grid, const struct turtle_voxel_opacity * opacity,
    struct turtle_trace_result * results);
TURTLE_API enum turtle_return turtle_stepper_trace_opacity_device(struct turtle_plan * plan,
    size_t n, const double * position, const double * direction,
    const struct turtle_trace_rule * rule, const struct turtle_voxel_grid * grid,
    const struct turtle_voxel_opacity * opacity, struct turtle_trace_result * results,
    void * stream);
TURTLE_API enum turtle_return turtle_stepper_trace_fans_opacity(struct turtle_plan * plan,
    const struct turtle_fans * fans, const struct turtle_trace_rule * rule,
    const struct turtle_voxel_grid * grid, const struct turtle_voxel_opacity * opacity,
    struct turtle_trace_result * results);
TURTLE_API enum turtle_return turtle_stepper_trace_fans_opacity_device(struct turtle_plan * plan,
    const struct turtle_fans * fans, const struct turtle_trace_rule * rule,
    const struct turtle_voxel_grid * grid, const struct turtle_voxel_opacity * opacity,
    struct turtle_trace_result * results, void * stream);

/* ---- one turtle_stepper_step for n independent particles -------------------
 * Same outputs as the scalar call (any output pointer may be NULL; direction
 * NULL = query mode, position untouched). `states` may be NULL: every particle
 * then starts from a reset stepper (exact when range <= 0). States may be destroyed
 * before or after the plan they were created for. */
TURTLE_API enum turtle_return turtle_states_create(
    struct turtle_plan * plan, size_t n, struct turtle_states ** states);
TURTLE_API void turtle_states_destroy(struct turtle_states ** states);
TURTLE_API enum turtle_return turtle_states_reset(struct turtle_states * states);
/* Bytes of HBM held per particle: the last sample (9 doubles), the stale-Jacobian mask and,
 * when the plan's range is > 0, the local approximations of the transforms the geometry
 * uses (15 doubles for a geodetic stack, 25 for a projected map over a stack ...). */
TURTLE_API size_t turtle_states_bytes_per_particle(const struct turtle_states * states);
TURTLE_API enum turtle_return turtle_stepper_step_batch(
    struct turtle_plan * plan, struct turtle_states * states, size_t n,
    double * position, const double * direction, double * latitude,
    double * longitude, double * altitude, double * elevation, double * step,
    int * index);
TURTLE_API enum turtle_return turtle_stepper_step_batch_device(
    struct turtle_plan * plan, struct turtle_states * states, size_t n,
    double * position, const double * direction, double * latitude,
    double * longitude, double * altitude, double * elevation, double * step,
    int * index, void * stream);

/* n_steps successive turtle_stepper_step calls per particle in ONE launch -- the inner loop
 * of a transport engine that draws a new direction every step (BASELINE configuration 4).
 * direction[j][i][3] is the direction of step j of particle i; the per-step outputs are
 * [n_steps][n] (elevation, index: [n_steps][n][2]; any may be NULL), position[n][3] is
 * advanced to the end of the walk. Same results as n_steps calls of
 * turtle_stepper_step_batch; what differs is the traffic: the particle's stepper state
 * (turtle_states, or a reset stepper when `states` is NULL) is read once, stays on chip for
 * all its steps and is written once, instead of crossing HBM both ways every step. */
TURTLE_API enum turtle_return turtle_stepper_walk_batch(
    struct turtle_plan * plan, struct turtle_states * states, size_t n, int n_steps,
    double * position, const double * direction, double * latitude,
    double * longitude, double * altitude, double * elevation, double * step,
    int * index);
TURTLE_API enum turtle_return turtle_stepper_walk_batch_device(
    struct turtle_plan * plan, struct turtle_states * states, size_t n, int n_steps,
    double * position, const double * direction, double * latitude,
    double * longitude, double * altitude, double * elevation, double * step,
    int * index, void * stream);

/* ---- ray origins (ref: turtle_stepper_position, src/turtle/stepper.c:877-931)
 * data_index[i] = -1 and position[i] untouched when (lat, lon) has no data. */
TURTLE_API enum turtle_return turtle_stepper_position_batch(
    struct turtle_plan * plan, size_t n, const double * latitude,
    const double * longitude, const double * height, int layer_index,
    double * position, int * data_index);

/* ---- frame transforms (ref: src/turtle/ecef.c:41-55,63-130,160-178) ---------
 * Run on the current CUDA device. Output pointers of to_geodetic may be NULL.
 * to_geodetic: the altitude has the bits of turtle_ecef_to_geodetic, latitude and
 * longitude are within 4 ulp of it, for points at least 50 km from the centre of the
 * Earth. Closer, the arguments of the arcsine in Olson's method leave the range its
 * device polynomial is fitted for and the latitude is not bounded (the reference's own
 * method returns NaN below about 40 km). Where x or y is denormal or infinite the
 * longitude is NaN (the device arctangent divides through a reciprocal). */
TURTLE_API enum turtle_return turtle_ecef_to_geodetic_batch(size_t n,
    const double * ecef, double * latitude, double * longitude,
    double * altitude);
TURTLE_API enum turtle_return turtle_ecef_to_geodetic_batch_device(size_t n,
    const double * ecef, double * latitude, double * longitude,
    double * altitude, void * stream);
TURTLE_API enum turtle_return turtle_ecef_from_geodetic_batch(size_t n,
    const double * latitude, const double * longitude,
    const double * elevation, double * ecef);
TURTLE_API enum turtle_return turtle_ecef_from_geodetic_batch_device(size_t n,
    const double * latitude, const double * longitude,
    const double * elevation, double * ecef, void * stream);
TURTLE_API enum turtle_return turtle_ecef_from_horizontal_batch(size_t n,
    const double * latitude, const double * longitude, const double * azimuth,
    const double * elevation, double * direction);
TURTLE_API enum turtle_return turtle_ecef_from_horizontal_batch_device(size_t n,
    const double * latitude, const double * longitude, const double * azimuth,
    const double * elevation, double * direction, void * stream);

/* ---- elevation queries (ref: turtle_map_elevation, src/turtle/map.c:229-277)
 * The map is mirrored on the current device on first use and after any
 * turtle_map_fill. z[i] is untouched where inside[i] == 0. */
TURTLE_API enum turtle_return turtle_map_elevation_batch(
    struct turtle_map * map, size_t n, const double * x, const double * y,
    double * z, int * inside);
TURTLE_API enum turtle_return turtle_map_elevation_batch_device(
    struct turtle_map * map, size_t n, const double * x, const double * y,
    double * z, int * inside, void * stream);
/* Node gathers of the batched elevation queries of `map` (the map-side twin of
 * turtle_plan_gather_set). 0 (default): four 16-bit loads from the row-major mirror -- two
 * 32-byte sectors per query. 1: ONE 8-byte load from a cell-packed second copy of the grid
 * (cell (ix, iy) = its four nodes; 4 x the bytes of the mirror, built on the device at the
 * next query) -- one sector per query, which is what a random-access query stream pays
 * for. Same bits either way. */
TURTLE_API void turtle_map_gather_set(struct turtle_map * map, int mode);
/* Fused ECEF -> geodetic -> (projection) -> bilinear elevation: one pass over the
 * points, no intermediate arrays in HBM. latitude/longitude/altitude may be NULL. */
TURTLE_API enum turtle_return turtle_map_elevation_ecef_batch(
    struct turtle_map * map, size_t n, const double * ecef, double * latitude,
    double * longitude, double * altitude, double * z, int * inside);
TURTLE_API enum turtle_return turtle_map_elevation_ecef_batch_device(
    struct turtle_map * map, size_t n, const double * ecef, double * latitude,
    double * longitude, double * altitude, double * z, int * inside,
    void * stream);

/* ---- projections (ref: turtle_projection_project / _unproject, src/turtle/projection.c:
 * 192-233; SURVEY.md 8f N3). Run on the current CUDA device. */
TURTLE_API enum turtle_return turtle_projection_project_batch(
    const struct turtle_projection * projection, size_t n, const double * latitude,
    const double * longitude, double * x, double * y);
TURTLE_API enum turtle_return turtle_projection_project_batch_device(
    const struct turtle_projection * projection, size_t n, const double * latitude,
    const double * longitude, double * x, double * y, void * stream);
TURTLE_API enum turtle_return turtle_projection_unproject_batch(
    const struct turtle_projection * projection, size_t n, const double * x,
    const double * y, double * latitude, double * longitude);
TURTLE_API enum turtle_return turtle_projection_unproject_batch_device(
    const struct turtle_projection * projection, size_t n, const double * x,
    const double * y, double * latitude, double * longitude, void * stream);

/* ---- gradients (ref: turtle_map_gradient, src/turtle/map.c:280-378; SURVEY.md 8f N1)
 * Same bits as the scalar call, including its first-row behaviour (map.c:353).
 * gx[i], gy[i] are untouched where inside[i] == 0. */
TURTLE_API enum turtle_return turtle_map_gradient_batch(
    struct turtle_map * map, size_t n, const double * x, const double * y,
    double * gx, double * gy, int * inside);
TURTLE_API enum turtle_return turtle_map_gradient_batch_device(
    struct turtle_map * map, size_t n, const double * x, const double * y,
    double * gx, double * gy, int * inside, void * stream);

/* ---- stack queries (ref: turtle_stack_elevation, src/turtle/stack.c:338-361, and
 * turtle_stack_gradient, stack.c:364-388; SURVEY.md 8f N1) on the resident tiles of a plan.
 * `stack` counts the stacks of the stepper in the order they were first added
 * (turtle_stepper_add_stack). The tile that answers an elevation query answers the gradient
 * query, with the bits of the scalar calls (turtle_map_gradient's first-row behaviour,
 * map.c:353, included). Outside of every tile: inside[i] = 0 and the outputs are 0
 * (stack.c:349-355,376-380); with inside == NULL that is not reported at all. */
TURTLE_API enum turtle_return turtle_stack_elevation_batch(struct turtle_plan * plan, int stack,
    size_t n, const double * latitude, const double * longitude, double * elevation,
    int * inside);
TURTLE_API enum turtle_return turtle_stack_elevation_batch_device(struct turtle_plan * plan,
    int stack, size_t n, const double * latitude, const double * longitude, double * elevation,
    int * inside, void * stream);
TURTLE_API enum turtle_return turtle_stack_gradient_batch(struct turtle_plan * plan, int stack,
    size_t n, const double * latitude, const double * longitude, double * glat, double * glon,
    int * inside);
TURTLE_API enum turtle_return turtle_stack_gradient_batch_device(struct turtle_plan * plan,
    int stack, size_t n, const double * latitude, const double * longitude, double * glat,
    double * glon, int * inside, void * stream);

/* ---- host bulk set-up ---------------------------------------------------------*/
/* turtle_map_fill for every node: elevation[iy * nx + ix] (ref: map.c:183-203).
 * Stops at the first node that turtle_map_fill rejects and returns its code. */
TURTLE_API enum turtle_return turtle_map_fill_batch(
    struct turtle_map * map, const double * elevation);
/* Same for rows [iy0, iy0 + n_rows): elevation[(iy - iy0) * nx + ix]. */
TURTLE_API enum turtle_return turtle_map_fill_rows(
    struct turtle_map * map, int iy0, int n_rows, const double * elevation);

/* Number of tiles of `stack` currently held on the HOST (what the reference's tests read
 * from `stack->tiles.size`, stack.h:34-52 -- the type is opaque here). */
TURTLE_API int turtle_stack_tiles_loaded(const struct turtle_stack * stack);

/* ---- device utilities -------------------------------------------------------*/
/* Number of CUDA devices visible (0 when there is no driver / GPU). */
TURTLE_API int turtle_b200_device_count(void);
/* Measured FP64 FMA rate of the current device in Gop/s (1 FMA = 1 op), from a
 * dependent-chain DFMA micro-benchmark kernel; used as the compute roofline. */
TURTLE_API double turtle_b200_dfma_peak(int repeats);
TURTLE_API const char * turtle_b200_version(void);
/* Registers per thread and static shared memory of a built kernel, by role: "trace_stack",
 * "trace", "trace_proj", "trace_lla", "trace_lla_proj", "trace_stack_stream", "walk",
 * "walk_proj", "walk_lla", "walk_lla_proj", "to_geodetic", "map_elevation",
 * "map_elevation_ecef". Returns 0, -1 for an unknown role, -2 without a device. The
 * measurement tools use it to check that a committed profile (profiles/) still describes
 * the kernel they are timing. */
TURTLE_API int turtle_b200_kernel_info(const char * name, int * registers, int * shared_bytes);
/* Device self test of the shared-reciprocal division used by the kernels against the
 * compiler's IEEE division on 2 * n random operand pairs: number of results that
 * differ in any bit (0 expected), -1 without a device. */
TURTLE_API long long turtle_b200_selftest_division(size_t n, uint64_t seed);

/* ---- resampling a geometry into a map (SURVEY.md section 8f, N3) ---------------------
 * The step that PRODUCES a high-resolution local map: examples/example-projection.c:88-104
 * walks the nodes of a projected map, un-projects each one, asks the tile stack for its
 * elevation and fills the node -- one scalar call chain per node. Here a kernel does it
 * for all nodes: node (x, y) -> inverse projection of `map` -> (latitude, longitude) ->
 * ground elevation of layer `layer` of the plan's geometry (the first data of the layer,
 * in the stepper's priority order, that holds the point, plus its offset; no geoid
 * undulation: the data's own datum) -> turtle_map_fill semantics for the node (quantised
 * to the map's 16-bit scale; TURTLE_RETURN_DOMAIN_ERROR if a value is outside of the
 * map's z span). Nodes where the layer has no data are left as they are and counted in
 * *outside (may be NULL). */
TURTLE_API enum turtle_return turtle_map_resample(struct turtle_map * map,
    struct turtle_plan * plan, int layer, size_t * outside);

/* ---- multi-GPU: result records written straight into a peer GPU's memory ----------
 * Rays shard across the GPUs of a box with the DEM replicated (SURVEY.md section 8e);
 * the only exchange of the path is the delivery of the fixed-size result records to the
 * rank that consumes them. Instead of a gather AFTER the kernel, the consumer allocates
 * the whole result array once, exports it (CUDA IPC), and every other process opens it
 * and passes `base + first_ray` as the `results` pointer of
 * turtle_stepper_trace_batch_device: the trace kernel then stores each record over
 * NVLink / NVSwitch the moment its ray ends, overlapped with the stepping of all other
 * rays. One process per GPU; all GPUs of the box must be visible to every process. */
#define TURTLE_B200_PEER_HANDLE_BYTES 64
/* cudaMalloc on the current device (an allocation of its own: exportable). */
TURTLE_API enum turtle_return turtle_b200_peer_alloc(size_t bytes, void ** device_pointer);
TURTLE_API enum turtle_return turtle_b200_peer_free(void * device_pointer);
/* Handle of an allocation made by turtle_b200_peer_alloc, to be sent to the peers. */
TURTLE_API enum turtle_return turtle_b200_peer_export(
    void * device_pointer, unsigned char handle[TURTLE_B200_PEER_HANDLE_BYTES]);
/* Map a peer's allocation into this process (current device must be able to reach the
 * owner over NVLink / PCIe peer access); close it before the owner frees it. */
TURTLE_API enum turtle_return turtle_b200_peer_open(
    const unsigned char handle[TURTLE_B200_PEER_HANDLE_BYTES], void ** device_pointer);
TURTLE_API enum turtle_return turtle_b200_peer_close(void * device_pointer);

#ifdef __cplusplus
}
#endif
#endif
