/*
 * tb_host.cpp -- the scalar turtle.h calls (set-up / cold path) of turtle-b200.
 *
 * These mirror the reference interface for the stepping path: same names,
 * argument meaning, return codes and error-message format. The arithmetic is
 * the host instantiation of tb_core.cuh, i.e. the very expressions the CUDA
 * kernels run. The batched hot path lives in tb_kernels.cu and never comes here.
 *
 * Error messages carry the reference's module name as the file tag
 * (e.g. `src/turtle/map.c`) so that callers matching the reference's message
 * format (tests/test-turtle.c:482-507) keep working.
 */
#include "tb_host.hpp"
#include "tb_io.hpp"
#include "turtle_b200.h"

#include <dirent.h>
#include <limits.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/stat.h>

#include <algorithm>
#include <mutex>
#include <new>

#define FN(f) ((turtle_function_t *)(f))
#define RAISE(fn, rc, file, ...) tbh::raise(FN(fn), rc, file, __LINE__, __VA_ARGS__)

/* ======================================================================== */
/* Error handling (ref: src/turtle/error.c)                                  */
/* ======================================================================== */

static void default_handler(enum turtle_return code, turtle_function_t * function,
    const char * message)
{
        fprintf(stderr, "A TURTLE library error occurred:\n%s\n", message);
        exit(EXIT_FAILURE);
}

static turtle_error_handler_t * g_handler = &default_handler;

extern "C" turtle_error_handler_t * turtle_error_handler_get(void)
{
        return g_handler;
}

extern "C" void turtle_error_handler_set(turtle_error_handler_t * handler)
{
        g_handler = handler;
}

enum turtle_return tbh::raise(turtle_function_t * fn, enum turtle_return rc,
    const char * file, int line, const char * format, ...)
{
        if ((g_handler == NULL) || (rc == TURTLE_RETURN_SUCCESS)) return rc;
        char body[1024];
        va_list ap;
        va_start(ap, format);
        vsnprintf(body, sizeof body, format, ap);
        va_end(ap);
        char message[1400];
        const char * name = turtle_error_function(fn);
        snprintf(message, sizeof message, "{ %s [#%d], %s:%d } %s",
            name ? name : "(null)", (int)rc, file, line, body);
        g_handler(rc, fn, message);
        return rc;
}

/* ======================================================================== */
/* Projections (ref: src/turtle/projection.c)                                */
/* ======================================================================== */

static const char * PROJ_C = "src/turtle/projection.c";

static int next_word(const char ** str)
{
        const char * p = *str;
        while (*p == ' ') p++;
        *str = p;
        int n = 0;
        while ((p[n] != ' ') && (p[n] != '\0')) n++;
        return n;
}

/* ref: turtle_projection_configure_, projection.c:98-172. Returns the code and
 * fills `msg` on failure; the caller raises under its own function name. */
static enum turtle_return projection_parse(
    struct turtle_projection * projection, const char * name, char * msg, size_t nmsg)
{
        projection->type = -1;
        projection->utm_longitude_0 = 0.;
        projection->utm_hemisphere = 0;
        projection->lambert_tag = 0;
        if (name == NULL) {
                projection->tag[0] = 0x0;
                return TURTLE_RETURN_SUCCESS;
        }
        const char * p = name;
        int n = next_word(&p);
        if (n == 0) {
                snprintf(msg, nmsg, "missing projection specifier");
                return TURTLE_RETURN_BAD_PROJECTION;
        } else if (strncmp(p, "Lambert", n) == 0) {
                projection->type = 0;
                p += n;
                n = next_word(&p);
                static const char * tags[6] = { "I", "II", "IIe", "III", "IV", "93" };
                for (int i = 0; i < 6; i++) {
                        if (strncmp(p, tags[i], n) == 0) {
                                projection->lambert_tag = i;
                                goto accept;
                        }
                }
        } else if (strncmp(p, "UTM", n) == 0) {
                projection->type = 1;
                p += n;
                int zone;
                char hemisphere;
                if (sscanf(p, "%d%c", &zone, &hemisphere) != 2) {
                        snprintf(msg, nmsg, "invalid UTM specifier `%s'", p);
                        return TURTLE_RETURN_BAD_PROJECTION;
                }
                if (hemisphere == '.') {
                        double longitude_0;
                        if (sscanf(p, "%lf%c", &longitude_0, &hemisphere) != 2) {
                                snprintf(msg, nmsg,
                                    "invalid extended UTM specifier `%s'", p);
                                return TURTLE_RETURN_BAD_PROJECTION;
                        }
                        projection->utm_longitude_0 = longitude_0;
                } else {
                        projection->utm_longitude_0 = 6. * zone - 183.;
                }
                if (hemisphere == 'N')
                        projection->utm_hemisphere = 1;
                else if (hemisphere == 'S')
                        projection->utm_hemisphere = -1;
                else {
                        snprintf(msg, nmsg, "invalid UTM hemisphere `%c'", hemisphere);
                        return TURTLE_RETURN_BAD_PROJECTION;
                }
                goto accept;
        }
        snprintf(msg, nmsg, "invalid projection `%s'", p);
        return TURTLE_RETURN_BAD_PROJECTION;
accept:
        strncpy(projection->tag, name, sizeof(projection->tag) - 1);
        projection->tag[sizeof(projection->tag) - 1] = 0x0;
        return TURTLE_RETURN_SUCCESS;
}

/* Lambert parameter sets, ref: projection.c:327-347 (I, II, IIe, III, IV, 93) */
static const double LAMBERT[6][6] = {
        { 0.08248325676, 0.7604059656, 11603796.98, 0.04079234433, 600000.0, 5657616.674 },
        { 0.08248325676, 0.7289686274, 11745793.39, 0.04079234433, 600000.0, 6199695.768 },
        { 0.08248325676, 0.7289686274, 11745793.39, 0.04079234433, 600000.0, 8199695.768 },
        { 0.08248325676, 0.6959127966, 11947992.52, 0.04079234433, 600000.0, 6791905.085 },
        { 0.08248325676, 0.6712679322, 12136281.99, 0.04079234433, 234.358, 7239161.542 },
        { 0.08181919112, 0.7253743710, 11755528.70, 0.05235987756, 700000.0, 12657560.145 }
};

/* UTM ellipsoid constants, ref: projection.c:380-391 / 420-431 */
static const double UTM_A = 6378.137E+03;
static const double UTM_F = 1. / 298.257223563;
static const double UTM_K0 = 0.9996;

void tbh::projection_to_desc(const struct turtle_projection * p, tb::ProjDesc * d)
{
        memset(d, 0x0, sizeof(*d));
        if ((p == NULL) || (p->type < 0)) {
                d->type = tb::PROJ_GEODETIC;
        } else if (p->type == 0) {
                const double * q = LAMBERT[p->lambert_tag];
                d->type = tb::PROJ_LAMBERT;
                d->e = q[0];
                d->n = q[1];
                d->C = q[2];
                d->lambda_c = q[3];
                d->xs = q[4];
                d->ys = q[5];
        } else {
                /* the call-invariant part of utm_ll_to_xy, same expressions */
                const double a = UTM_A, f = UTM_F, k0 = UTM_K0;
                const double n = f / (2. - f);
                const double A = a / (1. + n) * (1. + n * n * (0.25 + 0.0625 * n * n));
                d->type = tb::PROJ_UTM;
                d->lon0 = p->utm_longitude_0;
                d->E0 = 5E+05;
                d->N0 = (p->utm_hemisphere > 0) ? 0. : 1E+07;
                d->k0A = k0 * A;
                d->alpha[0] = n * (0.5 + n * (-2. / 3. + 5. / 16. * n));
                d->alpha[1] = n * n * (13. / 48. - 3. / 5. * n);
                d->alpha[2] = 61. / 240. * n * n * n;
                d->c = 2. * sqrt(n) / (1. + n);
                d->beta[0] = n * (0.5 + n * (-2. / 3. + 37. / 96. * n));
                d->beta[1] = n * n * (1. / 48. + 1. / 15. * n);
                d->beta[2] = 17. / 480. * n * n * n;
                d->delta[0] = n * (2. + n * (-2. / 3. - 2. * n));
                d->delta[1] = n * n * (7. / 3. - 8. / 5. * n);
                d->delta[2] = 56. / 15. * n * n * n;
        }
}

extern "C" enum turtle_return turtle_projection_create(
    struct turtle_projection ** projection, const char * name)
{
        *projection = NULL;
        struct turtle_projection tmp;
        char msg[256];
        enum turtle_return rc = projection_parse(&tmp, name, msg, sizeof msg);
        if (rc != TURTLE_RETURN_SUCCESS)
                return RAISE(&turtle_projection_create, rc, PROJ_C, "%s", msg);
        *projection = (struct turtle_projection *)malloc(sizeof(**projection));
        if (*projection == NULL)
                return RAISE(&turtle_projection_create, TURTLE_RETURN_MEMORY_ERROR,
                    PROJ_C, "could not allocate memory");
        memcpy(*projection, &tmp, sizeof(tmp));
        return TURTLE_RETURN_SUCCESS;
}

extern "C" void turtle_projection_destroy(struct turtle_projection ** projection)
{
        if ((projection == NULL) || (*projection == NULL)) return;
        free(*projection);
        *projection = NULL;
}

extern "C" enum turtle_return turtle_projection_configure(
    struct turtle_projection * projection, const char * name)
{
        char msg[256];
        enum turtle_return rc = projection_parse(projection, name, msg, sizeof msg);
        if (rc != TURTLE_RETURN_SUCCESS)
                return RAISE(&turtle_projection_configure, rc, PROJ_C, "%s", msg);
        return rc;
}

extern "C" const char * turtle_projection_name(
    const struct turtle_projection * projection)
{
        if ((projection == NULL) || (projection->type < 0)) return NULL;
        return projection->tag;
}

extern "C" enum turtle_return turtle_projection_project(
    const struct turtle_projection * projection, double latitude,
    double longitude, double * x, double * y)
{
        *x = 0.;
        *y = 0.;
        if (projection == NULL)
                return RAISE(&turtle_projection_project, TURTLE_RETURN_BAD_ADDRESS,
                    PROJ_C, "missing projection");
        if (projection->type < 0)
                return RAISE(&turtle_projection_project,
                    TURTLE_RETURN_BAD_PROJECTION, PROJ_C, "invalid projection");
        tb::ProjDesc d;
        tbh::projection_to_desc(projection, &d);
        tb::project(d, latitude, longitude, *x, *y);
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_projection_unproject(
    const struct turtle_projection * projection, double x, double y,
    double * latitude, double * longitude)
{
        *latitude = 0.;
        *longitude = 0.;
        if (projection == NULL)
                return RAISE(&turtle_projection_unproject, TURTLE_RETURN_BAD_ADDRESS,
                    PROJ_C, "missing projection");
        if (projection->type < 0)
                return RAISE(&turtle_projection_unproject,
                    TURTLE_RETURN_BAD_PROJECTION, PROJ_C, "invalid projection");
        tb::ProjDesc d;
        tbh::projection_to_desc(projection, &d);
        tb::unproject(d, x, y, *latitude, *longitude);
        return TURTLE_RETURN_SUCCESS;
}

/* ======================================================================== */
/* Maps (ref: src/turtle/map.c)                                              */
/* ======================================================================== */

static const char * MAP_C = "src/turtle/map.c";

static tb::MapDesc map_desc(const struct turtle_map * map)
{
        tb::MapDesc d;
        d.nodes = map->nodes.data();
        d.nx = map->nx;
        d.ny = map->ny;
        d.pitch = map->nx;
        d.kind = map->kind;
        d.x0 = map->x0;
        d.y0 = map->y0;
        d.dx = map->dx;
        d.dy = map->dy;
        d.z0 = map->z0;
        d.dz = map->dz;
        tb::map_desc_finish(d);
        return d;
}

static struct turtle_map * map_alloc(int nx, int ny)
{
        struct turtle_map * map = new (std::nothrow) turtle_map();
        if (map == NULL) return NULL;
        try {
                map->nodes.assign((size_t)nx * (size_t)ny, 0);
        } catch (...) {
                delete map;
                return NULL;
        }
        map->nx = nx;
        map->ny = ny;
        map->stack = NULL;
        map->version = 1;
        return map;
}

extern "C" enum turtle_return turtle_map_create(struct turtle_map ** map,
    const struct turtle_map_info * info, const char * projection)
{
        *map = NULL;
        if ((info->nx <= 0) || (info->ny <= 0) || (info->z[0] == info->z[1]))
                return RAISE(&turtle_map_create, TURTLE_RETURN_DOMAIN_ERROR, MAP_C,
                    "invalid input parameter(s)");
        struct turtle_projection proj;
        char msg[256];
        enum turtle_return rc = projection_parse(&proj, projection, msg, sizeof msg);
        if (rc != TURTLE_RETURN_SUCCESS)
                return RAISE(&turtle_map_create, rc, PROJ_C, "%s", msg);
        struct turtle_map * m = map_alloc(info->nx, info->ny);
        if (m == NULL)
                return RAISE(&turtle_map_create, TURTLE_RETURN_MEMORY_ERROR, MAP_C,
                    "could not allocate memory");
        /* ref: map.c:75-85 */
        m->x0 = info->x[0];
        m->y0 = info->y[0];
        m->z0 = info->z[0];
        m->dx = (info->nx > 1) ? (info->x[1] - info->x[0]) / (info->nx - 1) : 0.;
        m->dy = (info->ny > 1) ? (info->y[1] - info->y[0]) / (info->ny - 1) : 0.;
        m->dz = (info->z[1] - info->z[0]) / 65535;
        m->kind = tb::NODE_AFFINE_U16;
        m->projection = proj;
        strcpy(m->encoding, "none");
        *map = m;
        return TURTLE_RETURN_SUCCESS;
}

extern "C" void tb_map_release_mirrors(struct turtle_map * map); /* tb_kernels.cu */
extern "C" const char * tb_batch_function_name(turtle_function_t * caller);

extern "C" void turtle_map_destroy(struct turtle_map ** map)
{
        if ((map == NULL) || (*map == NULL)) return;
        struct turtle_map * m = *map;
        if (m->stack != NULL) {
                /* ref: map.c:103-109, the owning stack forgets the tile */
                struct turtle_stack * s = m->stack;
                for (size_t i = 0; i < s->tile.size(); i++) {
                        if (s->tile[i] == m) {
                                s->tile[i] = NULL;
                                s->mru.erase(std::remove(s->mru.begin(), s->mru.end(),
                                                 (int)i),
                                    s->mru.end());
                        }
                }
        }
        tb_map_release_mirrors(m);
        delete m;
        *map = NULL;
}

/* ref: turtle_map_load_, map.c:116-158 + the io plug-ins (tb_io.cpp). Nodes are kept
 * rows south first, native endian, whatever the file stored. */
static enum turtle_return map_load_file(struct turtle_map ** map, const char * path,
    turtle_function_t * caller)
{
        *map = NULL;
        tbio::Header h;
        tbio::RawLayout layout;
        tbio::Error err;
        std::vector<uint16_t> raw;
        if (tbio::read_map(path, h, layout, raw, err) != 0)
                return tbh::raise(caller, err.code, err.file, __LINE__, "%s", err.message.c_str());
        struct turtle_projection proj;
        char msg[256];
        enum turtle_return rc = projection_parse(
            &proj, h.projection.empty() ? NULL : h.projection.c_str(), msg, sizeof msg);
        if (rc != TURTLE_RETURN_SUCCESS) return tbh::raise(caller, rc, PROJ_C, __LINE__, "%s", msg);
        struct turtle_map * m = new (std::nothrow) turtle_map();
        if (m == NULL)
                return tbh::raise(caller, TURTLE_RETURN_MEMORY_ERROR, MAP_C, __LINE__,
                    "could not allocate memory for map `%s'", path);
        tbio::normalise(h, layout, raw);
        m->nodes.swap(raw);
        m->nx = h.nx;
        m->ny = h.ny;
        m->x0 = h.x0;
        m->y0 = h.y0;
        m->z0 = h.z0;
        m->dx = h.dx;
        m->dy = h.dy;
        m->dz = h.dz;
        m->kind = h.kind;
        m->projection = proj;
        m->stack = NULL;
        m->version = 1;
        snprintf(m->encoding, sizeof m->encoding, "%s", h.encoding.c_str());
        *map = m;
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_map_load(struct turtle_map ** map, const char * path)
{
        return map_load_file(map, path, FN(&turtle_map_load));
}

/* ref: turtle_map_dump, map.c:160-176 (`.png` and `.tif` have writers) */
extern "C" enum turtle_return turtle_map_dump(const struct turtle_map * map, const char * path)
{
        tbio::Header h;
        h.nx = map->nx;
        h.ny = map->ny;
        h.x0 = map->x0;
        h.y0 = map->y0;
        h.z0 = map->z0;
        h.dx = map->dx;
        h.dy = map->dy;
        h.dz = map->dz;
        h.kind = map->kind;
        const char * tag = turtle_projection_name(&map->projection);
        h.projection = (tag != NULL) ? tag : "";
        tbio::Error err;
        if (tbio::write_map(path, h, map->nodes, err) != 0)
                return tbh::raise(FN(&turtle_map_dump), err.code, err.file, __LINE__, "%s",
                    err.message.c_str());
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_map_fill(
    struct turtle_map * map, int ix, int iy, double elevation)
{
        if (map == NULL)
                return RAISE(&turtle_map_fill, TURTLE_RETURN_MEMORY_ERROR, MAP_C,
                    "could not allocate memory");
        if ((ix < 0) || (ix >= map->nx) || (iy < 0) || (iy >= map->ny))
                return RAISE(&turtle_map_fill, TURTLE_RETURN_DOMAIN_ERROR, MAP_C,
                    "point is outside of map");
        if ((map->dz <= 0.) && (elevation != map->z0))
                return RAISE(&turtle_map_fill, TURTLE_RETURN_DOMAIN_ERROR, MAP_C,
                    "inconsistent elevation value");
        if ((elevation < map->z0) || (elevation > map->z0 + 65535 * map->dz))
                return RAISE(&turtle_map_fill, TURTLE_RETURN_DOMAIN_ERROR, MAP_C,
                    "elevation is outside of map span");
        uint16_t raw;
        if (map->kind == tb::NODE_DIRECT_I16) {
                raw = (uint16_t)(int16_t)elevation;
        } else {
                const double d = round((elevation - map->z0) / map->dz); /* map.c:47-51 */
                raw = (uint16_t)d;
        }
        map->nodes[(size_t)iy * map->nx + ix] = raw;
        map->version++;
        return TURTLE_RETURN_SUCCESS;
}

/* Bulk variants of turtle_map_fill (turtle_b200.h). */
extern "C" enum turtle_return turtle_map_fill_rows(
    struct turtle_map * map, int iy0, int n_rows, const double * elevation)
{
        if (map == NULL) return turtle_map_fill(map, 0, 0, 0.);
        for (int iy = iy0; iy < iy0 + n_rows; iy++)
                for (int ix = 0; ix < map->nx; ix++) {
                        enum turtle_return rc = turtle_map_fill(
                            map, ix, iy, elevation[(size_t)(iy - iy0) * map->nx + ix]);
                        if (rc != TURTLE_RETURN_SUCCESS) return rc;
                }
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_map_fill_batch(
    struct turtle_map * map, const double * elevation)
{
        if (map == NULL) return turtle_map_fill(map, 0, 0, 0.);
        return turtle_map_fill_rows(map, 0, map->ny, elevation);
}

extern "C" enum turtle_return turtle_map_node(const struct turtle_map * map, int ix,
    int iy, double * x, double * y, double * elevation)
{
        if (map == NULL)
                return RAISE(&turtle_map_node, TURTLE_RETURN_MEMORY_ERROR, MAP_C,
                    "could not allocate memory");
        if ((ix < 0) || (ix >= map->nx) || (iy < 0) || (iy >= map->ny))
                return RAISE(&turtle_map_node, TURTLE_RETURN_DOMAIN_ERROR, MAP_C,
                    "point is outside of map");
        if (x != NULL) *x = map->x0 + ix * map->dx;
        if (y != NULL) *y = map->y0 + iy * map->dy;
        if (elevation != NULL) {
                const tb::MapDesc d = map_desc(map);
                *elevation = tb::node_value(d, map->nodes[(size_t)iy * map->nx + ix]);
        }
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_map_elevation(const struct turtle_map * map,
    double x, double y, double * z, int * inside)
{
        const tb::MapDesc d = map_desc(map);
        const int in = tb::map_elevation(d, x, y, *z);
        if (inside != NULL) {
                *inside = in;
                return TURTLE_RETURN_SUCCESS;
        }
        if (!in)
                return RAISE(&turtle_map_elevation, TURTLE_RETURN_DOMAIN_ERROR, MAP_C,
                    "point is outside of map");
        return TURTLE_RETURN_SUCCESS;
}

/* ref: turtle_map_gradient, map.c:388-393 (it registers turtle_map_elevation as the
 * failing function, which is kept) */
extern "C" enum turtle_return turtle_map_gradient(const struct turtle_map * map, double x,
    double y, double * gx, double * gy, int * inside)
{
        const tb::MapDesc d = map_desc(map);
        const int in = tb::map_gradient(d, x, y, *gx, *gy);
        if (inside != NULL) {
                *inside = in;
                return TURTLE_RETURN_SUCCESS;
        }
        if (!in)
                return RAISE(&turtle_map_elevation, TURTLE_RETURN_DOMAIN_ERROR, MAP_C,
                    "point is outside of map");
        return TURTLE_RETURN_SUCCESS;
}

extern "C" const struct turtle_projection * turtle_map_projection(
    const struct turtle_map * map)
{
        if ((map == NULL) || (map->projection.type < 0)) return NULL;
        return &map->projection;
}

extern "C" void turtle_map_meta(const struct turtle_map * map,
    struct turtle_map_info * info, const char ** projection)
{
        if (info != NULL) { /* ref: map.c:403-416 */
                info->nx = map->nx;
                info->ny = map->ny;
                info->x[0] = map->x0;
                info->x[1] = map->x0 + (map->nx - 1) * map->dx;
                info->y[0] = map->y0;
                info->y[1] = map->y0 + (map->ny - 1) * map->dy;
                info->z[0] = map->z0;
                info->z[1] = map->z0 + 65535 * map->dz;
                info->encoding = map->encoding;
        }
        if (projection != NULL) *projection = turtle_projection_name(&map->projection);
}

/* ======================================================================== */
/* ECEF (ref: src/turtle/ecef.c)                                             */
/* ======================================================================== */

extern "C" void turtle_ecef_from_geodetic(
    double latitude, double longitude, double elevation, double ecef[3])
{
        tb::ecef_from_geodetic(latitude, longitude, elevation, ecef);
}

extern "C" void turtle_ecef_to_geodetic(const double ecef[3], double * latitude,
    double * longitude, double * altitude)
{
        double la, lo, al;
        tb::ecef_to_geodetic(ecef, la, lo, al);
        if (latitude != NULL) *latitude = la;
        if (longitude != NULL) *longitude = lo;
        if (altitude != NULL) *altitude = al;
}

extern "C" void turtle_ecef_from_horizontal(double latitude, double longitude,
    double azimuth, double elevation, double direction[3])
{
        tb::ecef_from_horizontal(latitude, longitude, azimuth, elevation, direction);
}

extern "C" void turtle_ecef_to_horizontal(double latitude, double longitude,
    const double direction[3], double * azimuth, double * elevation)
{
        double az, el;
        if (!tb::ecef_to_horizontal(latitude, longitude, direction, az, el)) return;
        if (azimuth != NULL) *azimuth = az;
        if (elevation != NULL) *elevation = el;
}

/* ======================================================================== */
/* Stacks and clients (ref: src/turtle/stack.c, client.c)                    */
/* ======================================================================== */

static const char * STACK_C = "src/turtle/stack.c";

extern "C" enum turtle_return turtle_stack_create(struct turtle_stack ** stack,
    const char * path, int size, turtle_stack_locker_t * lock,
    turtle_stack_locker_t * unlock)
{
        *stack = NULL;
        if (((lock == NULL) && (unlock != NULL)) || ((unlock == NULL) && (lock != NULL)))
                return RAISE(&turtle_stack_create, TURTLE_RETURN_BAD_ADDRESS, STACK_C,
                    "inconsistent lock & unlock");

        DIR * dir = opendir(path);
        if (dir == NULL)
                return RAISE(&turtle_stack_create, TURTLE_RETURN_PATH_ERROR, STACK_C,
                    "could not access %s", path);

        /* first pass: tile spans and bounding box (ref: stack.c:59-132) */
        struct found { std::string path; double x0, y0; tb::MapDesc desc; };
        std::vector<found> files;
        double lat_min = DBL_MAX, long_min = DBL_MAX;
        double lat_max = -DBL_MAX, long_max = -DBL_MAX;
        double lat_delta = 0., long_delta = 0.;
        struct dirent * entry;
        enum turtle_return rc = TURTLE_RETURN_SUCCESS;
        const char * errmsg = NULL;
        while ((entry = readdir(dir)) != NULL) {
                std::string full = std::string(path) + "/" + entry->d_name;
                struct stat st;
                if ((stat(full.c_str(), &st) != 0) || S_ISDIR(st.st_mode)) continue;
                /* any of the five formats makes a tile (stack.c:76-91) */
                if (!tbio::known_extension(tbio::extension(entry->d_name))) continue;
                tbio::Header th;
                tbio::Error terr;
                if (tbio::read_header(full.c_str(), th, terr) != 0) {
                        closedir(dir);
                        return tbh::raise(FN(&turtle_stack_create), terr.code, terr.file, __LINE__,
                            "%s", terr.message.c_str());
                }
                const double x0 = th.x0, y0 = th.y0;
                const double dx = th.dx * (th.nx - 1);
                const double dy = th.dy * (th.ny - 1);
                if (long_delta == 0.)
                        long_delta = dx;
                else if (long_delta != dx) {
                        rc = TURTLE_RETURN_BAD_FORMAT;
                        errmsg = "inconsistent longitude span";
                        break;
                }
                if (lat_delta == 0.)
                        lat_delta = dy;
                else if (lat_delta != dy) {
                        rc = TURTLE_RETURN_BAD_FORMAT;
                        errmsg = "inconsistent latitude span";
                        break;
                }
                if (x0 < long_min) long_min = x0;
                if (y0 < lat_min) lat_min = y0;
                if (x0 + dx > long_max) long_max = x0 + dx;
                if (y0 + dy > lat_max) lat_max = y0 + dy;
                tb::MapDesc desc;
                memset(&desc, 0x0, sizeof desc);
                desc.nx = th.nx;
                desc.ny = th.ny;
                desc.x0 = th.x0;
                desc.y0 = th.y0;
                desc.dx = th.dx;
                desc.dy = th.dy;
                desc.z0 = th.z0;
                desc.dz = th.dz;
                desc.kind = th.kind;
                desc.pitch = th.nx;
                tb::map_desc_finish(desc);
                files.push_back({ full, x0, y0, desc });
        }
        closedir(dir);
        if (rc != TURTLE_RETURN_SUCCESS)
                return RAISE(&turtle_stack_create, rc, STACK_C, "%s", errmsg);

        int lat_n = 0, long_n = 0; /* ref: stack.c:134-148 */
        if ((lat_delta > 0.) && (long_delta > 0.)) {
                const double dx = (long_max - long_min) / long_delta;
                long_n = (int)(dx + FLT_EPSILON);
                if (fabs(long_n - dx) > FLT_EPSILON)
                        return RAISE(&turtle_stack_create, TURTLE_RETURN_BAD_FORMAT,
                            STACK_C, "invalid longitude grid");
                const double dy = (lat_max - lat_min) / lat_delta;
                lat_n = (int)(dy + FLT_EPSILON);
                if (fabs(lat_n - dy) > FLT_EPSILON)
                        return RAISE(&turtle_stack_create, TURTLE_RETURN_BAD_FORMAT,
                            STACK_C, "invalid latitude grid");
        }

        struct turtle_stack * s = new (std::nothrow) turtle_stack();
        if (s == NULL)
                return RAISE(&turtle_stack_create, TURTLE_RETURN_MEMORY_ERROR, STACK_C,
                    "could not allocate memory");
        s->max_size = (size > 0) ? size : INT_MAX;
        s->lock = lock;
        s->unlock = unlock;
        s->latitude_0 = lat_min;
        s->longitude_0 = long_min;
        s->latitude_delta = lat_delta;
        s->longitude_delta = long_delta;
        s->latitude_n = lat_n;
        s->longitude_n = long_n;
        s->root = path;
        *stack = s;
        /* a directory without tiles, or whose tiles have a null span (one row or column, no
         * pixel scale ...): an empty stack, as in the reference (stack.c:162-163) */
        if ((lat_n == 0) || (long_n == 0)) return TURTLE_RETURN_SUCCESS;
        s->path.assign((size_t)lat_n * long_n, std::string());
        s->tile.assign((size_t)lat_n * long_n, NULL);
        tb::MapDesc none;
        memset(&none, 0x0, sizeof none);
        s->header.assign((size_t)lat_n * long_n, none);
        for (size_t i = 0; i < files.size(); i++) { /* ref: stack.c:187-190 */
                const double fx = (files[i].x0 - long_min) / long_delta;
                const double fy = (files[i].y0 - lat_min) / lat_delta;
                if (!(fx >= 0.) || !(fx < long_n) || !(fy >= 0.) || !(fy < lat_n)) {
                        turtle_stack_destroy(stack);
                        return RAISE(&turtle_stack_create, TURTLE_RETURN_BAD_FORMAT, STACK_C,
                            "tile `%s' is off the grid of the stack", files[i].path.c_str());
                }
                const int ix = (int)fx, iy = (int)fy;
                s->path[(size_t)iy * long_n + ix] = files[i].path;
                s->header[(size_t)iy * long_n + ix] = files[i].desc;
        }
        return TURTLE_RETURN_SUCCESS;
}

static void stack_drop(struct turtle_stack * stack, int cell)
{
        struct turtle_map * m = stack->tile[cell];
        if (m == NULL) return;
        m->stack = NULL; /* no back search */
        stack->tile[cell] = NULL;
        stack->mru.erase(std::remove(stack->mru.begin(), stack->mru.end(), cell),
            stack->mru.end());
        turtle_map_destroy(&m);
}

extern "C" int turtle_stack_tiles_loaded(const struct turtle_stack * stack)
{
        return (stack == NULL) ? 0 : (int)stack->mru.size();
}

extern "C" void turtle_stack_destroy(struct turtle_stack ** stack)
{
        if ((stack == NULL) || (*stack == NULL)) return;
        for (size_t i = 0; i < (*stack)->tile.size(); i++) stack_drop(*stack, (int)i);
        delete *stack;
        *stack = NULL;
}

extern "C" enum turtle_return turtle_stack_clear(struct turtle_stack * stack)
{
        if ((stack->lock != NULL) && (stack->lock() != 0))
                return RAISE(&turtle_stack_clear, TURTLE_RETURN_LOCK_ERROR, STACK_C,
                    "could not acquire the lock");
        for (size_t i = 0; i < stack->tile.size(); i++) stack_drop(stack, (int)i);
        if ((stack->unlock != NULL) && (stack->unlock() != 0))
                return RAISE(&turtle_stack_clear, TURTLE_RETURN_UNLOCK_ERROR, STACK_C,
                    "could not release the lock");
        return TURTLE_RETURN_SUCCESS;
}

static void stack_touch(struct turtle_stack * stack, int cell)
{
        if (!stack->mru.empty() && (stack->mru[0] == cell)) return;
        stack->mru.erase(std::remove(stack->mru.begin(), stack->mru.end(), cell),
            stack->mru.end());
        stack->mru.insert(stack->mru.begin(), cell);
}

/* Load the tile of one grid cell; the least recently used tiles are evicted beyond
 * max_size (ref: stack.c:427-449). */
static enum turtle_return stack_load_cell(struct turtle_stack * stack, int cell,
    turtle_function_t * caller)
{
        if (stack->tile[cell] != NULL) return TURTLE_RETURN_SUCCESS;
        struct turtle_map * m;
        enum turtle_return rc = map_load_file(&m, stack->path[cell].c_str(), caller);
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        while ((int)stack->mru.size() >= stack->max_size && !stack->mru.empty())
                stack_drop(stack, stack->mru.back());
        m->stack = stack;
        stack->tile[cell] = m;
        stack->mru.insert(stack->mru.begin(), cell);
        return TURTLE_RETURN_SUCCESS;
}

enum turtle_return tbh::stack_load_all(struct turtle_stack * stack,
    turtle_function_t * caller)
{
        for (size_t i = 0; i < stack->path.size(); i++) {
                if (stack->path[i].empty()) continue;
                enum turtle_return rc = stack_load_cell(stack, (int)i, caller);
                if (rc != TURTLE_RETURN_SUCCESS) return rc;
        }
        return TURTLE_RETURN_SUCCESS;
}

/* ref: turtle_stack_load, stack.c:245-297: fill the stack up to max_size */
extern "C" enum turtle_return turtle_stack_load(struct turtle_stack * stack)
{
        if ((stack->latitude_n == 0) || (stack->longitude_n == 0))
                return TURTLE_RETURN_SUCCESS;
        if ((stack->lock != NULL) && (stack->lock() != 0))
                return RAISE(&turtle_stack_load, TURTLE_RETURN_LOCK_ERROR, STACK_C,
                    "could not acquire the lock");
        enum turtle_return rc = TURTLE_RETURN_SUCCESS;
        for (size_t i = 0; i < stack->path.size(); i++) {
                if ((int)stack->mru.size() >= stack->max_size) break;
                if (stack->path[i].empty() || (stack->tile[i] != NULL)) continue;
                rc = stack_load_cell(stack, (int)i, FN(&turtle_stack_load));
                if (rc != TURTLE_RETURN_SUCCESS) break;
        }
        if ((stack->unlock != NULL) && (stack->unlock() != 0))
                return RAISE(&turtle_stack_load, TURTLE_RETURN_UNLOCK_ERROR, STACK_C,
                    "could not release the lock");
        return rc;
}

/* The tile that answers a query at (latitude, longitude), with the ownership rules of
 * tb::stack_elevation, loading tiles on demand (and evicting beyond max_size, like the
 * reference: stack.c:413-449). *owner = its cell, or -1. */
static enum turtle_return stack_owner_scalar(struct turtle_stack * stack, double latitude,
    double longitude, int * owner_, turtle_function_t * caller)
{
        *owner_ = -1;
        if ((stack->latitude_n <= 0) || (stack->longitude_n <= 0) || isnan(latitude) ||
            isnan(longitude))
                return TURTLE_RETURN_SUCCESS;
        /* the candidate cell and, by rounding at a tile edge, its neighbours */
        double fx = (longitude - stack->longitude_0) / stack->longitude_delta;
        double fy = (latitude - stack->latitude_0) / stack->latitude_delta;
        if (!(fx >= 0.)) fx = 0.;
        if (!(fy >= 0.)) fy = 0.;
        const int cx = (fx < stack->longitude_n) ? (int)fx : stack->longitude_n - 1;
        const int cy = (fy < stack->latitude_n) ? (int)fy : stack->latitude_n - 1;
        int cells[9], n = 0;
        cells[n++] = cy * stack->longitude_n + cx;
        for (int jy = cy - 1; jy <= cy + 1; jy++)
                for (int jx = cx - 1; jx <= cx + 1; jx++) {
                        if ((jy < 0) || (jy >= stack->latitude_n) || (jx < 0) ||
                            (jx >= stack->longitude_n) || ((jx == cx) && (jy == cy)))
                                continue;
                        cells[n++] = jy * stack->longitude_n + jx;
                }
        int owner = -1;
        for (int k = 0; k < n; k++) {
                const int cell = cells[k];
                if (stack->path[cell].empty()) continue;
                /* ownership only needs the tile meta (x0, y0, dx, nx ...): the header
                 * read by turtle_stack_create when the tile is not loaded */
                if (stack->tile[cell] == NULL) {
                        if (!tb::tile_owns(stack->header[cell], latitude, longitude)) continue;
                        enum turtle_return rc = stack_load_cell(stack, cell, caller);
                        if (rc != TURTLE_RETURN_SUCCESS) return rc;
                } else if (!tb::tile_owns(map_desc(stack->tile[cell]), latitude, longitude))
                        continue;
                owner = cell;
                break;
        }
        if ((owner < 0) && !((longitude < stack->longitude_0) ||
                               (latitude < stack->latitude_0))) { /* ref: stack.c:413-425 */
                const double qx = (longitude - stack->longitude_0) / stack->longitude_delta;
                const double qy = (latitude - stack->latitude_0) / stack->latitude_delta;
                if ((qx < stack->longitude_n) && (qy < stack->latitude_n)) {
                        const int cell = (int)qy * stack->longitude_n + (int)qx;
                        if (!stack->path[cell].empty()) {
                                enum turtle_return rc = stack_load_cell(stack, cell, caller);
                                if (rc != TURTLE_RETURN_SUCCESS) return rc;
                                owner = cell;
                        }
                }
        }
        if (owner >= 0) stack_touch(stack, owner);
        *owner_ = owner;
        return TURTLE_RETURN_SUCCESS;
}

/* Scalar stack lookup (ref: turtle_stack_elevation, stack.c:338-361). */
static enum turtle_return stack_elevation_scalar(struct turtle_stack * stack,
    double latitude, double longitude, double * elevation, int * inside,
    turtle_function_t * caller)
{
        if (inside != NULL) *inside = 0;
        int owner;
        enum turtle_return rc = stack_owner_scalar(stack, latitude, longitude, &owner, caller);
        if (rc != TURTLE_RETURN_SUCCESS) {
                *elevation = 0.;
                return rc;
        }
        if (owner >= 0) {
                const int in = tb::map_elevation(map_desc(stack->tile[owner]), longitude,
                    latitude, *elevation);
                if (inside != NULL) {
                        *inside = in;
                        return TURTLE_RETURN_SUCCESS;
                }
                if (!in)
                        return tbh::raise(caller, TURTLE_RETURN_DOMAIN_ERROR, MAP_C, __LINE__,
                            "point is outside of map");
                return TURTLE_RETURN_SUCCESS;
        }
        *elevation = 0.; /* ref: stack.c:349-355 */
        if (inside != NULL) return TURTLE_RETURN_SUCCESS;
        return tbh::raise(caller, TURTLE_RETURN_PATH_ERROR, STACK_C, __LINE__,
            "missing elevation data in `%s'", stack->root.c_str());
}

extern "C" enum turtle_return turtle_stack_elevation(struct turtle_stack * stack,
    double latitude, double longitude, double * elevation, int * inside)
{
        return stack_elevation_scalar(stack, latitude, longitude, elevation, inside,
            FN(&turtle_stack_elevation));
}

/* ref: turtle_stack_gradient, stack.c:364-388: the tile that answers an elevation query
 * answers the gradient query (x = longitude, y = latitude). */
extern "C" enum turtle_return turtle_stack_gradient(struct turtle_stack * stack,
    double latitude, double longitude, double * glat, double * glon, int * inside)
{
        if (inside != NULL) *inside = 0;
        int owner;
        enum turtle_return rc = stack_owner_scalar(stack, latitude, longitude, &owner,
            FN(&turtle_stack_elevation));
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        int in = 0;
        if (owner >= 0)
                in = tb::map_gradient(map_desc(stack->tile[owner]), longitude, latitude, *glon,
                    *glat);
        if (!in) *glat = *glon = 0.;
        if (inside != NULL) {
                *inside = in;
                return TURTLE_RETURN_SUCCESS;
        }
        if (!in)
                return RAISE(&turtle_stack_elevation, TURTLE_RETURN_PATH_ERROR, STACK_C,
                    "missing elevation data in `%s'", stack->root.c_str());
        return TURTLE_RETURN_SUCCESS;
}

static const char * CLIENT_C = "src/turtle/client.c";

extern "C" enum turtle_return turtle_client_create(
    struct turtle_client ** client, struct turtle_stack * stack)
{
        *client = NULL;
        if (stack == NULL) /* ref: client.c:44-53 */
                return RAISE(&turtle_client_create, TURTLE_RETURN_BAD_ADDRESS, CLIENT_C,
                    "invalid null stack");
        if (stack->lock == NULL)
                return RAISE(&turtle_client_create, TURTLE_RETURN_BAD_ADDRESS, CLIENT_C,
                    "stack has no lock");
        *client = new (std::nothrow) turtle_client();
        if (*client == NULL)
                return RAISE(&turtle_client_create, TURTLE_RETURN_MEMORY_ERROR, CLIENT_C,
                    "could not allocate memory");
        (*client)->stack = stack;
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_client_destroy(struct turtle_client ** client)
{
        if ((client == NULL) || (*client == NULL)) return TURTLE_RETURN_SUCCESS;
        delete *client;
        *client = NULL;
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_client_clear(struct turtle_client * client)
{
        return TURTLE_RETURN_SUCCESS;
}

/* Same answer as the stack (ref: client.c:99-188), under the user's lock. */
extern "C" enum turtle_return turtle_client_elevation(struct turtle_client * client,
    double latitude, double longitude, double * elevation, int * inside)
{
        struct turtle_stack * stack = client->stack;
        if ((stack->lock != NULL) && (stack->lock() != 0))
                return RAISE(&turtle_client_elevation, TURTLE_RETURN_LOCK_ERROR, CLIENT_C,
                    "could not acquire the lock");
        enum turtle_return rc = stack_elevation_scalar(stack, latitude, longitude,
            elevation, inside, FN(&turtle_client_elevation));
        if ((stack->unlock != NULL) && (stack->unlock() != 0))
                return RAISE(&turtle_client_elevation, TURTLE_RETURN_UNLOCK_ERROR, CLIENT_C,
                    "could not release the lock");
        return rc;
}

/* ======================================================================== */
/* Stepper (ref: src/turtle/stepper.c)                                       */
/* ======================================================================== */

static const char * STEPPER_C = "src/turtle/stepper.c";

static void stepper_reset_history(struct turtle_stepper * stepper)
{
        tb::state_reset(stepper->state);
        /* every reference point (and the rest of the state, never read before it is
         * written) at DBL_MAX: stepper.c:602-615 */
        for (int i = 0; i < tb::LLA_ROWS_MAX; i++) stepper->lla[i] = DBL_MAX;
}

extern "C" enum turtle_return turtle_stepper_create(struct turtle_stepper ** stepper_)
{
        struct turtle_stepper * s = new (std::nothrow) turtle_stepper();
        if (s == NULL)
                return RAISE(&turtle_stepper_create, TURTLE_RETURN_MEMORY_ERROR, STEPPER_C,
                    "could not allocate memory");
        s->geoid = NULL;
        s->local_range = 1.; /* ref: stepper.c:558-560 */
        s->slope_factor = 0.4;
        s->resolution_factor = 1E-02;
        s->state.last.idx0 = s->state.last.idx1 = -1;
        s->state.last.elev0 = s->state.last.elev1 = 0.;
        s->state.last.lat = s->state.last.lon = s->state.last.alt = 0.;
        s->dirty = 1;
        s->lookup_rc = TURTLE_RETURN_SUCCESS;
        memset(&s->flat.G, 0x0, sizeof(s->flat.G));
        stepper_reset_history(s);
        *stepper_ = s;
        return TURTLE_RETURN_SUCCESS;
}

static std::mutex g_residency_mutex;

/* Drop the cached flattening before any change of the geometry. (The stepper holds no
 * claim on the tiles of its stacks: the scalar calls resolve them on demand, see
 * host_stack_lookup, so stacks and steppers may be destroyed in any order.) */
static void stepper_invalidate(struct turtle_stepper * s) { s->dirty = 1; }

extern "C" enum turtle_return turtle_stepper_destroy(struct turtle_stepper ** stepper)
{
        if ((stepper == NULL) || (*stepper == NULL)) return TURTLE_RETURN_SUCCESS;
        stepper_invalidate(*stepper);
        for (size_t i = 0; i < (*stepper)->data.size(); i++)
                turtle_client_destroy(&(*stepper)->data[i].client);
        delete *stepper;
        *stepper = NULL;
        return TURTLE_RETURN_SUCCESS;
}

extern "C" void turtle_stepper_geoid_set(
    struct turtle_stepper * stepper, struct turtle_map * geoid)
{
        stepper_invalidate(stepper);
        stepper->geoid = geoid;
        stepper_reset_history(stepper);
}

extern "C" struct turtle_map * turtle_stepper_geoid_get(
    const struct turtle_stepper * stepper)
{
        return stepper->geoid;
}

extern "C" double turtle_stepper_range_get(const struct turtle_stepper * stepper)
{
        return stepper->local_range;
}

extern "C" void turtle_stepper_range_set(struct turtle_stepper * stepper, double range)
{
        stepper->local_range = range;
        stepper->flat.G.range = range;
        stepper_reset_history(stepper);
}

extern "C" void turtle_stepper_reset(struct turtle_stepper * stepper)
{
        stepper_reset_history(stepper);
}

extern "C" double turtle_stepper_slope_get(const struct turtle_stepper * stepper)
{
        return stepper->slope_factor;
}

extern "C" void turtle_stepper_slope_set(struct turtle_stepper * stepper, double slope)
{
        stepper->slope_factor = slope;
        stepper->flat.G.slope = slope;
}

extern "C" double turtle_stepper_resolution_get(const struct turtle_stepper * stepper)
{
        return stepper->resolution_factor;
}

extern "C" void turtle_stepper_resolution_set(
    struct turtle_stepper * stepper, double resolution)
{
        stepper->resolution_factor = resolution;
        stepper->flat.G.resolution = resolution;
}

/* ref: stepper_add_layer, stepper.c:364-377: no-op while the top layer is empty */
extern "C" enum turtle_return turtle_stepper_add_layer(struct turtle_stepper * stepper)
{
        if (!stepper->layers.empty() && stepper->layers.back().empty())
                return TURTLE_RETURN_SUCCESS;
        stepper->layers.push_back(std::vector<tb_stepper_meta>());
        return TURTLE_RETURN_SUCCESS;
}

/* ref: add_data + add_meta, stepper.c:332-362, 390-409 */
static void stepper_attach(struct turtle_stepper * stepper, int data_index, double offset)
{
        if (stepper->layers.empty())
                stepper->layers.push_back(std::vector<tb_stepper_meta>());
        tb_stepper_meta meta = { data_index, offset };
        stepper->layers.back().push_back(meta);
}

static int stepper_transform(struct turtle_stepper * stepper, const char * name,
    const struct turtle_projection * projection)
{
        for (size_t i = 0; i < stepper->transforms.size(); i++)
                if (stepper->transforms[i].name == name) return (int)i;
        tb_stepper_transform t;
        t.name = name;
        tbh::projection_to_desc(projection, &t.proj);
        stepper->transforms.push_back(t);
        const int i = (int)stepper->transforms.size() - 1;
        if (i < tb::MAX_TRANSFORMS) /* stepper.c:349-351 (host blocks: LLA_BLOCK_MAX rows) */
                for (int k = 0; k < 3; k++) stepper->lla[tb::LLA_BLOCK_MAX * i + k] = DBL_MAX;
        return i;
}

extern "C" enum turtle_return turtle_stepper_add_stack(
    struct turtle_stepper * stepper, struct turtle_stack * stack, double offset)
{
        stepper_invalidate(stepper);
        int index = -1;
        for (size_t i = 0; i < stepper->data.size(); i++)
                if ((stepper->data[i].kind == tb::DATA_STACK) &&
                    (stepper->data[i].stack == stack))
                        index = (int)i;
        if (index < 0) {
                tb_stepper_data d = { tb::DATA_STACK, NULL, stack, NULL, 0 };
                if (stack->lock != NULL) { /* ref: stepper.c:432-436 */
                        enum turtle_return rc = turtle_client_create(&d.client, stack);
                        if (rc != TURTLE_RETURN_SUCCESS) return rc;
                }
                d.transform = stepper_transform(stepper, "geodetic", NULL);
                stepper->data.push_back(d);
                index = (int)stepper->data.size() - 1;
        }
        stepper_attach(stepper, index, offset);
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_stepper_add_map(
    struct turtle_stepper * stepper, struct turtle_map * map, double offset)
{
        stepper_invalidate(stepper);
        int index = -1;
        for (size_t i = 0; i < stepper->data.size(); i++)
                if ((stepper->data[i].kind == tb::DATA_MAP) && (stepper->data[i].map == map))
                        index = (int)i;
        if (index < 0) {
                tb_stepper_data d = { tb::DATA_MAP, map, NULL, NULL, 0 };
                const struct turtle_projection * projection = turtle_map_projection(map);
                const char * name = (projection == NULL) ?
                    "geodetic" :
                    turtle_projection_name(projection); /* stepper.c:494-498 */
                d.transform = stepper_transform(stepper, name, projection);
                stepper->data.push_back(d);
                index = (int)stepper->data.size() - 1;
        }
        stepper_attach(stepper, index, offset);
        return TURTLE_RETURN_SUCCESS;
}

extern "C" enum turtle_return turtle_stepper_add_flat(
    struct turtle_stepper * stepper, double offset)
{
        stepper_invalidate(stepper);
        int index = -1;
        for (size_t i = 0; i < stepper->data.size(); i++)
                if (stepper->data[i].kind == tb::DATA_FLAT) index = (int)i;
        if (index < 0) {
                tb_stepper_data d = { tb::DATA_FLAT, NULL, NULL, NULL, 0 };
                d.transform = stepper_transform(stepper, "geodetic", NULL);
                stepper->data.push_back(d);
                index = (int)stepper->data.size() - 1;
        }
        stepper_attach(stepper, index, offset);
        return TURTLE_RETURN_SUCCESS;
}

/* Steppers of different threads may share maps and stacks (one stepper per thread
 * is the reference's threading model, turtle.h:141-149): residency changes of a
 * stack are serialised here. */
/* Flatten the lists into tb::Geometry (host pointers). */
enum turtle_return tbh::stepper_flatten(struct turtle_stepper * s,
    turtle_function_t * caller)
{
        if (!s->dirty) {
                s->flat.G.range = s->local_range;
                s->flat.G.slope = s->slope_factor;
                s->flat.G.resolution = s->resolution_factor;
                return TURTLE_RETURN_SUCCESS;
        }
        enum turtle_return rc = tbh::flatten_into(s, s->flat, caller, 1, NULL);
        if (rc == TURTLE_RETURN_SUCCESS) s->dirty = 0;
        return rc;
}

/* Geodetic footprint of a projected map (tb::DataDesc::box): the border of the map is
 * walked node by node through the inverse projection; the box is widened by 1E-06 deg
 * (0.1 m) plus a bound on the bulge of an edge between two nodes, and dropped when the
 * footprint wraps in longitude, reaches +-180 deg or +-89 deg, or is not finite.
 *
 * The inverse UTM projection returns lon0 + atan2(...), which is not wrapped: a UTM 1N
 * map west of its zone unprojects to about -180.2 deg while its samples, from atan2, lie
 * at +179.8 deg and the projection, periodic in longitude, still sees them on the map. So
 * longitudes are brought into the (-180, 180] range of the samples first, and a footprint
 * that straddles or touches the antimeridian is not boxed at all. */
static void map_geodetic_box(const struct turtle_map * m, const tb::ProjDesc & P, tb::DataDesc & d)
{
        d.boxed = 0;
        d.box[0] = d.box[1] = d.box[2] = d.box[3] = 0.;
        if ((P.type == tb::PROJ_GEODETIC) || (m->nx < 2) || (m->ny < 2)) return;
        double la0 = DBL_MAX, la1 = -DBL_MAX, lo0 = DBL_MAX, lo1 = -DBL_MAX;
        const double x1 = m->x0 + m->dx * (m->nx - 1), y1 = m->y0 + m->dy * (m->ny - 1);
        for (int side = 0; side < 4; side++) {
                const int n = (side < 2) ? m->nx : m->ny;
                for (int k = 0; k < n; k++) {
                        const double x = (side < 2) ? m->x0 + k * m->dx : ((side == 2) ? m->x0 : x1);
                        const double y = (side < 2) ? ((side == 0) ? m->y0 : y1) : m->y0 + k * m->dy;
                        double la, lo;
                        tb::unproject(P, x, y, la, lo);
                        if (!isfinite(la) || !isfinite(lo)) return;
                        lo = remainder(lo, 360.); /* exact, in [-180, 180] */
                        la0 = std::min(la0, la);
                        la1 = std::max(la1, la);
                        lo0 = std::min(lo0, lo);
                        lo1 = std::max(lo1, lo);
                }
        }
        if ((lo1 - lo0 > 90.) || (la1 > 89.) || (la0 < -89.)) return;
        /* Between two border nodes h apart the extreme of latitude / longitude along the
         * edge can exceed both nodes by at most h^2 / 8 x the second derivative along the
         * edge, itself below 4 (1 + tan^2) / (R^2 cos) at the highest latitude of the
         * footprint (a generous bound for a conformal projection of the ellipsoid): the
         * box stays a superset of the footprint whatever the node spacing */
        const double phi = std::max(fabs(la0), fabs(la1)) * M_PI / 180.;
        const double h = std::max(fabs(m->dx), fabs(m->dy));
        const double curvature = 4. * (1. + tan(phi) * tan(phi)) /
            (TB_WGS84_B * TB_WGS84_B * cos(phi));
        const double margin = 1E-06 + 0.125 * h * h * curvature * 180. / M_PI;
        d.box[0] = la0 - margin;
        d.box[1] = la1 + margin;
        d.box[2] = lo0 - margin;
        d.box[3] = lo1 + margin;
        /* a footprint across the antimeridian has border nodes on both sides of it and
         * spans more than 90 deg after the wrap (dropped above); one that comes within
         * the margin of it may still bulge across */
        d.boxed = (d.box[2] > -180.) && (d.box[3] < 180.);
}

/* Does the closed footprint of a tile meet the region of a residency plan? */
static int tile_in_region(const tb::MapDesc & t, const struct turtle_residency * r)
{
        if (r == NULL) return 1;
        const double x1 = t.x0 + t.dx * t.nx1, y1 = t.y0 + t.dy * t.ny1;
        if (!isnan(r->longitude_min) && (x1 < r->longitude_min)) return 0;
        if (!isnan(r->longitude_max) && (t.x0 > r->longitude_max)) return 0;
        if (!isnan(r->latitude_min) && (y1 < r->latitude_min)) return 0;
        if (!isnan(r->latitude_max) && (t.y0 > r->latitude_max)) return 0;
        return 1;
}

/* The scalar calls resolve a stack query on the host like turtle_stack_elevation /
 * turtle_client_elevation do: tiles are loaded ON DEMAND and evicted beyond the `size`
 * given to turtle_stack_create (ref: stepper_step_stack / stepper_step_client,
 * stepper.c:199-225; stack.c:413-449). A load error is kept for turtle_stepper_step to
 * return. */
static int host_stack_lookup(void * context, int stack_index, double latitude,
    double longitude, double * z)
{
        struct turtle_stepper * s = (struct turtle_stepper *)context;
        int k = 0;
        for (size_t i = 0; i < s->data.size(); i++) {
                if (s->data[i].kind != tb::DATA_STACK) continue;
                if (k++ != stack_index) continue;
                int inside = 0;
                const enum turtle_return rc = (s->data[i].client != NULL) ?
                    turtle_client_elevation(s->data[i].client, latitude, longitude, z, &inside) :
                    turtle_stack_elevation(s->data[i].stack, latitude, longitude, z, &inside);
                if ((rc != TURTLE_RETURN_SUCCESS) && (s->lookup_rc == TURTLE_RETURN_SUCCESS))
                        s->lookup_rc = rc;
                return (rc == TURTLE_RETURN_SUCCESS) ? inside : 0;
        }
        return 0;
}

/* Flatten the lists into tb::Geometry.
 *   load_tiles = 1: the flattening of the scalar turtle.h calls (host): maps point to
 *                   host nodes, stacks are resolved through host_stack_lookup;
 *   load_tiles = 0: residency plan of a device -- tiles that are not on the host are
 *                   described from their file header only (F.src NULL, F.file set: the
 *                   freeze ingests them on the device), and tiles outside `region` are
 *                   left out of the plan (they answer `outside`). */
enum turtle_return tbh::flatten_into(struct turtle_stepper * s, tb_flat_geometry & F,
    turtle_function_t * caller, int load_tiles, const struct turtle_residency * region)
{
        std::lock_guard<std::mutex> guard(g_residency_mutex);
        F.maps.clear();
        F.src.clear();
        F.file.clear();
        F.tiles.clear();
        F.skipped = 0;
        tb::Geometry & G = F.G;
        memset(&G, 0x0, sizeof(G));

        size_t n_metas = 0;
        for (size_t i = 0; i < s->layers.size(); i++) n_metas += s->layers[i].size();
        size_t n_stacks = 0;
        for (size_t i = 0; i < s->data.size(); i++)
                if (s->data[i].kind == tb::DATA_STACK) n_stacks++;
        if ((s->layers.size() > tb::MAX_LAYERS) || (n_metas > tb::MAX_METAS) ||
            (s->data.size() > tb::MAX_DATA) ||
            (s->transforms.size() > tb::MAX_TRANSFORMS) || (n_stacks > tb::MAX_STACKS))
                return tbh::raise(caller, TURTLE_RETURN_MEMORY_ERROR, STEPPER_C, __LINE__,
                    "geometry too large (max %d layers, %d metas, %d data, %d transforms, "
                    "%d stacks)", tb::MAX_LAYERS, tb::MAX_METAS, tb::MAX_DATA,
                    tb::MAX_TRANSFORMS, tb::MAX_STACKS);

        G.n_layers = (int)s->layers.size();
        G.n_data = (int)s->data.size();
        G.n_transforms = (int)s->transforms.size();
        G.range = s->local_range;
        G.slope = s->slope_factor;
        G.resolution = s->resolution_factor;
        for (int t = 0; t < G.n_transforms; t++) G.transforms[t] = s->transforms[t].proj;

        for (int i = 0; i < G.n_data; i++) {
                const tb_stepper_data & d = s->data[i];
                G.data[i].kind = d.kind;
                G.data[i].transform = d.transform;
                G.data[i].ref = -1;
                if (d.kind == tb::DATA_MAP) {
                        G.data[i].ref = (int)F.maps.size();
                        F.maps.push_back(map_desc(d.map));
                        F.src.push_back(d.map);
                        F.file.push_back(std::string());
                        map_geodetic_box(d.map, G.transforms[d.transform], G.data[i]);
                } else if (d.kind == tb::DATA_STACK) {
                        struct turtle_stack * st = d.stack;
                        tb::StackDesc & S = G.stacks[G.n_stacks];
                        G.data[i].ref = G.n_stacks++;
                        S.lat0 = st->latitude_0;
                        S.dlat = st->latitude_delta;
                        S.lon0 = st->longitude_0;
                        S.dlon = st->longitude_delta;
                        S.inv_dlat = (st->latitude_delta > 0.) ? 1. / st->latitude_delta : 0.;
                        S.inv_dlon = (st->longitude_delta > 0.) ? 1. / st->longitude_delta : 0.;
                        S.nlat = st->latitude_n;
                        S.nlon = st->longitude_n;
                        S.tile0 = (int)F.tiles.size();
                        const tb::TileRec none = { NULL, 0., 0., -1, 0 };
                        const tb::MapDesc * first = NULL;
                        std::vector<tb::MapDesc> shapes(st->tile.size());
                        S.uniform = 1;
                        for (size_t c = 0; c < st->tile.size(); c++) {
                                const struct turtle_map * t = st->tile[c];
                                if (load_tiles || ((t == NULL) && st->path[c].empty())) {
                                        /* (host flattening: stacks are resolved through
                                         * G.host_stack, the tile table is not read) */
                                        F.tiles.push_back(none);
                                        continue;
                                }
                                /* a tile on the host is described by its map, else by
                                 * the header turtle_stack_create read from its file */
                                shapes[c] = (t != NULL) ? map_desc(t) : st->header[c];
                                if (!tile_in_region(shapes[c], region)) {
                                        F.tiles.push_back(none);
                                        F.skipped++;
                                        continue;
                                }
                                const tb::TileRec rec = { shapes[c].nodes, shapes[c].x0,
                                        shapes[c].y0, (int)F.maps.size(), 0 };
                                F.tiles.push_back(rec);
                                F.maps.push_back(shapes[c]);
                                F.src.push_back(st->tile[c]);
                                F.file.push_back((t != NULL) ? std::string() : st->path[c]);
                                if (first == NULL) first = &shapes[c];
                                if ((shapes[c].nx != first->nx) || (shapes[c].ny != first->ny) ||
                                    (shapes[c].dx != first->dx) || (shapes[c].dy != first->dy) ||
                                    (shapes[c].z0 != first->z0) || (shapes[c].dz != first->dz) ||
                                    (shapes[c].kind != first->kind))
                                        S.uniform = 0;
                        }
                        if (first != NULL) {
                                S.nx = first->nx;
                                S.ny = first->ny;
                                S.pitch = first->nx;
                                S.kind = first->kind;
                                S.dx = first->dx;
                                S.dy = first->dy;
                                S.z0 = first->z0;
                                S.dz = first->dz;
                                S.nx1 = (double)(first->nx - 1);
                                S.ny1 = (double)(first->ny - 1);
                                S.rdx = 1. / S.dx;
                                S.rdy = 1. / S.dy;
                        } else {
                                S.uniform = 0;
                        }
                        if (st->tile.empty()) { /* empty stack: 1 cell, no tile */
                                S.nlat = S.nlon = 1;
                                F.tiles.push_back(none);
                        }
                        S.nlat_d = (double)S.nlat;
                        S.nlon_d = (double)S.nlon;
                        /* do all tiles cover exactly their grid cell? (tb::stack_elevation) */
                        S.aligned = (S.dlat > 0.) && (S.dlon > 0.) && !st->tile.empty();
                        for (size_t c = 0; S.aligned && (c < st->tile.size()); c++) {
                                if (F.tiles[S.tile0 + c].map < 0) continue;
                                const tb::MapDesc * t = &shapes[c];
                                const double ix = (double)(c % (size_t)S.nlon);
                                const double iy = (double)(c / (size_t)S.nlon);
                                const double tol = 1E-09;
                                if (!(fabs((t->x0 - S.lon0) / S.dlon - ix) <= tol) ||
                                    !(fabs((t->y0 - S.lat0) / S.dlat - iy) <= tol) ||
                                    !(fabs((t->nx - 1) * t->dx / S.dlon - 1.) <= tol) ||
                                    !(fabs((t->ny - 1) * t->dy / S.dlat - 1.) <= tol))
                                        S.aligned = 0;
                        }
                }
        }
        G.geoid = -1;
        if (s->geoid != NULL) {
                G.geoid = (int)F.maps.size();
                F.maps.push_back(map_desc(s->geoid));
                F.src.push_back(s->geoid);
                F.file.push_back(std::string());
        }

        int first = 0;
        for (int L = 0; L < G.n_layers; L++) {
                const std::vector<tb_stepper_meta> & metas = s->layers[L];
                G.layers[L].first = first;
                G.layers[L].n = (int)metas.size();
                for (int k = 0; k < (int)metas.size(); k++) {
                        const tb_stepper_meta & m = metas[metas.size() - 1 - k];
                        G.metas[first + k].data = m.data;
                        G.metas[first + k].offset = m.offset;
                }
                first += (int)metas.size();
        }
        G.n_metas = first;
        G.maps = F.maps.data();
        G.tiles = F.tiles.data();
        /* per projected transform: the union of the footprints of its maps, widened by what
         * the local approximation can be off in latitude / longitude within its range */
        for (int t = 0; t < tb::MAX_TRANSFORMS; t++) {
                G.tboxed[t] = 0;
                G.tbox[t][0] = G.tbox[t][2] = DBL_MAX;
                G.tbox[t][1] = G.tbox[t][3] = -DBL_MAX;
        }
        for (int t = 0; t < G.n_transforms; t++) {
                if (G.transforms[t].type == tb::PROJ_GEODETIC) continue;
                int all = 1, any = 0;
                for (int i = 0; i < G.n_data; i++) {
                        if ((G.data[i].kind != tb::DATA_MAP) || (G.data[i].transform != t)) continue;
                        any = 1;
                        if (!G.data[i].boxed) all = 0;
                        G.tbox[t][0] = std::min(G.tbox[t][0], G.data[i].box[0]);
                        G.tbox[t][1] = std::max(G.tbox[t][1], G.data[i].box[1]);
                        G.tbox[t][2] = std::min(G.tbox[t][2], G.data[i].box[2]);
                        G.tbox[t][3] = std::max(G.tbox[t][3], G.data[i].box[3]);
                }
                /* (a sample in range is within r sqrt 3 of its reference point) */
                const double r = (G.range > 0.) ? G.range : 0.;
                const double rad = 180. / M_PI / TB_WGS84_B;
                const double slack = 4. * (r * r / TB_WGS84_B + 2. * r + 1E-03) * rad /
                    std::max(cos(89. * M_PI / 180.),
                        cos(std::max(fabs(G.tbox[t][0]), fabs(G.tbox[t][1])) * M_PI / 180.));
                G.tbox[t][0] -= slack;
                G.tbox[t][1] += slack;
                G.tbox[t][2] -= slack;
                G.tbox[t][3] += slack;
                /* Near the antimeridian the longitude a sample is culled with cannot be
                 * trusted: it may be linearised from a reference point whose finite
                 * difference Jacobian (10 m steps, stepper.c:144-162) jumps by 360 deg
                 * across the seam. A box that comes within the slack plus those 10 m of
                 * +-180 is dropped. So is one that reaches +-89 deg, the latitude up to
                 * which the slack above is conservative. */
                const double seam = slack + 40. * rad /
                    std::max(cos(89. * M_PI / 180.),
                        cos(std::max(fabs(G.tbox[t][0]), fabs(G.tbox[t][1])) * M_PI / 180.));
                G.tboxed[t] = any && all && isfinite(slack) &&
                    (G.tbox[t][2] - seam > -180.) && (G.tbox[t][3] + seam < 180.) &&
                    (G.tbox[t][0] > -89.) && (G.tbox[t][1] < 89.);
        }
        G.host_stack = load_tiles ? &host_stack_lookup : NULL;
        G.host_context = load_tiles ? (void *)s : NULL;
        tb::lla_layout(G, load_tiles);
        return TURTLE_RETURN_SUCCESS;
}

/* ref: sample_publish, stepper.c:758-778 */
static void publish(const struct turtle_stepper * s, double * latitude,
    double * longitude, double * altitude, double * elevation, int * index)
{
        const tb::Sample & last = s->state.last;
        if (latitude != NULL) *latitude = last.lat;
        if (longitude != NULL) *longitude = last.lon;
        if (altitude != NULL) *altitude = last.alt;
        if (elevation != NULL) {
                if (last.idx0 >= 0) {
                        elevation[0] = last.elev0;
                        elevation[1] = last.elev1;
                } else {
                        elevation[0] = 0.;
                        elevation[1] = 0.;
                }
        }
        if (index != NULL) {
                index[0] = last.idx0;
                index[1] = last.idx1;
        }
}

/* ref: turtle_stepper_step, stepper.c:780-875. One particle, on the host: the
 * set-up / debugging call. Batches go through turtle_stepper_*_batch (GPU). */
extern "C" enum turtle_return turtle_stepper_step(struct turtle_stepper * stepper,
    double * position, const double * direction, double * latitude,
    double * longitude, double * altitude, double * elevation,
    double * step_length, int * index)
{
        enum turtle_return rc = tbh::stepper_flatten(stepper, FN(&turtle_stepper_step));
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        const tb::Geometry & G = stepper->flat.G;
        stepper->lookup_rc = TURTLE_RETURN_SUCCESS;
        double ds;
        const tb::LlaView V = { stepper->lla, 1 };
        if (G.range > 0.)
                ds = tb::stepper_step<true>(G, V, stepper->state, position, direction);
        else
                ds = tb::stepper_step<false>(G, V, stepper->state, position, direction);
        if (stepper->lookup_rc != TURTLE_RETURN_SUCCESS)
                return stepper->lookup_rc; /* raised by the stack / client call already */
        publish(stepper, latitude, longitude, altitude, elevation, index);
        if (step_length != NULL) *step_length = ds;
        if ((stepper->state.last.idx0 < 0) && (index == NULL))
                return RAISE(&turtle_stepper_step, TURTLE_RETURN_DOMAIN_ERROR, STEPPER_C,
                    "no valid data");
        return TURTLE_RETURN_SUCCESS;
}

/* ref: turtle_stepper_position, stepper.c:877-931 */
extern "C" enum turtle_return turtle_stepper_position(struct turtle_stepper * stepper,
    double latitude, double longitude, double height, int layer_index,
    double * position, int * data_index)
{
        if ((layer_index < 0) || (layer_index >= (int)stepper->layers.size()))
                return RAISE(&turtle_stepper_position, TURTLE_RETURN_DOMAIN_ERROR,
                    STEPPER_C, "no valid data");
        enum turtle_return rc = tbh::stepper_flatten(stepper, FN(&turtle_stepper_position));
        if (rc != TURTLE_RETURN_SUCCESS) return rc;
        const tb::Geometry & G = stepper->flat.G;
        const tb::LayerDesc layer = G.layers[layer_index];
        stepper->lookup_rc = TURTLE_RETURN_SUCCESS;
        for (int k = 0; k < layer.n; k++) {
                const tb::MetaDesc & meta = G.metas[layer.first + k];
                const tb::DataDesc & d = G.data[meta.data];
                double z = 0.;
                int inside;
                if (d.kind == tb::DATA_FLAT) {
                        inside = 1;
                } else if (d.kind == tb::DATA_STACK) {
                        inside = tb::stack_elevation(G, G.stacks[d.ref], latitude, longitude, z);
                } else if (G.transforms[d.transform].type != tb::PROJ_GEODETIC) {
                        double x, y;
                        tb::project(G.transforms[d.transform], latitude, longitude, x, y);
                        inside = tb::map_elevation(G.maps[d.ref], x, y, z);
                } else {
                        inside = tb::map_elevation(G.maps[d.ref], longitude, latitude, z);
                }
                if (stepper->lookup_rc != TURTLE_RETURN_SUCCESS) return stepper->lookup_rc;
                if (!inside) continue;
                z += meta.offset;
                if (G.geoid >= 0) { /* ref: stepper.c:905-914 */
                        const double lo = (longitude >= 0) ? longitude : longitude + 360.;
                        double undulation;
                        if (tb::map_elevation(G.maps[G.geoid], lo, latitude, undulation))
                                z += undulation;
                }
                tb::ecef_from_geodetic(latitude, longitude, z + height, position);
                if (data_index != NULL) *data_index = k;
                return TURTLE_RETURN_SUCCESS;
        }
        if (data_index != NULL) {
                *data_index = -1;
                return TURTLE_RETURN_SUCCESS;
        }
        return RAISE(&turtle_stepper_position, TURTLE_RETURN_DOMAIN_ERROR, STEPPER_C,
            "no valid data");
}

/* ref: turtle_error_function, error.c:141-198 */
extern "C" const char * turtle_error_function(turtle_function_t * caller)
{
#define NAME(function) \
        if (caller == (turtle_function_t *)function) return #function
        NAME(turtle_client_clear);
        NAME(turtle_client_create);
        NAME(turtle_client_destroy);
        NAME(turtle_client_elevation);
        NAME(turtle_ecef_from_geodetic);
        NAME(turtle_ecef_from_horizontal);
        NAME(turtle_ecef_to_geodetic);
        NAME(turtle_ecef_to_horizontal);
        NAME(turtle_error_function);
        NAME(turtle_error_handler_get);
        NAME(turtle_error_handler_set);
        NAME(turtle_map_create);
        NAME(turtle_map_destroy);
        NAME(turtle_map_elevation);
        NAME(turtle_map_fill);
        NAME(turtle_map_gradient);
        NAME(turtle_map_load);
        NAME(turtle_map_dump);
        NAME(turtle_map_meta);
        NAME(turtle_map_node);
        NAME(turtle_map_projection);
        NAME(turtle_projection_configure);
        NAME(turtle_projection_create);
        NAME(turtle_projection_destroy);
        NAME(turtle_projection_name);
        NAME(turtle_projection_project);
        NAME(turtle_projection_unproject);
        NAME(turtle_stack_clear);
        NAME(turtle_stack_create);
        NAME(turtle_stack_destroy);
        NAME(turtle_stack_elevation);
        NAME(turtle_stack_gradient);
        NAME(turtle_stack_load);
        NAME(turtle_stepper_add_flat);
        NAME(turtle_stepper_add_layer);
        NAME(turtle_stepper_add_map);
        NAME(turtle_stepper_add_stack);
        NAME(turtle_stepper_create);
        NAME(turtle_stepper_destroy);
        NAME(turtle_stepper_geoid_get);
        NAME(turtle_stepper_geoid_set);
        NAME(turtle_stepper_range_get);
        NAME(turtle_stepper_range_set);
        NAME(turtle_stepper_position);
        NAME(turtle_stepper_step);
#undef NAME
        return tb_batch_function_name(caller);
}
