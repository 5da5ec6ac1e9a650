/*
 * turtle_oracle.c -- CPU RESTATEMENT of the reference's stepping path.
 *
 * TEST INFRASTRUCTURE ONLY. This file is the parity checker of turtle-b200: plain
 * C99 + glibc libm, compiled with -ffp-contract=off like the reference
 * (Makefile:2, -std=c99). It is never linked, imported or executed by the product
 * (turtle_b200/); only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline
 * / --impl reference legs use it, through oracle/trace_driver.c.
 *
 * It restates, from the reference's sources, the algorithm of
 *   turtle_stepper_step / stepper_sample / get_geographic  src/turtle/stepper.c
 *   turtle_ecef_*                                           src/turtle/ecef.c
 *   UTM / Lambert projections                               src/turtle/projection.c
 *   turtle_map_elevation                                    src/turtle/map.c
 *   stack tile lookup                                       src/turtle/stack.c
 *   the HGT node decoding                                   src/turtle/io/hgt.c
 * with arrays instead of linked lists and one translation unit instead of nine.
 * Unlike the product's core it keeps the reference's per-sample memo of data
 * results (stepper.c:173-197) and the MRU tile order (stack.c:300-335), so that
 * it can arbitrate when the product's simplifications are questioned.
 *
 * PINNING: tests/test_oracle.py checks this restatement bit-for-bit against the
 * compiled reference (oracle/_ref/libturtle_ref.so, when the reference's sources are
 * available), against the golden vectors under tests/golden/ that were generated
 * from the reference (tests/golden/make_golden.py), and against the closed-form
 * assertions of the reference's own test-suite (tests/test-turtle.c, listed in
 * SURVEY.md section 8c).
 *
 * It exports the subset of the turtle.h C ABI that trace_driver.c binds.
 */
#include <dirent.h>
#include <float.h>
#include <limits.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/stat.h>

#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif

enum { OK = 0, BAD_ADDRESS, BAD_EXTENSION, BAD_FORMAT, BAD_PROJECTION, BAD_JSON,
        DOMAIN_ERROR, LIBRARY_ERROR, LOCK_ERROR, MEMORY_ERROR, PATH_ERROR, UNLOCK_ERROR };

typedef void turtle_function_t(void);
typedef void turtle_error_handler_t(int, turtle_function_t *, const char *);
typedef int turtle_stack_locker_t(void);

static turtle_error_handler_t * handler = NULL;
void turtle_error_handler_set(turtle_error_handler_t * h) { handler = h; }

static int fail(int rc, void * fn, const char * message)
{
        if (handler != NULL) handler(rc, (turtle_function_t *)fn, message);
        return rc;
}

/* ====================================================================== */
/* ecef.c                                                                  */
/* ====================================================================== */

/* ecef.c:41-55 */
void turtle_ecef_from_geodetic(double latitude, double longitude, double elevation,
    double ecef[3])
{
        const double a = 6378137, e = 0.081819190842622; /* ecef.c:36-38 */
        const double s = sin(latitude * M_PI / 180.);
        const double c = cos(latitude * M_PI / 180.);
        const double R = a / sqrt(1. - e * e * s * s);
        ecef[0] = (R + elevation) * c * cos(longitude * M_PI / 180.);
        ecef[1] = (R + elevation) * c * sin(longitude * M_PI / 180.);
        ecef[2] = (R * (1. - e * e) + elevation) * s;
}

/* ecef.c:63-130 */
void turtle_ecef_to_geodetic(const double ecef[3], double * latitude,
    double * longitude, double * altitude)
{
        const double a = 6378137;
        const double e2 = 0.081819190842622 * 0.081819190842622;
        const double a1 = a * e2, a2 = a1 * a1, a3 = 0.5 * a1 * e2;
        const double a4 = 2.5 * a2, a5 = a1 + a3, a6 = 1. - e2;

        if ((ecef[0] == 0.) && (ecef[1] == 0.)) { /* ecef.c:77-84 */
                if (latitude) *latitude = (ecef[2] >= 0.) ? 90. : -90.;
                if (longitude) *longitude = 0.0;
                if (altitude) *altitude = fabs(ecef[2]) - 6356752.3142;
                return;
        }
        if (longitude) *longitude = atan2(ecef[1], ecef[0]) * 180. / M_PI;
        if (!latitude && !altitude) return;

        const double zp = fabs(ecef[2]);
        const double w2 = ecef[0] * ecef[0] + ecef[1] * ecef[1];
        const double w = sqrt(w2);
        const double z2 = ecef[2] * ecef[2];
        const double r2 = w2 + z2;
        const double r = sqrt(r2);
        const double s2 = z2 / r2;
        const double c2 = w2 / r2;
        double c, s, ss, la;
        if (c2 > 0.3) { /* ecef.c:101-108 */
                const double u = a2 / r;
                const double v = a3 - a4 / r;
                s = (zp / r) * (1. + c2 * (a1 + u + s2 * v) / r);
                la = asin(s);
                ss = s * s;
                c = sqrt(1. - ss);
        } else { /* ecef.c:109-115 */
                const double u = a2 / r;
                const double v = a3 - a4 / r;
                c = (w / r) * (1. - s2 * (a5 - u - c2 * v) / r);
                la = acos(c);
                ss = 1. - c * c;
                s = sqrt(ss);
        }
        const double g = 1. - e2 * ss; /* ecef.c:117-129 */
        const double rg = a / sqrt(g);
        const double rf = a6 * rg;
        const double u = w - rg * c;
        const double v = zp - rf * s;
        const double f = c * u + s * v;
        const double m = c * v - s * u;
        const double p = m / (rf / g + f);
        la += p;
        if (ecef[2] < 0.) la = -la;
        if (latitude) *latitude = la * 180. / M_PI;
        if (altitude) *altitude = f + 0.5 * m * p;
}

/* ecef.c:136-154 */
static void enu(double latitude, double longitude, double e[3], double n[3], double u[3])
{
        const double lambda = longitude * M_PI / 180.;
        const double phi = latitude * M_PI / 180.;
        const double sl = sin(lambda), cl = cos(lambda), sp = sin(phi), cp = cos(phi);
        e[0] = -sl, e[1] = cl, e[2] = 0.;
        n[0] = -cl * sp, n[1] = -sl * sp, n[2] = cp;
        u[0] = cl * cp, u[1] = sl * cp, u[2] = sp;
}

/* ecef.c:160-178 */
void turtle_ecef_from_horizontal(double latitude, double longitude, double azimuth,
    double elevation, double direction[3])
{
        double e[3], n[3], u[3];
        enu(latitude, longitude, e, n, u);
        const double az = azimuth * M_PI / 180.;
        const double el = elevation * M_PI / 180.;
        const double ce = cos(el);
        const double r[3] = { ce * sin(az), ce * cos(az), sin(el) };
        for (int i = 0; i < 3; i++) direction[i] = r[0] * e[i] + r[1] * n[i] + r[2] * u[i];
}

/* ecef.c:180-207 */
void turtle_ecef_to_horizontal(double latitude, double longitude,
    const double direction[3], double * azimuth, double * elevation)
{
        double e[3], n[3], u[3];
        enu(latitude, longitude, e, n, u);
        const double x = e[0] * direction[0] + e[1] * direction[1] + e[2] * direction[2];
        const double y = n[0] * direction[0] + n[1] * direction[1] + n[2] * direction[2];
        const double z = u[0] * direction[0] + u[1] * direction[1] + u[2] * direction[2];
        double r = direction[0] * direction[0] + direction[1] * direction[1] +
            direction[2] * direction[2];
        if (r <= FLT_EPSILON) return;
        r = sqrt(r);
        if (azimuth) *azimuth = atan2(x, y) * 180. / M_PI;
        if (elevation) {
                const double arg = z / r;
                *elevation = (arg > 1.) ? 90. : (arg < -1.) ? -90. : asin(arg) * 180. / M_PI;
        }
}

/* ====================================================================== */
/* projection.c                                                            */
/* ====================================================================== */

struct turtle_projection {
        int kind; /* -1 none, 0 Lambert, 1 UTM */
        double longitude_0;
        int hemisphere;
        int lambert;
        char tag[64];
};

static int word(const char ** s)
{
        while (**s == ' ') (*s)++;
        int n = 0;
        while (((*s)[n] != ' ') && ((*s)[n] != 0)) n++;
        return n;
}

/* projection.c:98-172 */
static int projection_configure(struct turtle_projection * p, const char * name)
{
        p->kind = -1;
        p->tag[0] = 0;
        if (name == NULL) return OK;
        const char * s = name;
        int n = word(&s);
        if (n == 0) return BAD_PROJECTION;
        if (strncmp(s, "Lambert", n) == 0) {
                static const char * tags[6] = { "I", "II", "IIe", "III", "IV", "93" };
                p->kind = 0;
                s += n;
                n = word(&s);
                int i;
                for (i = 0; i < 6; i++)
                        if (strncmp(s, tags[i], n) == 0) break;
                if (i == 6) return BAD_PROJECTION;
                p->lambert = i;
        } else if (strncmp(s, "UTM", n) == 0) {
                p->kind = 1;
                s += n;
                int zone;
                char h;
                if (sscanf(s, "%d%c", &zone, &h) != 2) return BAD_PROJECTION;
                if (h == '.') {
                        double l0;
                        if (sscanf(s, "%lf%c", &l0, &h) != 2) return BAD_PROJECTION;
                        p->longitude_0 = l0;
                } else
                        p->longitude_0 = 6. * zone - 183.;
                if (h == 'N')
                        p->hemisphere = 1;
                else if (h == 'S')
                        p->hemisphere = -1;
                else
                        return BAD_PROJECTION;
        } else
                return BAD_PROJECTION;
        strncpy(p->tag, name, sizeof(p->tag) - 1);
        p->tag[sizeof(p->tag) - 1] = 0;
        return OK;
}

int turtle_projection_create(struct turtle_projection ** projection, const char * name)
{
        struct turtle_projection tmp;
        *projection = NULL;
        const int rc = projection_configure(&tmp, name);
        if (rc != OK) return fail(rc, &turtle_projection_create, "invalid projection");
        *projection = malloc(sizeof(tmp));
        memcpy(*projection, &tmp, sizeof(tmp));
        return OK;
}

void turtle_projection_destroy(struct turtle_projection ** projection)
{
        if (projection && *projection) {
                free(*projection);
                *projection = NULL;
        }
}

/* projection.c:327-347: e, n, c, lambda_c, xs, ys for I, II, IIe, III, IV, 93 */
static const double lambert_set[6][6] = {
        { 0.08248325676, 0.7604059656, 11603796.98, 0.04079234433, 600000.0, 5657616.674 },
        { 0.08248325676, 0.7289686274, 11745793.39, 0.04079234433, 600000.0, 6199695.768 },
        { 0.08248325676, 0.7289686274, 11745793.39, 0.04079234433, 600000.0, 8199695.768 },
        { 0.08248325676, 0.6959127966, 11947992.52, 0.04079234433, 600000.0, 6791905.085 },
        { 0.08248325676, 0.6712679322, 12136281.99, 0.04079234433, 234.358, 7239161.542 },
        { 0.08181919112, 0.7253743710, 11755528.70, 0.05235987756, 700000.0, 12657560.145 } };

static void project(const struct turtle_projection * p, double latitude, double longitude,
    double * x, double * y)
{
        if (p->kind == 0) { /* projection.c:239-245, 286-295 */
                const double * q = lambert_set[p->lambert];
                const double e = q[0], n = q[1];
                const double phi = latitude * M_PI / 180.;
                const double s = sin(phi);
                const double L = log(tan(0.25 * M_PI + 0.5 * phi) *
                    pow((1. - e * s) / (1. + e * s), 0.5 * e));
                const double cenL = q[2] * exp(-n * L);
                const double lambda = longitude / 180. * M_PI;
                const double theta = n * (lambda - q[3]);
                *x = q[4] + cenL * sin(theta);
                *y = q[5] - cenL * cos(theta);
        } else { /* projection.c:377-408 */
                const double a = 6378.137E+03, f = 1. / 298.257223563;
                const double E0 = 5E+05, N0 = (p->hemisphere > 0) ? 0. : 1E+07, k0 = 0.9996;
                const double n = f / (2. - f);
                const double A = a / (1. + n) * (1. + n * n * (0.25 + 0.0625 * n * n));
                const double alpha[3] = { n * (0.5 + n * (-2. / 3. + 5. / 16. * n)),
                        n * n * (13. / 48. - 3. / 5. * n), 61. / 240. * n * n * n };
                const double c = 2. * sqrt(n) / (1. + n);
                const double s = sin(latitude * M_PI / 180.);
                const double t = sinh(atanh(s) - c * atanh(c * s));
                const double dl = (longitude - p->longitude_0) * M_PI / 180.;
                const double zeta = atan2(t, cos(dl));
                const double eta = atanh(sin(dl) / sqrt(1. + t * t));
                double xs = 0., ys = 0.;
                for (int i = 0; i < 3; i++) {
                        xs += alpha[i] * cos(2. * (i + 1) * zeta) * sinh(2. * (i + 1) * eta);
                        ys += alpha[i] * sin(2. * (i + 1) * zeta) * cosh(2. * (i + 1) * eta);
                }
                *x = E0 + k0 * A * (eta + xs);
                *y = N0 + k0 * A * (zeta + ys);
        }
}

static void unproject(const struct turtle_projection * p, double x, double y,
    double * latitude, double * longitude)
{
        if (p->kind == 0) { /* projection.c:254-268, 304-316 */
                const double * q = lambert_set[p->lambert];
                const double e = q[0], n = q[1];
                const double dx = x - q[4], dy = y - q[5];
                const double R = sqrt(dx * dx + dy * dy);
                const double gamma = atan2(dx, -dy);
                *longitude = (q[3] + gamma / n) * 180. / M_PI;
                const double L = -log(R / q[2]) / n;
                const double eL = exp(L);
                double phi0 = 2. * atan(eL) - 0.5 * M_PI;
                for (;;) {
                        const double s = sin(phi0);
                        const double phi1 =
                            2. * atan(pow((1. + e * s) / (1. - e * s), 0.5 * e) * eL) -
                            0.5 * M_PI;
                        if (fabs(phi1 - phi0) <= FLT_EPSILON) {
                                *latitude = phi1 / M_PI * 180.;
                                return;
                        }
                        phi0 = phi1;
                }
        } else { /* projection.c:417-448 */
                const double a = 6378.137E+03, f = 1. / 298.257223563;
                const double E0 = 5E+05, N0 = (p->hemisphere > 0) ? 0. : 1E+07, k0 = 0.9996;
                const double n = f / (2. - f);
                const double A = a / (1. + n) * (1. + n * n * (0.25 + 0.0625 * n * n));
                const double beta[3] = { n * (0.5 + n * (-2. / 3. + 37. / 96. * n)),
                        n * n * (1. / 48. + 1. / 15. * n), 17. / 480. * n * n * n };
                const double delta[3] = { n * (2. + n * (-2. / 3. - 2. * n)),
                        n * n * (7. / 3. - 8. / 5. * n), 56. / 15. * n * n * n };
                const double zeta0 = (y - N0) / (k0 * A);
                const double eta0 = (x - E0) / (k0 * A);
                double zeta = zeta0, eta = eta0;
                for (int i = 0; i < 3; i++) {
                        zeta -= beta[i] * sin(2. * (i + 1) * zeta0) * cosh(2. * (i + 1) * eta0);
                        eta -= beta[i] * cos(2. * (i + 1) * zeta0) * sinh(2. * (i + 1) * eta0);
                }
                const double chi = asin(sin(zeta) / cosh(eta));
                double s = 0.;
                for (int i = 0; i < 3; i++) s += delta[i] * sin(2. * (i + 1) * chi);
                *latitude = (chi + s) * 180. / M_PI;
                *longitude = p->longitude_0 + atan2(sinh(eta), cos(zeta)) * 180. / M_PI;
        }
}

/* projection.c:192-233 */
int turtle_projection_project(const struct turtle_projection * p, double latitude,
    double longitude, double * x, double * y)
{
        *x = *y = 0.;
        if (p == NULL) return fail(BAD_ADDRESS, &turtle_projection_project, "missing projection");
        if (p->kind < 0)
                return fail(BAD_PROJECTION, &turtle_projection_project, "invalid projection");
        project(p, latitude, longitude, x, y);
        return OK;
}

int turtle_projection_unproject(const struct turtle_projection * p, double x, double y,
    double * latitude, double * longitude)
{
        *latitude = *longitude = 0.;
        if (p == NULL)
                return fail(BAD_ADDRESS, &turtle_projection_unproject, "missing projection");
        if (p->kind < 0)
                return fail(BAD_PROJECTION, &turtle_projection_unproject, "invalid projection");
        unproject(p, x, y, latitude, longitude);
        return OK;
}

/* ====================================================================== */
/* map.c + io/hgt.c                                                        */
/* ====================================================================== */

struct turtle_map_info {
        int nx, ny;
        double x[2], y[2], z[2];
        const char * encoding;
};

struct turtle_map {
        int nx, ny;
        double x0, y0, z0, dx, dy, dz;
        int hgt; /* nodes are raw HGT file content: big-endian int16, north first */
        struct turtle_projection projection;
        uint16_t * data;
};

/* map.c:41-44 (default) and io/hgt.c:127-131 (HGT) */
static double get_z(const struct turtle_map * map, int ix, int iy)
{
        if (map->hgt) {
                iy = map->ny - 1 - iy;
                const uint16_t raw = map->data[(size_t)iy * map->nx + ix];
                return (int16_t)(uint16_t)((raw << 8) | (raw >> 8)); /* ntohs */
        }
        return map->z0 + map->data[(size_t)iy * map->nx + ix] * map->dz;
}

/* map.c:54-99 */
int turtle_map_create(struct turtle_map ** map, const struct turtle_map_info * info,
    const char * projection)
{
        *map = NULL;
        if ((info->nx <= 0) || (info->ny <= 0) || (info->z[0] == info->z[1]))
                return fail(DOMAIN_ERROR, &turtle_map_create, "invalid input parameter(s)");
        struct turtle_projection proj;
        if (projection_configure(&proj, projection) != OK)
                return fail(BAD_PROJECTION, &turtle_map_create, "invalid projection");
        struct turtle_map * m = calloc(1, sizeof(*m));
        m->data = calloc((size_t)info->nx * info->ny, sizeof(uint16_t));
        m->nx = info->nx;
        m->ny = info->ny;
        m->x0 = info->x[0];
        m->y0 = info->y[0];
        m->z0 = info->z[0];
        m->dx = (info->nx > 1) ? (info->x[1] - info->x[0]) / (info->nx - 1) : 0.;
        m->dy = (info->ny > 1) ? (info->y[1] - info->y[0]) / (info->ny - 1) : 0.;
        m->dz = (info->z[1] - info->z[0]) / 65535;
        m->projection = proj;
        *map = m;
        return OK;
}

void turtle_map_destroy(struct turtle_map ** map)
{
        if (map && *map) {
                free((*map)->data);
                free(*map);
                *map = NULL;
        }
}

/* map.c:183-203 with the default setter, map.c:47-51 */
int turtle_map_fill(struct turtle_map * map, int ix, int iy, double elevation)
{
        if (map == NULL) return fail(MEMORY_ERROR, &turtle_map_fill, "no map");
        if ((ix < 0) || (ix >= map->nx) || (iy < 0) || (iy >= map->ny))
                return fail(DOMAIN_ERROR, &turtle_map_fill, "point is outside of map");
        if ((map->dz <= 0.) && (elevation != map->z0))
                return fail(DOMAIN_ERROR, &turtle_map_fill, "inconsistent elevation value");
        if ((elevation < map->z0) || (elevation > map->z0 + 65535 * map->dz))
                return fail(DOMAIN_ERROR, &turtle_map_fill, "elevation is outside of map span");
        const double d = round((elevation - map->z0) / map->dz);
        map->data[(size_t)iy * map->nx + ix] = (uint16_t)d;
        return OK;
}

/* map.c:206-226 */
int turtle_map_node(const struct turtle_map * map, int ix, int iy, double * x, double * y,
    double * elevation)
{
        if ((map == NULL) || (ix < 0) || (ix >= map->nx) || (iy < 0) || (iy >= map->ny))
                return fail(DOMAIN_ERROR, &turtle_map_node, "point is outside of map");
        if (x) *x = map->x0 + ix * map->dx;
        if (y) *y = map->y0 + iy * map->dy;
        if (elevation) *elevation = get_z(map, ix, iy);
        return OK;
}

/* map.c:229-277 */
int turtle_map_elevation(const struct turtle_map * map, double x, double y, double * z,
    int * inside)
{
        int out = isnan(x) || isnan(y);
        double hx = 0., hy = 0.;
        if (!out) {
                hx = (x - map->x0) / map->dx;
                hy = (y - map->y0) / map->dy;
                out = (hx > map->nx - 1) || (hx < 0) || (hy > map->ny - 1) || (hy < 0);
        }
        if (out) {
                if (inside != NULL) {
                        *inside = 0;
                        return OK;
                }
                return fail(DOMAIN_ERROR, &turtle_map_elevation, "point is outside of map");
        }
        int ix = (int)hx, iy = (int)hy;
        if (ix == map->nx - 1) {
                ix--;
                hx = 1.;
        } else
                hx -= ix;
        if (iy == map->ny - 1) {
                iy--;
                hy = 1.;
        } else
                hy -= iy;
        const double z00 = get_z(map, ix, iy);
        const double z10 = get_z(map, ix + 1, iy);
        const double z01 = get_z(map, ix, iy + 1);
        const double z11 = get_z(map, ix + 1, iy + 1);
        *z = z00 * (1. - hx) * (1. - hy) + z01 * (1. - hx) * hy + z10 * hx * (1. - hy) +
            z11 * hx * hy;
        if (inside != NULL) *inside = 1;
        return OK;
}

/* map.c:280-378, first-row behaviour of :353 included (the y slope lands in *gx) */
int turtle_map_gradient(const struct turtle_map * map, double x, double y, double * gx,
    double * gy, int * inside)
{
        int out = isnan(x) || isnan(y);
        double hx = 0., hy = 0.;
        if (!out) {
                hx = (x - map->x0) / map->dx;
                hy = (y - map->y0) / map->dy;
                out = (hx > map->nx - 1) || (hx < 0) || (hy > map->ny - 1) || (hy < 0);
        }
        if (out) {
                if (inside != NULL) {
                        *inside = 0;
                        return OK;
                }
                return fail(DOMAIN_ERROR, &turtle_map_elevation, "point is outside of map");
        }
        int ix = (int)hx, iy = (int)hy;
        if (ix == map->nx - 1) {
                ix--;
                hx = 1.;
        } else
                hx -= ix;
        if (iy == map->ny - 1) {
                iy--;
                hy = 1.;
        } else
                hy -= iy;
        const double z00 = get_z(map, ix, iy), z10 = get_z(map, ix + 1, iy);
        const double z01 = get_z(map, ix, iy + 1), z11 = get_z(map, ix + 1, iy + 1);
        if (hx <= 0.5) {
                const double gx1 = (z10 - z00) * (1. - hy) + (z11 - z01) * hy;
                if (ix == 0) {
                        *gx = gx1 / map->dx;
                } else {
                        const double z_10 = get_z(map, ix - 1, iy), z_11 = get_z(map, ix - 1, iy + 1);
                        const double gx0 = (z00 - z_10) * (1. - hy) + (z01 - z_11) * hy;
                        const double ax = hx + 0.5;
                        *gx = (gx0 * (1. - ax) + gx1 * ax) / map->dx;
                }
        } else {
                const double gx0 = (z10 - z00) * (1. - hy) + (z11 - z01) * hy;
                if (ix == map->nx - 2) {
                        *gx = gx0 / map->dx;
                } else {
                        const double z20 = get_z(map, ix + 2, iy), z21 = get_z(map, ix + 2, iy + 1);
                        const double gx1 = (z20 - z10) * (1. - hy) + (z21 - z11) * hy;
                        const double ax = hx - 0.5;
                        *gx = (gx0 * (1. - ax) + gx1 * ax) / map->dx;
                }
        }
        if (hy <= 0.5) {
                const double gy1 = (z01 - z00) * (1. - hx) + (z11 - z10) * hx;
                if (iy == 0) {
                        *gx = gy1 / map->dy; /* map.c:353 */
                } else {
                        const double z0_1 = get_z(map, ix, iy - 1), z1_1 = get_z(map, ix + 1, iy - 1);
                        const double gy0 = (z00 - z0_1) * (1. - hx) + (z10 - z1_1) * hx;
                        const double ay = hy + 0.5;
                        *gy = (gy0 * (1. - ay) + gy1 * ay) / map->dy;
                }
        } else {
                const double gy0 = (z01 - z00) * (1. - hx) + (z11 - z10) * hx;
                if (iy == map->ny - 2) {
                        *gy = gy0 / map->dy;
                } else {
                        const double z02 = get_z(map, ix, iy + 2), z12 = get_z(map, ix + 1, iy + 2);
                        const double gy1 = (z02 - z01) * (1. - hx) + (z12 - z11) * hx;
                        const double ay = hy - 0.5;
                        *gy = (gy0 * (1. - ay) + gy1 * ay) / map->dy;
                }
        }
        if (inside != NULL) *inside = 1;
        return OK;
}

/* io/hgt.c:61-104 (file name -> grid) and :135-147 (raw read) */
static struct turtle_map * hgt_load(const char * path, int meta_only)
{
        const char * name = path;
        for (const char * p = path; *p; p++)
                if ((*p == '/') || (*p == '\\')) name = p + 1;
        if (strlen(name) < 8) return NULL;
        struct turtle_map * m = calloc(1, sizeof(*m));
        m->x0 = atoi(name + 4);
        if (name[3] == 'W')
                m->x0 = -m->x0;
        else if (name[3] != 'E')
                goto bad;
        m->y0 = atoi(name + 1);
        if (name[0] == 'S')
                m->y0 = -m->y0;
        else if (name[0] != 'N')
                goto bad;
        const char * ext = NULL;
        for (const char * p = name + 7; *p; p++)
                if (*p == '.') ext = p + 1;
        if (ext == NULL) goto bad;
        const int n = (int)(ext - name) - 8;
        m->nx = m->ny = ((n == 0) || (strncmp(name + 8, "SRTMGL1", n - 1) == 0)) ? 3601 : 1201;
        m->dx = 1. / (m->nx - 1);
        m->dy = 1. / (m->ny - 1);
        m->z0 = -32767.;
        m->dz = 1.;
        m->hgt = 1;
        m->projection.kind = -1;
        if (meta_only) return m;
        FILE * fid = fopen(path, "rb");
        if (fid == NULL) goto bad;
        const size_t count = (size_t)m->nx * m->ny;
        m->data = malloc(count * sizeof(uint16_t));
        const size_t got = fread(m->data, sizeof(uint16_t), count, fid);
        fclose(fid);
        if (got != count) {
                free(m->data);
                goto bad;
        }
        return m;
bad:
        free(m);
        return NULL;
}

/* ====================================================================== */
/* stack.c                                                                 */
/* ====================================================================== */

struct turtle_stack {
        turtle_stack_locker_t * lock; /* stack.h:40-42: guards the MRU list */
        turtle_stack_locker_t * unlock;
        double latitude_0, latitude_delta, longitude_0, longitude_delta;
        int latitude_n, longitude_n;
        char ** path;               /* per grid cell, NULL when no file */
        struct turtle_map ** tiles; /* loaded tiles in MRU order, tiles[0] = head */
        int * cell;                 /* grid cell of each loaded tile */
        int size;
};

static int is_hgt(const char * name)
{
        const char * ext = strrchr(name, '.');
        return (ext != NULL) && (strcmp(ext, ".hgt") == 0);
}

/* stack.c:46-201, HGT files only */
int turtle_stack_create(struct turtle_stack ** stack, const char * path, int size,
    turtle_stack_locker_t * lock, turtle_stack_locker_t * unlock)
{
        *stack = NULL;
        if ((lock == NULL) != (unlock == NULL))
                return fail(BAD_ADDRESS, &turtle_stack_create, "inconsistent lock & unlock");
        DIR * dir = opendir(path);
        if (dir == NULL) return fail(PATH_ERROR, &turtle_stack_create, "could not access path");
        double lat_min = DBL_MAX, long_min = DBL_MAX, lat_max = -DBL_MAX, long_max = -DBL_MAX;
        double lat_delta = 0., long_delta = 0.;
        struct dirent * entry;
        char full[4096];
        while ((entry = readdir(dir)) != NULL) { /* stack.c:71-128 */
                if (!is_hgt(entry->d_name)) continue;
                snprintf(full, sizeof full, "%s/%s", path, entry->d_name);
                struct turtle_map * meta = hgt_load(full, 1);
                if (meta == NULL) continue;
                const double dx = meta->dx * (meta->nx - 1);
                const double dy = meta->dy * (meta->ny - 1);
                int bad = 0;
                if (long_delta == 0.)
                        long_delta = dx;
                else if (long_delta != dx)
                        bad = 1;
                if (lat_delta == 0.)
                        lat_delta = dy;
                else if (lat_delta != dy)
                        bad = 1;
                if (bad) {
                        free(meta);
                        closedir(dir);
                        return fail(BAD_FORMAT, &turtle_stack_create, "inconsistent tile span");
                }
                if (meta->x0 < long_min) long_min = meta->x0;
                if (meta->y0 < lat_min) lat_min = meta->y0;
                if (meta->x0 + dx > long_max) long_max = meta->x0 + dx;
                if (meta->y0 + dy > lat_max) lat_max = meta->y0 + dy;
                free(meta);
        }
        int lat_n = 0, long_n = 0; /* stack.c:134-148 */
        if ((lat_delta > 0.) && (long_delta > 0.)) {
                const double dx = (long_max - long_min) / long_delta;
                long_n = (int)(dx + FLT_EPSILON);
                const double dy = (lat_max - lat_min) / lat_delta;
                lat_n = (int)(dy + FLT_EPSILON);
                if ((fabs(long_n - dx) > FLT_EPSILON) || (fabs(lat_n - dy) > FLT_EPSILON)) {
                        closedir(dir);
                        return fail(BAD_FORMAT, &turtle_stack_create, "invalid grid");
                }
        }
        struct turtle_stack * s = calloc(1, sizeof(*s));
        s->lock = lock;
        s->unlock = unlock;
        s->latitude_0 = lat_min;
        s->longitude_0 = long_min;
        s->latitude_delta = lat_delta;
        s->longitude_delta = long_delta;
        s->latitude_n = lat_n;
        s->longitude_n = long_n;
        const int cells = lat_n * long_n;
        s->path = calloc(cells > 0 ? cells : 1, sizeof(char *));
        s->tiles = calloc(cells > 0 ? cells : 1, sizeof(*s->tiles));
        s->cell = calloc(cells > 0 ? cells : 1, sizeof(int));
        rewinddir(dir);
        while ((entry = readdir(dir)) != NULL) { /* stack.c:170-196 */
                if (!is_hgt(entry->d_name)) continue;
                snprintf(full, sizeof full, "%s/%s", path, entry->d_name);
                struct turtle_map * meta = hgt_load(full, 1);
                if (meta == NULL) continue;
                const int ix = (int)((meta->x0 - long_min) / long_delta);
                const int iy = (int)((meta->y0 - lat_min) / lat_delta);
                s->path[iy * long_n + ix] = strdup(full);
                free(meta);
        }
        closedir(dir);
        *stack = s;
        return OK;
}

void turtle_stack_destroy(struct turtle_stack ** stack)
{
        if (!stack || !*stack) return;
        struct turtle_stack * s = *stack;
        for (int i = 0; i < s->size; i++) turtle_map_destroy(&s->tiles[i]);
        for (int i = 0; i < s->latitude_n * s->longitude_n; i++) free(s->path[i]);
        free(s->path);
        free(s->tiles);
        free(s->cell);
        free(s);
        *stack = NULL;
}

static void touch(struct turtle_stack * s, int k) /* stack.c:391-396 */
{
        struct turtle_map * m = s->tiles[k];
        const int c = s->cell[k];
        for (; k > 0; k--) {
                s->tiles[k] = s->tiles[k - 1];
                s->cell[k] = s->cell[k - 1];
        }
        s->tiles[0] = m;
        s->cell[0] = c;
}

/* turtle_stack_load_, stack.c:399-450. A tile that is already resident is not read
 * twice (the reference would load a duplicate with identical content). */
static int stack_load_at(struct turtle_stack * s, double latitude, double longitude)
{
        if ((longitude < s->longitude_0) || (latitude < s->latitude_0)) return 0;
        const int ix = (int)((longitude - s->longitude_0) / s->longitude_delta);
        if (ix >= s->longitude_n) return 0;
        const int iy = (int)((latitude - s->latitude_0) / s->latitude_delta);
        if (iy >= s->latitude_n) return 0;
        const int index = iy * s->longitude_n + ix;
        if (s->path[index] == NULL) return 0;
        for (int k = 0; k < s->size; k++)
                if (s->cell[k] == index) {
                        touch(s, k);
                        return 1;
                }
        struct turtle_map * m = hgt_load(s->path[index], 0);
        if (m == NULL) return 0;
        s->tiles[s->size] = m;
        s->cell[s->size] = index;
        touch(s, s->size++);
        return 1;
}

/* turtle_stack_load, stack.c:245-297: every tile of the grid */
int turtle_stack_load(struct turtle_stack * s)
{
        for (int iy = 0; iy < s->latitude_n; iy++)
                for (int ix = 0; ix < s->longitude_n; ix++)
                        stack_load_at(s, s->latitude_0 + (iy + 0.5) * s->latitude_delta,
                            s->longitude_0 + (ix + 0.5) * s->longitude_delta);
        return OK;
}

/* stack_get_map + turtle_stack_elevation, stack.c:300-361. When the stack was given
 * lock callbacks the MRU bookkeeping runs under the lock and the owning tile is
 * interpolated outside of it, which is what a turtle_client does (client.c:126-188;
 * tiles are never evicted here, so no reference counting is needed). */
int turtle_stack_elevation(struct turtle_stack * s, double latitude, double longitude,
    double * elevation, int * inside)
{
        if (inside != NULL) *inside = 0;
        if (s->lock != NULL) s->lock();
        int found = 0;
        for (int k = 0; k < s->size; k++) {
                const struct turtle_map * m = s->tiles[k];
                const double hx = (longitude - m->x0) / m->dx;
                const double hy = (latitude - m->y0) / m->dy;
                if ((hx >= 0.) && (hx < m->nx - 1) && (hy >= 0.) && (hy < m->ny - 1)) {
                        touch(s, k);
                        found = 1;
                        break;
                }
        }
        if (!found && !stack_load_at(s, latitude, longitude)) {
                if (s->unlock != NULL) s->unlock();
                *elevation = 0.;
                if (inside != NULL) return OK;
                return fail(PATH_ERROR, &turtle_stack_elevation, "missing elevation data");
        }
        const struct turtle_map * owner = s->tiles[0];
        if (s->unlock != NULL) s->unlock();
        return turtle_map_elevation(owner, longitude, latitude, elevation, inside);
}

/* turtle_stack_gradient, stack.c:364-388 */
int turtle_stack_gradient(struct turtle_stack * s, double latitude, double longitude,
    double * glat, double * glon, int * inside)
{
        if (inside != NULL) *inside = 0;
        if (s->lock != NULL) s->lock();
        int found = 0;
        for (int k = 0; k < s->size; k++) {
                const struct turtle_map * m = s->tiles[k];
                const double hx = (longitude - m->x0) / m->dx;
                const double hy = (latitude - m->y0) / m->dy;
                if ((hx >= 0.) && (hx < m->nx - 1) && (hy >= 0.) && (hy < m->ny - 1)) {
                        touch(s, k);
                        found = 1;
                        break;
                }
        }
        if (!found && !stack_load_at(s, latitude, longitude)) {
                if (s->unlock != NULL) s->unlock();
                *glat = *glon = 0.;
                if (inside != NULL) return OK;
                return fail(PATH_ERROR, &turtle_stack_elevation, "missing elevation data");
        }
        const struct turtle_map * owner = s->tiles[0];
        if (s->unlock != NULL) s->unlock();
        return turtle_map_gradient(owner, longitude, latitude, glon, glat, inside);
}

/* ====================================================================== */
/* stepper.c                                                               */
/* ====================================================================== */

#define MAXN 32

struct transform { /* stepper.h:45-58 */
        char name[64];
        double reference_ecef[3], reference_geographic[5], data[5][3];
        int updated;
        double geographic[5];
};

enum { FLAT, MAP, STACK };

struct data { /* stepper.h:60-79 */
        int kind;
        struct turtle_map * map;
        struct turtle_stack * stack;
        int transform;
        int updated, inside;
        double geographic[5], elevation;
};

struct meta {
        int data;
        double offset;
};

struct layer {
        struct meta meta[MAXN];
        int n;
};

struct sample { /* stepper.h:93-98 */
        double position[3], geographic[5], elevation[2];
        int index[2];
};

struct turtle_stepper { /* stepper.h:101-110 */
        struct data data[MAXN];
        int n_data;
        struct transform transforms[MAXN];
        int n_transforms;
        struct layer layers[MAXN];
        int n_layers;
        struct turtle_map * geoid;
        double local_range, slope_factor, resolution_factor;
        struct sample last;
};

static void reset_history(struct turtle_stepper * s) /* stepper.c:602-615 */
{
        for (int i = 0; i < 3; i++) s->last.position[i] = DBL_MAX;
        for (int t = 0; t < s->n_transforms; t++)
                for (int i = 0; i < 3; i++) s->transforms[t].reference_ecef[i] = DBL_MAX;
}

int turtle_stepper_create(struct turtle_stepper ** stepper) /* stepper.c:547-570 */
{
        struct turtle_stepper * s = calloc(1, sizeof(*s));
        s->local_range = 1.;
        s->slope_factor = 0.4;
        s->resolution_factor = 1E-02;
        s->last.index[0] = s->last.index[1] = -1;
        reset_history(s);
        *stepper = s;
        return OK;
}

int turtle_stepper_destroy(struct turtle_stepper ** stepper)
{
        if (stepper && *stepper) {
                free(*stepper);
                *stepper = NULL;
        }
        return OK;
}

void turtle_stepper_geoid_set(struct turtle_stepper * s, struct turtle_map * geoid)
{
        s->geoid = geoid;
        reset_history(s);
}
void turtle_stepper_range_set(struct turtle_stepper * s, double range)
{
        s->local_range = range;
        reset_history(s);
}
void turtle_stepper_reset(struct turtle_stepper * s) { reset_history(s); }
void turtle_stepper_slope_set(struct turtle_stepper * s, double slope) { s->slope_factor = slope; }
void turtle_stepper_resolution_set(struct turtle_stepper * s, double r) { s->resolution_factor = r; }

int turtle_stepper_add_layer(struct turtle_stepper * s) /* stepper.c:364-377 */
{
        if ((s->n_layers > 0) && (s->layers[s->n_layers - 1].n == 0)) return OK;
        if (s->n_layers >= MAXN) return fail(MEMORY_ERROR, &turtle_stepper_add_layer, "too many layers");
        s->layers[s->n_layers++].n = 0;
        return OK;
}

/* add_data + add_meta, stepper.c:332-362, 390-409 */
static int attach(struct turtle_stepper * s, int kind, struct turtle_map * map,
    struct turtle_stack * stack, const char * transform, double offset)
{
        int d;
        for (d = 0; d < s->n_data; d++)
                if ((s->data[d].kind == kind) && (s->data[d].map == map) &&
                    (s->data[d].stack == stack))
                        break;
        if (d == s->n_data) {
                if (s->n_data >= MAXN) return MEMORY_ERROR;
                int t;
                for (t = 0; t < s->n_transforms; t++)
                        if (strcmp(s->transforms[t].name, transform) == 0) break;
                if (t == s->n_transforms) {
                        strncpy(s->transforms[t].name, transform, 63);
                        for (int i = 0; i < 3; i++) s->transforms[t].reference_ecef[i] = DBL_MAX;
                        s->n_transforms++;
                }
                s->data[d].kind = kind;
                s->data[d].map = map;
                s->data[d].stack = stack;
                s->data[d].transform = t;
                s->n_data++;
        }
        if (s->n_layers == 0) turtle_stepper_add_layer(s);
        struct layer * layer = &s->layers[s->n_layers - 1];
        if (layer->n >= MAXN) return MEMORY_ERROR;
        layer->meta[layer->n].data = d;
        layer->meta[layer->n].offset = offset;
        layer->n++;
        return OK;
}

int turtle_stepper_add_flat(struct turtle_stepper * s, double offset)
{
        return attach(s, FLAT, NULL, NULL, "geodetic", offset);
}
int turtle_stepper_add_stack(struct turtle_stepper * s, struct turtle_stack * stack, double offset)
{
        return attach(s, STACK, NULL, stack, "geodetic", offset);
}
int turtle_stepper_add_map(struct turtle_stepper * s, struct turtle_map * map, double offset)
{
        return attach(s, MAP, map, NULL,
            (map->projection.kind < 0) ? "geodetic" : map->projection.tag, offset);
}

/* ecef_to_geodetic with the geoid, stepper.c:37-51 */
static void to_geodetic(struct turtle_stepper * s, const double * position, double * g)
{
        turtle_ecef_to_geodetic(position, g, g + 1, g + 2);
        if (s->geoid != NULL) {
                int inside;
                double undulation;
                const double lo = (g[1] >= 0) ? g[1] : g[1] + 360.;
                turtle_map_elevation(s->geoid, lo, g[0], &undulation, &inside);
                if (inside) g[2] -= undulation;
        }
}

/* compute_geodetic / compute_geomap, stepper.c:57-83 */
static void compute(struct turtle_stepper * s, struct data * d, const double * position,
    int n0, double * g)
{
        if (n0 == 0) to_geodetic(s, position, g);
        if ((d->kind == MAP) && (d->map->projection.kind >= 0))
                project(&d->map->projection, g[0], g[1], g + 3, g + 4);
}

/* get_geographic, stepper.c:85-171 */
static void get_geographic(struct turtle_stepper * s, struct data * d, const double * position,
    int n0, int n1, double * g)
{
        struct transform * t = &s->transforms[d->transform];
        if (t->updated) {
                memcpy(g + n0, t->geographic + n0, (n1 - n0) * sizeof(double));
                return;
        }
        if (s->local_range <= 0.) {
                compute(s, d, position, n0, g);
        } else {
                double local[3], range = 0.;
                for (int i = 0; i < 3; i++) {
                        double r = position[i] - t->reference_ecef[i];
                        local[i] = r;
                        r = fabs(r);
                        if (r > range) range = r;
                }
                if (range < s->local_range) {
                        for (int i = n0; i < n1; i++) {
                                g[i] = t->reference_geographic[i];
                                for (int j = 0; j < 3; j++) g[i] += t->data[i][j] * local[j];
                        }
                } else {
                        compute(s, d, position, n0, g);
                        double step = 0.;
                        for (int i = 0; i < 3; i++) {
                                const double q = fabs(position[i] - s->last.position[i]);
                                if (q > step) step = q;
                        }
                        if (step < 0.33 * s->local_range) {
                                memcpy(t->reference_ecef, position, 3 * sizeof(double));
                                memcpy(t->reference_geographic + n0, g + n0,
                                    (n1 - n0) * sizeof(double));
                                for (int i = 0; i < 3; i++) {
                                        double r[3] = { position[0], position[1], position[2] };
                                        r[i] += 10.;
                                        double g1[5];
                                        compute(s, d, r, 0, g1);
                                        for (int j = n0; j < n1; j++)
                                                t->data[j][i] = 0.1 * (g1[j] - g[j]);
                                }
                        }
                }
        }
        memcpy(t->geographic + n0, g + n0, (n1 - n0) * sizeof(double));
        t->updated = 1;
}

/* stepper_step and the four data steppers, stepper.c:173-264 */
static void data_step(struct turtle_stepper * s, struct data * d, const double * position,
    int has_geodetic, double * g, double * elevation, int * inside)
{
        if (d->updated) {
                memcpy(g, d->geographic, sizeof(d->geographic));
                *elevation = d->elevation;
                *inside = d->inside;
                return;
        }
        *inside = 0;
        if ((d->kind == MAP) && (d->map->projection.kind >= 0)) {
                get_geographic(s, d, position, has_geodetic ? 3 : 0, 5, g);
                turtle_map_elevation(d->map, g[3], g[4], elevation, inside);
        } else {
                if (!has_geodetic) get_geographic(s, d, position, 0, 3, g);
                if (d->kind == FLAT) {
                        *inside = 1;
                        *elevation = 0.;
                } else if (d->kind == MAP) {
                        turtle_map_elevation(d->map, g[1], g[0], elevation, inside);
                } else {
                        turtle_stack_elevation(d->stack, g[0], g[1], elevation, inside);
                }
        }
        d->updated = 1;
        memcpy(d->geographic, g, sizeof(d->geographic));
        d->elevation = *elevation;
        d->inside = *inside;
}

/* stepper_sample + check_layer, stepper.c:687-756 */
static void stepper_sample(struct turtle_stepper * s, const double * position,
    struct sample * sample)
{
        if ((position[0] == s->last.position[0]) && (position[1] == s->last.position[1]) &&
            (position[2] == s->last.position[2])) {
                if (sample != &s->last) memcpy(sample, &s->last, sizeof(*sample));
                return;
        }
        for (int t = 0; t < s->n_transforms; t++) s->transforms[t].updated = 0;
        for (int d = 0; d < s->n_data; d++) s->data[d].updated = 0;
        sample->index[0] = sample->index[1] = -1;
        sample->elevation[0] = -DBL_MAX;
        sample->elevation[1] = DBL_MAX;
        int has_geodetic = 0;
        for (int L = 0; L < s->n_layers; L++) {
                struct layer * layer = &s->layers[L];
                for (int k = 0; k < layer->n; k++) {
                        struct meta * meta = &layer->meta[layer->n - 1 - k];
                        int inside;
                        double elevation = 0.;
                        data_step(s, &s->data[meta->data], position, has_geodetic,
                            sample->geographic, &elevation, &inside);
                        if (sample == &s->last)
                                memcpy(s->last.position, position, sizeof(s->last.position));
                        has_geodetic = 1;
                        if (inside) {
                                elevation += meta->offset;
                                if (elevation >= sample->geographic[2]) {
                                        sample->index[0] = L;
                                        sample->index[1] = k;
                                        sample->elevation[1] = elevation;
                                        return;
                                }
                                sample->index[0] = L + 1;
                                sample->index[1] = k;
                                sample->elevation[0] = elevation;
                                break;
                        }
                }
        }
}

/* sample_publish, stepper.c:758-778 */
static void publish(struct turtle_stepper * s, double * latitude, double * longitude,
    double * altitude, double * elevation, int * index)
{
        if (latitude) *latitude = s->last.geographic[0];
        if (longitude) *longitude = s->last.geographic[1];
        if (altitude) *altitude = s->last.geographic[2];
        if (elevation) {
                elevation[0] = (s->last.index[0] >= 0) ? s->last.elevation[0] : 0.;
                elevation[1] = (s->last.index[0] >= 0) ? s->last.elevation[1] : 0.;
        }
        if (index) {
                index[0] = s->last.index[0];
                index[1] = s->last.index[1];
        }
}

/* turtle_stepper_step, stepper.c:780-875 */
int turtle_stepper_step(struct turtle_stepper * s, double * position, const double * direction,
    double * latitude, double * longitude, double * altitude, double * elevation,
    double * step_length, int * index)
{
        stepper_sample(s, position, &s->last);
        if (s->last.index[0] < 0) {
                publish(s, latitude, longitude, altitude, elevation, index);
                if (step_length) *step_length = 0;
                if (index == NULL) return fail(DOMAIN_ERROR, &turtle_stepper_step, "no valid data");
                return OK;
        }
        double ds = 0.; /* stepper.c:798-813 */
        for (int i = 0; i < 2; i++) {
                if ((s->last.index[0] == 0) && (i == 0))
                        continue;
                else if ((s->last.index[0] == s->n_layers) && (i == 1))
                        break;
                const double dsi = fabs(s->last.geographic[2] - s->last.elevation[i]);
                if ((dsi < ds) || (ds <= 0.)) ds = dsi;
        }
        ds *= s->slope_factor;
        if (ds < s->resolution_factor) ds = s->resolution_factor;
        if (direction == NULL) {
                publish(s, latitude, longitude, altitude, elevation, index);
                if (step_length) *step_length = ds;
                return OK;
        }
        for (int i = 0; i < 3; i++) position[i] += direction[i] * ds;
        const int medium0 = s->last.index[0];
        stepper_sample(s, position, &s->last);
        if (medium0 != s->last.index[0]) { /* stepper.c:832-864 */
                double ds0 = -ds, ds1 = 0.;
                struct sample sample2;
                memcpy(&sample2, &s->last, sizeof(sample2));
                while (ds1 - ds0 > 1E-08) {
                        const double ds2 = 0.5 * (ds0 + ds1);
                        double position2[3] = { position[0] + direction[0] * ds2,
                                position[1] + direction[1] * ds2,
                                position[2] + direction[2] * ds2 };
                        stepper_sample(s, position2, &sample2);
                        if (sample2.index[0] == medium0) {
                                ds0 = ds2;
                        } else {
                                ds1 = ds2;
                                memcpy(sample2.position, position2, sizeof(sample2.position));
                                memcpy(&s->last, &sample2, sizeof(s->last));
                        }
                }
                ds += ds1;
                for (int i = 0; i < 3; i++) position[i] += direction[i] * ds1;
        }
        publish(s, latitude, longitude, altitude, elevation, index);
        if (step_length) *step_length = ds;
        if ((s->last.index[0] < 0) && (index == NULL))
                return fail(DOMAIN_ERROR, &turtle_stepper_step, "no valid data");
        return OK;
}

/* turtle_stepper_position, stepper.c:877-931 (+ stepper_elevation_*, :266-324) */
int turtle_stepper_position(struct turtle_stepper * s, double latitude, double longitude,
    double height, int layer_index, double * position, int * data_index)
{
        if ((layer_index < 0) || (layer_index >= s->n_layers))
                return fail(DOMAIN_ERROR, &turtle_stepper_position, "no valid data");
        struct layer * layer = &s->layers[layer_index];
        for (int k = 0; k < layer->n; k++) {
                struct meta * meta = &layer->meta[layer->n - 1 - k];
                struct data * d = &s->data[meta->data];
                int inside = 0;
                double elevation = 0.;
                if (d->kind == FLAT) {
                        inside = 1;
                } else if (d->kind == STACK) {
                        turtle_stack_elevation(d->stack, latitude, longitude, &elevation, &inside);
                } else if (d->map->projection.kind >= 0) {
                        double x, y;
                        project(&d->map->projection, latitude, longitude, &x, &y);
                        turtle_map_elevation(d->map, x, y, &elevation, &inside);
                } else {
                        turtle_map_elevation(d->map, longitude, latitude, &elevation, &inside);
                }
                if (!inside) continue;
                elevation += meta->offset;
                if (s->geoid != NULL) {
                        int in;
                        double undulation;
                        const double lo = (longitude >= 0) ? longitude : longitude + 360.;
                        turtle_map_elevation(s->geoid, lo, latitude, &undulation, &in);
                        if (in) elevation += undulation;
                }
                turtle_ecef_from_geodetic(latitude, longitude, elevation + height, position);
                if (data_index) *data_index = k;
                return OK;
        }
        if (data_index) {
                *data_index = -1;
                return OK;
        }
        return fail(DOMAIN_ERROR, &turtle_stepper_position, "no valid data");
}
