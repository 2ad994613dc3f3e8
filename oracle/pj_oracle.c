/*
 * oracle/pj_oracle.c -- TEST INFRASTRUCTURE ONLY.  Never linked into libfimex_b200.so; only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load it.
 *
 * CPU restatement (plain C99 + libm) of the part of PROJ.4 that the reference's regridding path calls
 * through the classic proj_api.h API: pj_init_plus / pj_transform / pj_is_latlong / pj_free /
 * pj_strerrno / pj_errno (call sites: /root/reference/src/interpolation.c:355,366,396,402,408,
 * 623-644,681-700,734-773,1168-1185,1208-1233).
 *
 * Third-party dependency restated here: PROJ.4 "libproj", classic API.  The reference pins no
 * version (CMakeLists.txt:44 only looks for proj_api.h; README.md:16 says "proj-4 >= 4.4.9";
 * debian_bionic/control:22 => 4.9.3).  This file follows the PUBLISHED ALGORITHM of PROJ 4.9.x
 * (pj_init.c, pj_ell_set.c, pj_datum_set.c, pj_transform.c, pj_fwd.c, pj_inv.c, adjlon.c, dmstor.c,
 * aasincos.c, pj_tsfn.c, pj_phi2.c, pj_msfn.c, PJ_latlong.c, PJ_ob_tran.c, PJ_stere.c, PJ_lcc.c) as
 * recalled from its documentation / Snyder, "Map Projections - A Working Manual" (USGS PP 1395).
 * PROJ itself is not available in this image (no source, no binary, no pyproj), so this file cannot be compared with
 * libproj's output.  It is pinned instead by INDEPENDENT known answers (tests/proj_known_answers.py,
 * tests/test_proj_known_answers.py; the same assertions run against the GPU transforms):
 *   - Snyder's printed numerical examples, to the printed digits: Lambert conformal conic on the sphere and on the Clarke
 *     1866 ellipsoid (pp. 295-297), oblique stereographic on the sphere (pp. 312-313), polar stereographic on the
 *     International ellipsoid (p. 315), forward and inverse;
 *   - Snyder's equations (14-x, 15-x, 21-x) written out in numpy, on 2e4 random points per case, <= 1e-9 degree of arc:
 *     lcc and polar stere on sphere / WGS84 / Clarke 1866 / International, oblique stere on the sphere;
 *   - rotated pole (ob_tran +o_proj=longlat) against an explicit 3-D change of basis built from the CF definition of the
 *     rotated pole, 1e5 random points, <= 1e-12 degree away from the poles of both frames (<= 2e-11 degree of arc at them), and the very mesh of BASELINE
 *     config 2;
 *   - the reference's own tests at the PROJ boundary (test/testInterpolation.cc:265-278, 280-393, 396-512, 515-654;
 *     test/testInterpolator.cc:398-472), re-run in tests/test_oracle_golden.py and tests/test_gpu_parity.py.
 *   - 3- and 7-parameter datum shifts (+towgs84, +datum=WGS84|NAD83) against an independent geocentric reference
 *     (tests/datum_reference.py: geodetic -> ECEF, position-vector Helmert, PROJ 4's R^T inverse, Heikkinen's closed form
 *     polished by Newton in long double), <= 1e-11 degree of arc on random CRS pairs of all four families, plus the parser's
 *     +ellps / +datum / +towgs84 precedence and the early exits (tests/test_datum_reference_host.py).
 *   What remains UNPINNED: grid shifts (+nadgrids, refused) and the last-ulp behaviour of libproj itself (libm differences).
 *
 * Supported grammar (SURVEY.md 8a row P): +proj=latlong|longlat|latlon|lonlat, ob_tran (+o_proj one of
 * the four lat/long names, +o_lat_p, +o_lon_p), stere (+lat_0 +lon_0 +lat_ts | +k|+k_0), lcc (+lat_1
 * +lat_2 +lat_0 +lon_0), plus +x_0 +y_0 +a +b +rf +f +e +es +R +ellps=(sphere|WGS84|GRS80|bessel|
 * intl|clrk66|krass) +datum=(WGS84|NAD83) +towgs84 +units=(m|km) +to_meter +over +geoc +no_defs.
 */
#include "shim/proj_api.h"

#include <ctype.h>
#include <errno.h>
#include <stdio.h>
#include <string.h>

#define ORC_HALFPI 1.5707963267948966
#define ORC_FORTPI 0.78539816339744833
#define ORC_PI 3.14159265358979323846
#define ORC_TWOPI 6.2831853071795864769
#define ORC_SPI 3.14159265359 /* adjlon.c: deliberately short */

enum { PJD_UNKNOWN = 0, PJD_3PARAM = 1, PJD_7PARAM = 2, PJD_GRIDSHIFT = 3, PJD_WGS84 = 4 };
enum { KIND_LATLONG = 0, KIND_OB_TRAN = 1, KIND_STERE = 2, KIND_LCC = 3 };
enum { ST_S_POLE = 0, ST_N_POLE = 1, ST_OBLIQ = 2, ST_EQUIT = 3 };

#define MAX_PARAMS 64
#define MAX_TOKEN 128

typedef struct {
    char key[MAX_TOKEN];
    char val[MAX_TOKEN];
    int has_val;
} orc_param;

typedef struct {
    orc_param p[MAX_PARAMS];
    int n;
} orc_plist;

typedef struct orc_pj {
    int kind;
    int is_latlong;
    int over, geoc;
    double a, ra, es, e, one_es, rone_es, a_orig, es_orig;
    double lam0, phi0, x0, y0, k0, to_meter, fr_meter;
    int datum_type;
    double datum_params[7];
    /* stere */
    int mode;
    double phits, akm1, sinX1, cosX1;
    /* lcc */
    double phi1, phi2, n, rho0, c;
    int ellips;
    /* ob_tran (link is always a lat/long pseudo-projection here) */
    double lamp, cphip, sphip;
    int oblique;
    /* per-call error state (PROJ keeps it in the context) */
    int last_errno;
} orc_pj;

int pj_errno = 0;

/* ---------------------------------------------------------------- parameter list (pj_param.c) */

static const orc_param* pl_find(const orc_plist* pl, const char* key)
{
    for (int i = 0; i < pl->n; ++i)
        if (strcmp(pl->p[i].key, key) == 0)
            return &pl->p[i];
    return NULL;
}

static int pl_has(const orc_plist* pl, const char* key)
{
    return pl_find(pl, key) != NULL;
}

static int pl_append(orc_plist* pl, const char* key, const char* val)
{
    if (pl->n >= MAX_PARAMS)
        return -1;
    orc_param* q = &pl->p[pl->n++];
    snprintf(q->key, MAX_TOKEN, "%s", key);
    q->has_val = (val != NULL);
    snprintf(q->val, MAX_TOKEN, "%s", val ? val : "");
    return 0;
}

/* pj_init_plus: split on white space, strip the leading '+' of every token */
static int pl_parse(const char* def, orc_plist* pl)
{
    pl->n = 0;
    const char* s = def;
    while (*s) {
        while (*s && isspace((unsigned char)*s))
            ++s;
        if (!*s)
            break;
        char tok[2 * MAX_TOKEN];
        size_t len = 0;
        while (*s && !isspace((unsigned char)*s)) {
            if (len + 1 < sizeof(tok))
                tok[len++] = *s;
            ++s;
        }
        tok[len] = 0;
        const char* t = tok;
        if (*t == '+')
            ++t;
        if (!*t)
            continue;
        const char* eq = strchr(t, '=');
        char key[MAX_TOKEN];
        if (eq) {
            size_t kl = (size_t)(eq - t);
            if (kl >= MAX_TOKEN)
                kl = MAX_TOKEN - 1;
            memcpy(key, t, kl);
            key[kl] = 0;
            if (pl_append(pl, key, eq + 1))
                return -1;
        } else {
            if (pl_append(pl, t, NULL))
                return -1;
        }
    }
    return 0;
}

/* 'd' parameters: plain floating point numbers */
static double pl_double(const orc_plist* pl, const char* key, double dflt)
{
    const orc_param* q = pl_find(pl, key);
    if (!q || !q->has_val)
        return dflt;
    return strtod(q->val, NULL);
}

/* 'b' parameters: present without value, or value not starting with F/f => true */
static int pl_bool(const orc_plist* pl, const char* key)
{
    const orc_param* q = pl_find(pl, key);
    if (!q)
        return 0;
    if (!q->has_val || q->val[0] == 0)
        return 1;
    return !(q->val[0] == 'F' || q->val[0] == 'f');
}

/* dmstor.c: [+-]DDD[d MM['SS["]]][NnEeSsWw] or a plain number (degrees) or <number>r (radians) */
static double orc_dmstor(const char* is, int* err)
{
    static const double vm[3] = {.0174532925199432958, .0002908882086657216, .0000048481368110953599};
    const char* s = is;
    while (isspace((unsigned char)*s))
        ++s;
    int sign = '+';
    if (*s == '+' || *s == '-')
        sign = *s++;
    double v = 0.;
    int nl = 0, n = 0;
    for (; nl < 3; nl = n + 1) {
        if (!(isdigit((unsigned char)*s) || *s == '.'))
            break;
        /* proj_strtod: a 'd'/'D' terminates the number instead of starting an exponent */
        char buf[MAX_TOKEN];
        size_t bl = 0;
        const char* q = s;
        while (*q && bl + 1 < sizeof(buf) && *q != 'd' && *q != 'D' && *q != '\'' && *q != '"' && *q != 'r' && *q != 'R' &&
               !strchr("NnEeSsWw", *q))
            buf[bl++] = *q++;
        /* keep an exponent "e-5"/"E+3" that the loop above cut at 'e'/'E' */
        if ((*q == 'e' || *q == 'E') && (isdigit((unsigned char)q[1]) || ((q[1] == '+' || q[1] == '-') && isdigit((unsigned char)q[2])))) {
            buf[bl++] = *q++;
            while (*q && bl + 1 < sizeof(buf) && (isdigit((unsigned char)*q) || *q == '+' || *q == '-'))
                buf[bl++] = *q++;
        }
        buf[bl] = 0;
        char* endp = NULL;
        double tv = strtod(buf, &endp);
        s += (endp - buf);
        switch (*s) {
        case 'D':
        case 'd':
            n = 0;
            break;
        case '\'':
            n = 1;
            break;
        case '"':
            n = 2;
            break;
        case 'r':
        case 'R':
            if (nl) {
                *err = -16;
                return HUGE_VAL;
            }
            ++s;
            v = tv;
            n = 4;
            continue;
        default:
            v += tv * vm[nl];
            n = 4;
            continue;
        }
        if (n < nl) {
            *err = -16;
            return HUGE_VAL;
        }
        v += tv * vm[n];
        ++s;
    }
    if (*s) {
        const char* sym = "NnEeSsWw";
        const char* p = strchr(sym, *s);
        if (p) {
            sign = (p - sym) >= 4 ? '-' : '+';
            ++s;
        }
    }
    if (sign == '-')
        v = -v;
    return v;
}

/* 'r' parameters: angles through dmstor */
static double pl_angle(const orc_plist* pl, const char* key, int* err)
{
    const orc_param* q = pl_find(pl, key);
    if (!q || !q->has_val)
        return 0.;
    return orc_dmstor(q->val, err);
}

/* ---------------------------------------------------------------- small math helpers */

/* adjlon.c */
static double orc_adjlon(double lon)
{
    if (fabs(lon) <= ORC_SPI)
        return lon;
    lon += ORC_PI;
    lon -= ORC_TWOPI * floor(lon / ORC_TWOPI);
    lon -= ORC_PI;
    return lon;
}

/* aasincos.c */
static double orc_aasin(orc_pj* P, double v)
{
    double av = fabs(v);
    if (av >= 1.) {
        if (av > 1.00000000000001)
            P->last_errno = -19;
        return v < 0. ? -ORC_HALFPI : ORC_HALFPI;
    }
    return asin(v);
}

static double orc_aatan2(double n, double d)
{
    return (fabs(n) < 1e-50 && fabs(d) < 1e-50) ? 0. : atan2(n, d);
}

/* pj_tsfn.c */
static double orc_tsfn(double phi, double sinphi, double e)
{
    sinphi *= e;
    return tan(.5 * (ORC_HALFPI - phi)) / pow((1. - sinphi) / (1. + sinphi), .5 * e);
}

/* pj_msfn.c */
static double orc_msfn(double sinphi, double cosphi, double es)
{
    return cosphi / sqrt(1. - es * sinphi * sinphi);
}

/* pj_phi2.c */
static double orc_phi2(orc_pj* P, double ts, double e)
{
    double eccnth = .5 * e;
    double phi = ORC_HALFPI - 2. * atan(ts);
    int i = 15;
    double dphi;
    do {
        double con = e * sin(phi);
        dphi = ORC_HALFPI - 2. * atan(ts * pow((1. - con) / (1. + con), eccnth)) - phi;
        phi += dphi;
    } while (fabs(dphi) > 1.0e-10 && --i);
    if (i <= 0)
        P->last_errno = -18;
    return phi;
}

/* ---------------------------------------------------------------- ellipsoid + datum (pj_ell_set.c, pj_datum_set.c) */

typedef struct {
    const char* id;
    const char* major;
    const char* ell;
} orc_ellps;

static const orc_ellps orc_ellps_table[] = {
    {"sphere", "a=6370997.0", "b=6370997.0"},  {"WGS84", "a=6378137.0", "rf=298.257223563"},
    {"GRS80", "a=6378137.0", "rf=298.257222101"}, {"bessel", "a=6377397.155", "rf=299.1528128"},
    {"intl", "a=6378388.0", "rf=297."},        {"clrk66", "a=6378206.4", "b=6356583.8"},
    {"krass", "a=6378245.0", "rf=298.3"},      {NULL, NULL, NULL}};

static int orc_append_kv(orc_plist* pl, const char* kv)
{
    const char* eq = strchr(kv, '=');
    char key[MAX_TOKEN];
    size_t kl = (size_t)(eq - kv);
    memcpy(key, kv, kl);
    key[kl] = 0;
    return pl_append(pl, key, eq + 1);
}

static int orc_datum_set(orc_plist* pl, orc_pj* P)
{
    P->datum_type = PJD_UNKNOWN;
    const orc_param* d = pl_find(pl, "datum");
    if (d && d->has_val) {
        if (strcmp(d->val, "WGS84") == 0) {
            pl_append(pl, "ellps", "WGS84");
            pl_append(pl, "towgs84", "0,0,0");
        } else if (strcmp(d->val, "NAD83") == 0) {
            pl_append(pl, "ellps", "GRS80");
            pl_append(pl, "towgs84", "0,0,0");
        } else {
            return -9; /* unknown elliptical parameter name (datum table not restated) */
        }
    }
    if (pl_has(pl, "nadgrids")) {
        P->datum_type = PJD_GRIDSHIFT;
        return -38; /* grid shift files are out of scope */
    }
    const orc_param* t = pl_find(pl, "towgs84");
    if (t && t->has_val) {
        memset(P->datum_params, 0, sizeof(P->datum_params));
        const char* s = t->val;
        for (int i = 0; *s && i < 7; ++i) {
            P->datum_params[i] = strtod(s, NULL);
            while (*s && *s != ',')
                ++s;
            if (*s == ',')
                ++s;
        }
        if (P->datum_params[3] != 0. || P->datum_params[4] != 0. || P->datum_params[5] != 0. || P->datum_params[6] != 0.) {
            P->datum_type = PJD_7PARAM;
            const double sec2rad = 4.84813681109535993589914102357e-6;
            P->datum_params[3] *= sec2rad;
            P->datum_params[4] *= sec2rad;
            P->datum_params[5] *= sec2rad;
            P->datum_params[6] = (P->datum_params[6] / 1000000.0) + 1;
        } else {
            P->datum_type = PJD_3PARAM;
        }
    }
    return 0;
}

static int orc_ell_set(orc_plist* pl, double* a, double* es)
{
    *a = *es = 0.;
    if (pl_has(pl, "R")) {
        *a = pl_double(pl, "R", 0.);
    } else {
        const orc_param* el = pl_find(pl, "ellps");
        if (el && el->has_val) {
            const orc_ellps* t = orc_ellps_table;
            for (; t->id; ++t)
                if (strcmp(t->id, el->val) == 0)
                    break;
            if (!t->id)
                return -9;
            /* appended at the END: explicitly given +a/+b/+rf/+e found first still win */
            orc_append_kv(pl, t->major);
            orc_append_kv(pl, t->ell);
        }
        *a = pl_double(pl, "a", 0.);
        double b = 0.;
        if (pl_has(pl, "es")) {
            *es = pl_double(pl, "es", 0.);
        } else if (pl_has(pl, "e")) {
            double e = pl_double(pl, "e", 0.);
            *es = e * e;
        } else if (pl_has(pl, "rf")) {
            double rf = pl_double(pl, "rf", 0.);
            if (!rf)
                return -10;
            *es = 1. / rf;
            *es = *es * (2. - *es);
        } else if (pl_has(pl, "f")) {
            *es = pl_double(pl, "f", 0.);
            *es = *es * (2. - *es);
        } else if (pl_has(pl, "b")) {
            b = pl_double(pl, "b", 0.);
            *es = 1. - (b * b) / (*a * *a);
        }
        /* +R_A, +R_V, +R_a, +R_g, +R_h, +R_lat_a, +R_lat_g: not produced by Fimex, not restated */
    }
    if (*es < 0.)
        return -12;
    if (*a <= 0.)
        return -13;
    return 0;
}

/* ---------------------------------------------------------------- projection set-up (PJ_*.c ENTRY parts) */

static int orc_setup_stere(const orc_plist* pl, orc_pj* P, int* err)
{
    /* PJ_stere.c ENTRY0(stere) + setup() */
    P->phits = pl_has(pl, "lat_ts") ? pl_angle(pl, "lat_ts", err) : ORC_HALFPI;
    double t = fabs(P->phi0);
    if (fabs(t - ORC_HALFPI) < 1.e-10)
        P->mode = P->phi0 < 0. ? ST_S_POLE : ST_N_POLE;
    else
        P->mode = t > 1.e-10 ? ST_OBLIQ : ST_EQUIT;
    P->phits = fabs(P->phits);
    if (P->es != 0.) {
        double X;
        switch (P->mode) {
        case ST_N_POLE:
        case ST_S_POLE:
            if (fabs(P->phits - ORC_HALFPI) < 1.e-10) {
                P->akm1 = 2. * P->k0 / sqrt(pow(1 + P->e, 1 + P->e) * pow(1 - P->e, 1 - P->e));
            } else {
                t = sin(P->phits);
                P->akm1 = cos(P->phits) / orc_tsfn(P->phits, t, P->e);
                t *= P->e;
                P->akm1 /= sqrt(1. - t * t);
            }
            break;
        default: /* EQUIT, OBLIQ */
            t = sin(P->phi0);
            {
                double s = t * P->e;
                double ssfn = tan(.5 * (ORC_HALFPI + P->phi0)) * pow((1. - s) / (1. + s), .5 * P->e);
                X = 2. * atan(ssfn) - ORC_HALFPI;
            }
            t *= P->e;
            P->akm1 = 2. * P->k0 * cos(P->phi0) / sqrt(1. - t * t);
            P->sinX1 = sin(X);
            P->cosX1 = cos(X);
            break;
        }
    } else {
        switch (P->mode) {
        case ST_OBLIQ:
            P->sinX1 = sin(P->phi0); /* sinph0 */
            P->cosX1 = cos(P->phi0); /* cosph0 */
            /* fall through */
        case ST_EQUIT:
            P->akm1 = 2. * P->k0;
            break;
        default:
            P->akm1 = fabs(P->phits - ORC_HALFPI) >= 1.e-10 ? cos(P->phits) / tan(ORC_FORTPI - .5 * P->phits) : 2. * P->k0;
            break;
        }
    }
    return 0;
}

static int orc_setup_lcc(const orc_plist* pl, orc_pj* P, int* err)
{
    /* PJ_lcc.c ENTRY0(lcc) */
    P->phi1 = pl_angle(pl, "lat_1", err);
    if (pl_has(pl, "lat_2")) {
        P->phi2 = pl_angle(pl, "lat_2", err);
    } else {
        P->phi2 = P->phi1;
        if (!pl_has(pl, "lat_0"))
            P->phi0 = P->phi1;
    }
    if (fabs(P->phi1 + P->phi2) < 1.e-10)
        return -21;
    double sinphi = sin(P->phi1);
    double cosphi = cos(P->phi1);
    P->n = sinphi;
    int secant = fabs(P->phi1 - P->phi2) >= 1.e-10;
    P->ellips = (P->es != 0.);
    if (P->ellips) {
        double m1 = orc_msfn(sinphi, cosphi, P->es);
        double ml1 = orc_tsfn(P->phi1, sinphi, P->e);
        if (secant) {
            sinphi = sin(P->phi2);
            P->n = log(m1 / orc_msfn(sinphi, cos(P->phi2), P->es));
            P->n /= log(ml1 / orc_tsfn(P->phi2, sinphi, P->e));
        }
        P->rho0 = m1 * pow(ml1, -P->n) / P->n;
        P->c = P->rho0;
        P->rho0 *= (fabs(fabs(P->phi0) - ORC_HALFPI) < 1.e-10) ? 0. : pow(orc_tsfn(P->phi0, sin(P->phi0), P->e), P->n);
    } else {
        if (secant)
            P->n = log(cosphi / cos(P->phi2)) / log(tan(ORC_FORTPI + .5 * P->phi2) / tan(ORC_FORTPI + .5 * P->phi1));
        P->c = cosphi * pow(tan(ORC_FORTPI + .5 * P->phi1), P->n) / P->n;
        P->rho0 = (fabs(fabs(P->phi0) - ORC_HALFPI) < 1.e-10) ? 0. : P->c * pow(tan(ORC_FORTPI + .5 * P->phi0), -P->n);
    }
    return 0;
}

static int orc_is_latlong_name(const char* s)
{
    return strcmp(s, "latlong") == 0 || strcmp(s, "longlat") == 0 || strcmp(s, "latlon") == 0 || strcmp(s, "lonlat") == 0;
}

static int orc_setup_ob_tran(const orc_plist* pl, orc_pj* P, int* err)
{
    /* PJ_ob_tran.c ENTRY1(ob_tran): only the "+o_lat_p [+o_lon_p]" (new pole) form with a lat/long
     * link, which is what Fimex writes (RotatedLatitudeLongitudeProjection.cc:91-104) */
    const orc_param* o = pl_find(pl, "o_proj");
    if (!o || !o->has_val)
        return -26;
    if (!orc_is_latlong_name(o->val))
        return -5; /* other links are outside the hot path's grammar */
    P->es = 0.; /* force to spherical */
    P->e = 0.;
    P->one_es = P->rone_es = 1.;
    if (!pl_has(pl, "o_lat_p"))
        return -5; /* +o_alpha / +o_lon_1.. forms not restated */
    P->lamp = pl_angle(pl, "o_lon_p", err);
    double phip = pl_angle(pl, "o_lat_p", err);
    if (fabs(phip) > 1e-10) {
        P->oblique = 1;
        P->cphip = cos(phip);
        P->sphip = sin(phip);
    } else {
        P->oblique = 0;
    }
    return 0;
}

projPJ pj_init_plus(const char* definition)
{
    orc_plist pl;
    int err = 0;
    pj_errno = 0;
    if (!definition || pl_parse(definition, &pl) || pl.n == 0) {
        pj_errno = -1;
        return NULL;
    }
    if (pl_has(&pl, "init")) {
        pj_errno = -2; /* epsg-style init files not restated */
        return NULL;
    }
    const orc_param* pr = pl_find(&pl, "proj");
    if (!pr || !pr->has_val) {
        pj_errno = -4;
        return NULL;
    }
    orc_pj* P = (orc_pj*)calloc(1, sizeof(orc_pj));
    if (!P) {
        pj_errno = ENOMEM;
        return NULL;
    }
    if (orc_is_latlong_name(pr->val))
        P->kind = KIND_LATLONG;
    else if (strcmp(pr->val, "ob_tran") == 0)
        P->kind = KIND_OB_TRAN;
    else if (strcmp(pr->val, "stere") == 0)
        P->kind = KIND_STERE;
    else if (strcmp(pr->val, "lcc") == 0)
        P->kind = KIND_LCC;
    else {
        pj_errno = -5; /* unknown projection id */
        free(P);
        return NULL;
    }
    /* defaults of proj_def.dat, appended at the end unless +no_defs (pj_init.c get_defaults) */
    if (!pl_bool(&pl, "no_defs")) {
        /* get_opt: "don't default ellipse if datum, ellps or any earth model information is set" */
        if (!pl_has(&pl, "datum") && !pl_has(&pl, "ellps") && !pl_has(&pl, "a") && !pl_has(&pl, "b") && !pl_has(&pl, "rf") &&
            !pl_has(&pl, "f"))
            pl_append(&pl, "ellps", "WGS84");
        if (P->kind == KIND_LCC) {
            pl_append(&pl, "lat_1", "33");
            pl_append(&pl, "lat_2", "45");
        }
    }
    if ((err = orc_datum_set(&pl, P)) != 0)
        goto fail;
    if ((err = orc_ell_set(&pl, &P->a, &P->es)) != 0)
        goto fail;
    P->a_orig = P->a;
    P->es_orig = P->es;
    P->e = sqrt(P->es);
    P->ra = 1. / P->a;
    P->one_es = 1. - P->es;
    if (P->one_es == 0.) {
        err = -6;
        goto fail;
    }
    P->rone_es = 1. / P->one_es;
    if (P->datum_type == PJD_3PARAM && P->datum_params[0] == 0. && P->datum_params[1] == 0. && P->datum_params[2] == 0. &&
        P->a == 6378137.0 && fabs(P->es - 0.006694379990) < 0.000000000050)
        P->datum_type = PJD_WGS84;
    P->geoc = (P->es != 0. && pl_bool(&pl, "geoc"));
    P->over = pl_bool(&pl, "over");
    P->lam0 = pl_angle(&pl, "lon_0", &err);
    P->phi0 = pl_angle(&pl, "lat_0", &err);
    P->x0 = pl_double(&pl, "x_0", 0.);
    P->y0 = pl_double(&pl, "y_0", 0.);
    if (pl_has(&pl, "k_0"))
        P->k0 = pl_double(&pl, "k_0", 1.);
    else if (pl_has(&pl, "k"))
        P->k0 = pl_double(&pl, "k", 1.);
    else
        P->k0 = 1.;
    if (P->k0 <= 0.)
        err = -31;
    if (err)
        goto fail;
    P->to_meter = P->fr_meter = 1.;
    {
        const orc_param* u = pl_find(&pl, "units");
        if (u && u->has_val) {
            if (strcmp(u->val, "m") == 0)
                P->to_meter = 1.;
            else if (strcmp(u->val, "km") == 0)
                P->to_meter = 1000.;
            else {
                err = -7; /* unit table not restated beyond m/km */
                goto fail;
            }
            P->fr_meter = 1. / P->to_meter;
        } else if (pl_has(&pl, "to_meter")) {
            P->to_meter = pl_double(&pl, "to_meter", 1.);
            P->fr_meter = 1. / P->to_meter;
        }
    }
    if (pl_has(&pl, "pm")) {
        err = -46; /* prime meridians other than Greenwich not restated */
        goto fail;
    }
    switch (P->kind) {
    case KIND_LATLONG: /* PJ_latlong.c */
        P->is_latlong = 1;
        P->x0 = 0.;
        P->y0 = 0.;
        break;
    case KIND_OB_TRAN:
        err = orc_setup_ob_tran(&pl, P, &err);
        break;
    case KIND_STERE:
        err = orc_setup_stere(&pl, P, &err);
        break;
    case KIND_LCC:
        err = orc_setup_lcc(&pl, P, &err);
        break;
    }
    if (err)
        goto fail;
    return (projPJ)P;
fail:
    pj_errno = err;
    free(P);
    return NULL;
}

void pj_free(projPJ pj)
{
    free(pj);
}

int pj_is_latlong(projPJ pj)
{
    return pj == NULL || ((orc_pj*)pj)->is_latlong;
}

char* pj_strerrno(int err)
{
    static char buf[64];
    switch (err) {
    case 0:
        return NULL;
    case -4:
        return (char*)"projection not named";
    case -5:
        return (char*)"unknown projection id";
    case -9:
        return (char*)"unknown elliptical parameter name";
    case -13:
        return (char*)"major axis or radius = 0 or not given";
    case -14:
        return (char*)"latitude or longitude exceeded limits";
    case -15:
        return (char*)"invalid x or y";
    case -20:
        return (char*)"tolerance condition error";
    case -21:
        return (char*)"conic lat_1 = -lat_2";
    default:
        snprintf(buf, sizeof(buf), "proj (oracle restatement) error %d", err);
        return buf;
    }
}

/* ---------------------------------------------------------------- per-projection forward / inverse */

typedef struct {
    double x, y;
} orc_xy;
typedef struct {
    double lam, phi;
} orc_lp;

static orc_xy orc_stere_fwd(orc_pj* P, orc_lp lp)
{
    orc_xy xy = {0., 0.};
    if (P->es == 0.) { /* s_forward */
        double sinphi = sin(lp.phi), cosphi = cos(lp.phi);
        double coslam = cos(lp.lam), sinlam = sin(lp.lam);
        switch (P->mode) {
        case ST_EQUIT:
        case ST_OBLIQ:
            if (P->mode == ST_EQUIT)
                xy.y = 1. + cosphi * coslam;
            else
                xy.y = 1. + P->sinX1 * sinphi + P->cosX1 * cosphi * coslam;
            if (xy.y <= 1.e-10) {
                P->last_errno = -20;
                return xy;
            }
            xy.y = P->akm1 / xy.y;
            xy.x = xy.y * cosphi * sinlam;
            xy.y *= (P->mode == ST_EQUIT) ? sinphi : P->cosX1 * sinphi - P->sinX1 * cosphi * coslam;
            break;
        case ST_N_POLE:
            coslam = -coslam;
            lp.phi = -lp.phi;
            /* fall through */
        case ST_S_POLE:
            if (fabs(lp.phi - ORC_HALFPI) < 1.e-8) {
                P->last_errno = -20;
                return xy;
            }
            xy.y = P->akm1 * tan(ORC_FORTPI + .5 * lp.phi);
            xy.x = sinlam * xy.y;
            xy.y *= coslam;
            break;
        }
    } else { /* e_forward */
        double sinX = 0., cosX = 0., A;
        double coslam = cos(lp.lam), sinlam = sin(lp.lam), sinphi = sin(lp.phi);
        if (P->mode == ST_OBLIQ || P->mode == ST_EQUIT) {
            double s = sinphi * P->e;
            double ssfn = tan(.5 * (ORC_HALFPI + lp.phi)) * pow((1. - s) / (1. + s), .5 * P->e);
            double X = 2. * atan(ssfn) - ORC_HALFPI;
            sinX = sin(X);
            cosX = cos(X);
        }
        switch (P->mode) {
        case ST_OBLIQ:
            A = P->akm1 / (P->cosX1 * (1. + P->sinX1 * sinX + P->cosX1 * cosX * coslam));
            xy.y = A * (P->cosX1 * sinX - P->sinX1 * cosX * coslam);
            xy.x = A * cosX;
            break;
        case ST_EQUIT:
            A = 2. * P->akm1 / (1. + cosX * coslam);
            xy.y = A * sinX;
            xy.x = A * cosX;
            break;
        case ST_S_POLE:
            lp.phi = -lp.phi;
            coslam = -coslam;
            sinphi = -sinphi;
            /* fall through */
        case ST_N_POLE:
            xy.x = P->akm1 * orc_tsfn(lp.phi, sinphi, P->e);
            xy.y = -xy.x * coslam;
            break;
        }
        xy.x = xy.x * sinlam;
    }
    return xy;
}

static orc_lp orc_stere_inv(orc_pj* P, orc_xy xy)
{
    orc_lp lp = {0., 0.};
    if (P->es == 0.) { /* s_inverse */
        double rh = hypot(xy.x, xy.y);
        double c = 2. * atan(rh / P->akm1);
        double sinc = sin(c), cosc = cos(c);
        lp.lam = 0.;
        switch (P->mode) {
        case ST_EQUIT:
            if (fabs(rh) <= 1.e-10)
                lp.phi = 0.;
            else
                lp.phi = asin(xy.y * sinc / rh);
            if (cosc != 0. || xy.x != 0.)
                lp.lam = atan2(xy.x * sinc, cosc * rh);
            break;
        case ST_OBLIQ:
            if (fabs(rh) <= 1.e-10)
                lp.phi = P->phi0;
            else
                lp.phi = asin(cosc * P->sinX1 + xy.y * sinc * P->cosX1 / rh);
            c = cosc - P->sinX1 * sin(lp.phi);
            if (c != 0. || xy.x != 0.)
                lp.lam = atan2(xy.x * sinc * P->cosX1, c * rh);
            break;
        case ST_N_POLE:
            xy.y = -xy.y;
            /* fall through */
        case ST_S_POLE:
            if (fabs(rh) <= 1.e-10)
                lp.phi = P->phi0;
            else
                lp.phi = asin(P->mode == ST_S_POLE ? -cosc : cosc);
            lp.lam = (xy.x == 0. && xy.y == 0.) ? 0. : atan2(xy.x, xy.y);
            break;
        }
    } else { /* e_inverse */
        double cosphi, sinphi, tp = 0., phi_l = 0., halfe = 0., halfpi = 0.;
        double rho = hypot(xy.x, xy.y);
        switch (P->mode) {
        case ST_OBLIQ:
        case ST_EQUIT:
            tp = 2. * atan2(rho * P->cosX1, P->akm1);
            cosphi = cos(tp);
            sinphi = sin(tp);
            if (rho == 0.0)
                phi_l = asin(cosphi * P->sinX1);
            else
                phi_l = asin(cosphi * P->sinX1 + (xy.y * sinphi * P->cosX1 / rho));
            tp = tan(.5 * (ORC_HALFPI + phi_l));
            xy.x *= sinphi;
            xy.y = rho * P->cosX1 * cosphi - xy.y * P->sinX1 * sinphi;
            halfpi = ORC_HALFPI;
            halfe = .5 * P->e;
            break;
        case ST_N_POLE:
            xy.y = -xy.y;
            /* fall through */
        case ST_S_POLE:
            tp = -rho / P->akm1;
            phi_l = ORC_HALFPI - 2. * atan(tp);
            halfpi = -ORC_HALFPI;
            halfe = -.5 * P->e;
            break;
        }
        for (int i = 8; i--; phi_l = lp.phi) {
            sinphi = P->e * sin(phi_l);
            lp.phi = 2. * atan(tp * pow((1. + sinphi) / (1. - sinphi), halfe)) - halfpi;
            if (fabs(phi_l - lp.phi) < 1.e-10) {
                if (P->mode == ST_S_POLE)
                    lp.phi = -lp.phi;
                lp.lam = (xy.x == 0. && xy.y == 0.) ? 0. : atan2(xy.x, xy.y);
                return lp;
            }
        }
        P->last_errno = -20;
    }
    return lp;
}

static orc_xy orc_lcc_fwd(orc_pj* P, orc_lp lp)
{
    orc_xy xy = {0., 0.};
    double rho;
    if (fabs(fabs(lp.phi) - ORC_HALFPI) < 1.e-10) {
        if ((lp.phi * P->n) <= 0.) {
            P->last_errno = -20;
            return xy;
        }
        rho = 0.;
    } else {
        rho = P->c * (P->ellips ? pow(orc_tsfn(lp.phi, sin(lp.phi), P->e), P->n) : pow(tan(ORC_FORTPI + .5 * lp.phi), -P->n));
    }
    lp.lam *= P->n;
    xy.x = P->k0 * (rho * sin(lp.lam));
    xy.y = P->k0 * (P->rho0 - rho * cos(lp.lam));
    return xy;
}

static orc_lp orc_lcc_inv(orc_pj* P, orc_xy xy)
{
    orc_lp lp = {0., 0.};
    xy.x /= P->k0;
    xy.y /= P->k0;
    xy.y = P->rho0 - xy.y;
    double rho = hypot(xy.x, xy.y);
    if (rho != 0.0) {
        if (P->n < 0.) {
            rho = -rho;
            xy.x = -xy.x;
            xy.y = -xy.y;
        }
        if (P->ellips) {
            lp.phi = orc_phi2(P, pow(rho / P->c, 1. / P->n), P->e);
            if (lp.phi == HUGE_VAL) {
                P->last_errno = -20;
                return lp;
            }
        } else {
            lp.phi = 2. * atan(pow(P->c / rho, 1. / P->n)) - ORC_HALFPI;
        }
        lp.lam = atan2(xy.x, xy.y) / P->n;
    } else {
        lp.lam = 0.;
        lp.phi = P->n > 0. ? ORC_HALFPI : -ORC_HALFPI;
    }
    return lp;
}

/* PJ_ob_tran.c with a lat/long link: link->fwd is (lam/a, phi/a), link->inv is (x*a, y*a) */
static orc_xy orc_ob_tran_fwd(orc_pj* P, orc_lp lp)
{
    orc_xy xy;
    if (P->oblique) { /* o_forward */
        double coslam = cos(lp.lam);
        double sinphi = sin(lp.phi), cosphi = cos(lp.phi);
        double lam = orc_adjlon(orc_aatan2(cosphi * sin(lp.lam), P->sphip * cosphi * coslam + P->cphip * sinphi) + P->lamp);
        double phi = orc_aasin(P, P->sphip * sinphi - P->cphip * cosphi * coslam);
        lp.lam = lam;
        lp.phi = phi;
    } else { /* t_forward */
        double cosphi = cos(lp.phi), coslam = cos(lp.lam);
        double lam = orc_adjlon(orc_aatan2(cosphi * sin(lp.lam), sin(lp.phi)) + P->lamp);
        double phi = orc_aasin(P, -cosphi * coslam);
        lp.lam = lam;
        lp.phi = phi;
    }
    xy.x = lp.lam / P->a;
    xy.y = lp.phi / P->a;
    return xy;
}

static orc_lp orc_ob_tran_inv(orc_pj* P, orc_xy xy)
{
    orc_lp lp;
    lp.phi = xy.y * P->a;
    lp.lam = xy.x * P->a;
    if (lp.lam != HUGE_VAL) {
        if (P->oblique) { /* o_inverse */
            lp.lam -= P->lamp;
            double coslam = cos(lp.lam);
            double sinphi = sin(lp.phi), cosphi = cos(lp.phi);
            double phi = orc_aasin(P, P->sphip * sinphi + P->cphip * cosphi * coslam);
            double lam = orc_aatan2(cosphi * sin(lp.lam), P->sphip * cosphi * coslam - P->cphip * sinphi);
            lp.phi = phi;
            lp.lam = lam;
        } else { /* t_inverse */
            double cosphi = cos(lp.phi);
            double t = lp.lam - P->lamp;
            double lam = orc_aatan2(cosphi * sin(t), -sin(lp.phi));
            double phi = orc_aasin(P, cosphi * cos(t));
            lp.lam = lam;
            lp.phi = phi;
        }
    }
    return lp;
}

/* pj_fwd.c */
static orc_xy orc_fwd(orc_pj* P, orc_lp lp)
{
    orc_xy xy;
    double t = fabs(lp.phi) - ORC_HALFPI;
    if (t > 1.0e-12 || fabs(lp.lam) > 10.) {
        xy.x = xy.y = HUGE_VAL;
        P->last_errno = -14;
        return xy;
    }
    P->last_errno = 0;
    errno = 0;
    if (fabs(t) <= 1.0e-12)
        lp.phi = lp.phi < 0. ? -ORC_HALFPI : ORC_HALFPI;
    else if (P->geoc)
        lp.phi = atan(P->rone_es * tan(lp.phi));
    lp.lam -= P->lam0;
    if (!P->over)
        lp.lam = orc_adjlon(lp.lam);
    switch (P->kind) {
    case KIND_OB_TRAN:
        xy = orc_ob_tran_fwd(P, lp);
        break;
    case KIND_STERE:
        xy = orc_stere_fwd(P, lp);
        break;
    case KIND_LCC:
        xy = orc_lcc_fwd(P, lp);
        break;
    default: /* PJ_latlong.c forward (never reached through pj_transform) */
        xy.x = lp.lam / P->a;
        xy.y = lp.phi / P->a;
        break;
    }
    if (P->last_errno) {
        xy.x = xy.y = HUGE_VAL;
    } else {
        xy.x = P->fr_meter * (P->a * xy.x + P->x0);
        xy.y = P->fr_meter * (P->a * xy.y + P->y0);
    }
    return xy;
}

/* pj_inv.c */
static orc_lp orc_inv(orc_pj* P, orc_xy xy)
{
    orc_lp lp;
    if (xy.x == HUGE_VAL || xy.y == HUGE_VAL) {
        lp.lam = lp.phi = HUGE_VAL;
        P->last_errno = -15;
        return lp;
    }
    errno = 0;
    P->last_errno = 0;
    xy.x = (xy.x * P->to_meter - P->x0) * P->ra;
    xy.y = (xy.y * P->to_meter - P->y0) * P->ra;
    switch (P->kind) {
    case KIND_OB_TRAN:
        lp = orc_ob_tran_inv(P, xy);
        break;
    case KIND_STERE:
        lp = orc_stere_inv(P, xy);
        break;
    case KIND_LCC:
        lp = orc_lcc_inv(P, xy);
        break;
    default:
        lp.phi = xy.y * P->a;
        lp.lam = xy.x * P->a;
        break;
    }
    if (P->last_errno) {
        lp.lam = lp.phi = HUGE_VAL;
    } else {
        lp.lam += P->lam0;
        if (!P->over)
            lp.lam = orc_adjlon(lp.lam);
        if (P->geoc && fabs(fabs(lp.phi) - ORC_HALFPI) > 1.0e-12)
            lp.phi = atan(P->one_es * tan(lp.phi));
    }
    return lp;
}

/* ---------------------------------------------------------------- datum shift (pj_transform.c, geocent.c) */

static int orc_compare_datums(const orc_pj* s, const orc_pj* d)
{
    if (s->datum_type != d->datum_type)
        return 0;
    if (s->a_orig != d->a_orig || fabs(s->es_orig - d->es_orig) > 0.000000000050)
        return 0;
    if (s->datum_type == PJD_3PARAM)
        return s->datum_params[0] == d->datum_params[0] && s->datum_params[1] == d->datum_params[1] &&
               s->datum_params[2] == d->datum_params[2];
    if (s->datum_type == PJD_7PARAM) {
        for (int i = 0; i < 7; ++i)
            if (s->datum_params[i] != d->datum_params[i])
                return 0;
        return 1;
    }
    return 1;
}

static void orc_geodetic_to_geocentric(double a, double es, double* x, double* y, double* z)
{
    double lon = *x, lat = *y, h = *z;
    if (lat < -ORC_HALFPI && lat > -1.001 * ORC_HALFPI)
        lat = -ORC_HALFPI;
    else if (lat > ORC_HALFPI && lat < 1.001 * ORC_HALFPI)
        lat = ORC_HALFPI;
    else if (lat < -ORC_HALFPI || lat > ORC_HALFPI) {
        *x = *y = HUGE_VAL;
        return;
    }
    if (lon > ORC_PI)
        lon -= (2 * ORC_PI);
    double sin_lat = sin(lat), cos_lat = cos(lat);
    double rn = a / (sqrt(1.0e0 - es * sin_lat * sin_lat));
    *x = (rn + h) * cos_lat * cos(lon);
    *y = (rn + h) * cos_lat * sin(lon);
    *z = ((rn * (1 - es)) + h) * sin_lat;
}

static void orc_geocentric_to_geodetic(double a, double es, double* x, double* y, double* z)
{
    /* iterative method of geocent.c (genau = 1e-12, maxiter = 30) */
    const double genau = 1.E-12, genau2 = genau * genau;
    double X = *x, Y = *y, Z = *z;
    double b = a * sqrt(1. - es);
    double lon, lat, h;
    double P = sqrt(X * X + Y * Y);
    double RR = sqrt(X * X + Y * Y + Z * Z);
    if (P / a < genau) {
        lon = 0.;
        if (RR / a < genau) {
            *x = 0.;
            *y = ORC_HALFPI;
            *z = -b;
            return;
        }
    } else {
        lon = atan2(Y, X);
    }
    double CT = Z / RR, ST = P / RR;
    double RX = 1.0 / sqrt(1.0 - es * (2.0 - es) * ST * ST);
    double CPHI0 = ST * (1.0 - es) * RX;
    double SPHI0 = CT * RX;
    double CPHI, SPHI, SDPHI;
    int iter = 0;
    do {
        iter++;
        double RN = a / sqrt(1.0 - es * SPHI0 * SPHI0);
        h = P * CPHI0 + Z * SPHI0 - RN * (1.0 - es * SPHI0 * SPHI0);
        double RK = es * RN / (RN + h);
        RX = 1.0 / sqrt(1.0 - RK * (2.0 - RK) * ST * ST);
        CPHI = ST * (1.0 - RK) * RX;
        SPHI = CT * RX;
        SDPHI = SPHI * CPHI0 - CPHI * SPHI0;
        CPHI0 = CPHI;
        SPHI0 = SPHI;
    } while (SDPHI * SDPHI > genau2 && iter < 30);
    lat = atan(SPHI / fabs(CPHI));
    *x = lon;
    *y = lat;
    *z = h;
}

static int orc_datum_transform(const orc_pj* s, const orc_pj* d, long n, int off, double* x, double* y, double* z)
{
    if (s->datum_type == PJD_UNKNOWN || d->datum_type == PJD_UNKNOWN)
        return 0;
    if (orc_compare_datums(s, d))
        return 0;
    double src_a = s->a_orig, src_es = s->es_orig, dst_a = d->a_orig, dst_es = d->es_orig;
    int s37 = (s->datum_type == PJD_3PARAM || s->datum_type == PJD_7PARAM);
    int d37 = (d->datum_type == PJD_3PARAM || d->datum_type == PJD_7PARAM);
    if (!(src_es != dst_es || src_a != dst_a || s37 || d37))
        return 0;
    for (long i = 0; i < n; ++i) {
        double *px = &x[off * i], *py = &y[off * i];
        double zz = z ? z[off * i] : 0.;
        if (*px == HUGE_VAL)
            continue;
        orc_geodetic_to_geocentric(src_a, src_es, px, py, &zz);
        if (*px == HUGE_VAL)
            continue;
        if (s->datum_type == PJD_3PARAM) {
            *px += s->datum_params[0];
            *py += s->datum_params[1];
            zz += s->datum_params[2];
        } else if (s->datum_type == PJD_7PARAM) {
            const double* q = s->datum_params;
            double xo = q[6] * (*px - q[5] * *py + q[4] * zz) + q[0];
            double yo = q[6] * (q[5] * *px + *py - q[3] * zz) + q[1];
            double zo = q[6] * (-q[4] * *px + q[3] * *py + zz) + q[2];
            *px = xo;
            *py = yo;
            zz = zo;
        }
        if (d->datum_type == PJD_3PARAM) {
            *px -= d->datum_params[0];
            *py -= d->datum_params[1];
            zz -= d->datum_params[2];
        } else if (d->datum_type == PJD_7PARAM) {
            const double* q = d->datum_params;
            double xt = (*px - q[0]) / q[6];
            double yt = (*py - q[1]) / q[6];
            double zt = (zz - q[2]) / q[6];
            *px = xt + q[5] * yt - q[4] * zt;
            *py = -q[5] * xt + yt + q[3] * zt;
            zz = q[4] * xt - q[3] * yt + zt;
        }
        orc_geocentric_to_geodetic(dst_a, dst_es, px, py, &zz);
        if (z)
            z[off * i] = zz;
    }
    return 0;
}

/* ---------------------------------------------------------------- pj_transform.c */

static int orc_is_transient(int e)
{
    /* transient_error[] of pj_transform.c: -14 lat/lon limits, -15 invalid x/y, -17, -20 tolerance, -27, -45 */
    return e == -14 || e == -15 || e == -17 || e == -20 || e == -27 || e == -45;
}

int pj_transform(projPJ srcp, projPJ dstp, long point_count, int point_offset, double* x, double* y, double* z)
{
    orc_pj* src = (orc_pj*)srcp;
    orc_pj* dst = (orc_pj*)dstp;
    pj_errno = 0;
    if (point_offset == 0)
        point_offset = 1;
    if (!src->is_latlong) {
        for (long i = 0; i < point_count; ++i) {
            orc_xy in = {x[point_offset * i], y[point_offset * i]};
            if (in.x == HUGE_VAL)
                continue;
            orc_lp g = orc_inv(src, in);
            if (src->last_errno != 0) {
                int e = src->last_errno;
                if ((errno != 33 && errno != 34) && (e > 0 || e < -44 || point_count == 1 || !orc_is_transient(e))) {
                    pj_errno = e;
                    return e;
                }
                g.lam = HUGE_VAL;
                g.phi = HUGE_VAL;
            }
            x[point_offset * i] = g.lam;
            y[point_offset * i] = g.phi;
        }
    }
    if (orc_datum_transform(src, dst, point_count, point_offset, x, y, z) != 0)
        return pj_errno;
    if (!dst->is_latlong) {
        for (long i = 0; i < point_count; ++i) {
            orc_lp g = {x[point_offset * i], y[point_offset * i]};
            if (g.lam == HUGE_VAL)
                continue;
            orc_xy p = orc_fwd(dst, g);
            if (dst->last_errno != 0) {
                int e = dst->last_errno;
                if ((errno != 33 && errno != 34) && (e > 0 || e < -44 || point_count == 1 || !orc_is_transient(e))) {
                    pj_errno = e;
                    return e;
                }
                p.x = HUGE_VAL;
                p.y = HUGE_VAL;
            }
            x[point_offset * i] = p.x;
            y[point_offset * i] = p.y;
        }
    }
    return 0;
}
