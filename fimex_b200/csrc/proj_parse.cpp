// fimex_b200/csrc/proj_parse.cpp -- proj4-string -> ProjDef (host side of K1).
//
// The grammar is what Fimex itself writes and reads for the CRSs of the hot path
// (/root/reference/src/coordSys/ProjectionImpl.cc:116-160, RotatedLatitudeLongitudeProjection.cc:91-104,
// StereographicProjection.cc:86-95, PolarStereographicProjection.cc:38-50,
// LambertConformalConicProjection.cc:86-106, include/fimex/CDMconstants.h:118) plus the strings of the
// reference's tests (test/testInterpolation.cc:267-268,398-399; test/testInterpolator.cc:401-424).
// Semantics follow PROJ 4.9's pj_init: first occurrence of a key wins, +ellps/+datum/defaults are appended
// behind the user's keys, angles accept D[dM'S"][NSEW] or a trailing 'r' for radians.
#include "proj.cuh"

#include <cctype>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <utility>
#include <vector>

namespace fb {
namespace {

const double kHalfPi = 1.5707963267948966;
const double kFortPi = 0.78539816339744833;

struct KeyVals {
    std::vector<std::pair<std::string, std::string>> kv; // value "\x01" marks "no value"
    static constexpr const char* kNone = "\x01";

    const std::string* get(const std::string& k) const
    {
        for (const auto& p : kv)
            if (p.first == k)
                return &p.second;
        return nullptr;
    }
    bool has(const std::string& k) const { return get(k) != nullptr; }
    bool hasValue(const std::string& k) const
    {
        const std::string* v = get(k);
        return v && *v != kNone;
    }
    void add(const std::string& k, const std::string& v) { kv.emplace_back(k, v); }
    double num(const std::string& k, double dflt) const
    {
        const std::string* v = get(k);
        if (!v || *v == kNone)
            return dflt;
        return std::strtod(v->c_str(), nullptr);
    }
    bool flag(const std::string& k) const
    {
        const std::string* v = get(k);
        if (!v)
            return false;
        if (*v == kNone || v->empty())
            return true;
        return !((*v)[0] == 'F' || (*v)[0] == 'f');
    }
};

KeyVals tokenize(const char* def)
{
    KeyVals out;
    std::string s(def ? def : "");
    size_t i = 0;
    while (i < s.size()) {
        while (i < s.size() && std::isspace((unsigned char)s[i]))
            ++i;
        size_t j = i;
        while (j < s.size() && !std::isspace((unsigned char)s[j]))
            ++j;
        if (j > i) {
            std::string tok = s.substr(i, j - i);
            if (tok[0] == '+')
                tok.erase(0, 1);
            if (!tok.empty()) {
                const size_t eq = tok.find('=');
                if (eq == std::string::npos)
                    out.add(tok, KeyVals::kNone);
                else
                    out.add(tok.substr(0, eq), tok.substr(eq + 1));
            }
        }
        i = j;
    }
    return out;
}

// degrees-minutes-seconds (or radians with 'r') to radians
bool parseAngle(const std::string& text, double* out)
{
    static const double unit[3] = {.0174532925199432958, .0002908882086657216, .0000048481368110953599};
    const char* s = text.c_str();
    while (std::isspace((unsigned char)*s))
        ++s;
    bool neg = false;
    if (*s == '+' || *s == '-')
        neg = (*s++ == '-');
    double v = 0.;
    int next = 0;
    while (next < 3 && (std::isdigit((unsigned char)*s) || *s == '.')) {
        // a number; 'd'/'D' never starts an exponent here
        std::string numtxt;
        const char* q = s;
        while (std::isdigit((unsigned char)*q) || *q == '.')
            numtxt.push_back(*q++);
        if ((*q == 'e' || *q == 'E') && (std::isdigit((unsigned char)q[1]) || ((q[1] == '+' || q[1] == '-') && std::isdigit((unsigned char)q[2])))) {
            numtxt.push_back(*q++);
            if (*q == '+' || *q == '-')
                numtxt.push_back(*q++);
            while (std::isdigit((unsigned char)*q))
                numtxt.push_back(*q++);
        }
        const double tv = std::strtod(numtxt.c_str(), nullptr);
        s = q;
        int field;
        if (*s == 'd' || *s == 'D')
            field = 0;
        else if (*s == '\'')
            field = 1;
        else if (*s == '"')
            field = 2;
        else if (*s == 'r' || *s == 'R') {
            if (next != 0)
                return false;
            v = tv;
            ++s;
            break;
        } else {
            v += tv * unit[next];
            break;
        }
        if (field < next)
            return false;
        v += tv * unit[field];
        ++s;
        next = field + 1;
    }
    if (*s == 'S' || *s == 's' || *s == 'W' || *s == 'w')
        neg = true;
    else if (*s == 'N' || *s == 'n' || *s == 'E' || *s == 'e')
        neg = false;
    *out = neg ? -v : v;
    return true;
}

struct Ellipsoid {
    const char* id;
    double a;
    const char* shapeKey; // "b" or "rf"
    const char* shapeVal;
};
const Ellipsoid kEllipsoids[] = {
    {"sphere", 6370997.0, "b", "6370997.0"},   {"WGS84", 6378137.0, "rf", "298.257223563"}, {"GRS80", 6378137.0, "rf", "298.257222101"},
    {"bessel", 6377397.155, "rf", "299.1528128"}, {"intl", 6378388.0, "rf", "297."},         {"clrk66", 6378206.4, "b", "6356583.8"},
    {"krass", 6378245.0, "rf", "298.3"}};

bool isLatLongName(const std::string& n)
{
    return n == "latlong" || n == "longlat" || n == "latlon" || n == "lonlat";
}

int fail(char* err, int errlen, int code, const std::string& msg)
{
    if (err && errlen > 0)
        std::snprintf(err, (size_t)errlen, "%s (proj error %d)", msg.c_str(), code);
    return code;
}

} // namespace

int parse_proj(const char* definition, ProjDef* P, char* err, int errlen)
{
    std::memset(P, 0, sizeof(*P));
    KeyVals kv = tokenize(definition);
    if (kv.kv.empty())
        return fail(err, errlen, -1, "no arguments in projection definition");
    if (kv.has("init"))
        return fail(err, errlen, -2, "+init files are not supported");
    if (!kv.hasValue("proj"))
        return fail(err, errlen, -4, "projection not named");
    const std::string name = *kv.get("proj");
    if (isLatLongName(name))
        P->kind = PK_LATLONG;
    else if (name == "ob_tran")
        P->kind = PK_OB_TRAN;
    else if (name == "stere")
        P->kind = PK_STERE;
    else if (name == "lcc")
        P->kind = PK_LCC;
    else
        return fail(err, errlen, -5, "unknown projection id '" + name + "' (supported: latlong, ob_tran, stere, lcc)");

    if (!kv.flag("no_defs")) { // proj_def.dat defaults
        // pj_init does not default the ellipsoid when the string gives a datum or any earth figure: a
        // default +rf would otherwise win over a user's +b, and +datum=NAD83 would lose its GRS80
        if (!kv.has("datum") && !kv.has("ellps") && !kv.has("a") && !kv.has("b") && !kv.has("rf") && !kv.has("f"))
            kv.add("ellps", "WGS84");
        if (P->kind == PK_LCC) {
            kv.add("lat_1", "33");
            kv.add("lat_2", "45");
        }
    }

    // datum
    P->datum_kind = DK_UNKNOWN;
    if (kv.hasValue("datum")) {
        const std::string d = *kv.get("datum");
        if (d == "WGS84") {
            kv.add("ellps", "WGS84");
            kv.add("towgs84", "0,0,0");
        } else if (d == "NAD83") {
            kv.add("ellps", "GRS80");
            kv.add("towgs84", "0,0,0");
        } else {
            return fail(err, errlen, -9, "unsupported +datum=" + d);
        }
    }
    if (kv.has("nadgrids"))
        return fail(err, errlen, -38, "+nadgrids grid shifts are not supported");
    if (kv.hasValue("towgs84")) {
        const std::string t = *kv.get("towgs84");
        size_t pos = 0;
        for (int i = 0; i < 7 && pos <= t.size(); ++i) {
            P->datum[i] = std::strtod(t.c_str() + pos, nullptr);
            const size_t comma = t.find(',', pos);
            if (comma == std::string::npos)
                break;
            pos = comma + 1;
        }
        if (P->datum[3] != 0. || P->datum[4] != 0. || P->datum[5] != 0. || P->datum[6] != 0.) {
            P->datum_kind = DK_7PARAM;
            const double sec2rad = 4.84813681109535993589914102357e-6;
            P->datum[3] *= sec2rad;
            P->datum[4] *= sec2rad;
            P->datum[5] *= sec2rad;
            P->datum[6] = (P->datum[6] / 1000000.0) + 1;
        } else {
            P->datum_kind = DK_3PARAM;
        }
    }

    // ellipsoid
    double a = 0., es = 0.;
    if (kv.has("R")) {
        a = kv.num("R", 0.);
    } else {
        if (kv.hasValue("ellps")) {
            const std::string e = *kv.get("ellps");
            const Ellipsoid* found = nullptr;
            for (const auto& el : kEllipsoids)
                if (e == el.id)
                    found = &el;
            if (!found)
                return fail(err, errlen, -9, "unknown +ellps=" + e);
            char abuf[64];
            std::snprintf(abuf, sizeof(abuf), "%.17g", found->a);
            kv.add("a", abuf);
            kv.add(found->shapeKey, found->shapeVal);
        }
        a = kv.num("a", 0.);
        if (kv.has("es")) {
            es = kv.num("es", 0.);
        } else if (kv.has("e")) {
            const double e = kv.num("e", 0.);
            es = e * e;
        } else if (kv.has("rf")) {
            const double rf = kv.num("rf", 0.);
            if (rf == 0.)
                return fail(err, errlen, -10, "reciprocal flattening (1/f) = 0");
            es = 1. / rf;
            es = es * (2. - es);
        } else if (kv.has("f")) {
            es = kv.num("f", 0.);
            es = es * (2. - es);
        } else if (kv.has("b")) {
            const double b = kv.num("b", 0.);
            es = 1. - (b * b) / (a * a);
        }
    }
    if (es < 0.)
        return fail(err, errlen, -12, "squared eccentricity < 0");
    if (a <= 0.)
        return fail(err, errlen, -13, "major axis or radius = 0 or not given");
    P->a = P->a_orig = a;
    P->es = P->es_orig = es;
    P->e = std::sqrt(es);
    P->ra = 1. / a;
    P->one_es = 1. - es;
    if (P->one_es == 0.)
        return fail(err, errlen, -6, "effective eccentricity = 1");
    P->rone_es = 1. / P->one_es;
    if (P->datum_kind == DK_3PARAM && P->datum[0] == 0. && P->datum[1] == 0. && P->datum[2] == 0. && P->a == 6378137.0 &&
        std::fabs(P->es - 0.006694379990) < 0.000000000050)
        P->datum_kind = DK_WGS84;

    // general parameters
    P->geoc = (P->es != 0. && kv.flag("geoc")) ? 1 : 0;
    P->over = kv.flag("over") ? 1 : 0;
    auto angle = [&](const char* key, double* out) -> bool {
        *out = 0.;
        if (!kv.hasValue(key))
            return true;
        return parseAngle(*kv.get(key), out);
    };
    if (!angle("lon_0", &P->lam0) || !angle("lat_0", &P->phi0))
        return fail(err, errlen, -16, "malformed angle in +lon_0/+lat_0");
    P->x0 = kv.num("x_0", 0.);
    P->y0 = kv.num("y_0", 0.);
    P->k0 = kv.has("k_0") ? kv.num("k_0", 1.) : (kv.has("k") ? kv.num("k", 1.) : 1.);
    if (P->k0 <= 0.)
        return fail(err, errlen, -31, "k <= 0");
    P->to_meter = P->fr_meter = 1.;
    if (kv.hasValue("units")) {
        const std::string u = *kv.get("units");
        if (u == "m")
            P->to_meter = 1.;
        else if (u == "km")
            P->to_meter = 1000.;
        else
            return fail(err, errlen, -7, "unsupported +units=" + u);
        P->fr_meter = 1. / P->to_meter;
    } else if (kv.has("to_meter")) {
        P->to_meter = kv.num("to_meter", 1.);
        P->fr_meter = 1. / P->to_meter;
    }
    if (kv.has("pm"))
        return fail(err, errlen, -46, "+pm (prime meridian) is not supported");

    // projection specific
    switch (P->kind) {
    case PK_LATLONG:
        P->is_latlong = 1;
        P->x0 = P->y0 = 0.;
        break;
    case PK_OB_TRAN: {
        if (!kv.hasValue("o_proj"))
            return fail(err, errlen, -26, "ob_tran: no +o_proj");
        if (!isLatLongName(*kv.get("o_proj")))
            return fail(err, errlen, -5, "ob_tran: only +o_proj=longlat (rotated pole) is supported");
        if (!kv.has("o_lat_p"))
            return fail(err, errlen, -5, "ob_tran: only the +o_lat_p [+o_lon_p] form is supported");
        P->es = P->e = 0.;
        P->one_es = P->rone_es = 1.;
        double phip = 0.;
        if (!angle("o_lon_p", &P->ob_lamp) || !angle("o_lat_p", &phip))
            return fail(err, errlen, -16, "malformed angle in +o_lon_p/+o_lat_p");
        P->ob_oblique = std::fabs(phip) > 1e-10;
        if (P->ob_oblique) {
            P->ob_cphip = std::cos(phip);
            P->ob_sphip = std::sin(phip);
        }
        break;
    }
    case PK_STERE: {
        double phits = kHalfPi;
        if (kv.has("lat_ts") && !angle("lat_ts", &phits))
            return fail(err, errlen, -16, "malformed angle in +lat_ts");
        const double t0 = std::fabs(P->phi0);
        if (std::fabs(t0 - kHalfPi) < 1.e-10)
            P->st_mode = P->phi0 < 0. ? SM_SOUTH : SM_NORTH;
        else
            P->st_mode = t0 > 1.e-10 ? SM_OBLIQUE : SM_EQUATOR;
        phits = std::fabs(phits);
        const bool polar = (P->st_mode == SM_SOUTH || P->st_mode == SM_NORTH);
        if (P->es != 0.) {
            if (polar) {
                if (std::fabs(phits - kHalfPi) < 1.e-10) {
                    P->st_akm1 = 2. * P->k0 / std::sqrt(std::pow(1 + P->e, 1 + P->e) * std::pow(1 - P->e, 1 - P->e));
                } else {
                    double t = std::sin(phits);
                    const double se = t * P->e;
                    const double ts = std::tan(.5 * (kHalfPi - phits)) / std::pow((1. - se) / (1. + se), .5 * P->e);
                    P->st_akm1 = std::cos(phits) / ts;
                    t *= P->e;
                    P->st_akm1 /= std::sqrt(1. - t * t);
                }
            } else {
                double t = std::sin(P->phi0);
                const double se = t * P->e;
                const double X = 2. * std::atan(std::tan(.5 * (kHalfPi + P->phi0)) * std::pow((1. - se) / (1. + se), .5 * P->e)) - kHalfPi;
                t *= P->e;
                P->st_akm1 = 2. * P->k0 * std::cos(P->phi0) / std::sqrt(1. - t * t);
                P->st_sin1 = std::sin(X);
                P->st_cos1 = std::cos(X);
            }
        } else {
            if (polar) {
                P->st_akm1 = std::fabs(phits - kHalfPi) >= 1.e-10 ? std::cos(phits) / std::tan(kFortPi - .5 * phits) : 2. * P->k0;
            } else {
                if (P->st_mode == SM_OBLIQUE) {
                    P->st_sin1 = std::sin(P->phi0);
                    P->st_cos1 = std::cos(P->phi0);
                }
                P->st_akm1 = 2. * P->k0;
            }
        }
        break;
    }
    case PK_LCC: {
        double phi1 = 0., phi2 = 0.;
        if (!angle("lat_1", &phi1))
            return fail(err, errlen, -16, "malformed angle in +lat_1");
        if (kv.has("lat_2")) {
            if (!angle("lat_2", &phi2))
                return fail(err, errlen, -16, "malformed angle in +lat_2");
        } else {
            phi2 = phi1;
            if (!kv.has("lat_0"))
                P->phi0 = phi1;
        }
        if (std::fabs(phi1 + phi2) < 1.e-10)
            return fail(err, errlen, -21, "conic lat_1 = -lat_2");
        double sinphi = std::sin(phi1);
        const double cosphi = std::cos(phi1);
        double n = sinphi;
        const bool secant = std::fabs(phi1 - phi2) >= 1.e-10;
        P->lcc_ellips = (P->es != 0.) ? 1 : 0;
        auto tsfn = [&](double phi, double sp) {
            const double se = sp * P->e;
            return std::tan(.5 * (kHalfPi - phi)) / std::pow((1. - se) / (1. + se), .5 * P->e);
        };
        auto msfn = [&](double sp, double cp) { return cp / std::sqrt(1. - P->es * sp * sp); };
        if (P->lcc_ellips) {
            const double m1 = msfn(sinphi, cosphi);
            const double ml1 = tsfn(phi1, sinphi);
            if (secant) {
                sinphi = std::sin(phi2);
                n = std::log(m1 / msfn(sinphi, std::cos(phi2)));
                n /= std::log(ml1 / tsfn(phi2, sinphi));
            }
            P->lcc_rho0 = m1 * std::pow(ml1, -n) / n;
            P->lcc_c = P->lcc_rho0;
            P->lcc_rho0 *= (std::fabs(std::fabs(P->phi0) - kHalfPi) < 1.e-10) ? 0. : std::pow(tsfn(P->phi0, std::sin(P->phi0)), n);
        } else {
            if (secant)
                n = std::log(cosphi / std::cos(phi2)) / std::log(std::tan(kFortPi + .5 * phi2) / std::tan(kFortPi + .5 * phi1));
            P->lcc_c = cosphi * std::pow(std::tan(kFortPi + .5 * phi1), n) / n;
            P->lcc_rho0 = (std::fabs(std::fabs(P->phi0) - kHalfPi) < 1.e-10) ? 0. : P->lcc_c * std::pow(std::tan(kFortPi + .5 * P->phi0), -n);
        }
        P->lcc_n = n;
        break;
    }
    }
    return 0;
}

bool needs_datum_shift(const ProjDef& s, const ProjDef& d)
{
    if (s.datum_kind == DK_UNKNOWN || d.datum_kind == DK_UNKNOWN)
        return false;
    // identical datums
    if (s.datum_kind == d.datum_kind && s.a_orig == d.a_orig && std::fabs(s.es_orig - d.es_orig) <= 0.000000000050) {
        bool same = true;
        if (s.datum_kind == DK_3PARAM)
            same = s.datum[0] == d.datum[0] && s.datum[1] == d.datum[1] && s.datum[2] == d.datum[2];
        else if (s.datum_kind == DK_7PARAM)
            for (int i = 0; i < 7; ++i)
                same = same && s.datum[i] == d.datum[i];
        if (same)
            return false;
    }
    const bool s37 = s.datum_kind == DK_3PARAM || s.datum_kind == DK_7PARAM;
    const bool d37 = d.datum_kind == DK_3PARAM || d.datum_kind == DK_7PARAM;
    return s.es_orig != d.es_orig || s.a_orig != d.a_orig || s37 || d37;
}

} // namespace fb
