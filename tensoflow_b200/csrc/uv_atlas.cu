// UV atlas of box-projection charts and texture baking on the device.  The rules are stated in include/tensoflow_b200.h;
// oracle/torch_oracle_atlas.py restates them in numpy and the results here are bit-equal to it.  All fp64 arithmetic goes
// through __dadd_rn / __dsub_rn / __dmul_rn / __ddiv_rn / __dsqrt_rn in the oracle's operation order (no FMA contraction),
// every sum runs in a fixed order, and the only atomics are integer ones, so nothing depends on scheduling.
//
//   faces     per face the fp64 normal, its length, the initial class and the allowed classes; the half-edges
//   sort      a stable CUB radix sort of the half-edges by (min, max) vertex key: each edge's faces ascending
//   smooth    4 Jacobi passes over the edge neighbours
//   area      the projected area in fixed point (atomicMax of the largest, then an exact uint64 atomicAdd) -> s0
//   rounds    union-find over faces (union_find.cuh) -> charts numbered by root; chart boxes (ordered-uint atomics);
//             21 density trials, each a radix sort of the rectangles and one thread walking them (next-fit decreasing
//             height), with the bisection state kept on the device; texel coordinates; coverage in 8x8 tiles of the
//             faces' boxes (tile counts prefix-summed, one thread per tile); a second pass marks every face that covers a
//             centre some other face covers, and the next round's charts are computed at once, so the round ends with one
//             host read of (conflicting coverages, next chart count)
//   output    the (vertex, chart) corner keys radix-sorted, unique -> output vertices; one last host read of V'
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <algorithm>
#include "common.cuh"
#include "union_find.cuh"

namespace {

constexpr int SMOOTH_PASSES = 4;
constexpr int BISECTION_STEPS = 20;
constexpr int TILE = 8;

struct D3 {
    double x, y, z;
};

__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }

__device__ __forceinline__ int64_t gtid() { return blockIdx.x * (int64_t)blockDim.x + threadIdx.x; }
__device__ __forceinline__ int64_t gstride() { return (int64_t)gridDim.x * blockDim.x; }

__device__ __forceinline__ D3 load_p(const float* P, int32_t v) {
    return D3{(double)P[3 * (int64_t)v], (double)P[3 * (int64_t)v + 1], (double)P[3 * (int64_t)v + 2]};
}

// (b - a) x (c - a) of face f
__device__ __forceinline__ D3 face_normal(const float* P, const int32_t* F, int64_t f) {
    const D3 p0 = load_p(P, F[3 * f]), p1 = load_p(P, F[3 * f + 1]), p2 = load_p(P, F[3 * f + 2]);
    const D3 e1{dsub(p1.x, p0.x), dsub(p1.y, p0.y), dsub(p1.z, p0.z)};
    const D3 e2{dsub(p2.x, p0.x), dsub(p2.y, p0.y), dsub(p2.z, p0.z)};
    return D3{dsub(dmul(e1.y, e2.z), dmul(e1.z, e2.y)), dsub(dmul(e1.z, e2.x), dmul(e1.x, e2.z)),
              dsub(dmul(e1.x, e2.y), dmul(e1.y, e2.x))};
}

__device__ __forceinline__ double comp(const D3& n, int k) { return k == 0 ? n.x : (k == 1 ? n.y : n.z); }

// the projection (u, w) of position p for class c
__device__ __forceinline__ void project(const float* P, int32_t v, int c, float& u, float& w) {
    const int k = c >> 1, i1 = k == 2 ? 0 : k + 1, i2 = k == 0 ? 2 : k - 1;
    const float a = P[3 * (int64_t)v + i1], b = P[3 * (int64_t)v + i2];
    u = (c & 1) ? b : a;
    w = (c & 1) ? a : b;
}

// float <-> uint32 order-preserving maps for integer atomicMin / atomicMax
__device__ __forceinline__ uint32_t ord(float f) {
    const uint32_t b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float unord(uint32_t b) { return __uint_as_float((b & 0x80000000u) ? (b & 0x7fffffffu) : ~b); }

// the run [s, e) of sorted half-edge keys containing position p
__device__ __forceinline__ void run_of(const uint64_t* k, int64_t n, int64_t p, int64_t& s, int64_t& e) {
    const uint64_t key = k[p];
    s = p;
    while (s > 0 && k[s - 1] == key) --s;
    e = p + 1;
    while (e < n && k[e] == key) ++e;
}

__global__ void __launch_bounds__(256) ua_faces(const float* __restrict__ P, const int32_t* __restrict__ F, int64_t T,
                                                double* __restrict__ len, uint8_t* __restrict__ allowed, uint8_t* __restrict__ cls,
                                                uint64_t* __restrict__ he_k, uint32_t* __restrict__ he_v) {
    for (int64_t f = gtid(); f < T; f += gstride()) {
        const D3 n = face_normal(P, F, f);
        const double ln = __dsqrt_rn(dadd(dadd(dmul(n.x, n.x), dmul(n.y, n.y)), dmul(n.z, n.z)));
        len[f] = ln;
        const double ax = fabs(n.x), ay = fabs(n.y), az = fabs(n.z);
        int k = 0;
        double best = ax;
        if (ay > best) { k = 1; best = ay; }
        if (az > best) k = 2;
        cls[f] = (uint8_t)(2 * k + (comp(n, k) < 0.0 ? 1 : 0));
        const double half = dmul(ln, 0.5);
        uint8_t m = 0;
#pragma unroll
        for (int c = 0; c < 6; ++c) {
            const double v = (c & 1) ? -comp(n, c >> 1) : comp(n, c >> 1);
            if (v >= half) m |= (uint8_t)(1u << c);
        }
        allowed[f] = m;
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            const uint32_t a = (uint32_t)F[3 * f + j], b = (uint32_t)F[3 * f + (j == 2 ? 0 : j + 1)];
            he_k[3 * f + j] = ((uint64_t)min(a, b) << 32) | max(a, b);
            he_v[3 * f + j] = (uint32_t)(3 * f + j);
        }
    }
}

__global__ void __launch_bounds__(256) ua_positions(const uint32_t* __restrict__ he_v, int64_t n, int64_t* __restrict__ pos) {
    for (int64_t p = gtid(); p < n; p += gstride()) pos[he_v[p]] = p;
}

__device__ __forceinline__ void add6(double (&acc)[6], int c, double v) {
#pragma unroll
    for (int i = 0; i < 6; ++i)
        if (i == c) acc[i] = dadd(acc[i], v);
}

__global__ void __launch_bounds__(256) ua_smooth(const uint64_t* __restrict__ he_k, const uint32_t* __restrict__ he_v,
                                                 const int64_t* __restrict__ pos, int64_t T, const double* __restrict__ len,
                                                 const uint8_t* __restrict__ allowed, const uint8_t* __restrict__ cls_in,
                                                 uint8_t* __restrict__ cls_out) {
    const int64_t n = 3 * T;
    for (int64_t f = gtid(); f < T; f += gstride()) {
        double acc[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        const int own = cls_in[f];
        add6(acc, own, len[f]);
        for (int j = 0; j < 3; ++j) {
            const int64_t p = pos[3 * f + j];
            int64_t s, e;
            run_of(he_k, n, p, s, e);
            for (int64_t q = s; q < e; ++q) {
                if (q == p) continue;
                const int64_t g = he_v[q] / 3;
                add6(acc, cls_in[g], len[g]);
            }
        }
        int best = own;
        double bv = 0.0;
#pragma unroll
        for (int i = 0; i < 6; ++i)
            if (i == own) bv = acc[i];
        const uint8_t m = allowed[f];
#pragma unroll
        for (int i = 0; i < 6; ++i)
            if (((m >> i) & 1) && acc[i] > bv) { best = i; bv = acc[i]; }
        cls_out[f] = (uint8_t)best;
    }
}

// |n_k| of each face's class axis: pass 0 takes the largest (atomicMax of the fp64 bits, all >= 0), pass 1 sums
// rint(|n_k| / max * 2^32) exactly in uint64
template <int PASS>
__global__ void __launch_bounds__(256) ua_area(const float* __restrict__ P, const int32_t* __restrict__ F, int64_t T,
                                               const uint8_t* __restrict__ cls, unsigned long long* __restrict__ amax,
                                               unsigned long long* __restrict__ asum) {
    for (int64_t f = gtid(); f < T; f += gstride()) {
        const double a = fabs(comp(face_normal(P, F, f), cls[f] >> 1));
        if (PASS == 0) atomicMax(amax, (unsigned long long)__double_as_longlong(a));
        else atomicAdd(asum, __double2ull_rn(dmul(__ddiv_rn(a, __longlong_as_double((long long)*amax)), 4294967296.0)));
    }
}

// device state of the density search
struct Search {
    double s0, lo, hi, s_try, s;
    int32_t done, steps, nofit, total_steps;    // steps of this round's search, and of all rounds
};

__global__ void ua_search_init(const unsigned long long* __restrict__ amax, const unsigned long long* __restrict__ asum, int R,
                               Search* __restrict__ st) {
    const double m = __longlong_as_double((long long)*amax);
    const double A = dmul(dmul(__ull2double_rn(*asum), m), 0x1p-33);
    const double s0 = __ddiv_rn((double)R, __dsqrt_rn(A));
    st->s0 = s0;
    st->s_try = s0;
    st->s = 0.0;
    st->lo = 0.0;
    st->hi = s0;
    st->done = 0;
    st->steps = 0;
    st->total_steps = 0;
    st->nofit = !(m > 0.0);
}

__global__ void ua_search_restart(Search* __restrict__ st) {
    st->s_try = st->s0;
    st->lo = 0.0;
    st->hi = st->s0;
    st->done = 0;
    st->steps = 0;
}

__global__ void __launch_bounds__(256) ua_cc_init(int32_t* __restrict__ parent, int64_t T) {
    for (int64_t f = gtid(); f < T; f += gstride()) parent[f] = (int32_t)f;
}

// each half-edge joins its face to the next face of the run with the same class (neither solo): chains cover every such pair
__global__ void __launch_bounds__(256) ua_cc_link(const uint64_t* __restrict__ he_k, const uint32_t* __restrict__ he_v, int64_t n,
                                                  const uint8_t* __restrict__ cls, const uint8_t* __restrict__ solo, int32_t* parent) {
    for (int64_t p = gtid(); p < n; p += gstride()) {
        const int32_t f = (int32_t)(he_v[p] / 3);
        if (solo[f]) continue;
        const uint64_t key = he_k[p];
        for (int64_t q = p + 1; q < n && he_k[q] == key; ++q) {
            const int32_t g = (int32_t)(he_v[q] / 3);
            if (g == f || solo[g] || cls[g] != cls[f]) continue;
            tf_uf::unite(parent, f, g);
            break;
        }
    }
}

__global__ void __launch_bounds__(256) ua_cc_flatten(int32_t* parent, int64_t T, int32_t* __restrict__ is_root) {
    for (int64_t f = gtid(); f < T; f += gstride()) {
        const int32_t r = tf_uf::find(parent, (int32_t)f);
        tf_uf::set_parent(parent, (int32_t)f, r);
        is_root[f] = r == (int32_t)f;
    }
}

__global__ void __launch_bounds__(256) ua_chart_ids(const int32_t* __restrict__ parent, const int32_t* __restrict__ is_root,
                                                    const int32_t* __restrict__ rid, int64_t T, int32_t* __restrict__ chart,
                                                    int32_t* __restrict__ root_face, int64_t* __restrict__ n_charts) {
    for (int64_t f = gtid(); f < T; f += gstride()) {
        chart[f] = rid[parent[f]];
        if (is_root[f]) root_face[rid[f]] = (int32_t)f;
        if (f == T - 1) *n_charts = (int64_t)rid[f] + is_root[f];
    }
}

__global__ void __launch_bounds__(256) ua_bbox(const float* __restrict__ P, const int32_t* __restrict__ F, int64_t n,
                                               const uint8_t* __restrict__ cls, const int32_t* __restrict__ chart,
                                               uint32_t* __restrict__ bb) {
    for (int64_t i = gtid(); i < n; i += gstride()) {
        const int64_t f = i / 3;
        float u, w;
        project(P, F[i], cls[f], u, w);
        uint32_t* b = bb + 4 * (int64_t)chart[f];
        atomicMin(b, ord(u));
        atomicMax(b + 1, ord(u));
        atomicMin(b + 2, ord(w));
        atomicMax(b + 3, ord(w));
    }
}

__device__ __forceinline__ int32_t rect_in(uint32_t lo, uint32_t hi, double s, int R) {
    const double t = dmul(dsub((double)unord(hi), (double)unord(lo)), s);
    const double d = ceil(fmin(t, (double)R + 1.0));
    return d < 1.0 ? 1 : (int32_t)d;
}

// sort keys (0x7fff - h) << 46 | (0x7fff - w) << 31 | chart: ascending is (h desc, w desc, chart asc)
__global__ void __launch_bounds__(256) ua_rect_keys(const uint32_t* __restrict__ bb, int64_t C, int R, int pad, bool final_pass,
                                                    const Search* __restrict__ st, uint64_t* __restrict__ keys) {
    if (!final_pass && st->done) return;
    const double s = final_pass ? st->s : st->s_try;
    for (int64_t c = gtid(); c < C; c += gstride()) {
        const uint64_t w = rect_in(bb[4 * c], bb[4 * c + 1], s, R) + 2 * pad, h = rect_in(bb[4 * c + 2], bb[4 * c + 3], s, R) + 2 * pad;
        keys[c] = ((0x7fffull - h) << 46) | ((0x7fffull - w) << 31) | (uint64_t)c;
    }
}

// next-fit decreasing height over the sorted rectangles, one thread; then the bisection state moves on.  The final pass writes
// the rectangles (x0, y0, w, h) and the density the round uses.
__global__ void ua_nfdh(const uint64_t* __restrict__ keys, int64_t C, int R, bool final_pass, Search* __restrict__ st,
                        int32_t* __restrict__ rects) {
    if (!final_pass && st->done) return;
    int64_t x = 0, y = 0, shelf = 0;
    bool fits = true;
    for (int64_t i = 0; i < C; ++i) {
        const uint64_t k = keys[i];
        const int64_t c = (int64_t)(k & 0x7fffffffull), w = 0x7fff - (int64_t)((k >> 31) & 0x7fff), h = 0x7fff - (int64_t)(k >> 46);
        if (w > R) { fits = false; break; }
        if (x + w > R) { y += shelf; x = 0; shelf = 0; }
        if (shelf == 0) shelf = h;
        if (final_pass) {
            rects[4 * c] = (int32_t)x;
            rects[4 * c + 1] = (int32_t)y;
            rects[4 * c + 2] = (int32_t)w;
            rects[4 * c + 3] = (int32_t)h;
        }
        x += w;
        if (y + shelf > R) { fits = false; break; }
    }
    if (final_pass) return;
    ++st->steps;
    ++st->total_steps;
    if (st->steps == 1) {                          // the trial at s0
        if (fits) { st->done = 1; st->s = st->s0; return; }
    } else if (fits) st->lo = st->s_try;
    else st->hi = st->s_try;
    if (st->steps == BISECTION_STEPS + 1) {
        st->done = 1;
        st->s = st->lo;
        if (st->lo == 0.0) st->nofit = 1;
        return;
    }
    st->s_try = dmul(dadd(st->lo, st->hi), 0.5);
}

__global__ void __launch_bounds__(256) ua_corner_xy(const float* __restrict__ P, const int32_t* __restrict__ F, int64_t n,
                                                    const uint8_t* __restrict__ cls, const int32_t* __restrict__ chart,
                                                    const uint32_t* __restrict__ bb, const int32_t* __restrict__ rects, int pad,
                                                    const Search* __restrict__ st, float2* __restrict__ xy) {
    const double s = st->s;
    for (int64_t i = gtid(); i < n; i += gstride()) {
        const int64_t f = i / 3, c = chart[f];
        float u, w;
        project(P, F[i], cls[f], u, w);
        const double x = dadd((double)(rects[4 * c] + pad), dmul(dsub((double)u, (double)unord(bb[4 * c])), s));
        const double y = dadd((double)(rects[4 * c + 1] + pad), dmul(dsub((double)w, (double)unord(bb[4 * c + 2])), s));
        xy[i] = make_float2(__double2float_rn(x), __double2float_rn(y));
    }
}

// texel-centre box [i0, i0 + ni) x [j0, j0 + nj) of face f
__device__ __forceinline__ void centre_box(const float2* xy, int64_t f, int R, int32_t& i0, int32_t& ni, int32_t& j0, int32_t& nj) {
    const float2 a = xy[3 * f], b = xy[3 * f + 1], c = xy[3 * f + 2];
    const double xmin = fmin((double)a.x, fmin((double)b.x, (double)c.x)), xmax = fmax((double)a.x, fmax((double)b.x, (double)c.x));
    const double ymin = fmin((double)a.y, fmin((double)b.y, (double)c.y)), ymax = fmax((double)a.y, fmax((double)b.y, (double)c.y));
    const double lo_i = fmin(fmax(ceil(xmin - 0.5), 0.0), (double)(R - 1)), hi_i = fmin(fmax(floor(xmax - 0.5), -1.0), (double)(R - 1));
    const double lo_j = fmin(fmax(ceil(ymin - 0.5), 0.0), (double)(R - 1)), hi_j = fmin(fmax(floor(ymax - 0.5), -1.0), (double)(R - 1));
    i0 = (int32_t)lo_i;
    j0 = (int32_t)lo_j;
    ni = max(0, (int32_t)hi_i - i0 + 1);
    nj = max(0, (int32_t)hi_j - j0 + 1);
}

__global__ void __launch_bounds__(256) ua_tile_count(const float2* __restrict__ xy, int64_t T, int R, int64_t* __restrict__ cnt) {
    for (int64_t f = gtid(); f < T; f += gstride()) {
        int32_t i0, ni, j0, nj;
        centre_box(xy, f, R, i0, ni, j0, nj);
        cnt[f] = (int64_t)((ni + TILE - 1) / TILE) * ((nj + TILE - 1) / TILE);
    }
}

__global__ void ua_tile_total(const int64_t* __restrict__ cnt, const int64_t* __restrict__ off, int64_t T, int64_t* __restrict__ total) {
    *total = off[T - 1] + cnt[T - 1];
}

struct Edge {
    double e, dx, dy;
};

// the edge function of p -> q at (cx, cy), evaluated from the endpoint smaller in (x, y) order and negated for the other
// direction, so that the two faces of a shared edge see one value
__device__ __forceinline__ Edge edge_fn(double px, double py, double qx, double qy, double cx, double cy) {
    const bool bp = px < qx || (px == qx && py <= qy);
    const double bx = bp ? px : qx, by = bp ? py : qy, ox = bp ? qx : px, oy = bp ? qy : py;
    const double ex = dsub(ox, bx), ey = dsub(oy, by);
    const double e = dsub(dmul(ex, dsub(cy, by)), dmul(ey, dsub(cx, bx)));
    return bp ? Edge{e, ex, ey} : Edge{-e, -ex, -ey};
}

__device__ __forceinline__ bool inside(const Edge& g) { return g.e > 0.0 || (g.e == 0.0 && (g.dy < 0.0 || (g.dy == 0.0 && g.dx < 0.0))); }

// MODE 0: claim every covered texel (atomicCAS from -1) and mark the chart as hit; MODE 1: a face that finds another owner
// marks both solo and counts one conflict
template <int MODE>
__global__ void __launch_bounds__(256) ua_raster(const float2* __restrict__ xy, int64_t T, int R, const int64_t* __restrict__ off,
                                                 const int64_t* __restrict__ total, const int32_t* __restrict__ chart,
                                                 int32_t* owner, uint8_t* __restrict__ hit, uint8_t* __restrict__ solo,
                                                 unsigned long long* __restrict__ n_conf) {
    const int64_t items = *total;
    for (int64_t it = gtid(); it < items; it += gstride()) {
        int64_t lo = 0, hi = T - 1;                    // the last face with off <= it
        while (lo < hi) {
            const int64_t mid = (lo + hi + 1) >> 1;
            if (off[mid] <= it) lo = mid; else hi = mid - 1;
        }
        const int64_t f = lo;
        const int32_t r = (int32_t)(it - off[f]);      // fewer than (16384 / 8)^2 tiles per face
        int32_t i0, ni, j0, nj;
        centre_box(xy, f, R, i0, ni, j0, nj);
        const int32_t ntx = (ni + TILE - 1) / TILE;
        const int32_t ti = i0 + (r % ntx) * TILE, tj = j0 + (r / ntx) * TILE;
        const float2 fa = xy[3 * f], fb = xy[3 * f + 1], fc = xy[3 * f + 2];
        const double ax = fa.x, ay = fa.y;
        const Edge area = edge_fn(ax, ay, fb.x, fb.y, fc.x, fc.y);
        if (area.e == 0.0) continue;
        const bool flip = area.e < 0.0;
        const double bx = flip ? fc.x : fb.x, by = flip ? fc.y : fb.y, cx = flip ? fb.x : fc.x, cy = flip ? fb.y : fc.y;
        const int32_t ie = min(ti + TILE, i0 + ni), je = min(tj + TILE, j0 + nj);
        for (int32_t j = tj; j < je; ++j)
            for (int32_t i = ti; i < ie; ++i) {
                const double px = i + 0.5, py = j + 0.5;
                if (!inside(edge_fn(ax, ay, bx, by, px, py)) || !inside(edge_fn(bx, by, cx, cy, px, py)) ||
                    !inside(edge_fn(cx, cy, ax, ay, px, py)))
                    continue;
                const int64_t t = (int64_t)j * R + i;
                if (MODE == 0) {
                    atomicCAS(owner + t, -1, (int32_t)f);
                    hit[chart[f]] = 1;
                } else {
                    const int32_t o = owner[t];
                    if (o != (int32_t)f) {
                        solo[f] = 1;
                        solo[o] = 1;
                        atomicAdd(n_conf, 1ull);
                    }
                }
            }
    }
}

// a chart that covers no centre gets the texel under its root face's texel centroid, clamped into its rectangle's interior
__global__ void __launch_bounds__(256) ua_fallback(const float2* __restrict__ xy, int64_t C, int R, int pad,
                                                   const uint8_t* __restrict__ hit, const int32_t* __restrict__ root_face,
                                                   const int32_t* __restrict__ rects, int32_t* __restrict__ owner) {
    for (int64_t c = gtid(); c < C; c += gstride()) {
        if (hit[c]) continue;
        const int64_t f = root_face[c];
        const float2 a = xy[3 * f], b = xy[3 * f + 1], d = xy[3 * f + 2];
        const double cx = dmul(dadd(dadd((double)a.x, (double)b.x), (double)d.x), 1.0 / 3.0);
        const double cy = dmul(dadd(dadd((double)a.y, (double)b.y), (double)d.y), 1.0 / 3.0);
        const int32_t* q = rects + 4 * c;
        const int32_t i = (int32_t)fmin(fmax(floor(cx), (double)(q[0] + pad)), (double)(q[0] + q[2] - pad - 1));
        const int32_t j = (int32_t)fmin(fmax(floor(cy), (double)(q[1] + pad)), (double)(q[1] + q[3] - pad - 1));
        owner[(int64_t)j * R + i] = (int32_t)f;
    }
}

__global__ void __launch_bounds__(256) ua_corner_keys(const int32_t* __restrict__ F, const int32_t* __restrict__ chart, int64_t n,
                                                      uint64_t* __restrict__ keys, uint32_t* __restrict__ idx) {
    for (int64_t i = gtid(); i < n; i += gstride()) {
        keys[i] = ((uint64_t)(uint32_t)F[i] << 32) | (uint32_t)chart[i / 3];
        idx[i] = (uint32_t)i;
    }
}

__global__ void __launch_bounds__(256) ua_heads(const uint64_t* __restrict__ keys, int64_t n, int32_t* __restrict__ head) {
    for (int64_t p = gtid(); p < n; p += gstride()) head[p] = p == 0 || keys[p] != keys[p - 1];
}

__global__ void __launch_bounds__(256) ua_out_vertices(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ idx,
                                                       const int32_t* __restrict__ head, const int32_t* __restrict__ incl, int64_t n,
                                                       const float2* __restrict__ xy, int32_t* __restrict__ out_tri,
                                                       int64_t* __restrict__ out_vertex, float2* __restrict__ out_xy,
                                                       int64_t* __restrict__ n_out) {
    for (int64_t p = gtid(); p < n; p += gstride()) {
        const int32_t id = incl[p] - 1;
        const uint32_t corner = idx[p];
        out_tri[corner] = id;
        if (head[p]) {
            out_vertex[id] = (int64_t)(keys[p] >> 32);
            out_xy[id] = xy[corner];
        }
        if (p == n - 1) *n_out = incl[p];
    }
}

// ---- baking ----------------------------------------------------------------------------------------------------------

__global__ void __launch_bounds__(256) ua_texel_points(const float* __restrict__ P, const int32_t* __restrict__ F,
                                                       const float* __restrict__ xy, const int32_t* __restrict__ texel_tri, int R,
                                                       const int64_t* __restrict__ texels, int64_t n, float* __restrict__ out) {
    for (int64_t i = gtid(); i < n; i += gstride()) {
        const int64_t t = texels[i];
        const int64_t f = texel_tri[t];
        const int32_t va = F[3 * f], vb = F[3 * f + 1], vc = F[3 * f + 2];
        const double xa = xy[2 * (int64_t)va], ya = xy[2 * (int64_t)va + 1], xb = xy[2 * (int64_t)vb], yb = xy[2 * (int64_t)vb + 1];
        const double xc = xy[2 * (int64_t)vc], yc = xy[2 * (int64_t)vc + 1];
        const double px = (double)(t % R) + 0.5, py = (double)(t / R) + 0.5;
        const double area = dsub(dmul(dsub(xb, xa), dsub(yc, ya)), dmul(dsub(yb, ya), dsub(xc, xa)));
        double la = 1.0 / 3.0, lb = 1.0 / 3.0, lc = 1.0 / 3.0;
        if (area != 0.0) {
            double a = __ddiv_rn(dsub(dmul(dsub(xc, xb), dsub(py, yb)), dmul(dsub(yc, yb), dsub(px, xb))), area);
            double b = __ddiv_rn(dsub(dmul(dsub(xa, xc), dsub(py, yc)), dmul(dsub(ya, yc), dsub(px, xc))), area);
            double c = __ddiv_rn(dsub(dmul(dsub(xb, xa), dsub(py, ya)), dmul(dsub(yb, ya), dsub(px, xa))), area);
            a = fmax(a, 0.0);
            b = fmax(b, 0.0);
            c = fmax(c, 0.0);
            const double sm = dadd(dadd(a, b), c);
            if (sm > 0.0) {
                la = __ddiv_rn(a, sm);
                lb = __ddiv_rn(b, sm);
                lc = __ddiv_rn(c, sm);
            }
        }
        const D3 pa = load_p(P, va), pb = load_p(P, vb), pc = load_p(P, vc);
        out[3 * i] = __double2float_rn(dadd(dadd(dmul(la, pa.x), dmul(lb, pb.x)), dmul(lc, pc.x)));
        out[3 * i + 1] = __double2float_rn(dadd(dadd(dmul(la, pa.y), dmul(lb, pb.y)), dmul(lc, pc.y)));
        out[3 * i + 2] = __double2float_rn(dadd(dadd(dmul(la, pa.z), dmul(lb, pb.z)), dmul(lc, pc.z)));
    }
}

__global__ void __launch_bounds__(256) ua_scatter(const float* __restrict__ values, const int64_t* __restrict__ texels, int64_t n,
                                                  int C, const int32_t* __restrict__ texel_tri, const int32_t* __restrict__ chart,
                                                  float* __restrict__ tex, int32_t* __restrict__ tchart) {
    for (int64_t i = gtid(); i < n; i += gstride()) {
        const int64_t t = texels[i];
        for (int c = 0; c < C; ++c) tex[t * C + c] = values[i * C + c];
        tchart[t] = chart[texel_tri[t]];
    }
}

// one dilation pass: an empty texel inside the rectangle of a filled 8-neighbour's chart takes the fp32 mean of those
// neighbours, summed in row order
__global__ void __launch_bounds__(256) ua_dilate(const float* __restrict__ src, const int32_t* __restrict__ sch, int R, int C,
                                                 const int32_t* __restrict__ rects, float* __restrict__ dst, int32_t* __restrict__ dch) {
    const int64_t RR = (int64_t)R * R;
    for (int64_t t = gtid(); t < RR; t += gstride()) {
        const int32_t own = sch[t];
        const int32_t i = (int32_t)(t % R), j = (int32_t)(t / R);
        uint32_t mask = 0;
        int32_t cnt = 0, nc = -1;
        if (own < 0) {
            int b = 0;
            for (int dy = -1; dy <= 1; ++dy)
                for (int dx = -1; dx <= 1; ++dx) {
                    if (dx == 0 && dy == 0) continue;
                    const int32_t ni = i + dx, nj = j + dy;
                    if (ni >= 0 && ni < R && nj >= 0 && nj < R) {
                        const int32_t c = sch[(int64_t)nj * R + ni];
                        if (c >= 0) {
                            const int32_t* q = rects + 4 * (int64_t)c;
                            if (i >= q[0] && i < q[0] + q[2] && j >= q[1] && j < q[1] + q[3]) {
                                mask |= 1u << b;
                                ++cnt;
                                nc = c;
                            }
                        }
                    }
                    ++b;
                }
        }
        dch[t] = cnt > 0 ? nc : own;
        for (int c = 0; c < C; ++c) {
            if (cnt == 0) {
                dst[t * C + c] = src[t * C + c];
                continue;
            }
            float acc = 0.0f;
            int b = 0;
            for (int dy = -1; dy <= 1; ++dy)
                for (int dx = -1; dx <= 1; ++dx) {
                    if (dx == 0 && dy == 0) continue;
                    if ((mask >> b) & 1) acc = __fadd_rn(acc, src[((int64_t)(j + dy) * R + (i + dx)) * C + c]);
                    ++b;
                }
            dst[t * C + c] = __fdiv_rn(acc, (float)cnt);
        }
    }
}

unsigned grid_for(int64_t n) {
    const int64_t cap = (int64_t)tf_num_sms() * 8;
    return (unsigned)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, cap));
}

int key_bits(int64_t n) {
    int bits = 1;
    while ((int64_t(1) << bits) < n) ++bits;
    return bits;
}

constexpr size_t ALIGN = 256;
size_t up(size_t b) { return (b + ALIGN - 1) / ALIGN * ALIGN; }

struct Layout {
    size_t len, allowed, cls0, cls1, solo, parent, is_root, rid, chart0, chart1, root0, root1, tcnt, toff, hek0, hek1, hev0, hev1,
        pos, xy, bb, hit, rects, rkey0, rkey1, head, incl, counters, search, tmp, tmp_bytes, total;
};

int make_layout(int64_t V, int64_t T, Layout& L, const char* who) {
    const int64_t n = 3 * T;
    size_t b[5] = {0, 0, 0, 0, 0};
    cudaError_t e;
    {
        cub::DoubleBuffer<uint64_t> k(nullptr, nullptr);
        cub::DoubleBuffer<uint32_t> v(nullptr, nullptr);
        e = cub::DeviceRadixSort::SortPairs(nullptr, b[0], k, v, (int)n, 0, 32 + key_bits(V));
        TF_REQUIRE(e == cudaSuccess, "%s: radix sort sizing failed: %s", who, cudaGetErrorString(e));
        e = cub::DeviceRadixSort::SortKeys(nullptr, b[1], k, (int)T, 0, 61);
        TF_REQUIRE(e == cudaSuccess, "%s: radix sort sizing failed: %s", who, cudaGetErrorString(e));
    }
    e = cub::DeviceScan::ExclusiveSum(nullptr, b[2], (const int32_t*)nullptr, (int32_t*)nullptr, (int)T);
    TF_REQUIRE(e == cudaSuccess, "%s: scan sizing failed: %s", who, cudaGetErrorString(e));
    e = cub::DeviceScan::ExclusiveSum(nullptr, b[3], (const int64_t*)nullptr, (int64_t*)nullptr, (int)T);
    TF_REQUIRE(e == cudaSuccess, "%s: scan sizing failed: %s", who, cudaGetErrorString(e));
    e = cub::DeviceScan::InclusiveSum(nullptr, b[4], (const int32_t*)nullptr, (int32_t*)nullptr, (int)n);
    TF_REQUIRE(e == cudaSuccess, "%s: scan sizing failed: %s", who, cudaGetErrorString(e));
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += up(bytes); return o; };
    L.len = take(T * sizeof(double));
    L.allowed = take(T);
    L.cls0 = take(T);
    L.cls1 = take(T);
    L.solo = take(T);
    L.parent = take(T * sizeof(int32_t));
    L.is_root = take(T * sizeof(int32_t));
    L.rid = take(T * sizeof(int32_t));
    L.chart0 = take(T * sizeof(int32_t));
    L.chart1 = take(T * sizeof(int32_t));
    L.root0 = take(T * sizeof(int32_t));
    L.root1 = take(T * sizeof(int32_t));
    L.tcnt = take(T * sizeof(int64_t));
    L.toff = take(T * sizeof(int64_t));
    L.hek0 = take(n * sizeof(uint64_t));
    L.hek1 = take(n * sizeof(uint64_t));
    L.hev0 = take(n * sizeof(uint32_t));
    L.hev1 = take(n * sizeof(uint32_t));
    L.pos = take(n * sizeof(int64_t));
    L.xy = take(n * sizeof(float2));
    L.bb = take(T * 4 * sizeof(uint32_t));
    L.hit = take(T);
    L.rects = take(T * 4 * sizeof(int32_t));
    L.rkey0 = take(T * sizeof(uint64_t));
    L.rkey1 = take(T * sizeof(uint64_t));
    L.head = take(n * sizeof(int32_t));
    L.incl = take(n * sizeof(int32_t));
    L.counters = take(8 * sizeof(int64_t));
    L.search = take(sizeof(Search));
    L.tmp_bytes = *std::max_element(b, b + 5);
    L.tmp = take(L.tmp_bytes);
    L.total = off;
    return 0;
}

int check_sizes(int64_t V, int64_t T, int R, const char* who) {
    TF_REQUIRE(V > 0 && V < (int64_t(1) << 31), "%s: %lld vertices, need 0 < V < 2^31", who, (long long)V);
    TF_REQUIRE(T > 0 && T < (int64_t(1) << 31), "%s: %lld triangles, need 0 < T < 2^31", who, (long long)T);
    TF_REQUIRE(3 * T < (int64_t(1) << 31), "%s: %lld triangles, the sorts need 3 T < 2^31", who, (long long)T);
    TF_REQUIRE(R >= 16 && R <= 16384, "%s: resolution %d, need 16 <= R <= 16384", who, R);
    return 0;
}

}  // namespace

extern "C" TF_API int tf_uv_atlas_sizes(int64_t n_vertices, int64_t n_triangles, int32_t resolution, size_t* workspace_bytes) {
    TF_REQUIRE(workspace_bytes, "tf_uv_atlas_sizes: NULL pointer");
    if (check_sizes(n_vertices, n_triangles, resolution, "tf_uv_atlas_sizes")) return 1;
    Layout L;
    if (make_layout(n_vertices, n_triangles, L, "tf_uv_atlas_sizes")) return 1;
    *workspace_bytes = L.total;
    return 0;
}

extern "C" TF_API int tf_uv_atlas(const float* vertices, int64_t n_vertices, const int32_t* triangles, int64_t n_triangles,
                                  int32_t resolution, int32_t padding, void* workspace, size_t workspace_bytes, int32_t* out_chart,
                                  int32_t* out_triangles, int64_t* out_vertex_index, float* out_xy, int32_t* out_texel_tri,
                                  int32_t* out_rects, double* out_scale, int64_t* out_n_vertices, int64_t* out_n_charts,
                                  int32_t* out_rounds, int32_t* out_steps, tf_stream_t stream) {
    TF_REQUIRE(vertices && triangles && workspace && out_chart && out_triangles && out_vertex_index && out_xy && out_texel_tri &&
                   out_rects && out_scale && out_n_vertices && out_n_charts && out_rounds && out_steps,
               "tf_uv_atlas: NULL pointer");
    if (check_sizes(n_vertices, n_triangles, resolution, "tf_uv_atlas")) return 1;
    TF_REQUIRE(padding >= 1 && padding <= 16, "tf_uv_atlas: padding %d, need 1 <= padding <= 16", padding);
    const int64_t V = n_vertices, T = n_triangles, n = 3 * T;
    const int R = resolution, pad = padding;
    Layout L;
    if (make_layout(V, T, L, "tf_uv_atlas")) return 1;
    TF_REQUIRE(workspace_bytes >= L.total, "tf_uv_atlas: workspace of %zu bytes, %zu needed", workspace_bytes, L.total);
    char* ws = static_cast<char*>(workspace);
    auto at = [&](size_t o) { return static_cast<void*>(ws + o); };
    double* len = static_cast<double*>(at(L.len));
    uint8_t* allowed = static_cast<uint8_t*>(at(L.allowed));
    uint8_t* cls = static_cast<uint8_t*>(at(L.cls0));
    uint8_t* cls_alt = static_cast<uint8_t*>(at(L.cls1));
    uint8_t* solo = static_cast<uint8_t*>(at(L.solo));
    int32_t* parent = static_cast<int32_t*>(at(L.parent));
    int32_t* is_root = static_cast<int32_t*>(at(L.is_root));
    int32_t* rid = static_cast<int32_t*>(at(L.rid));
    int32_t* chart[2] = {static_cast<int32_t*>(at(L.chart0)), static_cast<int32_t*>(at(L.chart1))};
    int32_t* root_face[2] = {static_cast<int32_t*>(at(L.root0)), static_cast<int32_t*>(at(L.root1))};
    int64_t* tcnt = static_cast<int64_t*>(at(L.tcnt));
    int64_t* toff = static_cast<int64_t*>(at(L.toff));
    int64_t* pos = static_cast<int64_t*>(at(L.pos));
    float2* xy = static_cast<float2*>(at(L.xy));
    uint32_t* bb = static_cast<uint32_t*>(at(L.bb));
    uint8_t* hit = static_cast<uint8_t*>(at(L.hit));
    int32_t* rects = static_cast<int32_t*>(at(L.rects));
    int32_t* head = static_cast<int32_t*>(at(L.head));
    int32_t* incl = static_cast<int32_t*>(at(L.incl));
    // counters: [0], [1] chart counts of the two chart buffers, [2] conflicts, [3] n_vertices out, [4] amax bits, [5] area sum,
    // [6] tile total
    int64_t* counters = static_cast<int64_t*>(at(L.counters));
    unsigned long long* ull = reinterpret_cast<unsigned long long*>(counters);
    Search* search = static_cast<Search*>(at(L.search));
    void* tmp = at(L.tmp);
    const cudaStream_t s = (cudaStream_t)stream;
    int launches = 0;
    cudaError_t e = cudaSuccess;
    auto fail = [&](const char* what) {
        tf_count_launches(launches);
        tf_set_error("tf_uv_atlas: %s failed: %s", what, cudaGetErrorString(e));
        return 2;
    };
    const unsigned gt = grid_for(T), gn = grid_for(n);
    if ((e = cudaMemsetAsync(counters, 0, 8 * sizeof(int64_t), s)) != cudaSuccess || (e = cudaMemsetAsync(solo, 0, T, s)) != cudaSuccess)
        return fail("memset");

    cub::DoubleBuffer<uint64_t> hek(static_cast<uint64_t*>(at(L.hek0)), static_cast<uint64_t*>(at(L.hek1)));
    cub::DoubleBuffer<uint32_t> hev(static_cast<uint32_t*>(at(L.hev0)), static_cast<uint32_t*>(at(L.hev1)));
    ua_faces<<<gt, 256, 0, s>>>(vertices, triangles, T, len, allowed, cls, hek.Current(), hev.Current());
    ++launches;
    size_t tb = L.tmp_bytes;
    if ((e = cub::DeviceRadixSort::SortPairs(tmp, tb, hek, hev, (int)n, 0, 32 + key_bits(V), s)) != cudaSuccess) return fail("radix sort");
    const uint64_t* he_k = hek.Current();
    const uint32_t* he_v = hev.Current();
    ua_positions<<<gn, 256, 0, s>>>(he_v, n, pos);
    ++launches;
    for (int i = 0; i < SMOOTH_PASSES; ++i) {
        ua_smooth<<<gt, 256, 0, s>>>(he_k, he_v, pos, T, len, allowed, cls, cls_alt);
        std::swap(cls, cls_alt);
        ++launches;
    }
    ua_area<0><<<gt, 256, 0, s>>>(vertices, triangles, T, cls, ull + 4, ull + 5);
    ua_area<1><<<gt, 256, 0, s>>>(vertices, triangles, T, cls, ull + 4, ull + 5);
    ua_search_init<<<1, 1, 0, s>>>(ull + 4, ull + 5, R, search);
    launches += 3;

    // charts of the current solo set into buffer b; its count goes to counters[b]
    auto make_charts = [&](int b) -> bool {
        ua_cc_init<<<gt, 256, 0, s>>>(parent, T);
        ua_cc_link<<<gn, 256, 0, s>>>(he_k, he_v, n, cls, solo, parent);
        ua_cc_flatten<<<gt, 256, 0, s>>>(parent, T, is_root);
        size_t tb2 = L.tmp_bytes;
        if ((e = cub::DeviceScan::ExclusiveSum(tmp, tb2, is_root, rid, (int)T, s)) != cudaSuccess) return false;
        ua_chart_ids<<<gt, 256, 0, s>>>(parent, is_root, rid, T, chart[b], root_face[b], counters + b);
        launches += 4;
        return true;
    };
    int cur = 0;
    if (!make_charts(cur)) return fail("scan");
    int64_t C = 0;
    if ((e = cudaMemcpyAsync(&C, counters + cur, sizeof(int64_t), cudaMemcpyDeviceToHost, s)) != cudaSuccess) return fail("count read");
    if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return fail("charts");
    int32_t rounds = 0;
    for (;;) {
        const unsigned gc = grid_for(C);
        if ((e = cudaMemsetAsync(bb, 0, C * 4 * sizeof(uint32_t), s)) != cudaSuccess) return fail("memset");
        // minima start at 0xffffffff, maxima at 0
        for (int k = 0; k < 4; k += 2)
            if ((e = cudaMemset2DAsync(bb + k, 4 * sizeof(uint32_t), 0xff, sizeof(uint32_t), C, s)) != cudaSuccess) return fail("memset");
        ua_bbox<<<gn, 256, 0, s>>>(vertices, triangles, n, cls, chart[cur], bb);
        ua_search_restart<<<1, 1, 0, s>>>(search);
        launches += 2;
        cub::DoubleBuffer<uint64_t> rk(static_cast<uint64_t*>(at(L.rkey0)), static_cast<uint64_t*>(at(L.rkey1)));
        for (int step = 0; step <= BISECTION_STEPS + 1; ++step) {
            const bool final_pass = step == BISECTION_STEPS + 1;
            ua_rect_keys<<<gc, 256, 0, s>>>(bb, C, R, pad, final_pass, search, rk.Current());
            tb = L.tmp_bytes;
            if ((e = cub::DeviceRadixSort::SortKeys(tmp, tb, rk, (int)C, 0, 61, s)) != cudaSuccess) return fail("radix sort");
            ua_nfdh<<<1, 1, 0, s>>>(rk.Current(), C, R, final_pass, search, rects);
            launches += 2;
        }
        ua_corner_xy<<<gn, 256, 0, s>>>(vertices, triangles, n, cls, chart[cur], bb, rects, pad, search, xy);
        ua_tile_count<<<gt, 256, 0, s>>>(xy, T, R, tcnt);
        launches += 2;
        tb = L.tmp_bytes;
        if ((e = cub::DeviceScan::ExclusiveSum(tmp, tb, tcnt, toff, (int)T, s)) != cudaSuccess) return fail("scan");
        ua_tile_total<<<1, 1, 0, s>>>(tcnt, toff, T, counters + 6);
        if ((e = cudaMemsetAsync(out_texel_tri, 0xff, (size_t)R * R * sizeof(int32_t), s)) != cudaSuccess ||
            (e = cudaMemsetAsync(hit, 0, C, s)) != cudaSuccess || (e = cudaMemsetAsync(counters + 2, 0, sizeof(int64_t), s)) != cudaSuccess)
            return fail("memset");
        const unsigned gr = (unsigned)tf_num_sms() * 8;
        ua_raster<0><<<gr, 256, 0, s>>>(xy, T, R, toff, counters + 6, chart[cur], out_texel_tri, hit, solo, ull + 2);
        ua_raster<1><<<gr, 256, 0, s>>>(xy, T, R, toff, counters + 6, chart[cur], out_texel_tri, hit, solo, ull + 2);
        launches += 3;
        // the next round's charts, computed before the read so that the round costs one
        if (!make_charts(1 - cur)) return fail("scan");
        int64_t got[3] = {0, 0, 0};
        Search hs;
        if ((e = cudaMemcpyAsync(got, counters, 3 * sizeof(int64_t), cudaMemcpyDeviceToHost, s)) != cudaSuccess ||
            (e = cudaMemcpyAsync(&hs, search, sizeof(Search), cudaMemcpyDeviceToHost, s)) != cudaSuccess)
            return fail("count read");
        if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return fail("round");
        if (hs.nofit) {
            tf_count_launches(launches);
            tf_set_error("tf_uv_atlas: the %lld charts do not fit in a %dx%d atlas with padding %d", (long long)C, R, R, pad);
            return 3;
        }
        if (got[2] == 0) {
            *out_scale = hs.s;
            *out_steps = hs.total_steps;
            break;
        }
        cur = 1 - cur;
        C = got[cur];
        ++rounds;
    }
    ua_fallback<<<grid_for(C), 256, 0, s>>>(xy, C, R, pad, hit, root_face[cur], rects, out_texel_tri);
    // output vertices: unique (vertex, chart) corner keys; the half-edge buffers are free now
    cub::DoubleBuffer<uint64_t> ck(static_cast<uint64_t*>(at(L.hek0)), static_cast<uint64_t*>(at(L.hek1)));
    cub::DoubleBuffer<uint32_t> ci(static_cast<uint32_t*>(at(L.hev0)), static_cast<uint32_t*>(at(L.hev1)));
    ua_corner_keys<<<gn, 256, 0, s>>>(triangles, chart[cur], n, ck.Current(), ci.Current());
    launches += 2;
    tb = L.tmp_bytes;
    if ((e = cub::DeviceRadixSort::SortPairs(tmp, tb, ck, ci, (int)n, 0, 32 + key_bits(V), s)) != cudaSuccess) return fail("radix sort");
    ua_heads<<<gn, 256, 0, s>>>(ck.Current(), n, head);
    tb = L.tmp_bytes;
    if ((e = cub::DeviceScan::InclusiveSum(tmp, tb, head, incl, (int)n, s)) != cudaSuccess) return fail("scan");
    ua_out_vertices<<<gn, 256, 0, s>>>(ck.Current(), ci.Current(), head, incl, n, xy, out_triangles, out_vertex_index,
                                       reinterpret_cast<float2*>(out_xy), counters + 3);
    launches += 2;
    if ((e = cudaMemcpyAsync(out_chart, chart[cur], T * sizeof(int32_t), cudaMemcpyDeviceToDevice, s)) != cudaSuccess ||
        (e = cudaMemcpyAsync(out_rects, rects, C * 4 * sizeof(int32_t), cudaMemcpyDeviceToDevice, s)) != cudaSuccess)
        return fail("copy");
    int64_t nv = 0;
    if ((e = cudaMemcpyAsync(&nv, counters + 3, sizeof(int64_t), cudaMemcpyDeviceToHost, s)) != cudaSuccess) return fail("count read");
    if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return fail("output");
    tf_count_launches(launches);
    TF_CHECK_LAUNCH("tf_uv_atlas");
    *out_n_vertices = nv;
    *out_n_charts = C;
    *out_rounds = rounds;
    return 0;
}

extern "C" TF_API int tf_uv_texel_points(const float* vertices, const int32_t* triangles, const float* xy, const int32_t* texel_tri,
                                         int32_t resolution, const int64_t* texels, int64_t n, float* out_points, tf_stream_t stream) {
    TF_REQUIRE(n == 0 || (vertices && triangles && xy && texel_tri && texels && out_points), "tf_uv_texel_points: NULL pointer");
    TF_REQUIRE(resolution >= 16 && resolution <= 16384, "tf_uv_texel_points: resolution %d, need 16 <= R <= 16384", resolution);
    TF_REQUIRE(n >= 0, "tf_uv_texel_points: %lld texels, need >= 0", (long long)n);
    if (n == 0) return 0;
    ua_texel_points<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>(vertices, triangles, xy, texel_tri, resolution, texels, n, out_points);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_uv_texel_points");
    return 0;
}

extern "C" TF_API int tf_uv_fill_sizes(int32_t resolution, int32_t channels, size_t* workspace_bytes) {
    TF_REQUIRE(workspace_bytes, "tf_uv_fill_sizes: NULL pointer");
    TF_REQUIRE(resolution >= 16 && resolution <= 16384, "tf_uv_fill_sizes: resolution %d, need 16 <= R <= 16384", resolution);
    TF_REQUIRE(channels >= 1, "tf_uv_fill_sizes: %d channels, need >= 1", channels);
    const size_t RR = (size_t)resolution * resolution;
    *workspace_bytes = up(RR * channels * sizeof(float)) + 2 * up(RR * sizeof(int32_t));
    return 0;
}

extern "C" TF_API int tf_uv_fill(const float* values, const int64_t* texels, int64_t n, int32_t channels, const int32_t* texel_tri,
                                 const int32_t* chart, const int32_t* rects, int32_t resolution, int32_t padding, void* workspace,
                                 size_t workspace_bytes, float* out_texture, tf_stream_t stream) {
    TF_REQUIRE(texel_tri && chart && rects && workspace && out_texture && (n == 0 || (values && texels)), "tf_uv_fill: NULL pointer");
    size_t need = 0;
    if (tf_uv_fill_sizes(resolution, channels, &need)) return 1;
    TF_REQUIRE(padding >= 0 && padding <= 16, "tf_uv_fill: padding %d, need 0 <= padding <= 16", padding);
    TF_REQUIRE(n >= 0, "tf_uv_fill: %lld texels, need >= 0", (long long)n);
    TF_REQUIRE(workspace_bytes >= need, "tf_uv_fill: workspace of %zu bytes, %zu needed", workspace_bytes, need);
    const int R = resolution, C = channels;
    const size_t RR = (size_t)R * R;
    char* ws = static_cast<char*>(workspace);
    float* tex[2] = {out_texture, reinterpret_cast<float*>(ws)};
    int32_t* ch[2] = {reinterpret_cast<int32_t*>(ws + up(RR * C * sizeof(float))),
                      reinterpret_cast<int32_t*>(ws + up(RR * C * sizeof(float)) + up(RR * sizeof(int32_t)))};
    const cudaStream_t s = (cudaStream_t)stream;
    cudaError_t e;
    if ((e = cudaMemsetAsync(out_texture, 0, RR * C * sizeof(float), s)) != cudaSuccess ||
        (e = cudaMemsetAsync(ch[0], 0xff, RR * sizeof(int32_t), s)) != cudaSuccess) {
        tf_set_error("tf_uv_fill: memset failed: %s", cudaGetErrorString(e));
        return 2;
    }
    int launches = 0;
    if (n > 0) {
        ua_scatter<<<grid_for(n), 256, 0, s>>>(values, texels, n, C, texel_tri, chart, tex[0], ch[0]);
        ++launches;
    }
    int cur = 0;
    for (int p = 0; p < padding; ++p, cur = 1 - cur) {
        ua_dilate<<<grid_for((int64_t)RR), 256, 0, s>>>(tex[cur], ch[cur], R, C, rects, tex[1 - cur], ch[1 - cur]);
        ++launches;
    }
    if (cur == 1 && (e = cudaMemcpyAsync(out_texture, tex[1], RR * C * sizeof(float), cudaMemcpyDeviceToDevice, s)) != cudaSuccess) {
        tf_set_error("tf_uv_fill: copy failed: %s", cudaGetErrorString(e));
        return 2;
    }
    tf_count_launches(launches);
    TF_CHECK_LAUNCH("tf_uv_fill");
    return 0;
}
