// Mesh simplification on the device: Garland-Heckbert quadric-error edge collapse ("Surface Simplification Using Quadric Error
// Metrics", SIGGRAPH 1997), applied in rounds of collapses whose closed 1-rings are vertex-disjoint, so that a round needs no
// locks.  The rules are stated in include/tensoflow_b200.h; oracle/torch_oracle_simplify.py restates them in numpy and the
// result here is bit-equal to it.  All fp64 arithmetic goes through __dadd_rn / __dsub_rn / __dmul_rn / __ddiv_rn /
// __dsqrt_rn in the oracle's operation order: no FMA contraction, and every sum runs in a fixed order.
//
// One round over the current faces (T of them, input order):
//   emit     per face: the (vertex, face) pairs and the half-edges (min << 32 | max, face); faces with a repeated index lock
//            their vertices;
//   sort     two stable CUB radix sorts: the pairs by vertex (each vertex's faces ascending: its star) and the half-edges by key
//            (each edge's half-edges consecutive, in face order);
//   runs     star ranges per vertex, and the ends of every edge with a face count other than 2 locked;
//   quads    (first round only) per vertex the sum of its faces' unit-normal plane quadrics, in face order;
//   check    per edge of face count 2: link condition, apex valence, placement, fold-over, error bound -> fp32 cost key;
//   rank     a stable radix sort of the cost keys: ties by position, which is (a, b) order;
//   claim    the cheapest k valid edges (k from the valid count on the device) take atomicMin of their hashed priority on every
//            vertex of their closed 1-ring; an edge wins iff it holds all of them;
//   apply    winners move a, add Q_b to Q_a, drop their two faces and point the rest of star(b) at a;
//   compact  CUB select of the surviving faces; its count is read back to the host (cudaMemcpyAsync + stream synchronise) to
//            decide whether another round runs.
// The closed 1-ring of a winner holds every vertex its checks read and every face its collapse writes, so the collapses of one
// round commute.  Integer atomics only; the output does not depend on scheduling.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <algorithm>
#include "common.cuh"

namespace {

constexpr int BAND_SHIFT = 4;         // candidates per round: the cheapest sixteenth of the valid edges
constexpr double COND = 1e-6;         // det(A) > COND * trace(A)^3: closed-form placement
constexpr uint32_t NO_KEY = 0xffffffffu;

struct Tri {
    int32_t v[3];
};

struct D3 {
    double x, y, z;
};

__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }

__device__ __forceinline__ D3 load_p(const float* P, int32_t v) {
    return D3{(double)P[3 * (int64_t)v], (double)P[3 * (int64_t)v + 1], (double)P[3 * (int64_t)v + 2]};
}

// (p1 - p0) x (p2 - p0)
__device__ __forceinline__ D3 normal_of(const D3& p0, const D3& p1, const D3& p2) {
    const D3 e1{dsub(p1.x, p0.x), dsub(p1.y, p0.y), dsub(p1.z, p0.z)};
    const D3 e2{dsub(p2.x, p0.x), dsub(p2.y, p0.y), dsub(p2.z, p0.z)};
    return D3{dsub(dmul(e1.y, e2.z), dmul(e1.z, e2.y)), dsub(dmul(e1.z, e2.x), dmul(e1.x, e2.z)),
              dsub(dmul(e1.x, e2.y), dmul(e1.y, e2.x))};
}

// max(0, v^T Q v), Q = xx xy xz xd yy yz yd zz zd dd, rows summed left to right
__device__ __forceinline__ double quad_cost(const double* q, const D3& v) {
    const double r0 = dadd(dadd(dadd(dmul(q[0], v.x), dmul(q[1], v.y)), dmul(q[2], v.z)), q[3]);
    const double r1 = dadd(dadd(dadd(dmul(q[1], v.x), dmul(q[4], v.y)), dmul(q[5], v.z)), q[6]);
    const double r2 = dadd(dadd(dadd(dmul(q[2], v.x), dmul(q[5], v.y)), dmul(q[7], v.z)), q[8]);
    const double r3 = dadd(dadd(dadd(dmul(q[3], v.x), dmul(q[6], v.y)), dmul(q[8], v.z)), q[9]);
    const double c = dadd(dadd(dadd(dmul(v.x, r0), dmul(v.y, r1)), dmul(v.z, r2)), r3);
    return c < 0.0 ? 0.0 : c;
}

__device__ __forceinline__ D3 f32(const D3& v) {
    return D3{(double)__double2float_rn(v.x), (double)__double2float_rn(v.y), (double)__double2float_rn(v.z)};
}

// the position minimising v^T Q v, rounded to fp32, and its cost
__device__ __forceinline__ D3 placement(const double* q, const D3& pa, const D3& pb, double& cost) {
    const double xx = q[0], xy = q[1], xz = q[2], xd = q[3], yy = q[4], yz = q[5], yd = q[6], zz = q[7], zd = q[8];
    const double i00 = dsub(dmul(yy, zz), dmul(yz, yz));
    const double i01 = dsub(dmul(xz, yz), dmul(xy, zz));
    const double i02 = dsub(dmul(xy, yz), dmul(xz, yy));
    const double i11 = dsub(dmul(xx, zz), dmul(xz, xz));
    const double i12 = dsub(dmul(xy, xz), dmul(xx, yz));
    const double i22 = dsub(dmul(xx, yy), dmul(xy, xy));
    const double det = dadd(dadd(dmul(xx, i00), dmul(xy, i01)), dmul(xz, i02));
    const double tr = dadd(dadd(xx, yy), zz);
    D3 v;
    if (det > dmul(dmul(dmul(COND, tr), tr), tr)) {
        v = f32(D3{-__ddiv_rn(dadd(dadd(dmul(i00, xd), dmul(i01, yd)), dmul(i02, zd)), det),
                   -__ddiv_rn(dadd(dadd(dmul(i01, xd), dmul(i11, yd)), dmul(i12, zd)), det),
                   -__ddiv_rn(dadd(dadd(dmul(i02, xd), dmul(i12, yd)), dmul(i22, zd)), det)});
    } else {
        v = pa;
        double best = quad_cost(q, pa);
        const double cb = quad_cost(q, pb);
        if (cb < best) { v = pb; best = cb; }
        const D3 mid = f32(D3{dmul(dadd(pa.x, pb.x), 0.5), dmul(dadd(pa.y, pb.y), 0.5), dmul(dadd(pa.z, pb.z), 0.5)});
        if (quad_cost(q, mid) < best) v = mid;
    }
    cost = quad_cost(q, v);
    return v;
}

// splitmix64 finaliser
__device__ __forceinline__ uint64_t edge_hash(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

__device__ __forceinline__ bool is_run_of_two(const uint64_t* hk, int64_t i, int64_t n) {
    return (i == 0 || hk[i - 1] != hk[i]) && i + 1 < n && hk[i + 1] == hk[i] && !(i + 2 < n && hk[i + 2] == hk[i]);
}

__device__ __forceinline__ int64_t gtid() { return blockIdx.x * (int64_t)blockDim.x + threadIdx.x; }
__device__ __forceinline__ int64_t gstride() { return (int64_t)gridDim.x * blockDim.x; }

__global__ void __launch_bounds__(256) ms_emit(const Tri* __restrict__ F, int64_t T, uint32_t* __restrict__ vf_k,
                                               uint32_t* __restrict__ vf_v, uint64_t* __restrict__ he_k, uint32_t* __restrict__ he_v,
                                               uint8_t* __restrict__ keep, uint8_t* __restrict__ lock) {
    for (int64_t f = gtid(); f < T; f += gstride()) {
        const Tri t = F[f];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const uint32_t a = (uint32_t)t.v[k], b = (uint32_t)t.v[k == 2 ? 0 : k + 1];
            vf_k[3 * f + k] = a;
            vf_v[3 * f + k] = (uint32_t)f;
            he_k[3 * f + k] = ((uint64_t)min(a, b) << 32) | max(a, b);
            he_v[3 * f + k] = (uint32_t)f;
        }
        keep[f] = 1;
        if (t.v[0] == t.v[1] || t.v[1] == t.v[2] || t.v[0] == t.v[2]) lock[t.v[0]] = lock[t.v[1]] = lock[t.v[2]] = 1;
    }
}


// star ranges [vstart, vend) of the sorted (vertex, face) pairs; both ends of every edge whose face count is not 2 are locked
__global__ void __launch_bounds__(256) ms_runs(const uint32_t* __restrict__ vf_k, const uint64_t* __restrict__ he_k, int64_t n,
                                               int64_t* __restrict__ vstart, int64_t* __restrict__ vend, uint8_t* __restrict__ lock) {
    for (int64_t i = gtid(); i < n; i += gstride()) {
        const uint32_t v = vf_k[i];
        if (i == 0 || vf_k[i - 1] != v) vstart[v] = i;
        if (i == n - 1 || vf_k[i + 1] != v) vend[v] = i + 1;
        const uint64_t k = he_k[i];
        if ((i == 0 || he_k[i - 1] != k) && !is_run_of_two(he_k, i, n)) {
            lock[k >> 32] = 1;
            lock[k & 0xffffffffu] = 1;
        }
    }
}

// Q[v] = sum of the unit-normal plane quadrics of v's faces, in face order from 0 (a zero-length cross product adds nothing)
__global__ void __launch_bounds__(256) ms_quadrics(const float* __restrict__ P, const Tri* __restrict__ F,
                                                   const uint32_t* __restrict__ star, const int64_t* __restrict__ vstart,
                                                   const int64_t* __restrict__ vend, int64_t V, double* __restrict__ Q) {
    for (int64_t v = gtid(); v < V; v += gstride()) {
        double q[10];
#pragma unroll
        for (int k = 0; k < 10; ++k) q[k] = 0.0;
        for (int64_t j = vstart[v]; j < vend[v]; ++j) {
            const Tri t = F[star[j]];
            const D3 p0 = load_p(P, t.v[0]);
            const D3 n = normal_of(p0, load_p(P, t.v[1]), load_p(P, t.v[2]));
            const double ln = __dsqrt_rn(dadd(dadd(dmul(n.x, n.x), dmul(n.y, n.y)), dmul(n.z, n.z)));
            if (!(ln > 0.0)) continue;
            const double x = __ddiv_rn(n.x, ln), y = __ddiv_rn(n.y, ln), z = __ddiv_rn(n.z, ln);
            const double d = -dadd(dadd(dmul(x, p0.x), dmul(y, p0.y)), dmul(z, p0.z));
            const double e[10] = {dmul(x, x), dmul(x, y), dmul(x, z), dmul(x, d), dmul(y, y),
                                  dmul(y, z), dmul(y, d), dmul(z, z), dmul(z, d), dmul(d, d)};
#pragma unroll
            for (int k = 0; k < 10; ++k) q[k] = dadd(q[k], e[k]);
        }
#pragma unroll
        for (int k = 0; k < 10; ++k) Q[10 * v + k] = q[k];
    }
}

__device__ __forceinline__ bool face_has(const Tri& t, int32_t w) { return t.v[0] == w || t.v[1] == w || t.v[2] == w; }

// every face of star(s) other than f0, f1 keeps a normal within 90 degrees of its old one (a face whose old normal is zero is
// not constrained) when a and b move to v
__device__ __forceinline__ bool no_foldover(const float* P, const Tri* F, const uint32_t* star, int64_t s0, int64_t s1, uint32_t f0, uint32_t f1,
                            int32_t a, int32_t b, const D3& v) {
    for (int64_t j = s0; j < s1; ++j) {
        const uint32_t g = star[j];
        if (g == f0 || g == f1) continue;
        const Tri t = F[g];
        D3 p[3], q[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            p[k] = load_p(P, t.v[k]);
            q[k] = (t.v[k] == a || t.v[k] == b) ? v : p[k];
        }
        const D3 n0 = normal_of(p[0], p[1], p[2]);
        if (n0.x == 0.0 && n0.y == 0.0 && n0.z == 0.0) continue;
        const D3 n1 = normal_of(q[0], q[1], q[2]);
        if (!(dadd(dadd(dmul(n0.x, n1.x), dmul(n0.y, n1.y)), dmul(n0.z, n1.z)) > 0.0)) return false;
    }
    return true;
}

// Per sorted half-edge position i: the edge starting there, if it has exactly two faces, is checked; the cost key of a valid
// edge is its fp32 cost bits (costs are >= 0, so the unsigned order is the float order), NO_KEY otherwise.
__global__ void __launch_bounds__(256, 2) ms_check(const float* __restrict__ P, const double* __restrict__ Q, const Tri* __restrict__ F,
                                                const uint32_t* __restrict__ star, const int64_t* __restrict__ vstart,
                                                const int64_t* __restrict__ vend, const uint8_t* __restrict__ lock,
                                                const uint64_t* __restrict__ he_k, const uint32_t* __restrict__ he_f, int64_t n,
                                                double max_error, uint32_t* __restrict__ cost_key, uint32_t* __restrict__ cost_pos,
                                                float* __restrict__ place, unsigned long long* __restrict__ n_valid) {
    for (int64_t i = gtid(); i < n; i += gstride()) {
        cost_pos[i] = (uint32_t)i;
        cost_key[i] = NO_KEY;
        if (!is_run_of_two(he_k, i, n)) continue;
        const int32_t a = (int32_t)(he_k[i] >> 32), b = (int32_t)(he_k[i] & 0xffffffffu);
        if (lock[a] || lock[b]) continue;
        const uint32_t f0 = he_f[i], f1 = he_f[i + 1];
        const Tri t0 = F[f0], t1 = F[f1];
        const int32_t c0 = (int32_t)((int64_t)t0.v[0] + t0.v[1] + t0.v[2] - a - b);
        const int32_t c1 = (int32_t)((int64_t)t1.v[0] + t1.v[1] + t1.v[2] - a - b);
        if (c0 == c1 || vend[c0] - vstart[c0] <= 3 || vend[c1] - vstart[c1] <= 3) continue;
        // link condition: no vertex of star(a) other than a, b, c0, c1 is a vertex of star(b)
        const int64_t sa0 = vstart[a], sa1 = vend[a], sb0 = vstart[b], sb1 = vend[b];
        bool ok = true;
        for (int64_t j = sa0; j < sa1 && ok; ++j) {
            const Tri g = F[star[j]];
            for (int k = 0; k < 3 && ok; ++k) {
                const int32_t w = g.v[k];
                if (w == a || w == b || w == c0 || w == c1) continue;
                for (int64_t m = sb0; m < sb1; ++m)
                    if (face_has(F[star[m]], w)) { ok = false; break; }
            }
        }
        if (!ok) continue;
        double q[10];
#pragma unroll
        for (int k = 0; k < 10; ++k) q[k] = dadd(Q[10 * (int64_t)a + k], Q[10 * (int64_t)b + k]);
        double cost;
        const D3 v = placement(q, load_p(P, a), load_p(P, b), cost);
        if (!(__dsqrt_rn(cost) <= max_error)) continue;
        if (!no_foldover(P, F, star, sa0, sa1, f0, f1, a, b, v) || !no_foldover(P, F, star, sb0, sb1, f0, f1, a, b, v)) continue;
        cost_key[i] = __float_as_uint(__double2float_rn(cost));
        place[3 * i] = (float)v.x;
        place[3 * i + 1] = (float)v.y;
        place[3 * i + 2] = (float)v.z;
        atomicAdd(n_valid, 1ull);
    }
}

// k = min(max(1, n_valid >> BAND_SHIFT), need), 0 without a valid edge
__device__ __forceinline__ int64_t band(const unsigned long long* n_valid, int64_t need) {
    const int64_t nv = (int64_t)*n_valid;
    return nv == 0 ? 0 : min(max((int64_t)1, nv >> BAND_SHIFT), need);
}

__device__ __forceinline__ uint64_t priority(uint64_t key, int64_t rank) { return (edge_hash(key) >> 32 << 32) | (uint64_t)rank; }

// candidate `rank` (position e in the half-edge order) and the vertices of its closed 1-ring: `visit(w)` for every vertex of
// star(a) and star(b); stops early when visit returns false
template <typename Visit>
__device__ __forceinline__ bool for_ring(const Tri* F, const uint32_t* star, const int64_t* vstart, const int64_t* vend,
                                         int32_t a, int32_t b, Visit visit) {
    for (int s = 0; s < 2; ++s) {
        const int32_t x = s == 0 ? a : b;
        for (int64_t j = vstart[x]; j < vend[x]; ++j) {
            const Tri g = F[star[j]];
            if (!visit(g.v[0]) || !visit(g.v[1]) || !visit(g.v[2])) return false;
        }
    }
    return true;
}

__global__ void __launch_bounds__(256) ms_claim(const Tri* __restrict__ F, const uint32_t* __restrict__ star,
                                                const int64_t* __restrict__ vstart, const int64_t* __restrict__ vend,
                                                const uint64_t* __restrict__ he_k, const uint32_t* __restrict__ ranked,
                                                const unsigned long long* __restrict__ n_valid, int64_t need,
                                                unsigned long long* __restrict__ claim) {
    const int64_t k = band(n_valid, need);
    for (int64_t i = gtid(); i < k; i += gstride()) {
        const uint64_t key = he_k[ranked[i]];
        const unsigned long long p = priority(key, i);
        for_ring(F, star, vstart, vend, (int32_t)(key >> 32), (int32_t)(key & 0xffffffffu), [&](int32_t w) {
            atomicMin(claim + w, p);
            return true;
        });
    }
}

__global__ void __launch_bounds__(256) ms_win(const Tri* __restrict__ F, const uint32_t* __restrict__ star,
                                              const int64_t* __restrict__ vstart, const int64_t* __restrict__ vend,
                                              const uint64_t* __restrict__ he_k, const uint32_t* __restrict__ ranked,
                                              const unsigned long long* __restrict__ n_valid, int64_t need,
                                              const unsigned long long* __restrict__ claim, uint8_t* __restrict__ win) {
    const int64_t k = band(n_valid, need);
    for (int64_t i = gtid(); i < k; i += gstride()) {
        const uint64_t key = he_k[ranked[i]];
        const unsigned long long p = priority(key, i);
        win[i] = for_ring(F, star, vstart, vend, (int32_t)(key >> 32), (int32_t)(key & 0xffffffffu),
                          [&](int32_t w) { return claim[w] == p; });
    }
}

__global__ void __launch_bounds__(256) ms_apply(Tri* __restrict__ F, const uint32_t* __restrict__ star,
                                                const int64_t* __restrict__ vstart, const int64_t* __restrict__ vend,
                                                const uint64_t* __restrict__ he_k, const uint32_t* __restrict__ he_f,
                                                const uint32_t* __restrict__ ranked, const unsigned long long* __restrict__ n_valid,
                                                int64_t need, const uint8_t* __restrict__ win, const float* __restrict__ place,
                                                float* __restrict__ P, double* __restrict__ Q, uint8_t* __restrict__ keep) {
    const int64_t k = band(n_valid, need);
    for (int64_t i = gtid(); i < k; i += gstride()) {
        if (!win[i]) continue;
        const int64_t e = ranked[i];
        const uint64_t key = he_k[e];
        const int32_t a = (int32_t)(key >> 32), b = (int32_t)(key & 0xffffffffu);
        const uint32_t f0 = he_f[e], f1 = he_f[e + 1];
#pragma unroll
        for (int c = 0; c < 3; ++c) P[3 * (int64_t)a + c] = place[3 * e + c];
#pragma unroll
        for (int c = 0; c < 10; ++c) Q[10 * (int64_t)a + c] = dadd(Q[10 * (int64_t)a + c], Q[10 * (int64_t)b + c]);
        keep[f0] = 0;
        keep[f1] = 0;
        for (int64_t j = vstart[b]; j < vend[b]; ++j) {
            const uint32_t g = star[j];
            if (g == f0 || g == f1) continue;
#pragma unroll
            for (int c = 0; c < 3; ++c)
                if (F[g].v[c] == b) F[g].v[c] = a;
        }
    }
}

__global__ void __launch_bounds__(256) ms_mark_used(const Tri* __restrict__ F, int64_t T, int32_t* __restrict__ used) {
    for (int64_t f = gtid(); f < T; f += gstride()) {
        const Tri t = F[f];
        used[t.v[0]] = 1;
        used[t.v[1]] = 1;
        used[t.v[2]] = 1;
    }
}

__global__ void __launch_bounds__(256) ms_output(const float* __restrict__ P, const Tri* __restrict__ F, int64_t V, int64_t T,
                                                 const int32_t* __restrict__ used, const int32_t* __restrict__ new_index,
                                                 float* __restrict__ out_v, Tri* __restrict__ out_t) {
    for (int64_t v = gtid(); v < V; v += gstride())
        if (used[v]) {
            const int64_t o = new_index[v];
            out_v[3 * o] = P[3 * v];
            out_v[3 * o + 1] = P[3 * v + 1];
            out_v[3 * o + 2] = P[3 * v + 2];
        }
    for (int64_t f = gtid(); f < T; f += gstride()) {
        const Tri t = F[f];
        out_t[f] = Tri{{new_index[t.v[0]], new_index[t.v[1]], new_index[t.v[2]]}};
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
    size_t P, Q, lock, vstart, vend, claim, F0, F1, keep, vf_k0, vf_k1, vf_v0, vf_v1, he_k0, he_k1, he_v0, he_v1, ck0, ck1, cp0, cp1,
        place, win, counters, tmp, tmp_bytes, total;
};

// scratch layout for V vertices and T triangles; the CUB temporary storage is sized on the current device
int make_layout(int64_t V, int64_t T, Layout& L, const char* who) {
    const int64_t n = 3 * T;
    size_t b0 = 0, b1 = 0, b2 = 0, b3 = 0, b4 = 0;
    cudaError_t e;
    {
        cub::DoubleBuffer<uint32_t> k(nullptr, nullptr), v(nullptr, nullptr);
        e = cub::DeviceRadixSort::SortPairs(nullptr, b0, k, v, (int)n, 0, key_bits(V));
        TF_REQUIRE(e == cudaSuccess, "%s: radix sort sizing failed: %s", who, cudaGetErrorString(e));
        e = cub::DeviceRadixSort::SortPairs(nullptr, b1, k, v, (int)n, 0, 32);
        TF_REQUIRE(e == cudaSuccess, "%s: radix sort sizing failed: %s", who, cudaGetErrorString(e));
    }
    {
        cub::DoubleBuffer<uint64_t> k(nullptr, nullptr);
        cub::DoubleBuffer<uint32_t> v(nullptr, nullptr);
        e = cub::DeviceRadixSort::SortPairs(nullptr, b2, k, v, (int)n, 0, 32 + key_bits(V));
        TF_REQUIRE(e == cudaSuccess, "%s: radix sort sizing failed: %s", who, cudaGetErrorString(e));
    }
    e = cub::DeviceSelect::Flagged(nullptr, b3, (const Tri*)nullptr, (const uint8_t*)nullptr, (Tri*)nullptr, (int64_t*)nullptr, T);
    TF_REQUIRE(e == cudaSuccess, "%s: select sizing failed: %s", who, cudaGetErrorString(e));
    e = cub::DeviceScan::ExclusiveSum(nullptr, b4, (const int32_t*)nullptr, (int32_t*)nullptr, V);
    TF_REQUIRE(e == cudaSuccess, "%s: scan sizing failed: %s", who, cudaGetErrorString(e));
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += up(bytes); return o; };
    L.P = take(V * 3 * sizeof(float));
    L.Q = take(V * 10 * sizeof(double));
    L.lock = take(V);
    L.vstart = take(V * sizeof(int64_t));
    L.vend = take(V * sizeof(int64_t));
    L.claim = take(V * sizeof(uint64_t));
    L.F0 = take(T * sizeof(Tri));
    L.F1 = take(T * sizeof(Tri));
    L.keep = take(T);
    L.vf_k0 = take(n * sizeof(uint32_t));
    L.vf_k1 = take(n * sizeof(uint32_t));
    L.vf_v0 = take(n * sizeof(uint32_t));
    L.vf_v1 = take(n * sizeof(uint32_t));
    L.he_k0 = take(n * sizeof(uint64_t));
    L.he_k1 = take(n * sizeof(uint64_t));
    L.he_v0 = take(n * sizeof(uint32_t));
    L.he_v1 = take(n * sizeof(uint32_t));
    L.ck0 = take(n * sizeof(uint32_t));
    L.ck1 = take(n * sizeof(uint32_t));
    L.cp0 = take(n * sizeof(uint32_t));
    L.cp1 = take(n * sizeof(uint32_t));
    L.place = take(n * 3 * sizeof(float));
    L.win = take(n);
    L.counters = take(4 * sizeof(int64_t));
    L.tmp_bytes = std::max({b0, b1, b2, b3, b4});
    L.tmp = take(L.tmp_bytes);
    L.total = off;
    return 0;
}

int check_sizes(int64_t V, int64_t T, const char* who) {
    TF_REQUIRE(V > 0 && V < (int64_t(1) << 31), "%s: %lld vertices, need 0 < V < 2^31", who, (long long)V);
    TF_REQUIRE(T > 0 && T < (int64_t(1) << 31), "%s: %lld triangles, need 0 < T < 2^31", who, (long long)T);
    // the radix sorts run over 3 T half-edges with int item counts (about 310 B of workspace per triangle keeps T far below)
    TF_REQUIRE(3 * T < (int64_t(1) << 31), "%s: %lld triangles, the sorts need 3 T < 2^31", who, (long long)T);
    return 0;
}

}  // namespace

extern "C" TF_API int tf_mesh_simplify_sizes(int64_t n_vertices, int64_t n_triangles, size_t* workspace_bytes) {
    TF_REQUIRE(workspace_bytes, "tf_mesh_simplify_sizes: NULL pointer");
    if (check_sizes(n_vertices, n_triangles, "tf_mesh_simplify_sizes")) return 1;
    Layout L;
    if (make_layout(n_vertices, n_triangles, L, "tf_mesh_simplify_sizes")) return 1;
    *workspace_bytes = L.total;
    return 0;
}

extern "C" TF_API int tf_mesh_simplify(const float* vertices, int64_t n_vertices, const int32_t* triangles, int64_t n_triangles,
                                       int64_t target, double max_error, void* workspace, size_t workspace_bytes, float* out_vertices,
                                       int32_t* out_triangles, int64_t* out_n_vertices, int64_t* out_n_triangles, int32_t* out_rounds,
                                       tf_stream_t stream) {
    TF_REQUIRE(vertices && triangles && workspace && out_vertices && out_triangles && out_n_vertices && out_n_triangles && out_rounds,
               "tf_mesh_simplify: NULL pointer");
    if (check_sizes(n_vertices, n_triangles, "tf_mesh_simplify")) return 1;
    TF_REQUIRE(target >= 0, "tf_mesh_simplify: target %lld triangles, need >= 0", (long long)target);
    TF_REQUIRE(max_error >= 0.0, "tf_mesh_simplify: max_error %g, need >= 0 (+inf for no bound)", max_error);
    const int64_t V = n_vertices;
    Layout L;
    if (make_layout(V, n_triangles, L, "tf_mesh_simplify")) return 1;
    TF_REQUIRE(workspace_bytes >= L.total, "tf_mesh_simplify: workspace of %zu bytes, %zu needed", workspace_bytes, L.total);
    char* ws = static_cast<char*>(workspace);
    auto at = [&](size_t o) { return static_cast<void*>(ws + o); };
    float* P = static_cast<float*>(at(L.P));
    double* Q = static_cast<double*>(at(L.Q));
    uint8_t* lock = static_cast<uint8_t*>(at(L.lock));
    int64_t* vstart = static_cast<int64_t*>(at(L.vstart));
    int64_t* vend = static_cast<int64_t*>(at(L.vend));
    unsigned long long* claim = static_cast<unsigned long long*>(at(L.claim));
    Tri* F = static_cast<Tri*>(at(L.F0));
    Tri* F_alt = static_cast<Tri*>(at(L.F1));
    uint8_t* keep = static_cast<uint8_t*>(at(L.keep));
    uint8_t* win = static_cast<uint8_t*>(at(L.win));
    float* place = static_cast<float*>(at(L.place));
    int64_t* counters = static_cast<int64_t*>(at(L.counters));
    unsigned long long* n_valid = reinterpret_cast<unsigned long long*>(counters);
    int64_t* n_kept = counters + 1;
    void* tmp = at(L.tmp);
    const cudaStream_t s = (cudaStream_t)stream;
    int launches = 0;
    cudaError_t e = cudaSuccess;
    auto fail = [&](const char* what) {
        tf_count_launches(launches);
        tf_set_error("tf_mesh_simplify: %s failed: %s", what, cudaGetErrorString(e));
        return 2;
    };

    if ((e = cudaMemcpyAsync(P, vertices, V * 3 * sizeof(float), cudaMemcpyDeviceToDevice, s)) != cudaSuccess) return fail("copy");
    if ((e = cudaMemcpyAsync(F, triangles, n_triangles * sizeof(Tri), cudaMemcpyDeviceToDevice, s)) != cudaSuccess) return fail("copy");
    int64_t T = n_triangles;
    int32_t rounds = 0;
    bool first = true;
    while (T > target + 1) {
        const int64_t n = 3 * T;
        const unsigned gv = grid_for(V), gt = grid_for(T), gn = grid_for(n);
        if ((e = cudaMemsetAsync(lock, 0, V, s)) != cudaSuccess || (e = cudaMemsetAsync(vstart, 0, V * sizeof(int64_t), s)) != cudaSuccess ||
            (e = cudaMemsetAsync(vend, 0, V * sizeof(int64_t), s)) != cudaSuccess ||
            (e = cudaMemsetAsync(claim, 0xff, V * sizeof(uint64_t), s)) != cudaSuccess ||
            (e = cudaMemsetAsync(counters, 0, 4 * sizeof(int64_t), s)) != cudaSuccess)
            return fail("memset");
        ms_emit<<<gt, 256, 0, s>>>(F, T, static_cast<uint32_t*>(at(L.vf_k0)), static_cast<uint32_t*>(at(L.vf_v0)),
                                   static_cast<uint64_t*>(at(L.he_k0)), static_cast<uint32_t*>(at(L.he_v0)), keep, lock);
        ++launches;
        cub::DoubleBuffer<uint32_t> vfk(static_cast<uint32_t*>(at(L.vf_k0)), static_cast<uint32_t*>(at(L.vf_k1)));
        cub::DoubleBuffer<uint32_t> vfv(static_cast<uint32_t*>(at(L.vf_v0)), static_cast<uint32_t*>(at(L.vf_v1)));
        cub::DoubleBuffer<uint64_t> hek(static_cast<uint64_t*>(at(L.he_k0)), static_cast<uint64_t*>(at(L.he_k1)));
        cub::DoubleBuffer<uint32_t> hev(static_cast<uint32_t*>(at(L.he_v0)), static_cast<uint32_t*>(at(L.he_v1)));
        cub::DoubleBuffer<uint32_t> ck(static_cast<uint32_t*>(at(L.ck0)), static_cast<uint32_t*>(at(L.ck1)));
        cub::DoubleBuffer<uint32_t> cp(static_cast<uint32_t*>(at(L.cp0)), static_cast<uint32_t*>(at(L.cp1)));
        size_t tb = L.tmp_bytes;
        if ((e = cub::DeviceRadixSort::SortPairs(tmp, tb, vfk, vfv, (int)n, 0, key_bits(V), s)) != cudaSuccess) return fail("radix sort");
        tb = L.tmp_bytes;
        if ((e = cub::DeviceRadixSort::SortPairs(tmp, tb, hek, hev, (int)n, 0, 32 + key_bits(V), s)) != cudaSuccess) return fail("radix sort");
        const uint32_t* star = vfv.Current();
        const uint64_t* he_k = hek.Current();
        const uint32_t* he_f = hev.Current();
        ms_runs<<<gn, 256, 0, s>>>(vfk.Current(), he_k, n, vstart, vend, lock);
        ++launches;
        if (first) {
            ms_quadrics<<<gv, 256, 0, s>>>(P, F, star, vstart, vend, V, Q);
            ++launches;
            first = false;
        }
        ms_check<<<gn, 256, 0, s>>>(P, Q, F, star, vstart, vend, lock, he_k, he_f, n, max_error, ck.Current(), cp.Current(), place,
                                    n_valid);
        ++launches;
        tb = L.tmp_bytes;
        if ((e = cub::DeviceRadixSort::SortPairs(tmp, tb, ck, cp, (int)n, 0, 32, s)) != cudaSuccess) return fail("radix sort");
        const uint32_t* ranked = cp.Current();
        const int64_t need = (T - target) / 2;
        const unsigned gk = grid_for(std::min(n, need));
        ms_claim<<<gk, 256, 0, s>>>(F, star, vstart, vend, he_k, ranked, n_valid, need, claim);
        ms_win<<<gk, 256, 0, s>>>(F, star, vstart, vend, he_k, ranked, n_valid, need, claim, win);
        ms_apply<<<gk, 256, 0, s>>>(F, star, vstart, vend, he_k, he_f, ranked, n_valid, need, win, place, P, Q, keep);
        launches += 3;
        tb = L.tmp_bytes;
        if ((e = cub::DeviceSelect::Flagged(tmp, tb, F, keep, F_alt, n_kept, T, s)) != cudaSuccess) return fail("select");
        // the one host read of the round: whether it collapsed anything, and how many faces are left
        int64_t kept = 0;
        if ((e = cudaMemcpyAsync(&kept, n_kept, sizeof(int64_t), cudaMemcpyDeviceToHost, s)) != cudaSuccess) return fail("count read");
        if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return fail("round");
        if (kept == T) break;
        std::swap(F, F_alt);
        T = kept;
        ++rounds;
    }
    // output: surviving faces in order, referenced vertices in order, renumbered
    int32_t* used = reinterpret_cast<int32_t*>(vstart);
    int32_t* new_index = reinterpret_cast<int32_t*>(vend);
    if ((e = cudaMemsetAsync(used, 0, V * sizeof(int32_t), s)) != cudaSuccess) return fail("memset");
    ms_mark_used<<<grid_for(T), 256, 0, s>>>(F, T, used);
    size_t tb = L.tmp_bytes;
    if ((e = cub::DeviceScan::ExclusiveSum(tmp, tb, used, new_index, V, s)) != cudaSuccess) return fail("scan");
    ms_output<<<grid_for(std::max(V, T)), 256, 0, s>>>(P, F, V, T, used, new_index, out_vertices, reinterpret_cast<Tri*>(out_triangles));
    launches += 2;
    int32_t tail[2] = {0, 0};
    if ((e = cudaMemcpyAsync(&tail[0], used + V - 1, sizeof(int32_t), cudaMemcpyDeviceToHost, s)) != cudaSuccess ||
        (e = cudaMemcpyAsync(&tail[1], new_index + V - 1, sizeof(int32_t), cudaMemcpyDeviceToHost, s)) != cudaSuccess)
        return fail("count read");
    if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return fail("output");
    tf_count_launches(launches);
    TF_CHECK_LAUNCH("tf_mesh_simplify");
    *out_n_vertices = (int64_t)tail[0] + tail[1];
    *out_n_triangles = T;
    *out_rounds = rounds;
    return 0;
}
