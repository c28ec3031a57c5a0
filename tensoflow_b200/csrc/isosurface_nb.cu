// Narrow-band marching cubes: the mesh of tf_iso_* (isosurface.cu) for lattices of up to 4096 points per axis, with the
// field evaluated only in bricks of 8^3 cells around the surface.  Conventions and the band rule: include/tensoflow_b200.h
// ("narrow-band isosurface extraction"); oracle/torch_oracle_iso_nb.py restates them on the CPU.
//
// Brick (I, J, K), id (I*by + J)*bz + K, covers the points i0 .. i0 + ex (i0 = 8I, ex = min(8, nx-1-i0)) per axis and owns
// the cells i0 .. i0 + ex - 1 and the points i0 .. i0 + ex - 1 (the last brick on an axis also owns its end point).  The
// values of an active brick are a [9][9][9] block (z fastest) at its slot; positions past ex are clamped copies, never read.
// A segment is one (i, j) row of a brick, key (i*ny + j)*bz + K: in key order, then k, then axis (vertices) or case-table
// order (triangles), the items come out in the dense order, so the host sorts the segment keys and takes prefix sums of the
// per-segment counts, and the write passes place each item.  No atomics anywhere: the output is bit-reproducible.
//   tf_iso_nb_classify   thread per brick: active iff the corners straddle the threshold or one is within the band
//   tf_iso_nb_points     thread per brick point: lattice xyz from the axis tables
//   tf_iso_nb_grow       block per brick: flag inactive bricks that share a crossed lattice edge with it
//   tf_iso_nb_count      thread per segment: owned crossed edges, triangles of the row's cells, the segment key
//   tf_iso_nb_vertices   thread per segment: vertices, and idx = global id of each owned point's first vertex
//   tf_iso_nb_triangles  thread per segment: edge -> vertex id through the owner brick's slot and idx
#include "common.cuh"
#include "isosurface_table.cuh"

namespace {

constexpr int kB = 8;                 // cells per brick edge
constexpr int kP = kB + 1;            // points per brick edge
constexpr int kBP = kP * kP * kP;     // points per brick block
constexpr int kSeg = kP * kP;         // segments (rows) per brick
constexpr int kMaxAxis = 4096;

struct Lattice {
    int n[3];                          // points per axis
    int b[3];                          // bricks per axis
};

__host__ __device__ inline Lattice make_lattice(int nx, int ny, int nz) {
    Lattice L;
    L.n[0] = nx; L.n[1] = ny; L.n[2] = nz;
    for (int a = 0; a < 3; ++a) L.b[a] = (L.n[a] - 1 + kB - 1) / kB;
    return L;
}

struct Brick {
    int c[3];                          // brick coordinates
    int o[3];                          // first lattice point
    int e[3];                          // cells per axis (1..8)
    int own[3];                        // owned points per axis (e, or e + 1 for the last brick)
};

__device__ __forceinline__ Brick make_brick(const Lattice& L, int64_t id) {
    Brick B;
    B.c[2] = (int)(id % L.b[2]);
    B.c[1] = (int)(id / L.b[2] % L.b[1]);
    B.c[0] = (int)(id / ((int64_t)L.b[2] * L.b[1]));
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        B.o[a] = B.c[a] * kB;
        B.e[a] = min(kB, L.n[a] - 1 - B.o[a]);
        B.own[a] = B.e[a] + (B.c[a] == L.b[a] - 1);
    }
    return B;
}

__device__ __forceinline__ int lp(int x, int y, int z) { return (x * kP + y) * kP + z; }

// crossed edges of block point (x, y, z) inside the brick's closure: bit a = edge along axis a
__device__ __forceinline__ int nb_edge_bits(const float* v, const Brick& B, int x, int y, int z, float thr) {
    const bool in0 = v[lp(x, y, z)] < thr;
    int bits = 0;
    if (x < B.e[0] && (v[lp(x + 1, y, z)] < thr) != in0) bits |= 1;
    if (y < B.e[1] && (v[lp(x, y + 1, z)] < thr) != in0) bits |= 2;
    if (z < B.e[2] && (v[lp(x, y, z + 1)] < thr) != in0) bits |= 4;
    return bits;
}

__device__ __forceinline__ int nb_case(const float* v, int x, int y, int z, float thr) {
    int cs = 0;
#pragma unroll
    for (int c = 0; c < 8; ++c) cs |= (int)(v[lp(x + (c & 1), y + (c >> 1 & 1), z + (c >> 2 & 1))] < thr) << c;
    return cs;
}

__global__ void __launch_bounds__(256) nb_classify_kernel(const float* __restrict__ coarse, Lattice L, float thr, float band,
                                                          uint8_t* __restrict__ flags) {
    const int64_t id = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= (int64_t)L.b[0] * L.b[1] * L.b[2]) return;
    const int K = (int)(id % L.b[2]), J = (int)(id / L.b[2] % L.b[1]), I = (int)(id / ((int64_t)L.b[2] * L.b[1]));
    const int cy = L.b[1] + 1, cz = L.b[2] + 1;
    int n_in = 0;
    bool near = false;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        const float u = coarse[((int64_t)(I + (c & 1)) * cy + J + (c >> 1 & 1)) * cz + K + (c >> 2 & 1)];
        n_in += u < thr;
        near |= fabsf(__fsub_rn(u, thr)) < band;
    }
    flags[id] = (n_in > 0 && n_in < 8) || near;
}

__global__ void __launch_bounds__(256) nb_points_kernel(const float* __restrict__ ax, const float* __restrict__ ay,
                                                        const float* __restrict__ az, Lattice L, const int64_t* __restrict__ bricks,
                                                        int64_t n_bricks, float* __restrict__ xyz) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_bricks * kBP) return;
    const Brick B = make_brick(L, bricks[t / kBP]);
    const int p = (int)(t % kBP);
    const int x = min(p / (kP * kP), B.e[0]), y = min(p / kP % kP, B.e[1]), z = min(p % kP, B.e[2]);
    float* o = xyz + t * 3;
    o[0] = ax[B.o[0] + x];
    o[1] = ay[B.o[1] + y];
    o[2] = az[B.o[2] + z];
}

// A crossed lattice edge of the brick's closure that lies on its boundary is also in the closure of the bricks across that
// boundary (a face neighbour, or across a brick edge line, the two face neighbours and the diagonal one): the cells of those
// bricks around the edge carry triangles that use its vertex, so they join the band.  Flags: 0 inactive, 1 active, 2 newly
// flagged; every writer stores the same 2, so the result does not depend on the order of the stores.
__global__ void __launch_bounds__(256) nb_grow_kernel(const float* __restrict__ vals, const int64_t* __restrict__ bricks, Lattice L,
                                                      float thr, uint8_t* __restrict__ flags) {
    const int64_t id = bricks[blockIdx.x];
    const Brick B = make_brick(L, id);
    const float* v = vals + (int64_t)blockIdx.x * kBP;
    const int64_t stride[3] = {(int64_t)L.b[1] * L.b[2], L.b[2], 1};
    for (int p = threadIdx.x; p < kBP; p += blockDim.x) {
        const int l[3] = {p / (kP * kP), p / kP % kP, p % kP};
        if (l[0] > B.e[0] || l[1] > B.e[1] || l[2] > B.e[2]) continue;
        const int bits = nb_edge_bits(v, B, l[0], l[1], l[2], thr);
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            if (!(bits >> a & 1)) continue;
            const int b1 = a == 0 ? 1 : 0, b2 = a == 2 ? 1 : 2;           // the two axes across the edge
            int d1[2] = {0, 0}, d2[2] = {0, 0}, n1 = 1, n2 = 1;
            if (l[b1] == 0 && B.c[b1] > 0) d1[n1++] = -1;
            if (l[b1] == B.e[b1] && B.c[b1] + 1 < L.b[b1]) d1[n1++] = 1;
            if (l[b2] == 0 && B.c[b2] > 0) d2[n2++] = -1;
            if (l[b2] == B.e[b2] && B.c[b2] + 1 < L.b[b2]) d2[n2++] = 1;
            for (int s1 = 0; s1 < n1; ++s1)
                for (int s2 = 0; s2 < n2; ++s2) {
                    if (s1 == 0 && s2 == 0) continue;
                    const int64_t nb = id + d1[s1] * stride[b1] + d2[s2] * stride[b2];
                    if (flags[nb] == 0) flags[nb] = 2;
                }
        }
    }
}

__global__ void __launch_bounds__(256) nb_count_kernel(const float* __restrict__ vals, const int64_t* __restrict__ bricks, int64_t n_bricks,
                                                       Lattice L, float thr, int32_t* __restrict__ vert_count,
                                                       int32_t* __restrict__ tri_count, int64_t* __restrict__ keys) {
    __shared__ uint8_t s_count[256];
    for (int c = threadIdx.x; c < 256; c += blockDim.x) s_count[c] = kIsoTriCount[c];
    __syncthreads();
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_bricks * kSeg) return;
    const int64_t slot = t / kSeg;
    const int x = (int)(t % kSeg) / kP, y = (int)(t % kSeg) % kP;
    const Brick B = make_brick(L, bricks[slot]);
    const float* v = vals + slot * kBP;
    int nv = 0, nt = 0;
    int64_t key = INT64_MAX;
    if (x < B.own[0] && y < B.own[1]) {
        key = ((int64_t)(B.o[0] + x) * L.n[1] + B.o[1] + y) * L.b[2] + B.c[2];
        for (int z = 0; z < B.own[2]; ++z) nv += __popc(nb_edge_bits(v, B, x, y, z, thr));
        if (x < B.e[0] && y < B.e[1])
            for (int z = 0; z < B.e[2]; ++z) nt += s_count[nb_case(v, x, y, z, thr)];
    }
    vert_count[t] = nv;
    tri_count[t] = nt;
    keys[t] = key;
}

__global__ void __launch_bounds__(256) nb_vertices_kernel(const float* __restrict__ vals, const int64_t* __restrict__ bricks,
                                                          int64_t n_bricks, Lattice L, float thr, const int64_t* __restrict__ vert_offsets,
                                                          float* __restrict__ verts, int32_t* __restrict__ idx) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_bricks * kSeg) return;
    const int64_t slot = t / kSeg;
    const int x = (int)(t % kSeg) / kP, y = (int)(t % kSeg) % kP;
    const Brick B = make_brick(L, bricks[slot]);
    if (x >= B.own[0] || y >= B.own[1]) return;
    const float* v = vals + slot * kBP;
    int32_t* id = idx + slot * kBP;
    int64_t n = vert_offsets[t];
    for (int z = 0; z < B.own[2]; ++z) {
        id[lp(x, y, z)] = (int32_t)n;
        const int bits = nb_edge_bits(v, B, x, y, z, thr);
        if (!bits) continue;
        const float ua = v[lp(x, y, z)];
        const float pos[3] = {(float)(B.o[0] + x), (float)(B.o[1] + y), (float)(B.o[2] + z)};
        const float ub[3] = {v[lp(min(x + 1, kB), y, z)], v[lp(x, min(y + 1, kB), z)], v[lp(x, y, min(z + 1, kB))]};
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            if (!(bits >> a & 1)) continue;
            const float tt = __fdiv_rn(__fsub_rn(thr, ua), __fsub_rn(ub[a], ua));
            float* o = verts + n * 3;
            o[0] = a == 0 ? __fadd_rn(pos[0], tt) : pos[0];
            o[1] = a == 1 ? __fadd_rn(pos[1], tt) : pos[1];
            o[2] = a == 2 ? __fadd_rn(pos[2], tt) : pos[2];
            ++n;
        }
    }
}

__global__ void __launch_bounds__(256) nb_triangles_kernel(const float* __restrict__ vals, const int64_t* __restrict__ bricks,
                                                           int64_t n_bricks, Lattice L, float thr, const int32_t* __restrict__ slot_map,
                                                           const int64_t* __restrict__ tri_offsets, const int32_t* __restrict__ idx,
                                                           int32_t* __restrict__ tris) {
    __shared__ int8_t s_table[256][16];
    __shared__ uint8_t s_count[256];
    __shared__ uint8_t s_edge_start[12];
    for (int c = threadIdx.x; c < 256 * 16; c += blockDim.x) s_table[c >> 4][c & 15] = kIsoTriTable[c >> 4][c & 15];
    for (int c = threadIdx.x; c < 256; c += blockDim.x) s_count[c] = kIsoTriCount[c];
    if (threadIdx.x < 12) s_edge_start[threadIdx.x] = kIsoEdgeStart[threadIdx.x];
    __syncthreads();
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_bricks * kSeg) return;
    const int64_t slot = t / kSeg;
    const int x = (int)(t % kSeg) / kP, y = (int)(t % kSeg) % kP;
    const int64_t id = bricks[slot];
    const Brick B = make_brick(L, id);
    if (x >= B.e[0] || y >= B.e[1]) return;
    const float* v = vals + slot * kBP;
    const int64_t stride[3] = {(int64_t)L.b[1] * L.b[2], L.b[2], 1};
    int32_t* out = tris + tri_offsets[t] * 3;
    for (int z = 0; z < B.e[2]; ++z) {
        const int cs = nb_case(v, x, y, z, thr);
        const int n = s_count[cs];
        for (int m = 0; m < 3 * n; ++m) {
            const int e = s_table[cs][m];
            const int axis = e >> 2, c0 = s_edge_start[e];
            // the edge's lower point q, and the brick that owns q: local coordinate 8 is the next brick's 0 unless this
            // brick is the last on that axis (then q is its own end point)
            int q[3] = {x + (c0 & 1), y + (c0 >> 1 & 1), z + (c0 >> 2 & 1)};
            int64_t owner = id;
            Brick O = B;
            bool moved = false;
#pragma unroll
            for (int a = 0; a < 3; ++a)
                if (q[a] == kB && B.c[a] + 1 < L.b[a]) {
                    q[a] = 0;
                    owner += stride[a];
                    moved = true;
                }
            int64_t oslot = slot;
            if (moved) {
                oslot = slot_map[owner];            // active: the band is closed under shared crossed edges
                O = make_brick(L, owner);
            }
            int32_t vid = idx[oslot * kBP + lp(q[0], q[1], q[2])];
            if (axis > 0) {
                const int bits = nb_edge_bits(vals + oslot * kBP, O, q[0], q[1], q[2], thr);
                vid += (bits & 1) + (axis == 2 ? (bits >> 1 & 1) : 0);
            }
            out[m] = vid;
        }
        out += 3 * n;
    }
}

int nb_check(const char* what, int32_t nx, int32_t ny, int32_t nz) {
    TF_REQUIRE(nx >= 2 && ny >= 2 && nz >= 2 && nx <= kMaxAxis && ny <= kMaxAxis && nz <= kMaxAxis,
               "%s: every lattice axis needs 2 to %d points (got %d x %d x %d)", what, kMaxAxis, nx, ny, nz);
    return 0;
}

unsigned nb_blocks(int64_t threads) { return (unsigned)((threads + 255) / 256); }

}  // namespace

extern "C" TF_API int tf_iso_nb_classify(const float* coarse, int32_t nx, int32_t ny, int32_t nz, float threshold, float band,
                                         uint8_t* flags, tf_stream_t stream) {
    if (int rc = nb_check("tf_iso_nb_classify", nx, ny, nz)) return rc;
    TF_REQUIRE(coarse && flags, "tf_iso_nb_classify: NULL pointer");
    const Lattice L = make_lattice(nx, ny, nz);
    nb_classify_kernel<<<nb_blocks((int64_t)L.b[0] * L.b[1] * L.b[2]), 256, 0, (cudaStream_t)stream>>>(coarse, L, threshold, band, flags);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_iso_nb_classify");
    return 0;
}

extern "C" TF_API int tf_iso_nb_points(const float* ax, const float* ay, const float* az, int32_t nx, int32_t ny, int32_t nz,
                                       const int64_t* bricks, int64_t n_bricks, float* xyz, tf_stream_t stream) {
    if (int rc = nb_check("tf_iso_nb_points", nx, ny, nz)) return rc;
    TF_REQUIRE(n_bricks >= 0, "tf_iso_nb_points: negative brick count");
    if (n_bricks == 0) return 0;
    TF_REQUIRE(ax && ay && az && bricks && xyz, "tf_iso_nb_points: NULL pointer");
    nb_points_kernel<<<nb_blocks(n_bricks * kBP), 256, 0, (cudaStream_t)stream>>>(ax, ay, az, make_lattice(nx, ny, nz), bricks, n_bricks, xyz);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_iso_nb_points");
    return 0;
}

extern "C" TF_API int tf_iso_nb_grow(const float* values, const int64_t* bricks, int64_t n_bricks, int32_t nx, int32_t ny, int32_t nz,
                                     float threshold, uint8_t* flags, tf_stream_t stream) {
    if (int rc = nb_check("tf_iso_nb_grow", nx, ny, nz)) return rc;
    TF_REQUIRE(n_bricks >= 0 && n_bricks < ((int64_t)1 << 31), "tf_iso_nb_grow: brick count %lld out of range", (long long)n_bricks);
    if (n_bricks == 0) return 0;
    TF_REQUIRE(values && bricks && flags, "tf_iso_nb_grow: NULL pointer");
    nb_grow_kernel<<<(unsigned)n_bricks, 256, 0, (cudaStream_t)stream>>>(values, bricks, make_lattice(nx, ny, nz), threshold, flags);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_iso_nb_grow");
    return 0;
}

extern "C" TF_API int tf_iso_nb_count(const float* values, const int64_t* bricks, int64_t n_bricks, int32_t nx, int32_t ny, int32_t nz,
                                      float threshold, int32_t* vert_count, int32_t* tri_count, int64_t* keys, tf_stream_t stream) {
    if (int rc = nb_check("tf_iso_nb_count", nx, ny, nz)) return rc;
    TF_REQUIRE(n_bricks >= 0, "tf_iso_nb_count: negative brick count");
    if (n_bricks == 0) return 0;
    TF_REQUIRE(values && bricks && vert_count && tri_count && keys, "tf_iso_nb_count: NULL pointer");
    nb_count_kernel<<<nb_blocks(n_bricks * kSeg), 256, 0, (cudaStream_t)stream>>>(values, bricks, n_bricks, make_lattice(nx, ny, nz),
                                                                                 threshold, vert_count, tri_count, keys);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_iso_nb_count");
    return 0;
}

extern "C" TF_API int tf_iso_nb_vertices(const float* values, const int64_t* bricks, int64_t n_bricks, int32_t nx, int32_t ny, int32_t nz,
                                         float threshold, const int64_t* vert_offsets, float* vertices, int32_t* index, tf_stream_t stream) {
    if (int rc = nb_check("tf_iso_nb_vertices", nx, ny, nz)) return rc;
    TF_REQUIRE(n_bricks >= 0, "tf_iso_nb_vertices: negative brick count");
    if (n_bricks == 0) return 0;
    TF_REQUIRE(values && bricks && vert_offsets && vertices && index, "tf_iso_nb_vertices: NULL pointer");
    nb_vertices_kernel<<<nb_blocks(n_bricks * kSeg), 256, 0, (cudaStream_t)stream>>>(values, bricks, n_bricks, make_lattice(nx, ny, nz),
                                                                                    threshold, vert_offsets, vertices, index);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_iso_nb_vertices");
    return 0;
}

extern "C" TF_API int tf_iso_nb_triangles(const float* values, const int64_t* bricks, int64_t n_bricks, int32_t nx, int32_t ny, int32_t nz,
                                          float threshold, const int32_t* slot_map, const int64_t* tri_offsets, const int32_t* index,
                                          int32_t* triangles, tf_stream_t stream) {
    if (int rc = nb_check("tf_iso_nb_triangles", nx, ny, nz)) return rc;
    TF_REQUIRE(n_bricks >= 0, "tf_iso_nb_triangles: negative brick count");
    if (n_bricks == 0) return 0;
    TF_REQUIRE(values && bricks && slot_map && tri_offsets && index && triangles, "tf_iso_nb_triangles: NULL pointer");
    nb_triangles_kernel<<<nb_blocks(n_bricks * kSeg), 256, 0, (cudaStream_t)stream>>>(values, bricks, n_bricks, make_lattice(nx, ny, nz),
                                                                                     threshold, slot_map, tri_offsets, index, triangles);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_iso_nb_triangles");
    return 0;
}
