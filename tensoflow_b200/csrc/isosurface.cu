// Isosurface extraction (marching cubes) of a dense fp32 volume u[nx][ny][nz] (z fastest): the reference's
// `mcubes.marching_cubes(u, threshold)` (extract_mesh.py), which the shape stage uses to hand its zero level set to the
// material stage.  Conventions (oracle/torch_oracle_iso.py restates them on the CPU):
//   inside iff u < threshold; one vertex per crossed lattice edge, owned by the edge's lower point p = (i*ny + j)*nz + k and
//   ordered by (p, axis x/y/z); it lies at a_axis + t, t = (threshold - u_a) / (u_b - u_a), one rounding per op;
//   triangles ordered by cell (i*ny + j)*nz + k, then in the order of the generated case table (isosurface_table.cuh).
// Count / host prefix sum / write, one warp per (i, j) row of lattice points; a warp scan along the row places each
// lane's items, so the output order is fixed and no atomics are involved.
//   tf_iso_count      per row: owned crossed edges, triangles of the row's cells
//   tf_iso_vertices   vertices, and idx[p] = number of vertices owned by points before p (every p)
//   tf_iso_triangles  per cell: edge -> vertex id through idx, triangles from the table
// Vertex id of the edge (q, axis) from idx, with q + 1 the next point in memory order:
//   x: idx[q]    z: idx[q + 1] - 1    y: idx[q + 1] - 1 - (z edge of q crossed)
// (q's vertices are numbered x, y, z, so the z vertex is q's last and the y vertex precedes it when both exist).  A y or z
// edge of q implies q + 1 < nx*ny*nz, so idx[q + 1] always exists.
#include "common.cuh"
#include "isosurface_table.cuh"

namespace {

constexpr int kIsoWarps = 8;          // rows per 256-thread block

struct IsoRow {
    const float* r00;                  // row (i, j); r10 = (i+1, j), r01 = (i, j+1), r11 = (i+1, j+1) (aliases of r00 when absent)
    const float* r10;
    const float* r01;
    const float* r11;
    int i, j;
    bool hx, hy;                       // the +x / +y neighbour rows exist
};

__device__ __forceinline__ IsoRow iso_row(const float* u, int64_t row, int nx, int ny, int nz) {
    IsoRow r;
    r.i = (int)(row / ny);
    r.j = (int)(row % ny);
    r.hx = r.i + 1 < nx;
    r.hy = r.j + 1 < ny;
    r.r00 = u + row * nz;
    r.r10 = r.hx ? r.r00 + (int64_t)ny * nz : r.r00;
    r.r01 = r.hy ? r.r00 + nz : r.r00;
    r.r11 = r.hx && r.hy ? r.r00 + (int64_t)ny * nz + nz : r.r00;
    return r;
}

// owned crossed edges of point (i, j, k): bit a = edge along axis a
__device__ __forceinline__ int iso_edge_bits(const IsoRow& r, int k, int nz, float thr) {
    const bool in0 = r.r00[k] < thr;
    int bits = 0;
    if (r.hx && (r.r10[k] < thr) != in0) bits |= 1;
    if (r.hy && (r.r01[k] < thr) != in0) bits |= 2;
    if (k + 1 < nz && (r.r00[k + 1] < thr) != in0) bits |= 4;
    return bits;
}

// marching-cubes case of cell (i, j, k) (the caller ensures the cell exists): bit c = corner c inside
__device__ __forceinline__ int iso_case(const IsoRow& r, int k, float thr) {
    return (int)(r.r00[k] < thr) | (int)(r.r10[k] < thr) << 1 | (int)(r.r01[k] < thr) << 2 | (int)(r.r11[k] < thr) << 3 |
           (int)(r.r00[k + 1] < thr) << 4 | (int)(r.r10[k + 1] < thr) << 5 | (int)(r.r01[k + 1] < thr) << 6 |
           (int)(r.r11[k + 1] < thr) << 7;
}

__device__ __forceinline__ int warp_inclusive_scan(int v, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int n = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += n;
    }
    return v;
}

__global__ void __launch_bounds__(256) iso_count_kernel(const float* __restrict__ u, int nx, int ny, int nz, float thr,
                                                        int32_t* __restrict__ vert_count, int32_t* __restrict__ tri_count) {
    __shared__ uint8_t s_count[256];
    for (int c = threadIdx.x; c < 256; c += blockDim.x) s_count[c] = kIsoTriCount[c];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kIsoWarps + (threadIdx.x >> 5);
    if (row >= (int64_t)nx * ny) return;
    const IsoRow r = iso_row(u, row, nx, ny, nz);
    const bool cells = r.hx && r.hy;
    int nv = 0, nt = 0;
    for (int k = lane; k < nz; k += 32) {
        nv += __popc(iso_edge_bits(r, k, nz, thr));
        if (cells && k + 1 < nz) nt += s_count[iso_case(r, k, thr)];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        nv += __shfl_xor_sync(0xffffffffu, nv, o);
        nt += __shfl_xor_sync(0xffffffffu, nt, o);
    }
    if (lane == 0) {
        vert_count[row] = nv;
        tri_count[row] = nt;
    }
}

__global__ void __launch_bounds__(256) iso_vertices_kernel(const float* __restrict__ u, int nx, int ny, int nz, float thr,
                                                           const int64_t* __restrict__ vert_offsets, float* __restrict__ verts,
                                                           int32_t* __restrict__ idx) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kIsoWarps + (threadIdx.x >> 5);
    if (row >= (int64_t)nx * ny) return;
    const IsoRow r = iso_row(u, row, nx, ny, nz);
    int64_t base = vert_offsets[row];
    for (int k0 = 0; k0 < nz; k0 += 32) {
        const int k = k0 + lane;
        const int bits = k < nz ? iso_edge_bits(r, k, nz, thr) : 0;
        const int incl = warp_inclusive_scan(__popc(bits), lane);
        int64_t v = base + incl - __popc(bits);
        if (k < nz) idx[row * nz + k] = (int32_t)v;
        if (bits) {
            const float ua = r.r00[k];
            const float pos[3] = {(float)r.i, (float)r.j, (float)k};
            const float* nb[3] = {r.r10 + k, r.r01 + k, r.r00 + k + 1};
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                if (!(bits >> a & 1)) continue;
                const float t = __fdiv_rn(__fsub_rn(thr, ua), __fsub_rn(*nb[a], ua));
                float* o = verts + v * 3;
                o[0] = a == 0 ? __fadd_rn(pos[0], t) : pos[0];
                o[1] = a == 1 ? __fadd_rn(pos[1], t) : pos[1];
                o[2] = a == 2 ? __fadd_rn(pos[2], t) : pos[2];
                ++v;
            }
        }
        base += __shfl_sync(0xffffffffu, incl, 31);
    }
}

__global__ void __launch_bounds__(256) iso_triangles_kernel(const float* __restrict__ u, int nx, int ny, int nz, float thr,
                                                            const int64_t* __restrict__ tri_offsets, const int32_t* __restrict__ idx,
                                                            int32_t* __restrict__ tris) {
    __shared__ int8_t s_table[256][16];
    __shared__ uint8_t s_count[256];
    __shared__ uint8_t s_edge_start[12];
    for (int c = threadIdx.x; c < 256 * 16; c += blockDim.x) s_table[c >> 4][c & 15] = kIsoTriTable[c >> 4][c & 15];
    for (int c = threadIdx.x; c < 256; c += blockDim.x) s_count[c] = kIsoTriCount[c];
    if (threadIdx.x < 12) s_edge_start[threadIdx.x] = kIsoEdgeStart[threadIdx.x];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kIsoWarps + (threadIdx.x >> 5);
    if (row >= (int64_t)nx * ny) return;
    const IsoRow r = iso_row(u, row, nx, ny, nz);
    if (!(r.hx && r.hy)) return;                 // the last i and j rows own no cells (whole warp: no scan below)
    int64_t base = tri_offsets[row];
    for (int k0 = 0; k0 < nz - 1; k0 += 32) {
        const int k = k0 + lane;
        const int cs = k + 1 < nz ? iso_case(r, k, thr) : 0;
        const int n = s_count[cs];
        const int incl = warp_inclusive_scan(n, lane);
        int32_t* out = tris + (base + incl - n) * 3;
        for (int m = 0; m < 3 * n; ++m) {
            const int e = s_table[cs][m];
            const int axis = e >> 2, c0 = s_edge_start[e];
            const int64_t q = ((int64_t)(r.i + (c0 & 1)) * ny + r.j + (c0 >> 1 & 1)) * nz + k + (c0 >> 2 & 1);
            int32_t vid;
            if (axis == 0) {
                vid = idx[q];
            } else {
                vid = idx[q + 1] - 1;
                if (axis == 1 && k + (c0 >> 2 & 1) + 1 < nz && (u[q] < thr) != (u[q + 1] < thr)) vid -= 1;
            }
            out[m] = vid;
        }
        base += __shfl_sync(0xffffffffu, incl, 31);
    }
}

int iso_check(const char* what, const float* u, int32_t nx, int32_t ny, int32_t nz) {
    TF_REQUIRE(u, "%s: NULL volume", what);
    TF_REQUIRE(nx >= 2 && ny >= 2 && nz >= 2, "%s: every volume dimension must be >= 2 (got %d x %d x %d)", what, nx, ny, nz);
    TF_REQUIRE((int64_t)nx * ny * nz < ((int64_t)1 << 31), "%s: volume of %d x %d x %d points has 2^31 or more points", what, nx, ny, nz);
    return 0;
}

unsigned iso_blocks(int32_t nx, int32_t ny) { return (unsigned)(((int64_t)nx * ny + kIsoWarps - 1) / kIsoWarps); }

}  // namespace

extern "C" TF_API int tf_iso_count(const float* u, int32_t nx, int32_t ny, int32_t nz, float threshold, int32_t* vert_count,
                                   int32_t* tri_count, tf_stream_t stream) {
    if (int rc = iso_check("tf_iso_count", u, nx, ny, nz)) return rc;
    TF_REQUIRE(vert_count && tri_count, "tf_iso_count: NULL pointer");
    iso_count_kernel<<<iso_blocks(nx, ny), 32 * kIsoWarps, 0, (cudaStream_t)stream>>>(u, nx, ny, nz, threshold, vert_count, tri_count);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_iso_count");
    return 0;
}

extern "C" TF_API int tf_iso_vertices(const float* u, int32_t nx, int32_t ny, int32_t nz, float threshold, const int64_t* vert_offsets,
                                      float* vertices, int32_t* index_volume, tf_stream_t stream) {
    if (int rc = iso_check("tf_iso_vertices", u, nx, ny, nz)) return rc;
    TF_REQUIRE(vert_offsets && vertices && index_volume, "tf_iso_vertices: NULL pointer");
    iso_vertices_kernel<<<iso_blocks(nx, ny), 32 * kIsoWarps, 0, (cudaStream_t)stream>>>(u, nx, ny, nz, threshold, vert_offsets, vertices,
                                                                                         index_volume);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_iso_vertices");
    return 0;
}

extern "C" TF_API int tf_iso_triangles(const float* u, int32_t nx, int32_t ny, int32_t nz, float threshold, const int64_t* tri_offsets,
                                       const int32_t* index_volume, int32_t* triangles, tf_stream_t stream) {
    if (int rc = iso_check("tf_iso_triangles", u, nx, ny, nz)) return rc;
    TF_REQUIRE(tri_offsets && index_volume && triangles, "tf_iso_triangles: NULL pointer");
    iso_triangles_kernel<<<iso_blocks(nx, ny), 32 * kIsoWarps, 0, (cudaStream_t)stream>>>(u, nx, ny, nz, threshold, tri_offsets,
                                                                                          index_volume, triangles);
    tf_count_launches(1);
    TF_CHECK_LAUNCH("tf_iso_triangles");
    return 0;
}
