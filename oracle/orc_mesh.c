/* CPU ORACLE (test infrastructure only) -- marching-cubes mesh of the TSDF volume (dfusion.h df_extract_mesh).
 * Not in the reference (its next steps ask for a .ply / .obj export, Report.md:57): PARITY UNPINNED by construction.  A plain triple
 * loop over edges, then over cells, with the generated case table (dynamicfusion_b200/csrc/mc_table.h).  Built on its own into
 * liborc_mesh.so (together with orc_tsdf.c for the half conversion) by oracle/orc_mesh.py.  Vertex positions use edge_point below,
 * the same operations in the same order as orc_extract_cloud's interpolation (orc_tsdf.c), so a vertex on an edge the cloud also
 * emits equals that cloud point (tests/test_mesh_model.py checks it bit for bit). */
#include "orc_common.h"
#include <stdlib.h>
#include "../dynamicfusion_b200/csrc/mc_table.h"

static inline int active(uint32_t v) { int W; float F = orc_unpack_tsdf(v, &W); return W != 0 && F != 1.f; }
static inline int inside(uint32_t v) { return orc_unpack_tsdf(v, NULL) < 0.f; }

/* case of the cell with min corner (x, y, z), -1 when a corner is inactive */
static int cell_case(const orc_volume *vol, int x, int y, int z)
{
    const size_t sy = (size_t)vol->dims[0], sz = sy * vol->dims[1];
    const uint32_t *b = vol->data + x + sy * y + sz * z;
    int c = 0;
    for (int i = 0; i < 8; ++i) {
        uint32_t v = b[(i & 1) + ((i & 2) ? sy : 0) + ((i & 4) ? sz : 0)];
        if (!active(v)) return -1;
        c |= inside(v) << i;
    }
    return c;
}

/* the zero crossing of FullScan6 (tsdf_volume.cu:573-627) on the edge from voxel (x, y, z) (value F) along `axis`, then posed:
 * orc_extract_cloud's expression, operation for operation */
static orc_f3 edge_point(const orc_volume *vol, const orc_aff3f *pose, int x, int y, int z, int axis, float F, float Fn)
{
    orc_f3 V = f3(((float)x + 0.5f) * vol->voxel_size[0], ((float)y + 0.5f) * vol->voxel_size[1], ((float)z + 0.5f) * vol->voxel_size[2]);
    orc_f3 p = V;
    float d_inv = 1.f / (fabsf(F) + fabsf(Fn));
    if (axis == 0) { float Vn = V.x + vol->voxel_size[0]; p.x = (V.x * fabsf(Fn) + Vn * fabsf(F)) * d_inv; }
    if (axis == 1) { float Vn = V.y + vol->voxel_size[1]; p.y = (V.y * fabsf(Fn) + Vn * fabsf(F)) * d_inv; }
    if (axis == 2) { float Vn = V.z + vol->voxel_size[2]; p.z = (V.z * fabsf(Fn) + Vn * fabsf(F)) * d_inv; }
    return orc_aff_mul(pose, p);
}

static int cmp_key(const void *a, const void *b)
{
    uint32_t x = *(const uint32_t *)a, y = *(const uint32_t *)b;
    return x < y ? -1 : x > y;
}

/* counts[0] / [1] = true vertex / triangle totals; writes at most vcap vertices + keys and tcap triangles, none when the vertices overflow */
void orc_extract_mesh(orc_volume vol, orc_aff3f pose, float *vertices, uint32_t *keys, long long vcap, int32_t *tris, long long tcap,
                      long long *counts)
{
    const int D[3] = {vol.dims[0], vol.dims[1], vol.dims[2]};
    const size_t sy = (size_t)D[0], sz = sy * D[1];
    size_t cap = 1024, nv = 0;
    uint32_t *all = (uint32_t *)malloc(cap * sizeof(uint32_t));
    /* vertices: every edge (v, axis) whose endpoints differ in the inside test and that borders a meshed cell, ascending key */
    for (int z = 0; z < D[2]; ++z)
        for (int y = 0; y < D[1]; ++y)
            for (int x = 0; x < D[0]; ++x) {
                const uint32_t u = vol.data[x + sy * y + sz * z];
                for (int axis = 0; axis < 3; ++axis) {
                    const int p[3] = {x, y, z};
                    if (p[axis] + 1 >= D[axis]) continue;
                    const uint32_t n = vol.data[x + sy * y + sz * z + (axis == 0 ? 1 : axis == 1 ? sy : sz)];
                    if (inside(u) == inside(n)) continue;
                    int meshed = 0;
                    for (int j = 0; j < 2 && !meshed; ++j)
                        for (int k = 0; k < 2 && !meshed; ++k) {
                            int c[3] = {x, y, z};
                            const int a1 = axis == 0 ? 1 : 0, a2 = axis == 2 ? 1 : 2;     /* the two other axes */
                            c[a1] -= j; c[a2] -= k;
                            if (c[0] < 0 || c[1] < 0 || c[2] < 0 || c[0] >= D[0] - 1 || c[1] >= D[1] - 1 || c[2] >= D[2] - 1) continue;
                            const int cs = cell_case(&vol, c[0], c[1], c[2]);
                            meshed = cs > 0 && cs < 255;
                        }
                    if (!meshed) continue;
                    const uint32_t key = 3u * (uint32_t)(x + sy * y + sz * z) + (uint32_t)axis;
                    if (nv == cap) { cap *= 2; all = (uint32_t *)realloc(all, cap * sizeof(uint32_t)); }
                    all[nv] = key;
                    if ((long long)nv < vcap) {
                        orc_f3 q = edge_point(&vol, &pose, x, y, z, axis, orc_unpack_tsdf(u, NULL), orc_unpack_tsdf(n, NULL));
                        float *o = vertices + 4 * nv;
                        o[0] = q.x; o[1] = q.y; o[2] = q.z; o[3] = 0.f;
                        keys[nv] = key;
                    }
                    ++nv;
                }
            }
    /* triangles: meshed cells in ascending index, the case's triangles in table order */
    long long nt = 0;
    for (int z = 0; z < D[2] - 1; ++z)
        for (int y = 0; y < D[1] - 1; ++y)
            for (int x = 0; x < D[0] - 1; ++x) {
                const int cs = cell_case(&vol, x, y, z);
                if (cs <= 0 || cs >= 255) continue;
                for (int t = 0; t < df_mc_ntri[cs]; ++t, ++nt) {
                    if (nt >= tcap || (long long)nv > vcap) continue;
                    for (int q = 0; q < 3; ++q) {
                        const signed char *e = df_mc_edges[df_mc_tris[cs][3 * t + q]];
                        const uint32_t key = 3u * (uint32_t)((x + e[0]) + sy * (y + e[1]) + sz * (z + e[2])) + (uint32_t)e[3];
                        const uint32_t *hit = (const uint32_t *)bsearch(&key, all, nv, sizeof(uint32_t), cmp_key);
                        tris[3 * nt + q] = hit ? (int32_t)(hit - all) : -1;
                    }
                }
            }
    free(all);
    counts[0] = (long long)nv;
    counts[1] = nt;
}
