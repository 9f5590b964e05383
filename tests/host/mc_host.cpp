// Host reference of the isosurface stage (rho2sdf.jl_b200/csrc/r2s_surf.cu) for tests/isosurface_ref.py: the library's case table
// (r2s_mc.cuh, the same header) and a whole-grid extraction written out plainly from the output contract.  Built with -ffp-contract=off.
//
// Contract: one vertex per grid edge whose ends lie on different sides of iso (inside iff value >= iso), ordered by (linear id of the
// edge's lower point, axis x < y < z); triangles ordered by linear cell id, then by table order within the cell.
#include <stdint.h>
#include <string.h>
#include <vector>
#include "../../rho2sdf.jl_b200/csrc/r2s_mc.cuh"

typedef long long i64;

extern "C" void mc_host_table(uint8_t *out /* 256 x 16: count, then 15 edge ids */) {
  for (int c = 0; c < 256; c++) {
    const McCase m = mc_build_case(c);
    out[16 * c] = m.n;
    memcpy(out + 16 * c + 1, m.e, 15);
  }
}

extern "C" int mc_host_face_segments(int c, int f, int *seg) { return mc_face_segments(c, f, seg); }
extern "C" void mc_host_face(int f, int *cyc) { mc_face(f, cyc); }
extern "C" void mc_host_edge(int e, int *corner, int *axis) { *corner = mc_edge_corner(e); *axis = mc_edge_axis(e); }

struct Field {
  const float *v; i64 nx, ny, nz; float iso;
  bool in(i64 i, i64 j, i64 k) const { return v[(k * ny + j) * nx + i] >= iso; }
  float at(i64 i, i64 j, i64 k) const { return v[(k * ny + j) * nx + i]; }
  // crossing on the edge from (i,j,k) along axis a
  bool cross(i64 i, i64 j, i64 k, int a) const {
    const i64 p[3] = {i, j, k}, n[3] = {nx, ny, nz};
    if (p[a] + 1 >= n[a]) return false;
    return in(i, j, k) != in(i + (a == 0), j + (a == 1), k + (a == 2));
  }
  int crossings(i64 i, i64 j, i64 k) const { return cross(i, j, k, 0) + cross(i, j, k, 1) + cross(i, j, k, 2); }
  int cell_case(i64 i, i64 j, i64 k) const {
    int c = 0;
    for (int q = 0; q < 8; q++) c |= (int)in(i + (q & 1), j + (q >> 1 & 1), k + (q >> 2 & 1)) << q;
    return c;
  }
};

static McCase g_tab[256];
static void init_tab() { for (int c = 0; c < 256; c++) g_tab[c] = mc_build_case(c); }

extern "C" void mc_host_count(const float *v, i64 nx, i64 ny, i64 nz, float iso, i64 *nv, i64 *nt) {
  init_tab();
  const Field F{v, nx, ny, nz, iso};
  i64 a = 0, b = 0;
#pragma omp parallel for reduction(+ : a, b) schedule(dynamic, 16)
  for (i64 r = 0; r < ny * nz; r++) {
    const i64 j = r % ny, k = r / ny;
    for (i64 i = 0; i < nx; i++) {
      a += F.crossings(i, j, k);
      if (i + 1 < nx && j + 1 < ny && k + 1 < nz) b += g_tab[F.cell_case(i, j, k)].n;
    }
  }
  *nv = a; *nt = b;
}

// V[3 * nv] float, T[3 * nt] int32 (sizes from mc_host_count)
extern "C" void mc_host_extract(const float *v, i64 nx, i64 ny, i64 nz, const double *origin, const double *spacing, float iso, float *V, int32_t *T) {
  init_tab();
  const Field F{v, nx, ny, nz, iso};
  const i64 nrows = ny * nz;
  // first vertex id of every point row, first triangle id of every cell row
  std::vector<i64> vrow((size_t)nrows + 1, 0), trow((size_t)nrows + 1, 0);
#pragma omp parallel for schedule(dynamic, 16)
  for (i64 r = 0; r < nrows; r++) {
    const i64 j = r % ny, k = r / ny;
    i64 a = 0, b = 0;
    for (i64 i = 0; i < nx; i++) {
      a += F.crossings(i, j, k);
      if (i + 1 < nx && j + 1 < ny && k + 1 < nz) b += g_tab[F.cell_case(i, j, k)].n;
    }
    vrow[(size_t)r + 1] = a; trow[(size_t)r + 1] = b;
  }
  for (i64 r = 0; r < nrows; r++) { vrow[(size_t)r + 1] += vrow[(size_t)r]; trow[(size_t)r + 1] += trow[(size_t)r]; }
#pragma omp parallel
  {
    std::vector<i64> first[4];      // first vertex id of each point of the rows (j + dy, k + dz)
    for (auto &f : first) f.resize((size_t)nx);
#pragma omp for schedule(dynamic, 16)
    for (i64 r = 0; r < nrows; r++) {
      const i64 j = r % ny, k = r / ny;
      for (int q = 0; q < 4; q++) {
        const i64 jj = j + (q & 1), kk = k + (q >> 1);
        if (jj >= ny || kk >= nz) continue;
        i64 id = vrow[(size_t)(kk * ny + jj)];
        for (i64 i = 0; i < nx; i++) { first[q][(size_t)i] = id; id += F.crossings(i, jj, kk); }
      }
      // vertices of this row
      i64 id = vrow[(size_t)r];
      for (i64 i = 0; i < nx; i++)
        for (int a = 0; a < 3; a++)
          if (F.cross(i, j, k, a)) {
            mc_vertex(origin, spacing, i, j, k, a, F.at(i, j, k), F.at(i + (a == 0), j + (a == 1), k + (a == 2)), iso, V + 3 * id);
            id++;
          }
      if (j + 1 >= ny || k + 1 >= nz) continue;
      // triangles of this cell row
      i64 t = trow[(size_t)r];
      for (i64 i = 0; i + 1 < nx; i++) {
        const McCase &m = g_tab[F.cell_case(i, j, k)];
        for (int q = 0; q < 3 * m.n; q++) {
          const int e = m.e[q], c = mc_edge_corner(e), a = mc_edge_axis(e);
          const i64 pi = i + (c & 1), pj = j + (c >> 1 & 1), pk = k + (c >> 2 & 1);
          i64 vid = first[(c >> 1 & 1) | ((c >> 2 & 1) << 1)][(size_t)pi];
          for (int b = 0; b < a; b++) vid += F.cross(pi, pj, pk, b);
          T[3 * t + q] = (int32_t)vid;
        }
        t += m.n;
      }
    }
  }
}
