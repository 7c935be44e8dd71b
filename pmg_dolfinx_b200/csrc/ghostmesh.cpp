// Host-side ghost-layer builder for GENERAL (unstructured, arbitrarily numbered and oriented)
// conforming hexahedral meshes: from a global cell -> vertex table and a cell partition it produces,
// for one rank, everything the operator API takes -- the arrays the reference obtains from DOLFINx:
//   ghost_layer_mesh               src/mesh.hpp:16-98   every cell of another rank that shares a VERTEX
//                                                       with this rank's cells is ghosted here
//   compute_boundary_cells         src/mesh.hpp:105-143 lcells = owned cells without ghost dofs,
//                                                       bcells = the other owned cells + all ghost cells
//   tensor-product dofmaps         examples/pmg/main.cpp:83-87,199-213 (index = ix n^2 + iy n + iz)
//   geometry x / geometry dofmap   examples/pmg/main.cpp:217-256 (tp vertex order, src/mesh.hpp:75-84)
//   exterior-facet Dirichlet marker examples/pmg/main.cpp:122-124,173-185
//   IndexMap / Scatterer lists     src/vector.hpp:86-95
// Pure host code, no CUDA calls.  Unlike boxmesh.cpp nothing here assumes a box, a lexicographic
// numbering or aligned cell frames: shared edge and face dofs are numbered in a canonical frame of
// the entity (from its lowest global vertex towards the lower neighbour), so cells that see an
// entity with different local orientations agree on its dofs -- the job of DOLFINx's dof
// transformations for tensor-product Lagrange spaces, where GLL symmetry makes it a pure
// re-indexing.  Every rank is given the whole mesh description (there is no MPI here; the
// launcher reads or generates the mesh on every rank), so entity numbering and ownership need no
// communication.  Dof ownership: the lowest rank owning a cell that contains the dof's entity.
// Local numbering: owned dofs by global id, then ghosts by (owner, global id).
// Second-order (27-node) meshes (pmgx_ghostmesh_create_q2): the 8 corner nodes of every cell, renumbered densely in
// node-id order, are the vertices of all of the above; the geometry keeps all 27 nodes of each cell in the cell's
// own frame, and dof coordinates go through the triquadratic map.
#include "common.hpp"

#include <algorithm>
#include <array>
#include <cstring>
#include <map>
#include <memory>
#include <numeric>

namespace
{
using i64 = long long;

struct FaceKey
{
  std::array<i64, 4> v; // sorted vertex ids
  bool operator<(const FaceKey& o) const { return v < o.v; }
  bool operator==(const FaceKey& o) const { return v == o.v; }
};

// local vertex k = 4a + 2b + c  <->  (a,b,c) along (x,y,z)   (src/mesh.hpp:75-84)
inline int lv(int a, int b, int c) { return 4 * a + 2 * b + c; }

struct GSpace
{
  int P = 0;
  i64 n_owned = 0, n_ghost = 0, n_global = 0;
  std::vector<int32_t> dofmap;  // [n_cells][(P+1)^3]
  std::vector<int8_t> bc;       // [n_owned + n_ghost]
  std::vector<i64> l2g;
  std::vector<double> coords;   // [n][3]
  std::vector<int> send_ranks, send_offsets, recv_ranks, recv_offsets;
  std::vector<int32_t> send_idx, recv_idx;
};
} // namespace

struct pmgx_ghostmesh
{
  int rank = 0, nranks = 1;
  i64 n_cells_global = 0, n_vertices_global = 0;
  int npc = 8;                  // geometry nodes per cell: 8, or 27 (pmgx_ghostmesh_create_q2)
  // global description (kept: spaces are built lazily per degree)
  std::vector<i64> gcells;      // [ncg][8] vertex ids (the topology)
  std::vector<i64> gnodes;      // [ncg][27] global node ids of a 27-node mesh (empty with 8 nodes: gcells)
  std::vector<int> gowner;      // [ncg]
  std::vector<double> gcoords;  // [n_nodes][3], indexed by node id (the vertex id of an 8-node mesh)
  std::vector<uint64_t> vranks; // per global vertex: bit q set iff a cell owned by q contains it
  // global entity tables
  std::vector<uint64_t> edges;  // sorted unique (vmin << 32 | vmax)
  std::vector<FaceKey> faces;   // sorted unique
  std::vector<int> edge_owner, face_owner, vertex_owner;
  std::vector<char> vertex_bc, edge_bc, face_bc; // entity lies on an exterior facet
  // local part
  std::vector<i64> cells;       // global id of each local cell: owned first, then ghosts by (owner, id)
  i64 n_owned_cells = 0;
  std::vector<i64> lverts;      // global node id of each local geometry node
  std::vector<int32_t> geom_dofmap; // [n_cells][npc] local geometry node ids
  std::vector<int32_t> lcells, bcells;
  std::map<int, std::unique_ptr<GSpace>> spaces;

  i64 edge_index(i64 a, i64 b) const
  {
    const uint64_t k = ((uint64_t)std::min(a, b) << 32) | (uint64_t)std::max(a, b);
    return std::lower_bound(edges.begin(), edges.end(), k) - edges.begin();
  }
  i64 face_index(FaceKey k) const
  {
    std::sort(k.v.begin(), k.v.end());
    return std::lower_bound(faces.begin(), faces.end(), k) - faces.begin();
  }

  const i64* cell_nodes(i64 c) const { return npc == 8 ? &gcells[(size_t)c * 8] : &gnodes[(size_t)c * 27]; }
  GSpace& space(int P);
};

namespace
{
// the 12 edges and 6 faces of the reference hex as local vertex ids
void cell_edges(const i64* cv, std::array<std::array<i64, 2>, 12>& e)
{
  int k = 0;
  for (int b = 0; b < 2; ++b)
    for (int c = 0; c < 2; ++c)
      e[k++] = {cv[lv(0, b, c)], cv[lv(1, b, c)]}; // along x
  for (int a = 0; a < 2; ++a)
    for (int c = 0; c < 2; ++c)
      e[k++] = {cv[lv(a, 0, c)], cv[lv(a, 1, c)]}; // along y
  for (int a = 0; a < 2; ++a)
    for (int b = 0; b < 2; ++b)
      e[k++] = {cv[lv(a, b, 0)], cv[lv(a, b, 1)]}; // along z
}
void cell_faces(const i64* cv, std::array<FaceKey, 6>& f)
{
  int k = 0;
  for (int a = 0; a < 2; ++a)
    f[k++] = FaceKey{{cv[lv(a, 0, 0)], cv[lv(a, 1, 0)], cv[lv(a, 0, 1)], cv[lv(a, 1, 1)]}};
  for (int b = 0; b < 2; ++b)
    f[k++] = FaceKey{{cv[lv(0, b, 0)], cv[lv(1, b, 0)], cv[lv(0, b, 1)], cv[lv(1, b, 1)]}};
  for (int c = 0; c < 2; ++c)
    f[k++] = FaceKey{{cv[lv(0, 0, c)], cv[lv(1, 0, c)], cv[lv(0, 1, c)], cv[lv(1, 1, c)]}};
}
} // namespace

GSpace& pmgx_ghostmesh::space(int P)
{
  auto it = spaces.find(P);
  if (it != spaces.end())
    return *it->second;
  auto sp = std::make_unique<GSpace>();
  GSpace& s = *sp;
  s.P = P;
  const int n = P + 1, n3 = n * n * n;
  const i64 m = P - 1; // interior points per edge
  const i64 nvg = n_vertices_global, neg = (i64)edges.size(), nfg = (i64)faces.size();
  const i64 off_e = nvg, off_f = off_e + neg * m, off_c = off_f + nfg * m * m;
  s.n_global = off_c + n_cells_global * m * m * m;
  std::vector<double> pts, wts;
  pmgx::gll_points_weights(n, pts, wts);

  const i64 nc = (i64)cells.size();
  std::vector<i64> gdof((size_t)nc * n3);
  std::vector<int> down((size_t)nc * n3); // owner of each cell dof
  std::vector<char> isbc((size_t)nc * n3);
  for (i64 lc = 0; lc < nc; ++lc)
  {
    const i64 gc = cells[lc];
    const i64* cv = &gcells[(size_t)gc * 8];
    for (int ix = 0; ix < n; ++ix)
      for (int iy = 0; iy < n; ++iy)
        for (int iz = 0; iz < n; ++iz)
        {
          const int idx[3] = {ix, iy, iz};
          int fixed[3], nfixed = 0, freed[3], nfree = 0;
          for (int d = 0; d < 3; ++d)
          {
            if (idx[d] == 0 || idx[d] == P)
              fixed[nfixed++] = d;
            else
              freed[nfree++] = d;
          }
          // vertex of the cell at corner bits (a,b,c); free directions take the given bit
          auto corner = [&](int bit0, int bit1) -> i64
          {
            int abc[3];
            for (int d = 0; d < 3; ++d)
              abc[d] = idx[d] == P ? 1 : 0;
            if (nfree >= 1)
              abc[freed[0]] = bit0;
            if (nfree >= 2)
              abc[freed[1]] = bit1;
            return cv[lv(abc[0], abc[1], abc[2])];
          };
          const size_t slot = (size_t)lc * n3 + (size_t)(ix * n + iy) * n + iz;
          if (nfree == 0)
          {
            const i64 v = corner(0, 0);
            gdof[slot] = v;
            down[slot] = vertex_owner[v];
            isbc[slot] = vertex_bc[v];
          }
          else if (nfree == 1)
          {
            const i64 va = corner(0, 0), vb = corner(1, 0);
            const int t = idx[freed[0]];
            const i64 e = edge_index(va, vb);
            const i64 pos = va < vb ? t : P - t; // from the lower global vertex
            gdof[slot] = off_e + e * m + (pos - 1);
            down[slot] = edge_owner[e];
            isbc[slot] = edge_bc[e];
          }
          else if (nfree == 2)
          {
            const i64 f00 = corner(0, 0), f10 = corner(1, 0), f01 = corner(0, 1), f11 = corner(1, 1);
            const i64 fv[2][2] = {{f00, f01}, {f10, f11}}; // fv[a][b]: a along freed[0], b along freed[1]
            int oa = 0, ob = 0;
            for (int a = 0; a < 2; ++a)
              for (int b = 0; b < 2; ++b)
                if (fv[a][b] < fv[oa][ob])
                  oa = a, ob = b;
            const int s0 = idx[freed[0]], t0 = idx[freed[1]];
            const i64 so = oa ? P - s0 : s0, to = ob ? P - t0 : t0; // measured from the lowest vertex
            const i64 n1 = fv[1 - oa][ob], n2 = fv[oa][1 - ob];     // its neighbours along the two axes
            const i64 s1 = n1 < n2 ? so : to, t1 = n1 < n2 ? to : so;
            const i64 f = face_index(FaceKey{{f00, f10, f01, f11}});
            gdof[slot] = off_f + f * m * m + (s1 - 1) * m + (t1 - 1);
            down[slot] = face_owner[f];
            isbc[slot] = face_bc[f];
          }
          else
          {
            gdof[slot] = off_c + gc * m * m * m + ((i64)(ix - 1) * m + (iy - 1)) * m + (iz - 1);
            down[slot] = gowner[gc];
            isbc[slot] = 0;
          }
        }
  }
  // local numbering: owned by global id, ghosts by (owner, global id)
  struct Rec
  {
    int owner;
    i64 g;
    char bc;
  };
  std::vector<Rec> recs;
  recs.reserve(gdof.size());
  for (size_t i = 0; i < gdof.size(); ++i)
    recs.push_back({down[i] == rank ? -1 : down[i], gdof[i], isbc[i]});
  std::sort(recs.begin(), recs.end(), [](const Rec& a, const Rec& b) { return a.owner != b.owner ? a.owner < b.owner : a.g < b.g; });
  recs.erase(std::unique(recs.begin(), recs.end(), [](const Rec& a, const Rec& b) { return a.owner == b.owner && a.g == b.g; }),
             recs.end());
  const i64 nl = (i64)recs.size();
  s.l2g.resize((size_t)nl);
  s.bc.resize((size_t)nl);
  s.n_owned = 0;
  for (i64 i = 0; i < nl; ++i)
  {
    s.l2g[i] = recs[i].g;
    s.bc[i] = recs[i].bc;
    if (recs[i].owner == -1)
      ++s.n_owned;
  }
  s.n_ghost = nl - s.n_owned;
  // global -> local through two sorted ranges (owned block, then per-owner ghost blocks)
  std::map<i64, int32_t> g2l;
  for (i64 i = 0; i < nl; ++i)
    g2l[s.l2g[i]] = (int32_t)i;
  s.dofmap.resize(gdof.size());
  for (size_t i = 0; i < gdof.size(); ++i)
    s.dofmap[i] = g2l[gdof[i]];
  // dof coordinates: trilinear (8 nodes) or triquadratic (27 nodes) map of the first local cell that holds the dof
  s.coords.assign((size_t)nl * 3, 0.0);
  std::vector<char> have((size_t)nl, 0);
  for (i64 lc = 0; lc < nc; ++lc)
  {
    const i64* cv = cell_nodes(cells[lc]);
    for (int a = 0; a < n3; ++a)
    {
      const int32_t d = s.dofmap[(size_t)lc * n3 + a];
      if (have[d])
        continue;
      have[d] = 1;
      const double xi[3] = {pts[a / (n * n)], pts[(a / n) % n], pts[a % n]};
      if (npc == 8)
        for (int k = 0; k < 8; ++k)
        {
          const int ka = (k >> 2) & 1, kb = (k >> 1) & 1, kc = k & 1;
          const double w = (ka ? xi[0] : 1 - xi[0]) * (kb ? xi[1] : 1 - xi[1]) * (kc ? xi[2] : 1 - xi[2]);
          for (int dd = 0; dd < 3; ++dd)
            s.coords[(size_t)d * 3 + dd] += w * gcoords[(size_t)cv[k] * 3 + dd];
        }
      else
      {
        double l[3][3]; // quadratic Lagrange basis on {0, 1/2, 1} at xi[dir]
        for (int dir = 0; dir < 3; ++dir)
        {
          const double t = xi[dir];
          l[dir][0] = (2 * t - 1) * (t - 1), l[dir][1] = 4 * t * (1 - t), l[dir][2] = t * (2 * t - 1);
        }
        for (int k = 0; k < 27; ++k)
        {
          const double w = l[0][k / 9] * l[1][(k / 3) % 3] * l[2][k % 3];
          for (int dd = 0; dd < 3; ++dd)
            s.coords[(size_t)d * 3 + dd] += w * gcoords[(size_t)cv[k] * 3 + dd];
        }
      }
    }
  }
  // receive lists: ghosts are grouped by owner already
  s.recv_offsets.assign(1, 0);
  for (i64 i = s.n_owned; i < nl; ++i)
  {
    if (s.recv_ranks.empty() || s.recv_ranks.back() != recs[i].owner)
    {
      if (!s.recv_ranks.empty())
        s.recv_offsets.push_back((int)(i - s.n_owned));
      s.recv_ranks.push_back(recs[i].owner);
    }
    s.recv_idx.push_back((int32_t)(i - s.n_owned));
  }
  if (!s.recv_ranks.empty())
    s.recv_offsets.push_back((int)s.n_ghost);
  // send lists: a rank q holds my owned dof iff one of its local cells contains the dof's entity, i.e.
  // iff q touches a vertex of a cell containing it (all those cells are local here)
  std::vector<uint64_t> dest((size_t)s.n_owned, 0);
  for (i64 lc = 0; lc < nc; ++lc)
  {
    const i64* cv = &gcells[(size_t)cells[lc] * 8];
    uint64_t rc = 0;
    for (int k = 0; k < 8; ++k)
      rc |= vranks[cv[k]];
    rc &= ~(1ull << rank);
    if (!rc)
      continue;
    for (int a = 0; a < n3; ++a)
    {
      const int32_t d = s.dofmap[(size_t)lc * n3 + a];
      if (d < s.n_owned)
        dest[d] |= rc;
    }
  }
  s.send_offsets.assign(1, 0);
  for (int q = 0; q < nranks; ++q)
  {
    if (q == rank)
      continue;
    const size_t before = s.send_idx.size();
    for (i64 d = 0; d < s.n_owned; ++d) // owned dofs are in global-id order: what q's ghost ordering expects
      if (dest[d] & (1ull << q))
        s.send_idx.push_back((int32_t)d);
    if (s.send_idx.size() > before)
    {
      s.send_ranks.push_back(q);
      s.send_offsets.push_back((int)s.send_idx.size());
    }
  }
  GSpace& ref = *sp;
  spaces[P] = std::move(sp);
  return ref;
}

namespace
{
// Everything after the global vertex table M->gcells [n_cells][8] (vertex ids < n_vertices), M->gowner and
// M->gcoords are in place; fills the entity tables, the local cells and the local geometry of M->npc nodes per cell.
void build_ghostmesh(pmgx_ghostmesh* M, i64 n_vertices)
{
  const int rank = M->rank, nranks = M->nranks, npc = M->npc;
  const i64 n_cells = M->n_cells_global;
  M->n_vertices_global = n_vertices;
  for (int o : M->gowner)
    PMGX_REQUIRE(o >= 0 && o < nranks, "ghostmesh_create: cell owner out of range");
  // which ranks touch each vertex; vertex owner = lowest of them
  M->vranks.assign((size_t)n_vertices, 0);
  for (i64 c = 0; c < n_cells; ++c)
    for (int k = 0; k < 8; ++k)
      M->vranks[M->gcells[(size_t)c * 8 + k]] |= 1ull << M->gowner[c];
  M->vertex_owner.assign((size_t)n_vertices, 0);
  for (i64 v = 0; v < n_vertices; ++v)
  {
    PMGX_REQUIRE(M->vranks[v] != 0, "ghostmesh_create: vertex %lld belongs to no cell", v);
    M->vertex_owner[v] = __builtin_ctzll(M->vranks[v]);
  }
  // global edge and face tables with owners (lowest rank of a containing cell) and exterior marks
  {
    std::vector<std::pair<uint64_t, int>> el;
    std::vector<std::pair<FaceKey, int>> fl;
    el.reserve((size_t)n_cells * 12);
    fl.reserve((size_t)n_cells * 6);
    std::array<std::array<i64, 2>, 12> ce;
    std::array<FaceKey, 6> cf;
    for (i64 c = 0; c < n_cells; ++c)
    {
      const i64* cv = &M->gcells[(size_t)c * 8];
      cell_edges(cv, ce);
      cell_faces(cv, cf);
      for (auto& e : ce)
        el.emplace_back(((uint64_t)std::min(e[0], e[1]) << 32) | (uint64_t)std::max(e[0], e[1]), M->gowner[c]);
      for (auto& f : cf)
      {
        std::sort(f.v.begin(), f.v.end());
        fl.emplace_back(f, M->gowner[c]);
      }
    }
    std::sort(el.begin(), el.end());
    std::sort(fl.begin(), fl.end());
    for (size_t i = 0; i < el.size(); ++i)
      if (i == 0 || el[i].first != el[i - 1].first)
      {
        M->edges.push_back(el[i].first);
        M->edge_owner.push_back(el[i].second); // sorted by (key, owner): the first is the lowest rank
      }
    std::vector<int> fcount;
    for (size_t i = 0; i < fl.size(); ++i)
    {
      if (i == 0 || !(fl[i].first == fl[i - 1].first))
      {
        M->faces.push_back(fl[i].first);
        M->face_owner.push_back(fl[i].second);
        fcount.push_back(0);
      }
      ++fcount.back();
    }
    M->vertex_bc.assign((size_t)n_vertices, 0);
    M->edge_bc.assign(M->edges.size(), 0);
    M->face_bc.assign(M->faces.size(), 0);
    for (size_t f = 0; f < M->faces.size(); ++f)
    {
      PMGX_REQUIRE(fcount[f] <= 2, "ghostmesh_create: a face belongs to %d cells (non-conforming mesh)", fcount[f]);
      if (fcount[f] == 1)
        M->face_bc[f] = 1; // exterior facet (mesh::exterior_facet_indices)
    }
    // edges and vertices of exterior facets: walk the cells once more (the face's cyclic vertex order is
    // only known through a cell)
    for (i64 c = 0; c < n_cells; ++c)
    {
      const i64* cv = &M->gcells[(size_t)c * 8];
      cell_faces(cv, cf);
      for (auto& f : cf)
      {
        // f.v = {f00, f10, f01, f11}: edges 00-10, 00-01, 10-11, 01-11
        const i64 q[4] = {f.v[0], f.v[1], f.v[2], f.v[3]};
        if (!M->face_bc[M->face_index(f)])
          continue;
        for (int k = 0; k < 4; ++k)
          M->vertex_bc[q[k]] = 1;
        const int ep[4][2] = {{0, 1}, {0, 2}, {1, 3}, {2, 3}};
        for (auto& p : ep)
          M->edge_bc[M->edge_index(q[p[0]], q[p[1]])] = 1;
      }
    }
  }
  // local cells: owned, then the vertex-sharing ghost layer ordered by (owner, id)  (src/mesh.hpp:25-46)
  std::vector<std::pair<int, i64>> ghosts;
  for (i64 c = 0; c < n_cells; ++c)
  {
    if (M->gowner[c] == rank)
    {
      M->cells.push_back(c);
      continue;
    }
    bool touch = false;
    for (int k = 0; k < 8 && !touch; ++k)
      touch = (M->vranks[M->gcells[(size_t)c * 8 + k]] >> rank) & 1ull;
    if (touch)
      ghosts.emplace_back(M->gowner[c], c);
  }
  M->n_owned_cells = (i64)M->cells.size();
  std::sort(ghosts.begin(), ghosts.end());
  for (auto& g : ghosts)
    M->cells.push_back(g.second);
  // local geometry nodes (first-touch order) and the geometry dofmap
  {
    std::map<i64, int32_t> vmap;
    M->geom_dofmap.resize(M->cells.size() * npc);
    for (size_t lc = 0; lc < M->cells.size(); ++lc)
      for (int k = 0; k < npc; ++k)
      {
        const i64 v = M->cell_nodes(M->cells[lc])[k];
        auto it = vmap.find(v);
        if (it == vmap.end())
        {
          it = vmap.emplace(v, (int32_t)M->lverts.size()).first;
          M->lverts.push_back(v);
        }
        M->geom_dofmap[lc * npc + k] = it->second;
      }
  }
  // lcells / bcells (src/mesh.hpp:119-138): an owned cell is local iff every vertex of it is owned by this rank
  for (size_t lc = 0; lc < M->cells.size(); ++lc)
  {
    bool local = (i64)lc < M->n_owned_cells;
    for (int k = 0; k < 8 && local; ++k)
      local = M->vertex_owner[M->gcells[(size_t)M->cells[lc] * 8 + k]] == rank;
    (local ? M->lcells : M->bcells).push_back((int32_t)lc);
  }
}

void check_create_args(int rank, int nranks, long long n_cells, const long long* cells_h, const int* cell_owner_h,
                       long long n_nodes, const double* coords_h, pmgx_ghostmesh** out)
{
  PMGX_REQUIRE(out && cells_h && cell_owner_h && coords_h, "ghostmesh_create: null argument");
  PMGX_REQUIRE(nranks >= 1 && nranks <= 64 && rank >= 0 && rank < nranks, "ghostmesh_create: bad rank (1..64 ranks)");
  PMGX_REQUIRE(n_cells >= 0 && n_nodes >= 0 && n_nodes < (1ll << 32), "ghostmesh_create: bad sizes");
}
} // namespace

extern "C"
{
int pmgx_ghostmesh_create(int rank, int nranks, long long n_cells, const long long* cell_vertices_h,
                          const int* cell_owner_h, long long n_vertices, const double* coords_h,
                          pmgx_ghostmesh** out)
{
  PMGX_API_BEGIN
  check_create_args(rank, nranks, n_cells, cell_vertices_h, cell_owner_h, n_vertices, coords_h, out);
  std::unique_ptr<pmgx_ghostmesh> M(new pmgx_ghostmesh());
  M->rank = rank;
  M->nranks = nranks;
  M->n_cells_global = n_cells;
  M->gcells.assign(cell_vertices_h, cell_vertices_h + n_cells * 8);
  M->gowner.assign(cell_owner_h, cell_owner_h + n_cells);
  M->gcoords.assign(coords_h, coords_h + n_vertices * 3);
  for (i64 v : M->gcells)
    PMGX_REQUIRE(v >= 0 && v < n_vertices, "ghostmesh_create: vertex id out of range");
  build_ghostmesh(M.get(), n_vertices);
  *out = M.release();
  PMGX_API_END
}

int pmgx_ghostmesh_create_q2(int rank, int nranks, long long n_cells, const long long* cell_nodes_h,
                             const int* cell_owner_h, long long n_nodes, const double* coords_h,
                             pmgx_ghostmesh** out)
{
  PMGX_API_BEGIN
  check_create_args(rank, nranks, n_cells, cell_nodes_h, cell_owner_h, n_nodes, coords_h, out);
  std::unique_ptr<pmgx_ghostmesh> M(new pmgx_ghostmesh());
  M->rank = rank;
  M->nranks = nranks;
  M->npc = 27;
  M->n_cells_global = n_cells;
  M->gnodes.assign(cell_nodes_h, cell_nodes_h + n_cells * 27);
  M->gowner.assign(cell_owner_h, cell_owner_h + n_cells);
  M->gcoords.assign(coords_h, coords_h + n_nodes * 3);
  for (i64 v : M->gnodes)
    PMGX_REQUIRE(v >= 0 && v < n_nodes, "ghostmesh_create_q2: node id out of range");
  // the corners, node k = 18a + 6b + 2c for vertex 4a + 2b + c, renumbered densely in node-id order: the order
  // that fixes the entity frames is the node order, so every rank derives the same numbering
  static const int corner[8] = {0, 2, 6, 8, 18, 20, 24, 26};
  std::vector<i64> vid((size_t)n_nodes, -1);
  for (i64 c = 0; c < n_cells; ++c)
    for (int k = 0; k < 8; ++k)
    {
      const i64 v = M->gnodes[(size_t)c * 27 + corner[k]];
      for (int j = 0; j < k; ++j)
        PMGX_REQUIRE(M->gnodes[(size_t)c * 27 + corner[j]] != v, "ghostmesh_create_q2: cell %lld repeats corner node %lld", c, v);
      vid[v] = 0;
    }
  i64 nv = 0;
  for (i64& v : vid)
    if (v == 0)
      v = nv++;
  M->gcells.resize((size_t)n_cells * 8);
  for (i64 c = 0; c < n_cells; ++c)
    for (int k = 0; k < 8; ++k)
      M->gcells[(size_t)c * 8 + k] = vid[M->gnodes[(size_t)c * 27 + corner[k]]];
  build_ghostmesh(M.get(), nv);
  *out = M.release();
  PMGX_API_END
}

int pmgx_ghostmesh_nodes_per_cell(pmgx_ghostmesh* m) { return m ? m->npc : -1; }

int pmgx_ghostmesh_destroy(pmgx_ghostmesh* m)
{
  PMGX_API_BEGIN
  delete m;
  PMGX_API_END
}

int pmgx_ghostmesh_sizes(pmgx_ghostmesh* m, long long* out_h)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(m && out_h, "ghostmesh_sizes: null argument");
  out_h[0] = (long long)m->cells.size();
  out_h[1] = m->n_owned_cells;
  out_h[2] = (long long)m->lverts.size();
  out_h[3] = (long long)m->lcells.size();
  out_h[4] = (long long)m->bcells.size();
  PMGX_API_END
}

int pmgx_ghostmesh_geometry(pmgx_ghostmesh* m, double* xgeom_h, int32_t* geom_dofmap_h, long long* cell_gid_h)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(m, "ghostmesh_geometry: null mesh");
  if (xgeom_h)
    for (size_t v = 0; v < m->lverts.size(); ++v)
      for (int d = 0; d < 3; ++d)
        xgeom_h[v * 3 + d] = m->gcoords[(size_t)m->lverts[v] * 3 + d];
  if (geom_dofmap_h)
    std::copy(m->geom_dofmap.begin(), m->geom_dofmap.end(), geom_dofmap_h);
  if (cell_gid_h)
    std::copy(m->cells.begin(), m->cells.end(), cell_gid_h);
  PMGX_API_END
}

int pmgx_ghostmesh_cell_lists(pmgx_ghostmesh* m, int32_t* lcells_h, int32_t* bcells_h)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(m, "ghostmesh_cell_lists: null mesh");
  if (lcells_h)
    std::copy(m->lcells.begin(), m->lcells.end(), lcells_h);
  if (bcells_h)
    std::copy(m->bcells.begin(), m->bcells.end(), bcells_h);
  PMGX_API_END
}

int pmgx_ghostmesh_space_sizes(pmgx_ghostmesh* m, int degree, long long* out_h)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(m && out_h && degree >= 1 && degree <= PMGX_MAX_DEGREE, "ghostmesh_space_sizes: bad arguments");
  GSpace& s = m->space(degree);
  out_h[0] = s.n_owned;
  out_h[1] = s.n_ghost;
  out_h[2] = (long long)s.send_ranks.size();
  out_h[3] = (long long)s.send_idx.size();
  out_h[4] = (long long)s.recv_ranks.size();
  out_h[5] = (long long)s.recv_idx.size();
  out_h[6] = s.n_global;
  PMGX_API_END
}

int pmgx_ghostmesh_space(pmgx_ghostmesh* m, int degree, int32_t* dofmap_h, int8_t* bc_h, long long* l2g_h,
                         double* coords_h)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(m && degree >= 1 && degree <= PMGX_MAX_DEGREE, "ghostmesh_space: bad arguments");
  GSpace& s = m->space(degree);
  if (dofmap_h)
    std::copy(s.dofmap.begin(), s.dofmap.end(), dofmap_h);
  if (bc_h)
    std::copy(s.bc.begin(), s.bc.end(), bc_h);
  if (l2g_h)
    std::copy(s.l2g.begin(), s.l2g.end(), l2g_h);
  if (coords_h)
    std::copy(s.coords.begin(), s.coords.end(), coords_h);
  PMGX_API_END
}

int pmgx_ghostmesh_halo_lists(pmgx_ghostmesh* m, int degree, int* send_ranks_h, int* send_offsets_h,
                              int32_t* send_idx_h, int* recv_ranks_h, int* recv_offsets_h, int32_t* recv_idx_h)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(m && degree >= 1 && degree <= PMGX_MAX_DEGREE, "ghostmesh_halo_lists: bad arguments");
  GSpace& s = m->space(degree);
  if (send_ranks_h)
    std::copy(s.send_ranks.begin(), s.send_ranks.end(), send_ranks_h);
  if (send_offsets_h)
    std::copy(s.send_offsets.begin(), s.send_offsets.end(), send_offsets_h);
  if (send_idx_h)
    std::copy(s.send_idx.begin(), s.send_idx.end(), send_idx_h);
  if (recv_ranks_h)
    std::copy(s.recv_ranks.begin(), s.recv_ranks.end(), recv_ranks_h);
  if (recv_offsets_h)
    std::copy(s.recv_offsets.begin(), s.recv_offsets.end(), recv_offsets_h);
  if (recv_idx_h)
    std::copy(s.recv_idx.begin(), s.recv_idx.end(), recv_idx_h);
  PMGX_API_END
}
}
