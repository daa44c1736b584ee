// objects.cuh -- handle types behind the C ABI and the internal entry points
// each translation unit provides.
#pragma once
#include "collision.cuh"
#include "common.cuh"
#include "item_grid.cuh"
#include "tree.cuh"

struct rrtqx_range_result {
  rrtqx_ctx *ctx = nullptr;
  int64_t n_queries = 0;
  int64_t total = 0;
  bool has_dist = false;
  bool has_lists = false;
  rrtqx::DevBuf<int32_t> counts;
  rrtqx::DevBuf<int64_t> offsets;
  rrtqx::DevBuf<int32_t> idx;
  rrtqx::DevBuf<double> dist;
  // query sort scratch
  rrtqx::DevBuf<int32_t> qkey, qorder, qhist, qstart;
  rrtqx::DevBuf<int32_t> scan_tmp32;
  rrtqx::DevBuf<int64_t> scan_tmp64;
  rrtqx::DevBuf<double> qsorted;             // query coordinates in sorted order (valid when qbins > 0)
  int64_t qbins = 0;                        // bins of the last query sort (0: unsorted / iota order)
  bool qhist_clean = false;                 // qhist is all-zero (left so by the last complete sort)
  rrtqx::DevBuf<double> tq;                  // per-query thresholds T_lt(r_q)
  rrtqx::DevBuf<unsigned long long> cursor;  // fused kernel: [0] output cursor, [1] chunk counter
  // wrap-around trees through the pair kernel: virtual queries (real, ghost) and their per-identity results
  rrtqx::DevBuf<double> vq;
  rrtqx::DevBuf<int32_t> vorder, vcounts;
  rrtqx::DevBuf<int64_t> voffsets;
};

struct rrtqx_edges {
  rrtqx_tree *tree = nullptr;
  int64_t n_edges = 0;
  int64_t n_nodes = 0;  // tree size at upload
  bool has_parent = false;
  bool dirty = false;   // appended edges / parent updates not yet in the CSR
  int64_t n_parent = 0; // entries of parent[] that are initialised
  rrtqx::DevBuf<int32_t> src, dst;            // upload order (edge id = position)
  rrtqx::DevBuf<int32_t> row_ptr, cursor;     // CSR by start node
  rrtqx::DevBuf<int32_t> csr_dst, csr_eid;
  rrtqx::DevBuf<int32_t> parent;
  rrtqx::DevBuf<double> lmax;                 // per node: longest out/parent edge (cull bound)
  rrtqx::DevBuf<uint8_t> degenerate;          // per node: some edge has len == 0 or non-finite ends
  rrtqx::DevBuf<int32_t> scan_tmp;
  // per-item records of the two-stage collision kernels (collide_queue.cuh: ItemRecords), items = out-edges in
  // upload order, then one parent edge per node; rebuilt with the CSR
  rrtqx::DevBuf<float4> item_frec;
  rrtqx::DevBuf<double2> item_exact;
  // the same items sorted by the grid cell of their midpoint: obstacle-centric sweeps / checks (item_grid.cuh)
  rrtqx::ItemGridBufs igrid, igrid1;   // level 0: all items; level 1: the items too long for level 0
  // DubinsEdge trajectories (edge.trajectory[:,1:2]) of the ITEMS = out-edges in upload order, then one parent edge
  // per node: uploaded (traj_ptr / traj_xy) or solved on the device (`solved`); d_traj_* point at whichever is current
  rrtqx::DevBuf<int64_t> traj_ptr;
  rrtqx::DevBuf<double> traj_xy, solve_starts, solve_goals;
  struct rrtqx_dubins_result *solved = nullptr;
  const int64_t *d_traj_ptr = nullptr;
  const double *d_traj_xy = nullptr;
  int64_t traj_items = -1, traj_rows = 0;  // items the resident trajectories were made for (-1: none)
};

struct rrtqx_sweep_result {
  rrtqx_ctx *ctx = nullptr;
  int64_t n_edges = 0, n_nodes = 0;
  int64_t n_edge_hits = 0, n_node_hits = 0, n_candidates = 0, n_pair_tests = 0;
  rrtqx::DevBuf<uint8_t> edge_flag, node_flag;   // byte flags of the call in flight; zero again after sweep_finish
  bool flags_clean = false;                      // flag arrays and statistics are all-zero (left so by sweep_finish)
  rrtqx::DevBuf<int32_t> edge_scan, node_scan, edge_list, node_list, scan_tmp;
  rrtqx::DevBuf<unsigned long long> stats;
  // obstacle table of the sweep
  rrtqx::DevBuf<double4> ob_rec;
  rrtqx::DevBuf<double4> ob_par;  // (thr, thr_le, search_T_lt, search_range)
  rrtqx::DevBuf<double2> ob_thr, ob_ext, ob_thr2, ob_ext2;  // (thr, thr_le) / (T_lt(searchRange), searchRange)
  rrtqx::DevBuf<double4> ob_rec2;
  rrtqx::DevBuf<float4> ob_frec2;  // FP32 reject records of the binned obstacles
  rrtqx::DevBuf<int32_t> cstart;
  rrtqx::DevBuf<unsigned char> grid;
  rrtqx::DevBuf<int32_t> ids_stage, ids_stage2;
  rrtqx::DevBuf<uint8_t> inf_stage;
  rrtqx::DevBuf<unsigned char> filt2d;  // start-node filters of the Otte / Dubins sweeps (sweep2d.cu)
  rrtqx::DevBuf<int32_t> cand2d, cand2d_n;  // items admitted by the start-node filters of a call with few obstacles
};

namespace rrtqx {
// range.cu
void range_query(rrtqx_tree *t, const double *queries, int64_t nq, double r, const double *ranges, uint32_t flags,
                 rrtqx_range_result *res);
void nearest_query(rrtqx_tree *t, rrtqx_range_result *sortbuf, const double *queries, int64_t nq, int32_t *idx_out,
                   double *dist_out, DevBuf<int32_t> &idx_stage, DevBuf<double> &dist_stage);
void extend_query(rrtqx_tree *t, const rrtqx_spheres *S, const double *point, double range, double robot_radius,
                  uint32_t flags, int32_t capacity, int32_t *nearest_idx, double *nearest_dist,
                  uint8_t *point_collides, double *point_cert, int32_t *n_neighbors, int32_t *nbr_idx,
                  double *nbr_dist, uint8_t *fwd_collide, uint8_t *rev_collide);
void extend_query_dubins(rrtqx_tree *t, const rrtqx_polygons *P, double *point, double delta, double range,
                         double robot_radius, double min_turn_radius, uint32_t flags, int32_t capacity,
                         int32_t *nearest_idx, double *nearest_dist, int32_t *n_neighbors, int32_t *nbr_idx,
                         double *nbr_dist, double *edge_dist, int32_t *edge_type, uint8_t *edge_collide,
                         rrtqx_dubins_result **trajectories);
// collision.cu
void edge_check(rrtqx_ctx *ctx, const rrtqx_tree *tree, const rrtqx_spheres *spheres, const int32_t *src,
                const int32_t *dst, const double *starts, const double *ends, int64_t n_edges, double robot_radius,
                uint32_t flags, uint8_t *collide_out);
void edge_check_launch(rrtqx_ctx *ctx, const rrtqx_tree *tree, const rrtqx_spheres *spheres, const int32_t *src,
                       const int32_t *dst, const double *starts, const double *ends, int64_t n_edges,
                       double robot_radius, uint32_t flags, uint8_t *collide_out, const int32_t **bad_dev);
void node_check(rrtqx_ctx *ctx, const rrtqx_spheres *spheres, const double *points, int64_t n, double robot_radius,
                uint32_t flags, uint8_t *collide_out, double *cert_out);
// explicitEdgeCheck(S, edge) of every resident out-edge (collision.cu)
void edges_check(rrtqx_edges *E, const rrtqx_spheres *spheres, double robot_radius, uint32_t flags, uint8_t *collide_out);
// sweep.cu
void edges_upload(rrtqx_edges *E, const int32_t *src, const int32_t *dst, int64_t ne, const int32_t *parent,
                  int64_t n_parent);
void edges_append(rrtqx_edges *E, const int32_t *src, const int32_t *dst, int64_t n_new);
void edges_set_parents(rrtqx_edges *E, const int32_t *nodes, const int32_t *parents, int64_t n);
void edges_rebuild(rrtqx_edges *E);
void obstacle_add_sweep(rrtqx_edges *E, const rrtqx_spheres *S, const int32_t *ob_ids, int64_t n_obs,
                        double robot_radius, double delta, uint32_t flags, rrtqx_sweep_result *R);
void obstacle_remove_sweep(rrtqx_edges *E, const rrtqx_spheres *S, int32_t ob_id, const int32_t *other_ids,
                           int64_t n_others, const uint8_t *edge_dist_inf, double robot_radius, double delta,
                           uint32_t flags, rrtqx_sweep_result *R);
void sweep_prepare_result(rrtqx_edges *E, rrtqx_sweep_result *R);   // zeroed flag arrays for the current edge set
// flags -> ascending id lists + counts (one launch; cleans the flags); *extra_out = the device word *extra_dev
void sweep_finish(rrtqx_ctx *ctx, rrtqx_sweep_result *R, const int32_t *extra_dev = nullptr, int32_t *extra_out = nullptr);
void sweep_result_rebuild_flags(rrtqx_ctx *ctx, rrtqx_sweep_result *R);   // byte flags of the last result, from its lists
// sweep2d.cu
void edges_set_trajectories(rrtqx_edges *E, const int64_t *traj_ptr, const double *traj_xy);
void edges_solve_trajectories(rrtqx_edges *E, double min_turn_radius);
void obstacle_add_sweep_2d(rrtqx_edges *E, const rrtqx_polygons *P, const int32_t *ob_ids, int64_t n_obs,
                           double robot_radius, double delta, double min_turn_radius, uint32_t flags,
                           rrtqx_sweep_result *R);
void obstacle_remove_sweep_2d(rrtqx_edges *E, const rrtqx_polygons *P, int32_t ob_id, const int32_t *other_ids,
                              int64_t n_others, const uint8_t *edge_dist_inf, double robot_radius, double delta,
                              double min_turn_radius, uint32_t flags, rrtqx_sweep_result *R);
}  // namespace rrtqx
