# RRTQXGpu.jl -- Julia FFI module for librrtqx_b200.so (include/rrtqx_b200.h).
#
# Drop-in for the geometric inner loop of RRTQX_3D.  It provides, on top of `ccall`s into the hand-written
# sm_100a library and WITH THE REFERENCE'S ARGUMENT ORDER, the generic functions the planner calls:
#
#   kdInsert(KD, node), kdFindNearest(KD, q), kdFindWithinRange(KD, r, q), kdFindMoreWithinRange(KD, r, q, L)
#                                                                        (kdTree_general.jl:121,357,889,927)
#   explicitEdgeCheck(S, edge), explicitEdgeCheck(S, edge, ob)           (DRRT_Q.jl:1802; DRRT_SimpleEdge_functions.jl:210;
#                                                                         DRRT_DubinsEdge_functions.jl:750)
#   explicitPointCheck(S, p), explicitPointCheck3D, explicitNodeCheck(S, node), explicitNodeCheck3D
#                                                                        (DRRT_Q.jl:1520,1558,1594,1595)
#   findPointsInConflictWithObstacle(S, KD, ob, root)                    (DRRT_Q.jl:3195; DRRT.jl:3048)
#   addNewObstacle(S, KD, Q, ob, root, fileCounter, R)                   (DRRT_Q.jl:3220; DRRT.jl:3127)
#   removeObstacle(S, KD, Q, ob, root, hyberBallRad, timeElapsed, moveGoal)   (DRRT_Q.jl:3295; DRRT.jl:3202)
#   extend(S, KD, Q, newNode, closestNode, delta, hyberBallRad, moveGoal), findBestParent      (julia/extend_gpu.jl)
#
# The device objects that belong to a CSpace (obstacle mirror, resident edge set, the tree) are looked up from `S`
# in a module-level registry, so no call site of the planner changes its arguments:
#
#     include("RRTQXGpu.jl"); using .RRTQXGpu                    # after the reference's own includes
#     ctx = RRTQXGpu.Context(0)
#     KD  = RRTQXGpu.GpuKDTree{RRTNode{Float64}}(ctx, S.d, KDdist) # instead of KDTree{RRTNode{Float64}}(S.d, KDdist)
#     RRTQXGpu.attach!(S, KD)                                      # S -> (ctx, KD, obstacle mirror, edge mirror)
#     RRTQXGpu.install!()                                          # forwards Main's generic functions (see below)
#
# install!() adds methods to the reference's own generic functions in Main.  Those that take the tree dispatch on
# GpuKDTree (more specific than the reference's untyped methods, nothing is replaced); those that only take the
# CSpace (explicitEdgeCheck(S, edge), explicitPointCheck(S, p), ...) REPLACE the reference's methods and route an
# attached S to the GPU.  There is no CPU fallback: an S that was never attached is an error().
#
# popFromRangeList / emptyRangeList (kdTree_general.jl:774-787) are unchanged because the results are rebuilt as
# ordinary JLists with inHeap marks.
#
# NOTE: there is no Julia in the build image of this repository, so this file is written blind against Julia 1.0
# syntax and kept thin; all logic lives behind the C ABI, where it is tested (tests/, via the Python ctypes twin
# rrtqx_3d_b200/_abi.py which binds the same symbols with the same argument order).  julia/make_reference_vectors.jl
# is the script to run on the first machine that has Julia 1.x: it pins the CPU oracle against the real reference.

module RRTQXGpu

export Context, GpuKDTree, GpuObstacles, GpuPolygons, GpuEdges, GpuWorld, attach!, detach!, install!,
       kdInsert, kdInsertBatch, kdFindNearest, kdFindWithinRange, kdFindMoreWithinRange,
       kdFindWithinRangeBatch, kdFindNearestBatch,
       explicitEdgeCheck, explicitEdgeCheckBatch, explicitPointCheck, explicitPointCheck3D,
       explicitNodeCheck, explicitNodeCheck3D,
       findPointsInConflictWithObstacle, addNewObstacle, removeObstacle, syncObstacles!, syncPolygons!, syncEdges!,
       extendQuery, extendQueryMulti, kdInsertMulti, extendQueryDubinsMulti, dubinsEdgesFromQueryMulti!, pinnedVector

const LIB = get(ENV, "RRTQX_B200_LIB", joinpath(@__DIR__, "..", "rrtqx_3d_b200", "librrtqx_b200.so"))

const RANGE_WANT_DIST  = UInt32(1)
const RANGE_COUNT_ONLY = UInt32(2)
const CHECK_FMA_DOT       = UInt32(1)
const CHECK_IGNORE_ACTIVE = UInt32(2)
const CHECK_QUICK_PASS    = UInt32(4)
const EXTEND_SATURATE     = UInt32(8)
const SWEEP_REMOVED_INACTIVE = UInt32(16)

# ------------------------------------------------------------------ context
mutable struct Context
  h::Ptr{Cvoid}
  function Context(device::Integer = 0)
    isfile(LIB) || error("librrtqx_b200.so not found at $(LIB); build it first (no CPU fallback)")
    h = Ref{Ptr{Cvoid}}(C_NULL)
    st = ccall((:rrtqx_ctx_create, LIB), Int32, (Int32, Ptr{Cvoid}, Ref{Ptr{Cvoid}}), device, C_NULL, h)
    st == 0 || error("rrtqx_ctx_create: " * unsafe_string(ccall((:rrtqx_last_error, LIB), Cstring, (Ptr{Cvoid},), C_NULL)))
    c = new(h[])
    finalizer(x -> ccall((:rrtqx_ctx_destroy, LIB), Int32, (Ptr{Cvoid},), x.h), c)
    return c
  end
end

function check(ctx::Context, st::Int32)
  st == 0 && return nothing
  error("rrtqx status $(st): " * unsafe_string(ccall((:rrtqx_last_error, LIB), Cstring, (Ptr{Cvoid},), ctx.h)))
end

# Page-locked host memory (rrtqx_host_alloc): a Vector over pinned memory for arrays that are reused across calls.
# Ordinary Vectors work everywhere too, but the driver stages their copies at a fraction of the PCIe rate.
function pinnedVector(ctx::Context, ::Type{T}, n::Integer) where {T}
  p = Ref{Ptr{Cvoid}}(C_NULL)
  check(ctx, ccall((:rrtqx_host_alloc, LIB), Int32, (Ptr{Cvoid}, Int64, Ref{Ptr{Cvoid}}), ctx.h, Int64(n) * sizeof(T), p))
  v = unsafe_wrap(Array, Ptr{T}(p[]), Int(n))
  finalizer(x -> ccall((:rrtqx_host_free, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}), C_NULL, pointer(x)), v)
  return v
end

# --------------------------------------------------------------------- tree
# T is the node type (RRTNode{Float64}); nodes keep their own kd fields and are owned by Julia.
mutable struct GpuKDTree{T}
  ctx::Context
  h::Ptr{Cvoid}
  d::Int
  distanceFunction::Function      # kept for API compatibility; the device metric is KDdist = euclidianDist
  treeSize::Int
  numWraps::Int
  wraps::Array{Int}
  wrapPoints::Array{Float64}
  root::T
  nodes::Vector{T}                # device index (0-based) + 1 -> node
  index::IdDict{Any,Int32}        # node -> device index (RRTNode has no integer id)
  res::Base.RefValue{Ptr{Cvoid}}  # reusable rrtqx_range_result

  function GpuKDTree{T}(ctx::Context, d::Int, f::Function, wraps::Array{Int} = Int[],
                        wrapPoints::Array{Float64} = Float64[]) where {T}
    h = Ref{Ptr{Cvoid}}(C_NULL)
    w0 = Int32[w - 1 for w in wraps]   # the C ABI uses 0-based dimensions
    check(ctx, ccall((:rrtqx_tree_create, LIB), Int32,
                     (Ptr{Cvoid}, Int32, Int32, Ptr{Int32}, Ptr{Float64}, Ref{Ptr{Cvoid}}),
                     ctx.h, d, length(w0), w0, wrapPoints, h))
    t = new{T}(ctx, h[], d, f, 0, length(wraps), wraps, wrapPoints)
    t.nodes = Vector{T}()
    t.index = IdDict{Any,Int32}()
    t.res = Ref{Ptr{Cvoid}}(C_NULL)
    finalizer(t) do x
      x.res[] != C_NULL && ccall((:rrtqx_range_result_destroy, LIB), Int32, (Ptr{Cvoid},), x.res[])
      ccall((:rrtqx_tree_destroy, LIB), Int32, (Ptr{Cvoid},), x.h)
    end
    return t
  end
end

# keeps kdParent / kdChildL / kdChildR / kdSplit of the Julia nodes populated (saveRRTTree etc. walk them)
function refreshKdFields!(tree::GpuKDTree, first::Int, count::Int)
  parent = Vector{Int32}(undef, count); cl = similar(parent); cr = similar(parent); sp = similar(parent)
  check(tree.ctx, ccall((:rrtqx_tree_kd_fields, LIB), Int32,
                        (Ptr{Cvoid}, Int64, Int64, Ptr{Int32}, Ptr{Int32}, Ptr{Int32}, Ptr{Int32}),
                        tree.h, first, count, parent, cl, cr, sp))
  for k = 1:count
    n = tree.nodes[first + k]
    n.kdSplit = sp[k] + 1
    if parent[k] >= 0
      p = tree.nodes[parent[k] + 1]
      n.kdParent = p
      n.kdParentExist = true
      if n.position[p.kdSplit] < p.position[p.kdSplit]
        p.kdChildL = n; p.kdChildLExist = true
      else
        p.kdChildR = n; p.kdChildRExist = true
      end
    end
  end
end

# kdInsert (kdTree_general.jl:121-170)
function kdInsert(tree::GpuKDTree{T}, node::T) where {T}
  node.kdInTree && return
  node.kdInTree = true
  idx = Ref{Int32}(0)
  pos = vec(Array{Float64}(node.position))
  GC.@preserve pos check(tree.ctx, ccall((:rrtqx_tree_insert, LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ref{Int32}),
                                         tree.h, pos, idx))
  push!(tree.nodes, node)
  tree.index[node] = idx[]
  if tree.treeSize == 0
    tree.root = node
  end
  tree.treeSize += 1
  refreshKdFields!(tree, Int(idx[]), 1)
  return
end

# kdInsert(trees[i], nodes[i]) for every i in ONE launch (multirrtqx's agents in lock-step): the trees are distinct
# and of one context; each keeps nodes / index / root / treeSize and the kd fields exactly as kdInsert does
function kdInsertMulti(trees::Vector, nodes::Vector)
  keep = [i for i = 1:length(trees) if !nodes[i].kdInTree]
  isempty(keep) && return
  ts = trees[keep]; ns = nodes[keep]
  handles = Ptr{Cvoid}[t.h for t in ts]
  pos = Matrix{Float64}(undef, ts[1].d, length(ns))      # column-major d x n == row-major n x d for C
  for (k, n) in enumerate(ns); pos[:, k] = vec(n.position); end
  idx = Vector{Int32}(undef, length(ns))
  GC.@preserve handles pos idx check(ts[1].ctx, ccall((:rrtqx_tree_insert_multi, LIB), Int32,
      (Ptr{Ptr{Cvoid}}, Int32, Ptr{Float64}, Ptr{Int32}), handles, length(ns), pos, idx))
  for k = 1:length(ns)
    t = ts[k]; n = ns[k]
    n.kdInTree = true
    push!(t.nodes, n)
    t.index[n] = idx[k]
    if t.treeSize == 0
      t.root = n
    end
    t.treeSize += 1
    refreshKdFields!(t, Int(idx[k]), 1)
  end
  return
end

function kdInsertBatch(tree::GpuKDTree{T}, nodes::Vector{T}) where {T}
  new = [n for n in nodes if !n.kdInTree]
  isempty(new) && return
  pos = Matrix{Float64}(undef, tree.d, length(new))       # column-major d x n == row-major n x d for C
  for (k, n) in enumerate(new); pos[:, k] = vec(n.position); end
  first = Ref{Int32}(0)
  GC.@preserve pos check(tree.ctx, ccall((:rrtqx_tree_insert_batch, LIB), Int32,
                                         (Ptr{Cvoid}, Ptr{Float64}, Int64, Ref{Int32}), tree.h, pos, length(new), first))
  for (k, n) in enumerate(new)
    n.kdInTree = true
    push!(tree.nodes, n)
    tree.index[n] = first[] + Int32(k - 1)
  end
  if tree.treeSize == 0
    tree.root = new[1]
  end
  tree.treeSize += length(new)
  refreshKdFields!(tree, Int(first[]), length(new))
  return
end

# kdFindNearest (kdTree_general.jl:357-385) -> (node, dist)
function kdFindNearest(tree::GpuKDTree, queryPoint::Array{Float64})
  tree.treeSize == 0 && error("kdFindNearest on an empty tree")
  q = vec(Array{Float64}(queryPoint)); idx = Vector{Int32}(undef, 1); dist = Vector{Float64}(undef, 1)
  GC.@preserve q idx dist check(tree.ctx, ccall((:rrtqx_nearest_batch, LIB), Int32,
      (Ptr{Cvoid}, Ptr{Float64}, Int64, Ptr{Int32}, Ptr{Float64}), tree.h, q, 1, idx, dist))
  return (tree.nodes[idx[1] + 1], dist[1])
end

function kdFindNearestBatch(tree::GpuKDTree, queries::Matrix{Float64})   # d x nq (column per query)
  nq = size(queries, 2); idx = Vector{Int32}(undef, nq); dist = Vector{Float64}(undef, nq)
  GC.@preserve queries idx dist check(tree.ctx, ccall((:rrtqx_nearest_batch, LIB), Int32,
      (Ptr{Cvoid}, Ptr{Float64}, Int64, Ptr{Int32}, Ptr{Float64}), tree.h, queries, nq, idx, dist))
  return (idx .+ Int32(1), dist)
end

# batched range query -> (counts, offsets (1-based starts), idx (1-based), dist)
function kdFindWithinRangeBatch(tree::GpuKDTree, range::Float64, queries::Matrix{Float64};
                                ranges::Union{Nothing,Vector{Float64}} = nothing, wantDist::Bool = true)
  nq = size(queries, 2); total = Ref{Int64}(0)
  flags = wantDist ? RANGE_WANT_DIST : UInt32(0)
  rp = ranges === nothing ? Ptr{Float64}(C_NULL) : pointer(ranges)
  GC.@preserve queries ranges check(tree.ctx, ccall((:rrtqx_range_query_batch, LIB), Int32,
      (Ptr{Cvoid}, Ptr{Float64}, Int64, Float64, Ptr{Float64}, UInt32, Ref{Ptr{Cvoid}}, Ref{Int64}),
      tree.h, queries, nq, range, rp, flags, tree.res, total))
  counts = Vector{Int32}(undef, nq); offsets = Vector{Int64}(undef, nq)
  idx = Vector{Int32}(undef, total[]); dist = Vector{Float64}(undef, wantDist ? total[] : 0)
  GC.@preserve counts offsets idx dist begin
    check(tree.ctx, ccall((:rrtqx_range_result_layout, LIB), Int32, (Ptr{Cvoid}, Ptr{Int32}, Ptr{Int64}),
                          tree.res[], counts, offsets))
    check(tree.ctx, ccall((:rrtqx_range_result_fetch, LIB), Int32, (Ptr{Cvoid}, Ptr{Int32}, Ptr{Float64}),
                          tree.res[], idx, wantDist ? pointer(dist) : Ptr{Float64}(C_NULL)))
  end
  return (counts, offsets .+ 1, idx .+ Int32(1), dist)
end

# addToRangeList (kdTree_general.jl:765-771) is reused from the reference: it dedups through inHeap.
# kdFindMoreWithinRange (kdTree_general.jl:927-955)
function kdFindMoreWithinRange(tree::GpuKDTree, range::Float64, queryPoint::Array{Float64}, L)
  tree.treeSize == 0 && error("kdFindWithinRange on an empty tree")
  q = reshape(vec(Array{Float64}(queryPoint)), tree.d, 1)
  (counts, offsets, idx, dist) = kdFindWithinRangeBatch(tree, range, q)
  for k = 1:counts[1]
    Main.addToRangeList(L, tree.nodes[idx[offsets[1] + k - 1]], dist[offsets[1] + k - 1])
  end
  return L
end

# kdFindWithinRange (kdTree_general.jl:889-919)
function kdFindWithinRange(tree::GpuKDTree{T}, range::Float64, queryPoint::Array{Float64}) where {T}
  return kdFindMoreWithinRange(tree, range, queryPoint, Main.JList{T}())
end

# ---------------------------------------------------------------- obstacles
# device mirror of S.obstacles (List{SphereObstacle}), front-to-back order
mutable struct GpuObstacles
  ctx::Context
  h::Ptr{Cvoid}
  ids::IdDict{Any,Int32}          # obstacle -> device index
  radii::Vector{Float64}          # what the device holds (change detection)
  active::Vector{UInt8}
  function GpuObstacles(ctx::Context)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ctx, ccall((:rrtqx_spheres_create, LIB), Int32, (Ptr{Cvoid}, Ref{Ptr{Cvoid}}), ctx.h, h))
    o = new(ctx, h[], IdDict{Any,Int32}(), Float64[], UInt8[])
    finalizer(x -> ccall((:rrtqx_spheres_destroy, LIB), Int32, (Ptr{Cvoid},), x.h), o)
    return o
  end
end

# active[i] = !(obstacleUnused || lifeSpan <= 0): the early-out of explicitEdgeCheck3D (DRRT_Q.jl:1777).
# The obstacle list only grows and only radii / flags change in place (rrtqx.jl:462-530, obstacleAugmentation.jl),
# so an unchanged list costs one walk and no upload; a grown list is re-uploaded, changed radii / flags are patched.
function syncObstacles!(G::GpuObstacles, S)
  n = S.obstacles.length
  radii = Vector{Float64}(undef, n); active = Vector{UInt8}(undef, n)
  obs = Vector{Any}(undef, n)
  item = S.obstacles.front
  for i = 1:n
    ob = item.data
    obs[i] = ob
    radii[i] = ob.radius
    active[i] = (ob.obstacleUnused || ob.lifeSpan <= 0) ? 0x00 : 0x01
    item = item.child
  end
  same = n == length(G.radii)
  if same
    for i = 1:n
      if !haskey(G.ids, obs[i]) || G.ids[obs[i]] != Int32(i - 1)
        same = false
        break
      end
    end
  end
  if !same                                     # new / reordered list: full upload
    centers = Matrix{Float64}(undef, 3, n)
    empty!(G.ids)
    for i = 1:n
      centers[:, i] = obs[i].position[1:3]
      G.ids[obs[i]] = Int32(i - 1)
    end
    GC.@preserve centers radii active check(G.ctx, ccall((:rrtqx_spheres_upload, LIB), Int32,
        (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{UInt8}, Int64), G.h, centers, radii, active, n))
  elseif radii != G.radii || active != G.active  # in-place update of radius / flags
    GC.@preserve radii active check(G.ctx, ccall((:rrtqx_spheres_update, LIB), Int32,
        (Ptr{Cvoid}, Int64, Int64, Ptr{Float64}, Ptr{UInt8}), G.h, 0, n, radii, active))
  end
  G.radii = radii; G.active = active
  return G
end

# ------------------------------------------------------------------ polygons (Otte generation, DubinsEdge)
mutable struct GpuPolygons
  ctx::Context
  h::Ptr{Cvoid}
  ids::IdDict{Any,Int32}
  function GpuPolygons(ctx::Context)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ctx, ccall((:rrtqx_polygons_create, LIB), Int32, (Ptr{Cvoid}, Ref{Ptr{Cvoid}}), ctx.h, h))
    o = new(ctx, h[], IdDict{Any,Int32}())
    finalizer(x -> ccall((:rrtqx_polygons_destroy, LIB), Int32, (Ptr{Cvoid},), x.h), o)
    return o
  end
end

# Mirrors S.obstacles (Obstacle kinds 1 and 3, DRRT_data_structures.jl:135-265): bounding circles as the
# constructor computed them (ob.position, ob.radius), polygon vertices as a CSR.
function syncPolygons!(G::GpuPolygons, S)
  kinds = Int32[]; centers = Float64[]; radii = Float64[]; active = UInt8[]; vptr = Int64[0]; verts = Float64[]
  empty!(G.ids)
  item = S.obstacles.front
  for i = 1:S.obstacles.length
    ob = item.data
    G.ids[ob] = Int32(i - 1)
    push!(kinds, Int32(ob.kind)); push!(centers, ob.position[1], ob.position[2]); push!(radii, ob.radius)
    push!(active, (ob.obstacleUnused || ob.lifeSpan <= 0) ? 0x00 : 0x01)
    if ob.kind == 3
      for r = 1:size(ob.polygon, 1)
        push!(verts, ob.polygon[r, 1], ob.polygon[r, 2])
      end
    end
    push!(vptr, length(verts) ÷ 2)
    item = item.child
  end
  GC.@preserve kinds centers radii active vptr verts check(G.ctx, ccall((:rrtqx_polygons_upload, LIB), Int32,
      (Ptr{Cvoid}, Ptr{Int32}, Ptr{Float64}, Ptr{Float64}, Ptr{UInt8}, Ptr{Int64}, Ptr{Float64}, Int64),
      G.h, kinds, centers, radii, active, vptr, verts, length(kinds)))
  return G
end

# -------------------------------------------------------------- resident edge set
mutable struct GpuEdges
  tree::GpuKDTree
  h::Ptr{Cvoid}
  items::Vector{Any}              # edge id + 1 -> JListNode holding the edge
  res::Base.RefValue{Ptr{Cvoid}}
  function GpuEdges(tree::GpuKDTree)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(tree.ctx, ccall((:rrtqx_edges_create, LIB), Int32, (Ptr{Cvoid}, Ref{Ptr{Cvoid}}), tree.h, h))
    e = new(tree, h[], Vector{Any}(), Ref{Ptr{Cvoid}}(C_NULL))
    finalizer(e) do x
      x.res[] != C_NULL && ccall((:rrtqx_sweep_result_destroy, LIB), Int32, (Ptr{Cvoid},), x.res[])
      ccall((:rrtqx_edges_destroy, LIB), Int32, (Ptr{Cvoid},), x.h)
    end
    return e
  end
end

# mirrors every node's out-edges in the order of RRTNodeNeighborIterator (DRRT_Q.jl:2408-2431):
# InitialNeighborListOut, then rrtNeighborsOut; plus the parent edges.  With withTrajectories (DubinsEdge) the
# planner's own edge.trajectory rows are uploaded too (items = out-edges, then one parent edge per node), so the
# Dubins sweeps decide on exactly the points the reference would test.
function syncEdges!(E::GpuEdges; withTrajectories::Bool = false)
  tree = E.tree
  src = Int32[]; dst = Int32[]; empty!(E.items)
  nn = length(tree.nodes)
  parent = fill(Int32(-1), nn)
  for n in tree.nodes
    for lst in (n.InitialNeighborListOut, n.rrtNeighborsOut)
      item = lst.front
      for k = 1:lst.length
        push!(src, tree.index[n]); push!(dst, tree.index[item.data.endNode]); push!(E.items, item)
        item = item.child
      end
    end
    if n.rrtParentUsed
      parent[tree.index[n] + 1] = tree.index[n.rrtParentEdge.endNode]
    end
  end
  GC.@preserve src dst parent check(tree.ctx, ccall((:rrtqx_edges_upload, LIB), Int32,
      (Ptr{Cvoid}, Ptr{Int32}, Ptr{Int32}, Int64, Ptr{Int32}, Int64), E.h, src, dst, length(src), parent, length(parent)))
  if withTrajectories
    ne = length(src)
    ptr = Vector{Int64}(undef, ne + nn + 1); ptr[1] = 0
    for (i, it) in enumerate(E.items)
      ptr[i + 1] = ptr[i] + size(it.data.trajectory, 1)
    end
    for (v, n) in enumerate(tree.nodes)
      ptr[ne + v + 1] = ptr[ne + v] + (n.rrtParentUsed ? size(n.rrtParentEdge.trajectory, 1) : 0)
    end
    xy = Matrix{Float64}(undef, 2, ptr[ne + nn + 1])
    for (i, it) in enumerate(E.items)
      xy[:, ptr[i]+1:ptr[i+1]] = permutedims(it.data.trajectory[:, 1:2])
    end
    for (v, n) in enumerate(tree.nodes)
      if n.rrtParentUsed
        xy[:, ptr[ne+v]+1:ptr[ne+v+1]] = permutedims(n.rrtParentEdge.trajectory[:, 1:2])
      end
    end
    GC.@preserve ptr xy check(tree.ctx, ccall((:rrtqx_edges_set_trajectories, LIB), Int32,
        (Ptr{Cvoid}, Ptr{Int64}, Ptr{Float64}), E.h, ptr, xy))
  end
  return E
end

function fetchSweep(E::GpuEdges)
  ne = Ref{Int64}(0); nn = Ref{Int64}(0)
  check(E.tree.ctx, ccall((:rrtqx_sweep_result_sizes, LIB), Int32,
                          (Ptr{Cvoid}, Ref{Int64}, Ref{Int64}, Ptr{Int64}, Ptr{Int64}), E.res[], ne, nn, C_NULL, C_NULL))
  edges = Vector{Int32}(undef, ne[]); nodes = Vector{Int32}(undef, nn[])
  GC.@preserve edges nodes check(E.tree.ctx, ccall((:rrtqx_sweep_result_fetch, LIB), Int32,
                                                   (Ptr{Cvoid}, Ptr{Int32}, Ptr{Int32}), E.res[], edges, nodes))
  return (edges, nodes)
end

# ------------------------------------------------------------------ neighbour-graph residency
# Edges the planner creates in one iteration (makeNeighborOf / makeInitialOutNeighborOf,
# DRRT_Q.jl:2589-2593) are appended to the resident set instead of re-uploading the graph; parent
# edges are re-pointed in place (makeParentOf, DRRT_Q.jl:1841-1856).  `srcIdx`/`dstIdx` are 0-based
# device node indices (KD.index[node]); edge ids continue the order of E.items.
function appendEdges!(E::GpuEdges, newEdges::Vector, srcIdx::Vector{Int32}, dstIdx::Vector{Int32})
  append!(E.items, newEdges)
  GC.@preserve srcIdx dstIdx check(E.tree.ctx, ccall((:rrtqx_edges_append, LIB), Int32,
      (Ptr{Cvoid}, Ptr{Int32}, Ptr{Int32}, Int64), E.h, srcIdx, dstIdx, length(srcIdx)))
end

function setParents!(E::GpuEdges, nodeIdx::Vector{Int32}, parentIdx::Vector{Int32})   # parent -1: rrtParentUsed = false
  GC.@preserve nodeIdx parentIdx check(E.tree.ctx, ccall((:rrtqx_edges_set_parents, LIB), Int32,
      (Ptr{Cvoid}, Ptr{Int32}, Ptr{Int32}, Int64), E.h, nodeIdx, parentIdx, length(nodeIdx)))
end

# ------------------------------------------------------------------ CSpace -> device objects
# Everything the reference-order entry points need is found from `S`: the planner's call sites keep their
# arguments (explicitEdgeCheck(S, edge), addNewObstacle(S, KD, Q, ob, root, fileCounter, R), ...).
mutable struct GpuWorld
  ctx::Context
  KD::GpuKDTree
  spheres::GpuObstacles           # mirror of S.obstacles when they are SphereObstacles (QX-3D generation)
  polygons::GpuPolygons           # mirror of S.obstacles when they are Obstacles (Otte generation, DubinsEdge)
  edges::GpuEdges                 # resident out-edge lists + parents
  edgesStale::Bool                # the graph changed since the last syncEdges!
  single::GpuObstacles            # one-obstacle set for explicitEdgeCheck(S, edge, ob)
  pinned::Dict{Symbol,Any}        # pinned scratch arrays reused across calls (extendQuery)
end

const WORLDS = IdDict{Any,GpuWorld}()

function attach!(S, KD::GpuKDTree)
  W = GpuWorld(KD.ctx, KD, GpuObstacles(KD.ctx), GpuPolygons(KD.ctx), GpuEdges(KD), true, GpuObstacles(KD.ctx),
               Dict{Symbol,Any}())
  WORLDS[S] = W
  return W
end
detach!(S) = delete!(WORLDS, S)
function world(S)
  haskey(WORLDS, S) || error("this CSpace is not attached to a GPU context: RRTQXGpu.attach!(S, KD) first (there is no CPU fallback)")
  return WORLDS[S]
end
# the planner tells the mirror that neighbour lists / parents changed (extend_gpu.jl does it for its own edits);
# the next sweep re-syncs
markEdgesStale!(S) = (world(S).edgesStale = true; nothing)

isPolygonWorld(S) = S.obstacles.length > 0 && (:polygon in fieldnames(typeof(S.obstacles.front.data)))
isDubinsEdge(edge) = :trajectory in fieldnames(typeof(edge))

# ------------------------------------------------------------------ collision checks, reference order
# explicitEdgeCheck(S, edge) (DRRT_Q.jl:1802-1826 / DRRT.jl:1660-1678): OR over the obstacle list
function explicitEdgeCheck(S, edge)
  S.inWarmupTime && return false
  W = world(S)
  if isDubinsEdge(edge)
    syncPolygons!(W.polygons, S)
    return explicitEdgeCheckBatch(W.polygons, S, Any[edge])[1]
  end
  syncObstacles!(W.spheres, S)
  return segmentCheck(W.spheres, S, edge)
end

# explicitEdgeCheck(S, edge, ob): ONE obstacle (DRRT_SimpleEdge_functions.jl:210 -> explicitEdgeCheck3D
# DRRT_Q.jl:1775; DRRT_DubinsEdge_functions.jl:750).  No warm-up short-circuit here, as in the reference.
function explicitEdgeCheck(S, edge, ob)
  W = world(S)
  if isDubinsEdge(edge)
    one = GpuPolygons(W.ctx)
    kinds = Int32[ob.kind]; centers = Float64[ob.position[1], ob.position[2]]; radii = Float64[ob.radius]
    active = UInt8[(ob.obstacleUnused || ob.lifeSpan <= 0) ? 0x00 : 0x01]
    verts = Float64[]
    if ob.kind == 3
      for r = 1:size(ob.polygon, 1)
        push!(verts, ob.polygon[r, 1], ob.polygon[r, 2])
      end
    end
    vptr = Int64[0, length(verts) ÷ 2]
    GC.@preserve kinds centers radii active vptr verts check(W.ctx, ccall((:rrtqx_polygons_upload, LIB), Int32,
        (Ptr{Cvoid}, Ptr{Int32}, Ptr{Float64}, Ptr{Float64}, Ptr{UInt8}, Ptr{Int64}, Ptr{Float64}, Int64),
        one.h, kinds, centers, radii, active, vptr, verts, 1))
    return dubinsCheck(one, S, Any[edge])[1]
  end
  c = Array{Float64}(vec(ob.position)[1:3]); r = Float64[ob.radius]
  a = UInt8[(ob.obstacleUnused || ob.lifeSpan <= 0) ? 0x00 : 0x01]
  GC.@preserve c r a check(W.ctx, ccall((:rrtqx_spheres_upload, LIB), Int32,
      (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{UInt8}, Int64), W.single.h, c, r, a, 1))
  return segmentCheck(W.single, S, edge)
end

function segmentCheck(G::GpuObstacles, S, edge, flags::UInt32 = UInt32(0))
  s = vec(Array{Float64}(edge.startNode.position))[1:3]; e = vec(Array{Float64}(edge.endNode.position))[1:3]
  out = Vector{UInt8}(undef, 1)
  GC.@preserve s e out check(G.ctx, ccall((:rrtqx_segment_check_batch, LIB), Int32,
      (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Float64, UInt32, Ptr{UInt8}),
      G.ctx.h, G.h, s, e, 1, S.robotRadius, flags, out))
  return out[1] != 0x00
end

# batched explicitEdgeCheck over edges between tree nodes given as 1-based index vectors (SimpleEdge)
function explicitEdgeCheckBatch(S, tree::GpuKDTree, src::Vector{Int32}, dst::Vector{Int32}, flags::UInt32 = UInt32(0))
  out = Vector{UInt8}(undef, length(src))
  S.inWarmupTime && return fill!(out, 0x00)
  G = syncObstacles!(world(S).spheres, S)
  s0 = src .- Int32(1); d0 = dst .- Int32(1)
  GC.@preserve s0 d0 out check(G.ctx, ccall((:rrtqx_edge_check_batch, LIB), Int32,
      (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Int32}, Ptr{Int32}, Int64, Float64, UInt32, Ptr{UInt8}),
      tree.h, G.h, s0, d0, length(src), S.robotRadius, flags, out))
  return out
end

function pointCheck(S, point::Array{Float64}, flags::UInt32)
  S.inWarmupTime && return (false, Inf)
  G = syncObstacles!(world(S).spheres, S)
  p = vec(Array{Float64}(point))[1:3]; out = Vector{UInt8}(undef, 1); cert = Vector{Float64}(undef, 1)
  GC.@preserve p out cert check(G.ctx, ccall((:rrtqx_node_check_batch, LIB), Int32,
      (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}, Int64, Float64, UInt32, Ptr{UInt8}, Ptr{Float64}),
      G.ctx.h, G.h, p, 1, S.robotRadius, flags, out, cert))
  return (out[1] != 0x00, cert[1])
end
explicitPointCheck(S, point::Array{Float64}) = pointCheck(S, point, CHECK_QUICK_PASS)   # DRRT_Q.jl:1520
explicitPointCheck3D(S, point::Array{Float64}) = pointCheck(S, point, UInt32(0))        # DRRT_Q.jl:1558
explicitNodeCheck(S, node) = explicitPointCheck(S, node.position)                       # DRRT_Q.jl:1594
explicitNodeCheck3D(S, node) = explicitPointCheck3D(S, node.position)                   # DRRT_Q.jl:1595

# ------------------------------------------------------------------ obstacle sweeps, reference order
# findPointsInConflictWithObstacle (DRRT_Q.jl:3195-3215; Otte DRRT.jl:3048-3064), spaces without time
function findPointsInConflictWithObstacle(S, KD::GpuKDTree, ob, root)
  S.spaceHasTime && error("this type of obstacle not coded for this type of space")
  if !S.spaceHasTheta
    searchRange = S.robotRadius + S.delta + ob.radius
    return kdFindWithinRange(KD, searchRange, Array{Float64}(ob.position))
  end
  searchRange = S.robotRadius + S.delta + ob.radius + pi          # Dubins robot without time, [x y 0.0 theta]
  obsCenterDubins = Float64[ob.position[1] ob.position[2] 0.0 pi]
  return kdFindWithinRange(KD, searchRange, obsCenterDubins)
end

function ensureEdges!(W::GpuWorld, withTrajectories::Bool)
  if W.edgesStale
    syncEdges!(W.edges; withTrajectories = withTrajectories)
    W.edgesStale = false
  end
  return W.edges
end

# addNewObstacle (DRRT_Q.jl:3220-3290; Otte DRRT.jl:3127-3197): the GPU returns the blocked edge ids and the
# orphaned node ids, the reference's list surgery is applied here unchanged.
function addNewObstacle(S, KD::GpuKDTree, Q, ob, root, fileCounter::Int, R)
  W = world(S)
  ob.obstacleUnused = false
  poly = isPolygonWorld(S)
  E = ensureEdges!(W, poly)
  if ob.lifeSpan > 0
    if poly
      syncPolygons!(W.polygons, S)
      ids = Int32[W.polygons.ids[ob]]
      GC.@preserve ids check(KD.ctx, ccall((:rrtqx_obstacle_add_sweep_2d, LIB), Int32,
          (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Int32}, Int64, Float64, Float64, Float64, UInt32, Ref{Ptr{Cvoid}}),
          E.h, W.polygons.h, ids, 1, S.robotRadius, S.delta, S.minTurningRadius, UInt32(0), E.res))
    else
      syncObstacles!(W.spheres, S)
      ids = Int32[W.spheres.ids[ob]]
      GC.@preserve ids check(KD.ctx, ccall((:rrtqx_obstacle_add_sweep, LIB), Int32,
          (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Int32}, Int64, Float64, Float64, UInt32, Ref{Ptr{Cvoid}}),
          E.h, W.spheres.h, ids, 1, S.robotRadius, S.delta, UInt32(0), E.res))
    end
    (blocked, orphans) = fetchSweep(E)
    for e in blocked
      E.items[e + 1].data.dist = Inf                                   # :3248-3249
    end
    for v in orphans                                                   # :3257-3270
      thisNode = KD.nodes[v + 1]
      Main.JlistRemove(thisNode.rrtParentEdge.endNode.SuccessorList, thisNode.successorListItemInParent)
      thisNode.rrtParentEdge.endNode = thisNode
      thisNode.rrtParentEdge.dist = Inf
      thisNode.rrtParentUsed = false
      Main.verifyInOSQueue(Q, thisNode)
    end
    if length(orphans) > 0
      idx = Int32[v for v in orphans]
      setParents!(E, idx, fill(Int32(-1), length(idx)))                # keep the resident parents in step
    end
  end
  if R.robotEdgeUsed && explicitEdgeCheck(S, R.robotEdge, ob)          # :3287-3289 (per-obstacle form: no warm-up test)
    R.currentMoveInvalid = true
  end
end

# removeObstacle.  SphereObstacle worlds follow this fork (DRRT_Q.jl:3295-3362: the obstacle is disabled BEFORE the
# loop, so nothing is ever restored -- reproduced by RRTQX_SWEEP_REMOVED_INACTIVE); Obstacle worlds follow the
# Otte generation (DRRT.jl:3202-3268: still active while tested).  qxSemantics overrides the choice.
function removeObstacle(S, KD::GpuKDTree, Q, ob, root, hyberBallRad::Float64, timeElapsed::Float64, moveGoal;
                        qxSemantics::Union{Nothing,Bool} = nothing)
  W = world(S)
  poly = isPolygonWorld(S)
  qx = qxSemantics === nothing ? !poly : qxSemantics
  E = ensureEdges!(W, poly)
  ids = poly ? syncPolygons!(W.polygons, S).ids : syncObstacles!(W.spheres, S).ids
  obId = ids[ob]
  if qx
    ob.expired = true
    ob.obstacleUnused = true                                           # DRRT_Q.jl:3301-3302
  end
  others = Int32[]
  item = S.obstacles.front
  for i = 1:S.obstacles.length
    o = item.data
    if o != ob && !o.obstacleUnused && o.lifeSpan > 0 && o.startTime <= timeElapsed <= (o.startTime + o.lifeSpan)
      push!(others, ids[o])
    end
    item = item.child
  end
  inf = UInt8[(it.data.dist == Inf) ? 0x01 : 0x00 for it in E.items]
  if poly
    GC.@preserve others inf check(KD.ctx, ccall((:rrtqx_obstacle_remove_sweep_2d, LIB), Int32,
        (Ptr{Cvoid}, Ptr{Cvoid}, Int32, Ptr{Int32}, Int64, Ptr{UInt8}, Float64, Float64, Float64, UInt32, Ref{Ptr{Cvoid}}),
        E.h, W.polygons.h, obId, others, length(others), inf, S.robotRadius, S.delta, S.minTurningRadius, UInt32(0), E.res))
  else
    flags = qx ? SWEEP_REMOVED_INACTIVE : UInt32(0)
    GC.@preserve others inf check(KD.ctx, ccall((:rrtqx_obstacle_remove_sweep, LIB), Int32,
        (Ptr{Cvoid}, Ptr{Cvoid}, Int32, Ptr{Int32}, Int64, Ptr{UInt8}, Float64, Float64, UInt32, Ref{Ptr{Cvoid}}),
        E.h, W.spheres.h, obId, others, length(others), inf, S.robotRadius, S.delta, flags, E.res))
  end
  (restored, requeue) = fetchSweep(E)
  for e in restored
    E.items[e + 1].data.dist = E.items[e + 1].data.distOriginal        # :3340-3346
  end
  for v in requeue                                                     # :3352-3357
    thisNode = KD.nodes[v + 1]
    Main.recalculateLMCMineVTwo(Q, thisNode, root, hyberBallRad)
    if thisNode.rrtTreeCost != thisNode.rrtLMC && Main.lessQ(thisNode, moveGoal)
      Main.verifyInQueue(Q, thisNode)
    end
  end
  ob.obstacleUnused = true
end

# ------------------------------------------------------------------ fused per-iteration query
# One launch for what extend() asks of the geometry per sample (rrtqx.jl:926-950, DRRT_Q.jl:2551-2637):
# nearest node, explicitNodeCheck of the sample, the shrinking-ball neighbours with their keys, and
# explicitEdgeCheck of every new edge in both directions.  Result arrays are pinned and reused across calls; the
# returned views are valid until the next extendQuery on the same CSpace.  julia/extend_gpu.jl is the consumer.
function extendQuery(S, tree::GpuKDTree, point::Array{Float64}, range::Float64; capacity::Int = 8192)
  W = world(S)
  G = syncObstacles!(W.spheres, S)
  if !haskey(W.pinned, :idx) || length(W.pinned[:idx]) < capacity
    W.pinned[:idx] = pinnedVector(W.ctx, Int32, capacity); W.pinned[:dist] = pinnedVector(W.ctx, Float64, capacity)
    W.pinned[:fwd] = pinnedVector(W.ctx, UInt8, capacity); W.pinned[:rev] = pinnedVector(W.ctx, UInt8, capacity)
  end
  idx = W.pinned[:idx]::Vector{Int32}; dist = W.pinned[:dist]::Vector{Float64}
  fwd = W.pinned[:fwd]::Vector{UInt8}; rev = W.pinned[:rev]::Vector{UInt8}
  nearestIdx = Ref{Int32}(0); nearestDist = Ref{Float64}(0.0)
  collides = Ref{UInt8}(0); cert = Ref{Float64}(0.0); n = Ref{Int32}(0)
  p = vec(Array{Float64}(point))
  GC.@preserve p idx dist fwd rev check(tree.ctx, ccall((:rrtqx_extend_query, LIB), Int32,
      (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}, Float64, Float64, UInt32, Int32, Ref{Int32}, Ref{Float64}, Ref{UInt8},
       Ref{Float64}, Ref{Int32}, Ptr{Int32}, Ptr{Float64}, Ptr{UInt8}, Ptr{UInt8}),
      tree.h, G.h, p, range, S.robotRadius, CHECK_QUICK_PASS, Int32(length(idx)), nearestIdx, nearestDist, collides, cert, n,
      idx, dist, fwd, rev))
  n[] <= length(idx) || return extendQuery(S, tree, point, range; capacity = 2 * Int(n[]))   # grow and repeat (rare)
  k = min(Int(n[]), length(idx))            # never slice past the buffers
  warm = S.inWarmupTime                     # obstacles are ignored during warm-up (DRRT_Q.jl:1805-1807, 1523-1525)
  return (tree.nodes[nearestIdx[] + 1], nearestDist[], warm ? false : collides[] != 0, warm ? Inf : cert[],
          view(idx, 1:k), view(dist, 1:k), warm ? falses(k) : view(fwd, 1:k) .!= 0, warm ? falses(k) : view(rev, 1:k) .!= 0)
end

# extendQuery for many planners in lock-step (multirrtqx's agents, rrtqx.jl:331,915): agent i is (Ss[i], trees[i],
# points[i], ranges[i]), each with its own CSpace and tree.  One launch and one host wait serve the whole round; each
# agent gets the tuple extendQuery returns, warm-up handling included.  The views stay valid until the next
# extendQueryMulti on the same first CSpace.  An agent whose ball holds more than `capacity` nodes is repeated alone
# with extendQuery (rare).  The agents share one robot radius (the C call takes one).
function extendQueryMulti(Ss::Vector, trees::Vector, points::Vector, ranges::Vector{Float64}; capacity::Int = 8192)
  n = length(trees)
  n == 0 && return Any[]
  rho = Ss[1].robotRadius
  all(S -> S.robotRadius == rho, Ss) || error("extendQueryMulti: the agents' robot radii differ")
  sets = Ptr{Cvoid}[syncObstacles!(world(S).spheres, S).h for S in Ss]
  handles = Ptr{Cvoid}[t.h for t in trees]
  P = Matrix{Float64}(undef, trees[1].d, n)               # column-major d x n == row-major n x d for C
  for i = 1:n; P[:, i] = vec(points[i]); end
  W = world(Ss[1])
  if !haskey(W.pinned, :mIdx) || length(W.pinned[:mIdx]) < n * capacity
    W.pinned[:mIdx] = pinnedVector(W.ctx, Int32, n * capacity); W.pinned[:mDist] = pinnedVector(W.ctx, Float64, n * capacity)
    W.pinned[:mFwd] = pinnedVector(W.ctx, UInt8, n * capacity); W.pinned[:mRev] = pinnedVector(W.ctx, UInt8, n * capacity)
  end
  idx = W.pinned[:mIdx]::Vector{Int32}; dist = W.pinned[:mDist]::Vector{Float64}
  fwd = W.pinned[:mFwd]::Vector{UInt8}; rev = W.pinned[:mRev]::Vector{UInt8}
  nearestIdx = Vector{Int32}(undef, n); nearestDist = Vector{Float64}(undef, n)
  collides = Vector{UInt8}(undef, n); cert = Vector{Float64}(undef, n); cnt = Vector{Int32}(undef, n)
  GC.@preserve sets handles P ranges idx dist fwd rev nearestIdx nearestDist collides cert cnt check(trees[1].ctx,
      ccall((:rrtqx_extend_query_multi, LIB), Int32,
            (Ptr{Ptr{Cvoid}}, Ptr{Ptr{Cvoid}}, Int32, Ptr{Float64}, Ptr{Float64}, Float64, UInt32, Int32, Ptr{Int32},
             Ptr{Float64}, Ptr{UInt8}, Ptr{Float64}, Ptr{Int32}, Ptr{Int32}, Ptr{Float64}, Ptr{UInt8}, Ptr{UInt8}),
            handles, sets, n, P, ranges, rho, CHECK_QUICK_PASS, Int32(capacity), nearestIdx, nearestDist, collides,
            cert, cnt, idx, dist, fwd, rev))
  out = Vector{Any}(undef, n)
  for i = 1:n
    S = Ss[i]; c = Int(cnt[i])
    if c > capacity                          # overflow: this agent alone, with room for its whole ball
      out[i] = extendQuery(S, trees[i], points[i], ranges[i]; capacity = 2 * c)
      continue
    end
    r = (i - 1) * capacity + 1 : (i - 1) * capacity + c
    warm = S.inWarmupTime                    # obstacles are ignored during warm-up (DRRT_Q.jl:1805-1807, 1523-1525)
    out[i] = (trees[i].nodes[nearestIdx[i] + 1], nearestDist[i], warm ? false : collides[i] != 0, warm ? Inf : cert[i],
              view(idx, r), view(dist, r), warm ? falses(c) : view(fwd, r) .!= 0, warm ? falses(c) : view(rev, r) .!= 0)
  end
  return out
end

# ------------------------------------------------------------------ Dubins edges (2-D polygon world)
const DUBINS_TYPES = ("rsl", "rsr", "rlr", "lsr", "lsl", "lrl")

# calculateTrajectory(S, edge::DubinsEdge) for a batch of edges (DRRT_DubinsEdge_functions.jl:329-709, space
# without time): sets dist / distOriginal / Wdist / dubinsType / trajectory on every edge.
function calculateTrajectoryBatch(ctx::Context, S, edges::Vector)
  n = length(edges)
  starts = Matrix{Float64}(undef, 4, n); goals = Matrix{Float64}(undef, 4, n)
  for (i, e) in enumerate(edges)
    starts[:, i] = e.startNode.position[1:4]; goals[:, i] = e.endNode.position[1:4]
  end
  res = Ref{Ptr{Cvoid}}(C_NULL)
  GC.@preserve starts goals check(ctx, ccall((:rrtqx_dubins_trajectory_batch, LIB), Int32,
      (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Float64, Ref{Ptr{Cvoid}}), ctx.h, starts, goals, n, S.minTurningRadius, res))
  ne = Ref{Int64}(0); nr = Ref{Int64}(0)
  check(ctx, ccall((:rrtqx_dubins_result_sizes, LIB), Int32, (Ptr{Cvoid}, Ref{Int64}, Ref{Int64}), res[], ne, nr))
  dist = Vector{Float64}(undef, n); typ = Vector{Int32}(undef, n); ptr = Vector{Int64}(undef, n + 1)
  xy = Matrix{Float64}(undef, 2, nr[])
  GC.@preserve dist typ ptr xy check(ctx, ccall((:rrtqx_dubins_result_fetch, LIB), Int32,
      (Ptr{Cvoid}, Ptr{Float64}, Ptr{Int32}, Ptr{Int64}, Ptr{Float64}), res[], dist, typ, ptr, xy))
  ccall((:rrtqx_dubins_result_destroy, LIB), Int32, (Ptr{Cvoid},), res[])
  for (i, e) in enumerate(edges)
    setDubinsTrajectory!(e, dist[i], typ[i], xy, ptr[i], ptr[i+1])
  end
end

# What calculateTrajectory sets on a DubinsEdge, from a device solve: dist = distOriginal = Wdist, dubinsType and
# trajectory = rows first+1:last of xy (2 x rows, 0-based CSR bounds), as the reference builds it (rows x 2)
function setDubinsTrajectory!(e, dist::Float64, typ::Integer, xy::AbstractMatrix{Float64}, first::Integer, last::Integer)
  e.dubinsType = typ < 0 ? "xxx" : DUBINS_TYPES[typ + 1]
  e.Wdist = dist; e.dist = dist; e.distOriginal = dist
  e.trajectory = permutedims(xy[:, first+1:last])
end

# The DubinsEdge iteration in one call (rrtqx_extend_query_dubins): kdFindNearest, saturate(point, nearest, S.delta)
# when `saturate` (DRRT_DubinsEdge_functions.jl:70-95), kdFindWithinRange(range) with the theta ghost, and for every
# neighbour calculateTrajectory + explicitEdgeCheck of edge(new -> n) (findBestParent, DRRT_Q.jl:1949-1960) and
# edge(n -> new) (:2600-2603).  Returns (nearest node, its distance, the (saturated) point, neighbour ids (0-based)
# and keys, per-edge dist / type codes / collision flags with edge 2i-1 = new -> n_i and 2i = n_i -> new).  Arrays
# are pinned and reused; the views are valid until the next call on the same CSpace.  The rows stay on the device
# until dubinsEdgesFromQuery! puts them onto edge objects.  Collision flags are false during warm-up.
function extendQueryDubins(S, tree::GpuKDTree, point::Array{Float64}, range::Float64; saturate::Bool = false,
                           capacity::Int = 8192)
  W = world(S)
  G = syncPolygons!(W.polygons, S)
  if !haskey(W.pinned, :didx) || length(W.pinned[:didx]) < capacity
    W.pinned[:didx] = pinnedVector(W.ctx, Int32, capacity); W.pinned[:ddist] = pinnedVector(W.ctx, Float64, capacity)
    W.pinned[:dedist] = pinnedVector(W.ctx, Float64, 2 * capacity)
    W.pinned[:detype] = pinnedVector(W.ctx, Int32, 2 * capacity)
    W.pinned[:decol] = pinnedVector(W.ctx, UInt8, 2 * capacity)
  end
  if !haskey(W.pinned, :dres)
    r = Ref{Ptr{Cvoid}}(C_NULL)
    W.pinned[:dres] = r
    finalizer(x -> x[] != C_NULL && ccall((:rrtqx_dubins_result_destroy, LIB), Int32, (Ptr{Cvoid},), x[]), r)
  end
  idx = W.pinned[:didx]::Vector{Int32}; dist = W.pinned[:ddist]::Vector{Float64}
  edist = W.pinned[:dedist]::Vector{Float64}; etype = W.pinned[:detype]::Vector{Int32}
  ecol = W.pinned[:decol]::Vector{UInt8}; res = W.pinned[:dres]::Base.RefValue{Ptr{Cvoid}}
  nearestIdx = Ref{Int32}(0); nearestDist = Ref{Float64}(0.0); n = Ref{Int32}(0)
  p = Vector{Float64}(vec(point)[1:4])
  flags = saturate ? EXTEND_SATURATE : UInt32(0)
  GC.@preserve p idx dist edist etype ecol check(tree.ctx, ccall((:rrtqx_extend_query_dubins, LIB), Int32,
      (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}, Float64, Float64, Float64, Float64, UInt32, Int32, Ref{Int32},
       Ref{Float64}, Ref{Int32}, Ptr{Int32}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{UInt8}, Ref{Ptr{Cvoid}}),
      tree.h, G.h, p, S.delta, range, S.robotRadius, S.minTurningRadius, flags, Int32(length(idx)), nearestIdx,
      nearestDist, n, idx, dist, edist, etype, ecol, res))
  n[] <= length(idx) || return extendQueryDubins(S, tree, point, range; saturate = saturate, capacity = 2 * Int(n[]))
  k = min(Int(n[]), length(idx))            # never slice past the buffers
  warm = S.inWarmupTime                     # obstacles are ignored during warm-up (DRRT.jl:1660-1678)
  return (tree.nodes[nearestIdx[] + 1], nearestDist[], p, view(idx, 1:k), view(dist, 1:k), view(edist, 1:2k),
          view(etype, 1:2k), warm ? falses(2k) : view(ecol, 1:2k) .!= 0)
end

# Puts the device solve of the last extendQueryDubins on S onto DubinsEdge objects: edges[e] receives edge e of
# that call (edges[2i-1] = new -> n_i, edges[2i] = n_i -> new; `nothing` entries are skipped).
function dubinsEdgesFromQuery!(S, edges::Vector)
  W = world(S)
  res = W.pinned[:dres]::Base.RefValue{Ptr{Cvoid}}
  ne = Ref{Int64}(0); nr = Ref{Int64}(0)
  check(W.ctx, ccall((:rrtqx_dubins_result_sizes, LIB), Int32, (Ptr{Cvoid}, Ref{Int64}, Ref{Int64}), res[], ne, nr))
  length(edges) <= ne[] || error("the last extendQueryDubins produced $(ne[]) edges, not $(length(edges))")
  dist = Vector{Float64}(undef, ne[]); typ = Vector{Int32}(undef, ne[]); ptr = Vector{Int64}(undef, ne[] + 1)
  xy = Matrix{Float64}(undef, 2, nr[])
  GC.@preserve dist typ ptr xy check(W.ctx, ccall((:rrtqx_dubins_result_fetch, LIB), Int32,
      (Ptr{Cvoid}, Ptr{Float64}, Ptr{Int32}, Ptr{Int64}, Ptr{Float64}), res[], dist, typ, ptr, xy))
  for (i, e) in enumerate(edges)
    e === nothing || setDubinsTrajectory!(e, dist[i], typ[i], xy, ptr[i], ptr[i+1])
  end
  return edges
end

# extendQueryDubins for many Dubins planners in lock-step (the city-block instances of config C5): agent i is
# (Ss[i], trees[i], points[i], ranges[i]), each with its own CSpace and tree.  One call and one host wait serve the
# whole round; each agent gets the tuple extendQueryDubins returns, warm-up handling included.  The views and the
# device solve stay valid until the next extendQueryDubinsMulti on the same first CSpace; dubinsEdgesFromQueryMulti!
# puts an agent's solved edges onto its DubinsEdge objects.  An agent whose ball holds more than `capacity` nodes is
# repeated alone with extendQueryDubins (rare; Dubins balls hold about 16 nodes), and its edges then come from
# dubinsEdgesFromQuery! on its CSpace.  The agents share one robot radius, turning radius and delta (the C call takes
# one of each).
function extendQueryDubinsMulti(Ss::Vector, trees::Vector, points::Vector, ranges::Vector{Float64};
                                saturate::Bool = false, capacity::Int = 1024)
  n = length(trees)
  n == 0 && return Any[]
  S1 = Ss[1]
  all(S -> S.robotRadius == S1.robotRadius, Ss) || error("extendQueryDubinsMulti: the agents' robot radii differ")
  all(S -> S.minTurningRadius == S1.minTurningRadius, Ss) ||
    error("extendQueryDubinsMulti: the agents' turning radii differ")
  all(S -> S.delta == S1.delta, Ss) || error("extendQueryDubinsMulti: the agents' delta differ")
  sets = Ptr{Cvoid}[syncPolygons!(world(S).polygons, S).h for S in Ss]
  handles = Ptr{Cvoid}[t.h for t in trees]
  P = Matrix{Float64}(undef, 4, n)                        # column-major 4 x n == row-major n x 4 for C
  for i = 1:n; P[:, i] = vec(points[i])[1:4]; end
  W = world(S1)
  if !haskey(W.pinned, :mdIdx) || length(W.pinned[:mdIdx]) < n * capacity
    W.pinned[:mdIdx] = pinnedVector(W.ctx, Int32, n * capacity); W.pinned[:mdDist] = pinnedVector(W.ctx, Float64, n * capacity)
    W.pinned[:mdEdist] = pinnedVector(W.ctx, Float64, 2 * n * capacity)
    W.pinned[:mdEtype] = pinnedVector(W.ctx, Int32, 2 * n * capacity)
    W.pinned[:mdEcol] = pinnedVector(W.ctx, UInt8, 2 * n * capacity)
  end
  if !haskey(W.pinned, :mdRes)
    r = Ref{Ptr{Cvoid}}(C_NULL)
    W.pinned[:mdRes] = r
    finalizer(x -> x[] != C_NULL && ccall((:rrtqx_dubins_result_destroy, LIB), Int32, (Ptr{Cvoid},), x[]), r)
  end
  idx = W.pinned[:mdIdx]::Vector{Int32}; dist = W.pinned[:mdDist]::Vector{Float64}
  edist = W.pinned[:mdEdist]::Vector{Float64}; etype = W.pinned[:mdEtype]::Vector{Int32}
  ecol = W.pinned[:mdEcol]::Vector{UInt8}; res = W.pinned[:mdRes]::Base.RefValue{Ptr{Cvoid}}
  nearestIdx = Vector{Int32}(undef, n); nearestDist = Vector{Float64}(undef, n); cnt = Vector{Int32}(undef, n)
  flags = saturate ? EXTEND_SATURATE : UInt32(0)
  GC.@preserve sets handles P ranges idx dist edist etype ecol nearestIdx nearestDist cnt check(trees[1].ctx,
      ccall((:rrtqx_extend_query_dubins_multi, LIB), Int32,
            (Ptr{Ptr{Cvoid}}, Ptr{Ptr{Cvoid}}, Int32, Ptr{Float64}, Ptr{Float64}, Float64, Float64, Float64, UInt32,
             Int32, Ptr{Int32}, Ptr{Float64}, Ptr{Int32}, Ptr{Int32}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32},
             Ptr{UInt8}, Ref{Ptr{Cvoid}}),
            handles, sets, n, P, ranges, S1.delta, S1.robotRadius, S1.minTurningRadius, flags, Int32(capacity),
            nearestIdx, nearestDist, cnt, idx, dist, edist, etype, ecol, res))
  first = Vector{Int}(undef, n)                           # agent i's first edge (0-based) in the packed solve
  alone = falses(n)
  out = Vector{Any}(undef, n)
  f = 0
  for i = 1:n
    S = Ss[i]; c = Int(cnt[i])
    first[i] = f
    f += 2 * min(c, capacity)
    if c > capacity                          # overflow: this agent alone, with room for its whole ball
      out[i] = extendQueryDubins(S, trees[i], points[i], ranges[i]; saturate = saturate, capacity = 2 * c)
      alone[i] = true
      continue
    end
    r = (i - 1) * capacity + 1 : (i - 1) * capacity + c
    re = 2 * (i - 1) * capacity + 1 : 2 * (i - 1) * capacity + 2 * c
    warm = S.inWarmupTime                    # obstacles are ignored during warm-up (DRRT.jl:1660-1678)
    out[i] = (trees[i].nodes[nearestIdx[i] + 1], nearestDist[i], P[:, i], view(idx, r), view(dist, r), view(edist, re),
              view(etype, re), warm ? falses(2 * c) : view(ecol, re) .!= 0)
  end
  W.pinned[:mdFirst] = first; W.pinned[:mdAlone] = alone; W.pinned[:mdFetched] = nothing
  return out
end

# Puts agent i's device solve of the last extendQueryDubinsMulti whose first CSpace was S onto DubinsEdge objects:
# edges[e] receives the agent's edge e (edges[2k-1] = new -> n_k, edges[2k] = n_k -> new; `nothing` entries are
# skipped).  The packed solve is fetched once per call and shared by the agents.
function dubinsEdgesFromQueryMulti!(S, i::Int, edges::Vector)
  W = world(S)
  (W.pinned[:mdAlone]::BitVector)[i] &&
    error("agent $i was repeated alone by extendQueryDubinsMulti: its edges come from dubinsEdgesFromQuery!")
  if W.pinned[:mdFetched] === nothing
    res = W.pinned[:mdRes]::Base.RefValue{Ptr{Cvoid}}
    ne = Ref{Int64}(0); nr = Ref{Int64}(0)
    check(W.ctx, ccall((:rrtqx_dubins_result_sizes, LIB), Int32, (Ptr{Cvoid}, Ref{Int64}, Ref{Int64}), res[], ne, nr))
    dist = Vector{Float64}(undef, ne[]); typ = Vector{Int32}(undef, ne[]); ptr = Vector{Int64}(undef, ne[] + 1)
    xy = Matrix{Float64}(undef, 2, nr[])
    GC.@preserve dist typ ptr xy check(W.ctx, ccall((:rrtqx_dubins_result_fetch, LIB), Int32,
        (Ptr{Cvoid}, Ptr{Float64}, Ptr{Int32}, Ptr{Int64}, Ptr{Float64}), res[], dist, typ, ptr, xy))
    W.pinned[:mdFetched] = (dist, typ, ptr, xy)
  end
  dist, typ, ptr, xy = W.pinned[:mdFetched]
  first = (W.pinned[:mdFirst]::Vector{Int})[i]
  last = i < length(W.pinned[:mdFirst]) ? W.pinned[:mdFirst][i + 1] : length(dist)
  length(edges) <= last - first || error("agent $i has $(last - first) edges in the last call, not $(length(edges))")
  for (k, e) in enumerate(edges)
    j = first + k                            # 1-based index of the packed edge
    e === nothing || setDubinsTrajectory!(e, dist[j], typ[j], xy, ptr[j], ptr[j+1])
  end
  return edges
end

# Dubins explicitEdgeCheck OR-ed over the obstacle list of G for a batch (DRRT_DubinsEdge_functions.jl:750-774);
# no warm-up test (the per-obstacle form of the reference has none)
function dubinsCheck(G::GpuPolygons, S, edges::Vector)
  n = length(edges)
  starts = Matrix{Float64}(undef, 2, n); ends = Matrix{Float64}(undef, 2, n); ptr = Vector{Int64}(undef, n + 1); ptr[1] = 0
  for (i, e) in enumerate(edges)
    starts[:, i] = e.startNode.position[1:2]; ends[:, i] = e.endNode.position[1:2]
    ptr[i + 1] = ptr[i] + size(e.trajectory, 1)
  end
  xy = Matrix{Float64}(undef, 2, ptr[n + 1])
  for (i, e) in enumerate(edges)
    xy[:, ptr[i]+1:ptr[i+1]] = permutedims(e.trajectory[:, 1:2])
  end
  out = Vector{UInt8}(undef, n)
  GC.@preserve starts ends ptr xy out check(G.ctx, ccall((:rrtqx_dubins_edge_check_batch, LIB), Int32,
      (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{Float64}, Int64, Float64, Float64, UInt32, Ptr{UInt8}),
      G.h, starts, ends, ptr, xy, n, S.robotRadius, S.minTurningRadius, UInt32(0), out))
  return out .!= 0
end
# explicitEdgeCheck(S, edge) for a batch of Dubins edges (DRRT.jl:1660-1678: false during warm-up)
explicitEdgeCheckBatch(G::GpuPolygons, S, edges::Vector) = S.inWarmupTime ? falses(length(edges)) : dubinsCheck(G, S, edges)

# saturate(newPoint, closestPoint, delta), DubinsEdge version (DRRT_DubinsEdge_functions.jl:70-95): in place.
function saturateDubins!(ctx::Context, newPoint::Array{Float64}, closestPoint::Array{Float64}, delta::Float64)
  p = vec(newPoint); c = vec(closestPoint)
  GC.@preserve p c check(ctx, ccall((:rrtqx_dubins_saturate_batch, LIB), Int32,
      (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Float64), ctx.h, p, c, 1, delta))
  newPoint[:] = p
end

# ------------------------------------------------------------------ hooking into the planner
# install!() makes the planner's unqualified calls reach this module.  Call it once, after the reference's includes
# (it refers to the reference's CSpace / Edge / SimpleEdge / DubinsEdge / rrtXQueue types in Main) and after
# include("extend_gpu.jl") if the fused extend is wanted.  Methods that take the tree are more specific than the
# reference's (KD::GpuKDTree) and replace nothing; methods that take only the CSpace replace the reference's methods
# of the same signature -- from then on every CSpace must be attach!ed (there is no CPU fallback).
function install!()
  @eval Main begin
    kdInsert(tree::RRTQXGpu.GpuKDTree, node) = RRTQXGpu.kdInsert(tree, node)
    kdFindNearest(tree::RRTQXGpu.GpuKDTree, queryPoint::Array{Float64}) = RRTQXGpu.kdFindNearest(tree, queryPoint)
    kdFindWithinRange(tree::RRTQXGpu.GpuKDTree, range::Float64, queryPoint::Array{Float64}) =
      RRTQXGpu.kdFindWithinRange(tree, range, queryPoint)
    kdFindMoreWithinRange(tree::RRTQXGpu.GpuKDTree, range::Float64, queryPoint::Array{Float64}, L) =
      RRTQXGpu.kdFindMoreWithinRange(tree, range, queryPoint, L)
    findPointsInConflictWithObstacle(S, KD::RRTQXGpu.GpuKDTree, ob, root) =
      RRTQXGpu.findPointsInConflictWithObstacle(S, KD, ob, root)
    addNewObstacle(S, KD::RRTQXGpu.GpuKDTree, Q, ob, root, fileCounter::Int, R) =
      RRTQXGpu.addNewObstacle(S, KD, Q, ob, root, fileCounter, R)
    removeObstacle(S, KD::RRTQXGpu.GpuKDTree, Q, ob, root, hyberBallRad::Float64, timeElapsed::Float64, moveGoal) =
      RRTQXGpu.removeObstacle(S, KD, Q, ob, root, hyberBallRad, timeElapsed, moveGoal)
    # replaced: same signatures as DRRT_Q.jl:1802,1520,1558,1594,1595 and the per-edge-type methods
    explicitEdgeCheck(C::CSpace{T}, edge::Edge) where {T} = RRTQXGpu.explicitEdgeCheck(C, edge)
    explicitEdgeCheck(S::CSpace{T}, edge::Edge, obstacle::OT) where {T, OT} = RRTQXGpu.explicitEdgeCheck(S, edge, obstacle)
    explicitPointCheck(S::CSpace{T}, point::Array{Float64}) where {T} = RRTQXGpu.explicitPointCheck(S, point)
    explicitPointCheck3D(S::CSpace{T}, point::Array{Float64}) where {T} = RRTQXGpu.explicitPointCheck3D(S, point)
    explicitNodeCheck(S::CSpace{T}, node) where {T} = RRTQXGpu.explicitNodeCheck(S, node)
    explicitNodeCheck3D(S::CSpace{T}, node) where {T} = RRTQXGpu.explicitNodeCheck3D(S, node)
  end
  if isdefined(RRTQXGpu, :extendRRTx)
    @eval Main begin
      extend(S, KD::RRTQXGpu.GpuKDTree, Q::rrtXQueue, newNode, closestNode, delta::Float64, hyberBallRad::Float64, moveGoal) =
        RRTQXGpu.extendRRTx(S, KD, Q, newNode, closestNode, delta, hyberBallRad, moveGoal)
    end
  end
  return nothing
end

isfile(joinpath(@__DIR__, "extend_gpu.jl")) && include("extend_gpu.jl")

end # module
