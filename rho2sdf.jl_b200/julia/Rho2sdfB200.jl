# Rho2sdfB200.jl -- Julia host side of the B200 hot path: keeps the reference's names and signatures
# (src/RhoToSDF.jl:116-304, src/MeshGrid, src/SignedDistances, src/SdfSmoothing) and `ccall`s libr2s.so (include/r2s.h).
#
# NOT EXECUTED IN THE BUILD IMAGE (no Julia toolchain there): it is the binding a maintainer drops into the reference
# next to src/RhoToSDF.jl; the Python mirror in rho2sdf.jl_b200/__init__.py binds the very same entry points and is what
# the tests exercise.  There is no CPU fallback: every call errors if the library or a CUDA device is missing.
module Rho2sdfB200

using Rho2sdf                      # the reference package: Mesh, Grid, Rho2sdfOptions, HEX8/TET4, grid set-up, exports
using Rho2sdf.MeshGrid: Mesh, Grid, generateGridPoints
using Rho2sdf.ElementTypes: AbstractElement, HEX8, TET4

export rho2sdf, rho2sdf_hex8, rho2sdf_tet4, evalDistances, Sign_Detection, remove_sdf_artifacts!, RBFs_smoothing,
       DenseInNodes, find_threshold_for_volume, calculate_volume_from_sdf, isosurface, export_isosurface, sample_sdf, sample_sdf_lattice, rbf_weights

const LIB = get(ENV, "R2S_LIBRARY", joinpath(@__DIR__, "..", "libr2s.so"))

# mirror of r2s_params / r2s_report (include/r2s.h); field order and types must match the C structs
struct R2SParams
  rho_t::Cdouble; delta_factor::Cdouble; remove_artifacts::Int32; artifact_threshold::Cdouble; artifact_min_ratio::Cdouble
  rbf_interp::Int32; smooth::Int32; rbf_cut::Cdouble; target_volume::Cdouble; final_volume::Int32
end
mutable struct R2SReport
  n_solid::Int64; n_crossing::Int64; n_active::Int64; n_pairs::Int64; n_not_converged::Int64; n_newton_iters::Int64; n_flipped::Int64
  cg_iters::Int32; bisections::Int32; th::Cfloat; volume::Cfloat
  ms_bin::Cfloat; ms_project::Cfloat; ms_assemble::Cfloat; ms_sign::Cfloat; ms_cc::Cfloat; ms_rbf_prep::Cfloat; ms_cg::Cfloat; ms_lsf::Cfloat
  ms_threshold::Cfloat; ms_fine::Cfloat; ms_volume::Cfloat; ms_total::Cfloat
  launches::Int64; collectives::Int64; cg_probe::NTuple{4,Cfloat}; n_pairs_pruned::Int64; ms_solve::Cfloat; ms_scan::Cfloat
  R2SReport() = new(0, 0, 0, 0, 0, 0, 0, 0, 0, 0f0, 0f0, 0f0, 0f0, 0f0, 0f0, 0f0, 0f0, 0f0, 0f0, 0f0, 0f0, 0f0, 0f0, 0, 0, (0f0, 0f0, 0f0, 0f0), 0, 0f0, 0f0)
end

mutable struct Context
  h::Ptr{Cvoid}
  function Context(device::Integer=0)
    ref = Ref{Ptr{Cvoid}}(C_NULL)
    rc = ccall((:r2s_create, LIB), Cint, (Ref{Ptr{Cvoid}}, Cint, Ptr{Cvoid}), ref, device, C_NULL)
    (rc != 0 || ref[] == C_NULL) && error("r2s_create failed (rc=$rc): no usable CUDA device -- libr2s has no CPU fallback")
    c = new(ref[])
    finalizer(x -> (x.h != C_NULL && ccall((:r2s_destroy, LIB), Cvoid, (Ptr{Cvoid},), x.h); x.h = C_NULL), c)
    return c
  end
end
check(c::Context, rc) = rc == 0 ? nothing : error(unsafe_string(ccall((:r2s_last_error, LIB), Cstring, (Ptr{Cvoid},), c.h)))   # mirrors the reference's error(...)

# One device context per Mesh object, held WEAKLY: when the Mesh is garbage collected its entry disappears and the Context's finalizer
# frees the device memory (an IdDict would pin every mesh ever used).  release!(mesh) frees it right away.
const CONTEXTS = WeakKeyDict{Any,Context}()
function release!(mesh::Mesh)
  c = pop!(CONTEXTS, mesh, nothing)
  c === nothing || finalize(c)
  return nothing
end

function context(mesh::Mesh)
  get!(CONTEXTS, mesh) do
    c = Context()
    # mesh.X is 3 x nnp Float64, mesh.IEN is nen x nel Int64 with 1-based ids: already the layout r2s_set_mesh takes
    check(c, ccall((:r2s_set_mesh, LIB), Cint, (Ptr{Cvoid}, Cint, Int64, Ptr{Cdouble}, Int64, Ptr{Int64}),
                   c.h, mesh.nen, mesh.nnp, mesh.X, mesh.nel, mesh.IEN))
    c
  end
end
function use_grid(c::Context, grid::Grid)
  # the Grid fields exactly as the reference's ctor computed them (src/MeshGrid/Grid.jl:10-34): no re-derivation on the C side
  check(c, ccall((:r2s_set_grid, LIB), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Int64}, Cdouble),
                 c.h, Vector{Float64}(grid.AABB_min), Vector{Float64}(grid.AABB_max), Vector{Int64}(grid.N), grid.cell_size))
end

# ---- src/MeshGrid/NodalDensities.jl:89-109, Isocontour_volume.jl:77-154 -----------------------------------------------
function DenseInNodes(mesh::Mesh, rho::Vector{Float64})
  c = context(mesh); out = Vector{Float64}(undef, mesh.nnp)
  check(c, ccall((:r2s_nodal_densities, LIB), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Ptr{Cdouble}), c.h, rho, out))
  return out
end
function find_threshold_for_volume(mesh::Mesh, nodal_values::Vector{Float64}; tolerance::Float64=1e-4, max_iterations::Int=60)
  c = context(mesh); out = Ref{Cdouble}(0.0)
  check(c, ccall((:r2s_find_threshold, LIB), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Cdouble, Cdouble, Cint, Ref{Cdouble}),
                 c.h, nodal_values, mesh.V_domain * mesh.V_frac, tolerance, max_iterations, out))
  return out[]
end

# ---- src/SignedDistances/sdfOnDensityField.jl:139-486 ---------------------------------------------------------------------
# points = the grid's own point set: the grid entry point (faster, same result); any other 3 x n points: the points entry point, binned in
# the grid's frame like the reference's LinkedList(grid, points) (rule in include/r2s.h)
is_grid_points(grid::Grid, points::Matrix{Float64}) = size(points, 2) == grid.ngp && points == generateGridPoints(grid)
function evalDistances(mesh::Mesh, grid::Grid, points::Matrix{Float64}, ρₙ::Vector{Float64}, ρₜ::Float64; delta_factor::Float64=1.1)
  c = context(mesh); use_grid(c, grid)
  if is_grid_points(grid, points)
    dist = Vector{Float64}(undef, grid.ngp); xp = zeros(Float64, 3, grid.ngp)
    check(c, ccall((:r2s_eval_distances, LIB), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Cdouble, Cdouble, Ptr{Cdouble}, Ptr{Cdouble}), c.h, ρₙ, ρₜ, delta_factor, dist, xp))
    return dist, xp
  end
  size(points, 1) == 3 || error("points must be a 3 x n matrix")
  n = size(points, 2); dist = Vector{Float64}(undef, n); xp = zeros(Float64, 3, n)
  check(c, ccall((:r2s_eval_distances_points, LIB), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Cdouble, Cdouble, Ptr{Cdouble}, Int64, Ptr{Cdouble}, Ptr{Cdouble}),
                 c.h, ρₙ, ρₜ, delta_factor, points, n, dist, xp))
  return dist, xp
end
# ---- src/SignedDistances/SignDetection.jl:275-283 -----------------------------------------------------------------------
function Sign_Detection(mesh::Mesh, grid::Grid, points::Matrix{Float64}, ρₙ::Vector{Float64}, ρₜ::Float64)
  c = context(mesh); use_grid(c, grid)
  if is_grid_points(grid, points)
    signs = Vector{Float64}(undef, grid.ngp)
    check(c, ccall((:r2s_sign_detection, LIB), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Cdouble, Ptr{Cdouble}), c.h, ρₙ, ρₜ, signs))
    return signs
  end
  size(points, 1) == 3 || error("points must be a 3 x n matrix")
  n = size(points, 2); signs = Vector{Float64}(undef, n)
  check(c, ccall((:r2s_sign_detection_points, LIB), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Cdouble, Ptr{Cdouble}, Int64, Ptr{Cdouble}), c.h, ρₙ, ρₜ, points, n, signs))
  return signs
end
# ---- src/SignedDistances/SdfArtifactRemoval.jl:134-245 ------------------------------------------------------------------
function remove_sdf_artifacts!(sdf_values::Vector{Float64}, grid::Grid; threshold::Float64=0.0, min_component_ratio::Float64=0.01, ctx::Context=Context())
  length(sdf_values) == grid.ngp || error("SDF values length ($(length(sdf_values))) doesn't match grid points ($(grid.ngp))")
  use_grid(ctx, grid); flipped = Ref{Int64}(0)
  check(ctx, ccall((:r2s_remove_artifacts, LIB), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Cdouble, Cdouble, Ref{Int64}), ctx.h, sdf_values, threshold, min_component_ratio, flipped))
  return Int(flipped[])
end
# ---- src/SdfSmoothing/RBFs4Smoothing.jl:321-377 ----------------------------------------------------------------------------
"fine_grid stand-in: same indexing as create_smooth_grid's Array{Vector{Float32},3} (RBFs4Smoothing.jl:60-74) without 10^9 heap vectors"
struct LazyFineGrid <: AbstractArray{Vector{Float32},3}
  xmin::NTuple{3,Float32}; dx::Float32; dims::NTuple{3,Int}
end
Base.size(g::LazyFineGrid) = g.dims
Base.getindex(g::LazyFineGrid, i::Int, j::Int, k::Int) = Float32[g.xmin[1] + Float32(i - 1) * g.dx, g.xmin[2] + Float32(j - 1) * g.dx, g.xmin[3] + Float32(k - 1) * g.dx]
function fine_grid_of(grid::Grid, smooth::Int)
  dims = Tuple(Int.(grid.N .* smooth .+ 1)); xmin = Float32.(grid.AABB_min)
  dx = (Float32(grid.AABB_max[1]) - xmin[1]) / Float32(dims[1] - 1)
  return LazyFineGrid(Tuple(xmin), dx, dims)
end
function RBFs_smoothing(mesh::Mesh, dist::Vector{Float64}, my_grid::Grid, Is_interpolation::Bool, smooth::Int, taskName::String, threshold::Float64=1e-3)
  c = context(mesh); use_grid(c, my_grid)
  dims = Tuple(Int.(my_grid.N .* smooth .+ 1)); fine = Array{Float32,3}(undef, dims)
  th = Ref{Cfloat}(0f0); vol = Ref{Cfloat}(0f0)
  check(c, ccall((:r2s_rbf_smoothing, LIB), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Cint, Cint, Cdouble, Cdouble, Ptr{Cfloat}, Ref{Cfloat}, Ref{Cfloat}),
                 c.h, dist, Is_interpolation, smooth, threshold, mesh.V_frac * mesh.V_domain, fine, th, vol))
  return fine, fine_grid_of(my_grid, smooth)
end

# ---- src/SdfSmoothing/CalcVolumeFromSDF.jl:26-125 (stand-alone volume tool, test/ConvergenceTests/*) --------------------------------------
function calculate_volume_from_sdf(fine_sdf::Array{Float32,3}, fine_grid::AbstractArray{Vector{Float32},3}; iso_threshold::Float32=0.0f0, detailed_quad_order::Int=9,
                                   ctx::Context=Context())
  nx, ny, nz = size(fine_sdf)
  size(fine_grid) == (nx, ny, nz) || error("Dimensions of fine_sdf and fine_grid must match")
  edge = Float32(sqrt(sum(abs2, fine_grid[2, 1, 1] .- fine_grid[1, 1, 1])))          # :37-38
  v = Ref{Cdouble}(0.0)
  check(ctx, ccall((:r2s_volume_from_sdf, LIB), Cint, (Ptr{Cvoid}, Ptr{Cfloat}, Int64, Int64, Int64, Cfloat, Cfloat, Cint, Ref{Cdouble}),
                   ctx.h, fine_sdf, nx, ny, nz, edge, iso_threshold, detailed_quad_order, v))
  return Float32(v[])
end

# ---- all GPUs of the box from this one process: r2s_multi (include/r2s.h) ----------------------------------------------------------
mutable struct MultiContext
  h::Ptr{Cvoid}; n::Int
  function MultiContext(devices::Vector{<:Integer})
    ref = Ref{Ptr{Cvoid}}(C_NULL)
    rc = ccall((:r2s_multi_create, LIB), Cint, (Ref{Ptr{Cvoid}}, Ptr{Cint}, Cint), ref, Cint.(devices), length(devices))
    (rc != 0 || ref[] == C_NULL) && error("r2s_multi_create failed (rc=$rc): no usable CUDA devices / no peer access -- libr2s has no CPU fallback")
    m = new(ref[], length(devices))
    finalizer(x -> (x.h != C_NULL && ccall((:r2s_multi_destroy, LIB), Cvoid, (Ptr{Cvoid},), x.h); x.h = C_NULL), m)
    return m
  end
end
mcheck(m::MultiContext, rc) = rc == 0 ? nothing : error(unsafe_string(ccall((:r2s_multi_last_error, LIB), Cstring, (Ptr{Cvoid},), m.h)))
"GPUs rho2sdf() uses: ENV[\"R2S_DEVICES\"] = \"0,1,2,3\" (default: device 0 only)"
devices_from_env() = haskey(ENV, "R2S_DEVICES") ? parse.(Int, split(ENV["R2S_DEVICES"], ",")) : [0]

# ---- src/DataExport/ExportToVTI.jl:22-67 (SURVEY 8f-1): host array -> .vti; `export_device_vti` streams the device-resident result ---
function exportSdfToVTI(filename::String, grid::Grid, values::Vector{<:AbstractFloat}, value_label::String, smooth::Union{Int,Nothing}=nothing)
  sm = isnothing(smooth) ? 1 : smooth
  dims = Int.(grid.N .* sm .+ 1)
  length(values) == prod(dims) || error("Values vector length ($(length(values))) doesn't match grid dimensions ($(prod(dims))).")
  vals = eltype(values) == Float32 ? values : Float64.(values)
  path = endswith(filename, ".vti") ? filename : filename * ".vti"
  rc = ccall((:r2s_write_vti_host, LIB), Cint, (Cstring, Cstring, Ptr{Cvoid}, Cint, Int64, Int64, Int64, Ptr{Cdouble}, Ptr{Cdouble}),
             path, value_label, vals, eltype(vals) == Float64, dims[1], dims[2], dims[3], Float64.(grid.AABB_min), fill(grid.cell_size / sm, 3))
  rc == 0 || error("exportSdfToVTI: cannot write $path (code $rc)")
  return path
end
export_device_vti(mesh::Mesh, filename::String; label::String="distance", fine::Bool=true) =
  (c = context(mesh); check(c, ccall((:r2s_export_vti, LIB), Cint, (Ptr{Cvoid}, Cstring, Cstring, Cint), c.h, filename, label, fine ? 1 : 0)); filename)

# ---- the zero surface of the smoothed SDF (csrc/r2s_surf.cu; the reference leaves it to src/Visualizations / ParaView) -----------------
# Vertices 3 x nv Float32, triangles 3 x nt Int32 with 1-BASED vertex ids, counter-clockwise seen from outside {fine_sdf >= iso}.
surface_format(path::String) = endswith(lowercase(path), ".stl") ? 0 : endswith(lowercase(path), ".ply") ? 1 :
                               error("export_isosurface: the file name must end in .stl (binary STL) or .ply (binary PLY): $path")
function download_surface(c::Context, nv::Int64, nt::Int64)
  V = Matrix{Float32}(undef, 3, nv); T = Matrix{Int32}(undef, 3, nt)
  check(c, ccall((:r2s_download_isosurface, LIB), Cint, (Ptr{Cvoid}, Ptr{Cfloat}, Ptr{Int32}), c.h, V, T))
  return V, T .+ Int32(1)
end
"surface of the fine_sdf the last RBFs_smoothing call on `mesh` left on the device (frame: AABB_min, cell_size / smooth)"
function isosurface(mesh::Mesh; iso::Float32=0f0)
  c = context(mesh); nv = Ref{Int64}(0); nt = Ref{Int64}(0)
  check(c, ccall((:r2s_isosurface, LIB), Cint, (Ptr{Cvoid}, Cfloat, Ref{Int64}, Ref{Int64}), c.h, iso, nv, nt))
  return download_surface(c, nv[], nt[])
end
"surface of a host field; the frame is read off fine_grid (its first point and its steps along the three axes)"
function isosurface(fine_sdf::Array{Float32,3}, fine_grid::AbstractArray{Vector{Float32},3}; iso::Float32=0f0, ctx::Context=Context())
  nx, ny, nz = size(fine_sdf)
  size(fine_grid) == (nx, ny, nz) || error("Dimensions of fine_sdf and fine_grid must match")
  p0 = Float64.(fine_grid[1, 1, 1])
  h = [Float64(fine_grid[2, 1, 1][1]) - p0[1], Float64(fine_grid[1, 2, 1][2]) - p0[2], Float64(fine_grid[1, 1, 2][3]) - p0[3]]
  nv = Ref{Int64}(0); nt = Ref{Int64}(0)
  check(ctx, ccall((:r2s_isosurface_from_sdf, LIB), Cint, (Ptr{Cvoid}, Ptr{Cfloat}, Int64, Int64, Int64, Ptr{Cdouble}, Ptr{Cdouble}, Cfloat, Ref{Int64}, Ref{Int64}),
                   ctx.h, fine_sdf, nx, ny, nz, p0, h, iso, nv, nt))
  return download_surface(ctx, nv[], nt[])
end
"extract the surface on the device of `mesh` and write it as binary STL (.stl) or binary little-endian PLY (.ply)"
function export_isosurface(mesh::Mesh, path::String; iso::Float32=0f0)
  c = context(mesh); fmt = surface_format(path); nv = Ref{Int64}(0); nt = Ref{Int64}(0)
  check(c, ccall((:r2s_isosurface, LIB), Cint, (Ptr{Cvoid}, Cfloat, Ref{Int64}, Ref{Int64}), c.h, iso, nv, nt))
  check(c, ccall((:r2s_export_isosurface, LIB), Cint, (Ptr{Cvoid}, Cstring, Cint), c.h, path, fmt))
  return path
end

# ---- the smoothed SDF as a continuous function: rbf_interpolation_kdtree (src/SdfSmoothing/RBFs4Smoothing.jl:219-248) on the GPU ----------
# th + sum_c w_c exp(-(|x - c| / cell_size)^2) over the coarse points within the cut radius, for the field the last RBFs_smoothing call on
# `mesh` left on the device (exact arithmetic: include/r2s.h)
"values (Float32, n) at the columns of points (3 x n); with gradient=true also the analytic gradients (3 x n Float32)"
function sample_sdf(mesh::Mesh, points::Matrix{Float64}; gradient::Bool=false)
  size(points, 1) == 3 || error("sample_sdf: points must be a 3 x n matrix")
  c = context(mesh); n = size(points, 2)
  values = Vector{Float32}(undef, n); grads = gradient ? Matrix{Float32}(undef, 3, n) : nothing
  check(c, ccall((:r2s_sample_sdf, LIB), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Int64, Ptr{Cfloat}, Ptr{Cfloat}),
                 c.h, points, n, values, gradient ? grads : C_NULL))
  return gradient ? (values, grads) : values
end
"values on the lattice origin + (i - 1) .* spacing, i = 1 .. dims per axis (Float32 arithmetic), as an Array{Float32,3} of size dims"
function sample_sdf_lattice(mesh::Mesh, origin::AbstractVector{<:Real}, spacing::AbstractVector{<:Real}, dims::NTuple{3,Int})
  c = context(mesh); out = Array{Float32,3}(undef, dims)
  check(c, ccall((:r2s_sample_sdf_lattice, LIB), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Int64}, Ptr{Cfloat}),
                 c.h, Vector{Float64}(origin), Vector{Float64}(spacing), Int64[dims...], out))
  return out
end
"(weights on the coarse grid of `grid`, th): the definition of the continuous field"
function rbf_weights(mesh::Mesh, grid)
  c = context(mesh); w = Array{Float32,3}(undef, Tuple(Int.(grid.N .+ 1))); th = Ref{Cfloat}(0f0)
  check(c, ccall((:r2s_download_rbf_weights, LIB), Cint, (Ptr{Cvoid}, Ptr{Cfloat}, Ref{Cfloat}), c.h, w, th))
  return w, th[]
end

# ---- src/RhoToSDF.jl:116-242: same preamble as the reference, the timed region (:164-227) is ONE library call ---------------
function rho2sdf(taskName::String, X::Vector{Vector{Float64}}, IEN::Vector{Vector{Int64}}, rho::Vector{Float64}; options::Rho2sdfOptions=Rho2sdfOptions(),
                 devices::Vector{Int}=devices_from_env(), export_surface::Union{String,Nothing}=nothing)
  element_type = options.element_type
  mesh = Mesh(X, IEN, rho, Rho2sdf.ShapeFunctions.shape_functions; element_type=element_type)                  # :128
  sdf_grid = options.sdf_grid_setup == :manual ? Rho2sdf.MeshGrid.interactive_sdf_grid_setup(mesh) : Rho2sdf.MeshGrid.noninteractive_sdf_grid_setup(mesh)   # :141-145
  ρₙ = DenseInNodes(mesh, rho)                                                                                  # :148
  ρₜ = options.threshold_density === nothing ? find_threshold_for_volume(mesh, ρₙ) : options.threshold_density   # :151-156
  smooth = options.rbf_grid == :fine ? 2 : 1                                                                    # :222
  p = R2SParams(ρₜ, 1.1, options.remove_artifacts, 0.0, options.artifact_min_component_ratio, options.rbf_interp, smooth, 1e-3, mesh.V_frac * mesh.V_domain, 1)
  dims = Tuple(Int.(sdf_grid.N .* smooth .+ 1))
  sdf_dists = Vector{Float64}(undef, sdf_grid.ngp); fine_sdf = Array{Float32,3}(undef, dims); rep = R2SReport()
  if length(devices) > 1
    # ONE call, all GPUs: the library cuts the coarse planes into z-slabs, one per device, and fills the whole-grid arrays
    m = MultiContext(devices)
    mcheck(m, ccall((:r2s_multi_set_mesh, LIB), Cint, (Ptr{Cvoid}, Cint, Int64, Ptr{Cdouble}, Int64, Ptr{Int64}), m.h, mesh.nen, mesh.nnp, mesh.X, mesh.nel, mesh.IEN))
    mcheck(m, ccall((:r2s_multi_set_grid, LIB), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Int64}, Cdouble),
                    m.h, Vector{Float64}(sdf_grid.AABB_min), Vector{Float64}(sdf_grid.AABB_max), Vector{Int64}(sdf_grid.N), sdf_grid.cell_size))
    mcheck(m, ccall((:r2s_multi_pipeline, LIB), Cint, (Ptr{Cvoid}, Ref{R2SParams}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cfloat}, Ref{R2SReport}), m.h, p, ρₙ, sdf_dists, fine_sdf, rep))
    if export_surface !== nothing      # the zero surface of the fine SDF, extracted on all slabs, one file
      fmt = surface_format(export_surface); nv = Ref{Int64}(0); nt = Ref{Int64}(0)
      mcheck(m, ccall((:r2s_multi_isosurface, LIB), Cint, (Ptr{Cvoid}, Cfloat, Ref{Int64}, Ref{Int64}), m.h, 0f0, nv, nt))
      mcheck(m, ccall((:r2s_multi_export_isosurface, LIB), Cint, (Ptr{Cvoid}, Cstring, Cint), m.h, export_surface, fmt))
    end
    finalize(m)
  else
    c = context(mesh); use_grid(c, sdf_grid)
    check(c, ccall((:r2s_pipeline, LIB), Cint, (Ptr{Cvoid}, Ref{R2SParams}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cfloat}, Ref{R2SReport}), c.h, p, ρₙ, sdf_dists, fine_sdf, rep))
    export_surface === nothing || export_isosurface(mesh, export_surface)      # before release!(mesh): the field is on that context
  end
  fine_grid = fine_grid_of(sdf_grid, smooth)
  Rho2sdf.export_sdf_results_with_element_type(fine_sdf, fine_grid, sdf_grid, taskName, smooth, options.rbf_interp, element_type)   # :230-238 (unchanged, Julia)
  release!(mesh)                                                                                                # the Mesh is local to this call: free its device context now
  return fine_sdf, fine_grid, sdf_grid, sdf_dists                                                               # :241
end
rho2sdf_hex8(taskName, X, IEN, rho; kwargs...) = rho2sdf(taskName, X, IEN, rho; options=Rho2sdfOptions(; element_type=HEX8, kwargs...))    # :284-293
rho2sdf_tet4(taskName, X, IEN, rho; kwargs...) = rho2sdf(taskName, X, IEN, rho; options=Rho2sdfOptions(; element_type=TET4, kwargs...))    # :295-304

end # module
