# KDEB200.jl -- Julia `ccall` binding of libkdeb200.so (include/kdeb200.h).
#
# NOT RUNNABLE IN THE BUILD IMAGE (no julia binary there); it is the binding a maintainer of
# KernelDensityEstimate.jl adds to re-point the three seams of SURVEY.md 8b at the B200 library.
# kerneldensityestimate.jl_b200/api.py is the line-for-line Python mirror that the test-suite
# exercises; keep the two in sync.
#
#   seam S1  gibbs1(...)                 src/MSGibbs01.jl:527-629  ->  KDEB200.gibbs1!
#   seam S2  evaluate(bd, loc, p, ...)   src/DualTree01.jl:303-346 ->  KDEB200.evaluate!
#   seam S3  entropy(bd) / nLOO_LL       src/DualTree01.jl:505-508, src/CrossValidation.jl:15-24
#                                                                    ->  KDEB200.entropy
module KDEB200

using KernelDensityEstimate
const KDE = KernelDensityEstimate

const LIB = get(ENV, "KDEB200_LIB", "libkdeb200.so")

# nonzero return code -> the reference's error convention (error(...) => ErrorException)
function check(rc::Cint)
  rc == 0 && return nothing
  error(unsafe_string(ccall((:kdeb200_last_error, LIB), Cstring, ())))
end

init(device::Integer=0) = check(ccall((:kdeb200_init, LIB), Cint, (Cint,), device))

# One Julia process drives `ngpus` GPUs (0 = all visible): afterwards gibbs1!, evaluate!, entropy and lcv_bandwidths
# shard their samples / query points / leaf rows over the set inside the library -- no MPI, no second process.
init_multi(ngpus::Integer=0) = check(ccall((:kdeb200_init_multi, LIB), Cint, (Cint,), ngpus))
function multi_count()
  n = Ref{Cint}(0)
  check(ccall((:kdeb200_multi_count, LIB), Cint, (Ref{Cint},), n))
  Int(n[])
end

# setForceEvalDirect!(flag) of the reference (src/DualTree01.jl:3-9): false selects the error-bounded pruned kernel
# (every value within 1e-13 of the brute-force sum; the reference's dual tree: errTol = 1e-3) for evaluate!
setForceEvalDirect!(flag::Bool) = check(ccall((:kdeb200_set_pruning, LIB), Cint, (Cint,), flag ? 1 : 2))

# Arithmetic of the Gibbs label probabilities: 0 = FP64 (default; labels identical to the reference under injected
# randU / randN), 1 = packed FP32 on large calls (free-running statistical mode only, ~3x the sample rate)
set_gibbs_precision!(precision::Int) = check(ccall((:kdeb200_set_gibbs_precision, LIB), Cint, (Cint,), precision))
function gibbs_f32_slow_draws()
  n = Ref{Culonglong}(0)
  check(ccall((:kdeb200_gibbs_f32_slow_draws, LIB), Cint, (Ref{Culonglong},), n))
  return Int(n[])
end
# FP64 (default) calls: (lane-draws, warp-draws) whose label neither the certified FP32 nor the certified warp-parallel
# FP64 sums could decide, so that they were summed serially in node order, since the last call
function gibbs_exact_tier3()
  n, w = Ref{Culonglong}(0), Ref{Culonglong}(0)
  check(ccall((:kdeb200_gibbs_exact_tier3, LIB), Cint, (Ref{Culonglong}, Ref{Culonglong}), n, w))
  return Int(n[]), Int(w[])
end

# ---- S0: device-resident BallTreeDensity -------------------------------------------------
mutable struct DeviceTree
  h::Ptr{Cvoid}
  # gibbs=false: leaf records only (evaluate / entropy / nLOO_LL never touch the level records)
  function DeviceTree(bd::BallTreeDensity; gibbs::Bool=true)
    bd.multibandwidth == 0 || error("kdeb200: multibandwidth != 0 is not supported")
    bt = bd.bt
    out = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve bd begin
      if gibbs
        check(ccall((:kdeb200_tree_create, LIB), Cint,
                    (Cint, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{Int64}, Ptr{Int64},
                     Ref{Ptr{Cvoid}}),
                    bt.dims, bt.num_points, bd.means, bd.bandwidth, bt.weights, bt.left_child, bt.right_child,
                    bt.permutation, out))
      else
        check(ccall((:kdeb200_tree_create_eval, LIB), Cint,
                    (Cint, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ref{Ptr{Cvoid}}),
                    bt.dims, bt.num_points, bd.means, bd.bandwidth, bt.weights, bt.permutation, out))
      end
    end
    t = new(out[])
    finalizer(x -> ccall((:kdeb200_tree_destroy, LIB), Cint, (Ptr{Cvoid},), x.h), t)
    return t
  end
end

euclidean(addop, diffop) = all(f -> f === (+), addop) && all(f -> f === (-), diffop)

# ---- S1: gibbs1 -------------------------------------------------------------------------
# Same positional arguments as KDE.gibbs1; writes pts (d*Np) and ind (Ndens x Np) in place.
# randU / randN === nothing selects the library's Philox streams (keyed by `seed`).
# Ndens: 1..64 (KDEB200_MAX_DENS_LARGE), like the reference's any number of incoming messages; products of more than 16
# densities run a kernel of their own with the same labels and points, and refuse degenerate (zero / non-finite /
# out-of-range) bandwidths with an error instead of the reference's NaN rules.
function gibbs1!(Ndens::Int, trees::Vector{BallTreeDensity}, Np::Int, Niter::Int,
                 pts::Vector{Float64}, ind::Matrix{Int},
                 randU::Union{Nothing,Vector{Float64}}, randN::Union{Nothing,Vector{Float64}};
                 addop=(+,), diffop=(-,), getMu=(KDE.getEuclidMu,), getLambda=(KDE.getEuclidLambda,),
                 glbs=nothing, addEntropy::Bool=true, ndims::Int=maximum(Ndim.(trees)),
                 partialDimMask::AbstractVector{<:BitVector}=[trues(ndims) for i in 1:Ndens],
                 seed::UInt64=rand(UInt64))
  (euclidean(addop, diffop) && all(f -> f === KDE.getEuclidMu, getMu) &&
   all(f -> f === KDE.getEuclidLambda, getLambda)) ||
    error("kdeb200: only the default Euclidean (+,-) manifold is supported on the B200 path")
  dts = [DeviceTree(t) for t in trees]
  hs = Ptr{Cvoid}[d.h for d in dts]
  mask = UInt8[partialDimMask[j][k] ? 0x01 : 0x00 for k in 1:ndims, j in 1:Ndens]  # [j*d + k], column-major
  uptr = randU === nothing ? Ptr{Float64}(C_NULL) : pointer(randU)
  nptr = randN === nothing ? Ptr{Float64}(C_NULL) : pointer(randN)
  # glbs.recordChoosen (src/MSGibbs01.jl:29-31, examples/ExtractingLabels.jl): the library records
  # permutation[ind[j]] of the last sampleIndex call of every level into an Int64 array [Nlevels, Ndens, Np]
  # (C order [sample][density][level]); it is unpacked into glbs.labelsChoosen[sample][density][level] below.
  record = glbs !== nothing && glbs.recordChoosen
  nlev = Ref{Cint}(0)
  GC.@preserve dts hs check(ccall((:kdeb200_gibbs_sizes, LIB), Cint,
    (Ptr{Ptr{Cvoid}}, Cint, Cint, Ref{Cint}, Ptr{Int64}, Ptr{Int64}, Ptr{Int64}),
    hs, Ndens, Niter, nlev, C_NULL, C_NULL, C_NULL))
  rec = record ? Array{Int64,3}(undef, Int(nlev[]), Ndens, Np) : Array{Int64,3}(undef, 0, 0, 0)
  GC.@preserve dts hs mask randU randN pts ind rec begin
    check(ccall((:kdeb200_gibbs, LIB), Cint,
                (Ptr{Ptr{Cvoid}}, Cint, Int64, Cint, Cint, Ptr{UInt8}, Ptr{Float64}, Int64, Ptr{Float64}, Int64,
                 UInt64, Int64, Int64, Ptr{Float64}, Ptr{Int64}, Ptr{Int64}),
                hs, Ndens, Np, Niter, addEntropy, mask, uptr, randU === nothing ? 0 : length(randU),
                nptr, randN === nothing ? 0 : length(randN), seed, 0, Np, pts, ind,
                record ? pointer(rec) : Ptr{Int64}(C_NULL)))
  end
  if record   # same nesting as the reference fills it at :109-112 (entries of levels never visited are absent)
    for s in 1:Np
      glbs.labelsChoosen[s] = Dict{Int,Dict{Int,Int}}()
      for j in 1:Ndens
        glbs.labelsChoosen[s][j] = Dict{Int,Int}()
        for l in 1:Int(nlev[])
          rec[l, j, s] >= 0 && (glbs.labelsChoosen[s][j][l] = rec[l, j, s])
        end
      end
    end
  end
  nothing
end

# ---- S2: evaluate -------------------------------------------------------------------------
# p is filled in the original order of `locations`' points (bd === locations => leave-one-out).
function evaluate!(bd::BallTreeDensity, locations::BallTreeDensity, p::Vector{Float64},
                   maxErr::Float64=1e-3, addop=(+,), diffop=(-,); precision::Int=0)
  bd.bt.dims == locations.bt.dims || error("evaluate -- dimensions of two BallTreeDensities must match")
  euclidean(addop, diffop) || error("kdeb200: only the default Euclidean (+,-) manifold is supported")
  dt = DeviceTree(bd; gibbs=false)
  if bd === locations
    GC.@preserve dt p check(ccall((:kdeb200_eval, LIB), Cint,
      (Ptr{Cvoid}, Ptr{Float64}, Int64, Cint, Cint, Ptr{Float64}), dt.h, C_NULL, Npts(bd), 1, precision, p))
  else
    pos = getPoints(locations)   # d x M, original order
    GC.@preserve dt pos p check(ccall((:kdeb200_eval, LIB), Cint,
      (Ptr{Cvoid}, Ptr{Float64}, Int64, Cint, Cint, Ptr{Float64}), dt.h, pos, size(pos, 2), 0, precision, p))
  end
  nothing
end

function evaluateDualTree(bd::BallTreeDensity, pos::Matrix{Float64}, lvFlag::Bool=false; precision::Int=0)
  bd.bt.dims == size(pos, 1) || error("bd and pos must have the same dimension")
  dt = DeviceTree(bd; gibbs=false)
  M = lvFlag ? Npts(bd) : size(pos, 2)
  p = zeros(M)
  GC.@preserve dt pos p check(ccall((:kdeb200_eval, LIB), Cint,
    (Ptr{Cvoid}, Ptr{Float64}, Int64, Cint, Cint, Ptr{Float64}), dt.h, pos, M, lvFlag, precision, p))
  return p
end

# ---- S3: leave-one-out entropy (one launch, one scalar back) ------------------------------------
function entropy(bd::BallTreeDensity, dt::DeviceTree=DeviceTree(bd; gibbs=false))
  H = Ref{Float64}(0.0)
  bw = bd.bandwidthMin[1:bd.bt.dims]     # the (possibly alpha^2-scaled) leaf variances
  GC.@preserve dt bw check(ccall((:kdeb200_loo_entropy, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ref{Float64}),
                                 dt.h, bw, H))
  return H[]
end

# the bandwidth loop of kde!(points) (src/KDE01.jl:13-23) in one call; N <= 512: one kernel launch
function lcv_bandwidths(points::Matrix{Float64})
  d, N = size(points)
  bw = zeros(d)
  GC.@preserve points bw check(ccall((:kdeb200_kde_lcv, LIB), Cint,
    (Cint, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Cint}), d, N, points, bw, C_NULL))
  return bw
end

# multi-GPU form (one Julia process per GPU): this process owns leaf rows j0+1:j1 of every nLOO_LL evaluation;
# `allreduce` is a C-callable that sums the partial likelihood and maxes the zero flag over the processes, e.g.
#   function ar(ps::Ptr{Float64}, pf::Ptr{Cint}, ::Ptr{Cvoid})::Cint
#     unsafe_store!(ps, MPI.Allreduce(unsafe_load(ps), +, comm)); unsafe_store!(pf, MPI.Allreduce(unsafe_load(pf), max, comm)); 0
#   end
#   lcv_bandwidths_sharded(points, j0, j1, @cfunction(ar, Cint, (Ptr{Float64}, Ptr{Cint}, Ptr{Cvoid})))
function lcv_bandwidths_sharded(points::Matrix{Float64}, j0::Integer, j1::Integer, allreduce::Ptr{Cvoid})
  d, N = size(points)
  bw = zeros(d)
  GC.@preserve points bw check(ccall((:kdeb200_kde_lcv_sharded, LIB), Cint,
    (Cint, Int64, Ptr{Float64}, Int64, Int64, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}, Ptr{Cint}),
    d, N, points, j0, j1, allreduce, C_NULL, bw, C_NULL))
  return bw
end

# `*` (src/MSGibbs01.jl:707-726) in one call: product samples + the LOOCV bandwidths of kde!(pGM); up to 512 samples never
# leave the device between the Gibbs kernel and the refit.  Returns the product density.
function product(trees::Vector{BallTreeDensity}; addEntropy::Bool=true, Niter::Int=5, seed::UInt64=rand(UInt64))
  Np = round(Int, sum(Npts.(trees)) / length(trees))
  d = Ndim(trees[1])
  dts = [DeviceTree(t) for t in trees]
  hs = Ptr{Cvoid}[t.h for t in dts]
  pts = zeros(d, Np); bw = zeros(d)
  GC.@preserve dts hs pts bw check(ccall((:kdeb200_product_kde, LIB), Cint,
    (Ptr{Ptr{Cvoid}}, Cint, Int64, Cint, Cint, Ptr{UInt8}, UInt64, Ptr{Float64}, Ptr{Int64}, Ptr{Float64}, Ptr{Cint}),
    hs, length(trees), Np, Niter, addEntropy, C_NULL, seed, pts, C_NULL, bw, C_NULL))
  return kde!(pts, bw)
end

# Many independent gibbs1 problems in one call (kdeb200_gibbs_batch: one launch per dimension, one CTA per 128 samples).
# tree_lists[i], Np[i]: problem i.  pts[i] (d_i*Np[i]) and ind[i] (Ndens_i x Np[i]) are filled in place, each equal to
# gibbs1!'s result for that problem alone.  partialDimMasks, randU, randN: nothing, or one entry (or nothing) per problem;
# a problem without streams draws from Philox(seeds[i]).
function gibbs1_batch!(tree_lists::Vector{Vector{BallTreeDensity}}, Np::Vector{Int}, Niter::Int,
                       pts::Vector{Vector{Float64}}, ind::Vector{Matrix{Int}};
                       addEntropy::Bool=true, partialDimMasks=nothing, randU=nothing, randN=nothing,
                       seeds::Vector{UInt64}=rand(UInt64, length(tree_lists)))
  n = length(tree_lists)
  ndens = Cint[length(ts) for ts in tree_lists]
  dims = [Ndim(ts[1]) for ts in tree_lists]
  dts = [DeviceTree(t) for ts in tree_lists for t in ts]
  hs = Ptr{Cvoid}[d.h for d in dts]
  mask = partialDimMasks === nothing ? UInt8[] :
    reduce(vcat, [m === nothing ? ones(UInt8, ndens[i] * dims[i]) :
                  UInt8[m[j][k] ? 0x01 : 0x00 for k in 1:dims[i], j in 1:ndens[i]] for (i, m) in enumerate(partialDimMasks)])
  U = randU === nothing ? Float64[] : reduce(vcat, [u === nothing ? Float64[] : u for u in randU]; init=Float64[])
  G = randN === nothing ? Float64[] : reduce(vcat, [g === nothing ? Float64[] : g for g in randN]; init=Float64[])
  nU = randU === nothing ? Int64[] : Int64[u === nothing ? 0 : length(u) for u in randU]
  nN = randN === nothing ? Int64[] : Int64[g === nothing ? 0 : length(g) for g in randN]
  P = zeros(sum(dims .* Np)); I = zeros(Int64, sum(ndens .* Np))
  GC.@preserve dts hs mask U G nU nN P I begin
    check(ccall((:kdeb200_gibbs_batch, LIB), Cint,
                (Cint, Ptr{Cint}, Ptr{Ptr{Cvoid}}, Ptr{Int64}, Cint, Cint, Ptr{UInt8}, Ptr{Float64}, Ptr{Int64},
                 Ptr{Float64}, Ptr{Int64}, Ptr{UInt64}, Ptr{Float64}, Ptr{Int64}),
                n, ndens, hs, Int64.(Np), Niter, addEntropy, partialDimMasks === nothing ? C_NULL : mask,
                randU === nothing ? C_NULL : U, randU === nothing ? C_NULL : nU,
                randN === nothing ? C_NULL : G, randN === nothing ? C_NULL : nN, seeds, P, I))
  end
  p0 = 0; i0 = 0
  for i in 1:n
    pts[i] .= P[p0+1:p0+dims[i]*Np[i]]
    ind[i] .= reshape(I[i0+1:i0+ndens[i]*Np[i]], Int(ndens[i]), Np[i])
    p0 += dims[i] * Np[i]; i0 += ndens[i] * Np[i]
  end
  nothing
end

# [product(ts; addEntropy, seed=s) for (ts, s) in zip(tree_lists, seeds)] with the Gibbs steps and the LOOCV refits in
# one call (kdeb200_product_kde_batch); what `*` answers on the host (one density without entropy, fewer than two
# product samples) is answered the same way here.
function product_batch(tree_lists::Vector{Vector{BallTreeDensity}}; addEntropy::Bool=true,
                       seeds::Vector{UInt64}=rand(UInt64, length(tree_lists)))
  res = Vector{BallTreeDensity}(undef, length(tree_lists))
  dev = Int[]
  for (i, ts) in enumerate(tree_lists)
    numpts = round(Int, sum(Npts.(ts)) / length(ts))
    if length(ts) == 1 && !addEntropy
      res[i] = kde!(getPoints(ts[1]))
    elseif numpts < 2
      d = Ndim(ts[1]); pts = zeros(d * numpts); ind = zeros(Int, length(ts), numpts)
      gibbs1!(length(ts), ts, numpts, 5, pts, ind, nothing, nothing; addEntropy=addEntropy, seed=seeds[i])
      res[i] = kde!(reshape(pts, d, numpts))
    else
      push!(dev, i)
    end
  end
  isempty(dev) && return res
  ndens = Cint[length(tree_lists[i]) for i in dev]
  dims = [Ndim(tree_lists[i][1]) for i in dev]
  Np = Int64[round(Int, sum(Npts.(tree_lists[i])) / length(tree_lists[i])) for i in dev]
  dts = [DeviceTree(t) for i in dev for t in tree_lists[i]]
  hs = Ptr{Cvoid}[d.h for d in dts]
  sd = seeds[dev]
  P = zeros(sum(dims .* Np)); bw = zeros(sum(dims))
  GC.@preserve dts hs sd P bw check(ccall((:kdeb200_product_kde_batch, LIB), Cint,
    (Cint, Ptr{Cint}, Ptr{Ptr{Cvoid}}, Ptr{Int64}, Cint, Cint, Ptr{UInt8}, Ptr{UInt64}, Ptr{Float64}, Ptr{Int64},
     Ptr{Float64}, Ptr{Cint}),
    length(dev), ndens, hs, Np, 5, addEntropy, C_NULL, sd, P, C_NULL, bw, C_NULL))
  p0 = 0; b0 = 0
  for (k, i) in enumerate(dev)
    res[i] = kde!(reshape(P[p0+1:p0+dims[k]*Np[k]], dims[k], Np[k]), bw[b0+1:b0+dims[k]])
    p0 += dims[k] * Np[k]; b0 += dims[k]
  end
  return res
end

# [evaluateDualTree(bd, pos, lv) for (bd, pos, lv) in zip(densities, positions, lvFlags)] in one call (kdeb200_eval_batch:
# one brute-force launch per dimension and leave-one-out flag).  positions[i] is d_i x M_i; a leave-one-out problem
# ignores its entry.  Each result is bit for bit the single call's (pruning modes 0 and 1).
function evaluate_batch(densities::Vector{BallTreeDensity}, positions::Vector{Matrix{Float64}},
                        lvFlags::Vector{Bool}=fill(false, length(densities)))
  n = length(densities)
  for i in 1:n
    lvFlags[i] || Ndim(densities[i]) == size(positions[i], 1) ||
      error("evaluate_batch: problem $(i-1): bd and pos must have the same dimension")
  end
  dts = [DeviceTree(bd; gibbs=false) for bd in densities]
  hs = Ptr{Cvoid}[d.h for d in dts]
  M = Int64[lvFlags[i] ? Npts(densities[i]) : size(positions[i], 2) for i in 1:n]
  loo = Cint[lv ? 1 : 0 for lv in lvFlags]
  Q = reduce(vcat, [vec(positions[i]) for i in 1:n if !lvFlags[i]]; init=Float64[])
  P = zeros(sum(M; init=0))
  GC.@preserve dts hs M loo Q P check(ccall((:kdeb200_eval_batch, LIB), Cint,
    (Cint, Ptr{Ptr{Cvoid}}, Ptr{Int64}, Ptr{Cint}, Ptr{Float64}, Cint, Ptr{Float64}), n, hs, M, loo, Q, 0, P))
  res = Vector{Vector{Float64}}(undef, n)
  o = 0
  for i in 1:n
    res[i] = P[o+1:o+M[i]]
    o += M[i]
  end
  return res
end

# [lcv_bandwidths(p) for p in point_sets] in one call (kdeb200_kde_lcv_batch): sets of at most 512 points in one launch,
# larger ones by the bandwidth loop one after the other.  kde!(p, bw) then builds each density as kde!(p) does.
function kde_lcv_batch(point_sets::Vector{Matrix{Float64}})
  n = length(point_sets)
  d = Cint[size(p, 1) for p in point_sets]
  N = Int64[size(p, 2) for p in point_sets]
  pts = reduce(vcat, [vec(p) for p in point_sets]; init=Float64[])
  bw = zeros(sum(d; init=0))
  GC.@preserve d N pts bw check(ccall((:kdeb200_kde_lcv_batch, LIB), Cint,
    (Cint, Ptr{Cint}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Ptr{Cint}), n, d, N, pts, bw, C_NULL))
  res = Vector{Vector{Float64}}(undef, n)
  b0 = 0
  for i in 1:n
    res[i] = bw[b0+1:b0+d[i]]
    b0 += d[i]
  end
  return res
end

# sample(npd, Npts) (src/KDE01.jl:164-183) on the device; Philox(seed) variates (Julia's RNG streams can be injected as
# randU (Npts) / randN (d x Npts) through the C entry point directly)
function sample(npd::BallTreeDensity, Np::Int; seed::UInt64=rand(UInt64))
  dt = DeviceTree(npd; gibbs=false)
  pts = zeros(Ndim(npd), Np); ind = zeros(Int, Np)
  GC.@preserve dt pts ind check(ccall((:kdeb200_sample, LIB), Cint,
    (Ptr{Cvoid}, Int64, UInt64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}), dt.h, Np, seed, C_NULL, C_NULL, pts, ind))
  return pts, ind
end

# [sample(p, n; seed=s) for (p, n, s) in zip(densities, Np, seeds)] in one call (kdeb200_sample_batch: one launch for
# every problem of at most 2048 samples).  Each result is bit for bit the single call's.
function sample_batch(densities::Vector{BallTreeDensity}, Np::Vector{Int};
                      seeds::Vector{UInt64}=rand(UInt64, length(densities)))
  n = length(densities)
  (length(Np) == n && length(seeds) == n) || error("sample_batch: need one Np and one seed per density")
  dts = [DeviceTree(p; gibbs=false) for p in densities]
  hs = Ptr{Cvoid}[d.h for d in dts]
  dims = [Ndim(p) for p in densities]
  N64 = Int64.(Np)
  P = zeros(sum(dims .* N64; init=0)); ind = zeros(Int64, sum(N64; init=0))
  GC.@preserve dts hs N64 seeds P ind check(ccall((:kdeb200_sample_batch, LIB), Cint,
    (Cint, Ptr{Ptr{Cvoid}}, Ptr{Int64}, Ptr{UInt64}, Ptr{Float64}, Ptr{Int64}, Ptr{Float64}, Ptr{Int64}, Ptr{Float64},
     Ptr{Int64}), n, hs, N64, seeds, C_NULL, C_NULL, C_NULL, C_NULL, P, ind))
  res = Vector{Tuple{Matrix{Float64},Vector{Int}}}(undef, n)
  p0 = 0; i0 = 0
  for i in 1:n
    res[i] = (reshape(P[p0+1:p0+dims[i]*N64[i]], dims[i], N64[i]), Int.(ind[i0+1:i0+N64[i]]))
    p0 += dims[i] * N64[i]; i0 += N64[i]
  end
  return res
end

# [resample(p, n) with Philox(seed)] for many densities in one call (kdeb200_resample_batch): the samples as
# sample_batch draws them, then the kde! LOOCV bandwidths of every sample set (Np <= 512 without the samples leaving the
# device); kde!(points, bw) then builds each density as kde!(points) does.
function resample_batch(densities::Vector{BallTreeDensity}, Np::Vector{Int}=[Npts(p) for p in densities];
                        seeds::Vector{UInt64}=rand(UInt64, length(densities)))
  n = length(densities)
  (length(Np) == n && length(seeds) == n) || error("resample_batch: need one Np and one seed per density")
  dts = [DeviceTree(p; gibbs=false) for p in densities]
  hs = Ptr{Cvoid}[d.h for d in dts]
  dims = [Ndim(p) for p in densities]
  N64 = Int64.(Np)
  P = zeros(sum(dims .* N64; init=0)); bw = zeros(sum(dims; init=0))
  GC.@preserve dts hs N64 seeds P bw check(ccall((:kdeb200_resample_batch, LIB), Cint,
    (Cint, Ptr{Ptr{Cvoid}}, Ptr{Int64}, Ptr{UInt64}, Ptr{Float64}, Ptr{Int64}, Ptr{Float64}, Ptr{Int64}, Ptr{Float64},
     Ptr{Int64}, Ptr{Float64}, Ptr{Cint}), n, hs, N64, seeds, C_NULL, C_NULL, C_NULL, C_NULL, P, C_NULL, bw, C_NULL))
  res = Vector{BallTreeDensity}(undef, n)
  p0 = 0; b0 = 0
  for i in 1:n
    res[i] = kde!(reshape(P[p0+1:p0+dims[i]*N64[i]], dims[i], N64[i]), bw[b0+1:b0+dims[i]])
    p0 += dims[i] * N64[i]; b0 += dims[i]
  end
  return res
end

# every 1-D marginal on its own grid in one launch (getKDEMax, src/DualTree01.jl:558-569): grids is G x d (column k = the
# abscissae of dimension k, i.e. the C side's d x G row-major), result likewise
function eval_marginals(p::BallTreeDensity, grids::Matrix{Float64})
  dt = DeviceTree(p; gibbs=false)
  out = similar(grids)
  GC.@preserve dt grids out check(ccall((:kdeb200_eval_marginals, LIB), Cint,
    (Ptr{Cvoid}, Ptr{Float64}, Int64, Ptr{Float64}), dt.h, grids, size(grids, 1), out))
  return out
end

# nLOO_LL with the device tree reused across the ~20 golden-section steps of one ksize call
function nLOO_LL(alpha::Float64, bd::BallTreeDensity, dt::DeviceTree)
  a2 = alpha^2
  KDE.updateBandwidth!(bd, bd.bandwidth * a2)
  H = entropy(bd, dt)
  KDE.updateBandwidth!(bd, bd.bandwidth / a2)
  return H
end

end # module
