# BulkLMMB200.jl — Julia shim over libblmm_b200.so (include/blmm_b200.h).
#
# Keeps the reference's public API for the multi-trait genome-scan path and replaces the bodies by
# `ccall`s into the sm_100a CUDA library:
#
#     bulkscan(Y, G, K; ...), bulkscan(Y, G, Covar, K; ...)          src/bulkscan.jl:81-162
#     bulkscan_null / bulkscan_null_grid / bulkscan_alt_grid         src/bulkscan.jl:188-526
#     scan(y, g, K; permutation_test = true, nperms, rndseed, ...)   src/scan.jl:94-271, 485-557
#     calcKinship(geno)                                              src/kinship.jl:4-14
#     transform_rotation(y, g, K; ...)                               src/transform_helpers.jl:1-54
#
# STATUS: EXPERIMENTAL.  Julia is not installed in the build image, so this file has been written against the C
# header but NOT executed there; tests/cabi_smoke.c drives the same entry points with hand-built structs exactly as
# these `ccall`s do (no Python in between).  The same ABI is exercised end to end from Python ctypes
# (bulklmm.jl_b200/blmm_b200/_lib.py, tests/test_gpu_*.py); the struct layouts below mirror
# `_lib.Problem` / `_lib.Opts` field by field.  See INTEGRATION.md for how a maintainer wires it in.
module BulkLMMB200

using LinearAlgebra, Random, Statistics

export bulkscan, bulkscan_peaks, bulkscan_null, bulkscan_null_grid, bulkscan_alt_grid, scan, calcKinship, transform_rotation, Context,
       get_thresholds, thresholds_from_max, lod2log10p, readBXDpheno, readBXDgeno, readGenoProb_ExcludeComplements

const libblmm = get(ENV, "BLMM_B200_LIB", "libblmm_b200.so")

# ---- mirrors of include/blmm_b200.h ------------------------------------------------------------------
const BLMM_MEM_HOST = Cint(0)
const METHOD_NULL_GRID, METHOD_ALT_GRID, METHOD_NULL_EXACT = Cint(0), Cint(1), Cint(2)
const H2PANEL_REFERENCE, H2PANEL_ARGMAX = Cint(0), Cint(1)
const DECOMP_EIGEN, DECOMP_SVD = Cint(0), Cint(1)

struct BlmmProblem            # blmm_problem
    n::Int64; p::Int64; m::Int64; c::Int64
    Y::Ptr{Float64}; G::Ptr{Float64}; Covar::Ptr{Float64}; U::Ptr{Float64}; lambda::Ptr{Float64}
    obs_weights::Ptr{Float64}   # C_NULL or the `weights` keyword (rows scaled on the device)
end

struct BlmmOpts               # blmm_opts
    method::Int32; reml::Int32
    prior_variance::Float64; prior_sample_size::Float64
    h2_grid::Ptr{Float64}; ngrid::Int32
    optim_interval::Int32; h2_panel_mode::Int32; mem_space::Int32
    ld_out::Int64
    chisq_df::Int32; reserved::Int32
    log10p_out::Ptr{Float64}    # `output_pvals`: -log10 p of every LOD, written next to L
end
BlmmOpts(method, reml, pv, pss, grid, ngrid, oi, mode, ms, ld) =
    BlmmOpts(method, reml, pv, pss, grid, ngrid, oi, mode, ms, ld, Int32(0), Int32(0), Ptr{Float64}(C_NULL))

mutable struct Context
    handle::Ptr{Cvoid}
    # One GPU (`Context(0)`), or several GPUs of this box behind one context (`Context([0, 1, 2, 3])`,
    # blmm_create_multi): the library then shards traits / permutation columns over them — the GPU analogue of the
    # reference's `nb` trait blocks (src/bulkscan.jl:263-309) — and every GPU writes its slab of the result arrays.
    function Context(device::Integer = 0)
        h = Ref{Ptr{Cvoid}}(C_NULL)
        st = ccall((:blmm_create, libblmm), Cint, (Ref{Ptr{Cvoid}}, Cint), h, device)
        st == 0 || error("blmm_create failed (status $st): no usable sm_100 (B200) device")
        ctx = new(h[])
        finalizer(c -> ccall((:blmm_destroy, libblmm), Cvoid, (Ptr{Cvoid},), c.handle), ctx)
        return ctx
    end
    function Context(devices::AbstractVector{<:Integer})
        h = Ref{Ptr{Cvoid}}(C_NULL)
        devs = Cint.(collect(devices))
        st = ccall((:blmm_create_multi, libblmm), Cint, (Ref{Ptr{Cvoid}}, Ptr{Cint}, Cint), h, devs, length(devs))
        st == 0 || error("blmm_create_multi failed (status $st)")
        ctx = new(h[])
        finalizer(c -> ccall((:blmm_destroy, libblmm), Cvoid, (Ptr{Cvoid},), c.handle), ctx)
        return ctx
    end
end
device_count(ctx::Context) = Int(ccall((:blmm_device_count, libblmm), Cint, (Ptr{Cvoid},), ctx.handle))

# `ndev` keyword of the scan entry points: 1 = the default one-GPU context; N > 1 = a cached context over GPUs 0..N-1
const _default_ctx = Ref{Union{Nothing, Context}}(nothing)
const _multi_ctx = Dict{Int, Context}()
default_context() = (_default_ctx[] === nothing && (_default_ctx[] = Context(0)); _default_ctx[])
context_for(ndev::Integer) = ndev <= 1 ? default_context() : get!(() -> Context(collect(0:ndev-1)), _multi_ctx, Int(ndev))

# The library reports the reference's own error strings; re-throw them as `error(msg)` so that code and
# tests matching on `e.msg` keep working (e.g. "Dimension mismatch.", src/transform_helpers.jl:9-11).
function check(ctx::Context, st::Cint)
    st == 0 && return nothing
    msg = unsafe_string(ccall((:blmm_last_error, libblmm), Cstring, (Ptr{Cvoid},), ctx.handle))
    throw(error(msg))
end

# ---- setup -------------------------------------------------------------------------------------------
function calcKinship(geno::Array{Float64, 2}; ctx::Context = default_context())
    (n, p) = size(geno)
    K = Array{Float64, 2}(undef, n, n)
    GC.@preserve geno K check(ctx, ccall((:blmm_kinship, libblmm), Cint,
        (Ptr{Cvoid}, Int64, Int64, Ptr{Float64}, Ptr{Float64}, Cint), ctx.handle, n, p, geno, K, BLMM_MEM_HOST))
    return K
end

function decompose(K::Array{Float64, 2}; decomp_scheme::String = "eigen", ctx::Context = default_context())
    decomp_scheme in ("eigen", "svd") ||
        throw(error("Please choose either `eigen` or `svd` for decomposition of the kinship matrix."))
    n = size(K, 1)
    U = Array{Float64, 2}(undef, n, n); lambda = Array{Float64, 1}(undef, n); nneg = Ref{Cint}(0)
    GC.@preserve K U lambda check(ctx, ccall((:blmm_decompose, libblmm), Cint,
        (Ptr{Cvoid}, Int64, Ptr{Float64}, Cint, Ptr{Float64}, Ptr{Float64}, Ref{Cint}, Cint),
        ctx.handle, n, K, decomp_scheme == "eigen" ? DECOMP_EIGEN : DECOMP_SVD, U, lambda, nneg, BLMM_MEM_HOST))
    nneg[] > 0 && @warn "Negative eigenvalues exist. The kinship matrix supplied may not be SPD."
    return U, lambda
end

function transform_rotation(y::Array{Float64, 2}, g::Array{Float64, 2}, K::Array{Float64, 2};
                            addIntercept::Bool = true, decomp_scheme::String = "eigen",
                            ctx::Context = default_context())
    n = size(y, 1)
    if (size(g, 1) != n) | (size(K, 1) != n)
        throw(error("Dimension mismatch."))
    end
    X = addIntercept ? [ones(n, 1) g] : g
    U, lambda = decompose(K; decomp_scheme = decomp_scheme, ctx = ctx)
    Y0 = similar(y); X0 = similar(X)
    prob = BlmmProblem(n, 0, size(y, 2), size(X, 2), pointer(y), C_NULL, pointer(X), pointer(U), pointer(lambda), C_NULL)
    GC.@preserve y X U lambda Y0 X0 check(ctx, ccall((:blmm_rotate, libblmm), Cint,
        (Ptr{Cvoid}, Ref{BlmmProblem}, Ptr{Float64}, Ptr{Float64}, Cint), ctx.handle, prob, Y0, X0, BLMM_MEM_HOST))
    return Y0, X0, lambda
end

# Argument plumbing shared by the scan entry points: the intercept column.  The observation weights
# (src/bulkscan.jl:231-250, 351-370, 457-476; src/scan.jl:204-222) cross the ABI as
# blmm_problem.obs_weights — Y, G and Covar are row-scaled on the device — and only the n x n kinship
# becomes W*K*W up front (blmm_weight_kinship) because it feeds the decomposition.
function prep(Y, G, Covar, K, weights, addIntercept; ctx::Context = default_context())
    n = size(Y, 1)
    if (size(G, 1) != n) | (size(K, 1) != n)
        throw(error("Dimension mismatch."))
    end
    C = addIntercept ? [ones(n, 1) Covar] : Covar
    K = Array{Float64, 2}(K)
    w = Float64[]
    if !ismissing(weights)
        length(weights) == n || throw(error("Dimension mismatch."))
        w = Array{Float64, 1}(weights)
        Kw = similar(K)
        GC.@preserve K w Kw check(ctx, ccall((:blmm_weight_kinship, libblmm), Cint,
            (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Cint), ctx.handle, n, K, w, Kw, BLMM_MEM_HOST))
        K = Kw
    end
    return Array{Float64, 2}(Y), Array{Float64, 2}(G), Array{Float64, 2}(C), K, w
end
wptr(w::Array{Float64, 1}) = isempty(w) ? Ptr{Float64}(C_NULL) : pointer(w)

function run_bulkscan(method::Cint, Y, G, C, K, w, grid::Array{Float64, 1}; reml, prior_variance, prior_sample_size,
                      optim_interval, decomp_scheme, h2_panel_mode = H2PANEL_REFERENCE, output_pvals = false,
                      chisq_df = 1, ctx = default_context())
    (n, m) = size(Y); p = size(G, 2)
    U, lambda = decompose(K; decomp_scheme = decomp_scheme, ctx = ctx)
    L = Array{Float64, 2}(undef, p, m)
    H = method == METHOD_ALT_GRID ? Array{Float64, 2}(undef, p, m) : Array{Float64, 1}(undef, m)
    P = output_pvals ? Array{Float64, 2}(undef, p, m) : Array{Float64, 2}(undef, 0, 0)
    prob = BlmmProblem(n, p, m, size(C, 2), pointer(Y), pointer(G), pointer(C), pointer(U), pointer(lambda), wptr(w))
    opts = BlmmOpts(method, reml, prior_variance, prior_sample_size, pointer(grid), length(grid), optim_interval,
                    h2_panel_mode, BLMM_MEM_HOST, 0, output_pvals ? Int32(chisq_df) : Int32(0), Int32(0),
                    output_pvals ? pointer(P) : Ptr{Float64}(C_NULL))
    GC.@preserve Y G C U lambda w grid L H P check(ctx, ccall((:blmm_bulkscan, libblmm), Cint,
        (Ptr{Cvoid}, Ref{BlmmProblem}, Ref{BlmmOpts}, Ptr{Float64}, Ptr{Float64}), ctx.handle, prob, opts, L, H))
    return L, H, P
end

# NamedTuple assembly of src/bulkscan.jl:154-160 (p-values only on request)
pack(names::NTuple{2, Symbol}, L, H, P, output_pvals, chisq_df) = output_pvals ?
    NamedTuple{(names..., :log10Pvals_mat, :Chisq_df)}((L, H, P, chisq_df)) : NamedTuple{names}((L, H))

# ---- bulkscan family (src/bulkscan.jl) ------------------------------------------------------------------
function bulkscan_null_grid(Y::Array{Float64, 2}, G::Array{Float64, 2}, Covar::Array{Float64, 2},
                            K::Array{Float64, 2}, grid_list::Array{Float64, 1};
                            weights::Union{Missing, Array{Float64, 1}} = missing, addIntercept::Bool = true,
                            prior_variance::Float64 = 1.0, prior_sample_size::Float64 = 0.0, reml::Bool = false,
                            decomp_scheme::String = "eigen", output_pvals::Bool = false, chisq_df::Int64 = 1,
                            ndev::Int64 = 1)
    ctx = context_for(ndev)
    Ys, Gs, Cs, Ks, w = prep(Y, G, Covar, K, weights, addIntercept; ctx = ctx)
    L, h2, P = run_bulkscan(METHOD_NULL_GRID, Ys, Gs, Cs, Ks, w, grid_list; reml = reml, prior_variance = prior_variance,
                            prior_sample_size = prior_sample_size, optim_interval = 1, decomp_scheme = decomp_scheme,
                            output_pvals = output_pvals, chisq_df = chisq_df, ctx = ctx)
    return pack((:L, :h2_null_list), L, h2, P, output_pvals, chisq_df)
end
bulkscan_null_grid(Y, G, K, grid_list; kw...) =
    bulkscan_null_grid(Y, G, ones(size(Y, 1), 1), K, grid_list; addIntercept = false, kw...)

function bulkscan_alt_grid(Y::Array{Float64, 2}, G::Array{Float64, 2}, Covar::Array{Float64, 2},
                            K::Array{Float64, 2}, hsq_list::Array{Float64, 1};
                            weights::Union{Missing, Array{Float64, 1}} = missing, addIntercept::Bool = true,
                            prior_variance::Float64 = 1.0, prior_sample_size::Float64 = 0.0, reml::Bool = false,
                            decomp_scheme::String = "eigen", output_pvals::Bool = false, chisq_df::Int64 = 1,
                            ndev::Int64 = 1)
    ctx = context_for(ndev)
    Ys, Gs, Cs, Ks, w = prep(Y, G, Covar, K, weights, addIntercept; ctx = ctx)
    L, h2, P = run_bulkscan(METHOD_ALT_GRID, Ys, Gs, Cs, Ks, w, hsq_list; reml = reml, prior_variance = prior_variance,
                            prior_sample_size = prior_sample_size, optim_interval = 1, decomp_scheme = decomp_scheme,
                            output_pvals = output_pvals, chisq_df = chisq_df, ctx = ctx)
    return pack((:L, :h2_panel), L, h2, P, output_pvals, chisq_df)
end
bulkscan_alt_grid(Y, G, K, hsq_list; kw...) =
    bulkscan_alt_grid(Y, G, ones(size(Y, 1), 1), K, hsq_list; addIntercept = false, kw...)

function bulkscan_null(Y::Array{Float64, 2}, G::Array{Float64, 2}, Covar::Array{Float64, 2}, K::Array{Float64, 2};
                       nb::Int64 = Threads.nthreads(), nt_blas::Int64 = 1,   # CPU threading knobs: accepted, unused
                       weights::Union{Missing, Array{Float64, 1}} = missing, addIntercept::Bool = true,
                       prior_variance::Float64 = 1.0, prior_sample_size::Float64 = 0.0, reml::Bool = false,
                       optim_interval::Int64 = 1, decomp_scheme::String = "eigen", output_pvals::Bool = false,
                       chisq_df::Int64 = 1, ndev::Int64 = 1)
    ctx = context_for(ndev)
    Ys, Gs, Cs, Ks, w = prep(Y, G, Covar, K, weights, addIntercept; ctx = ctx)
    L, h2, P = run_bulkscan(METHOD_NULL_EXACT, Ys, Gs, Cs, Ks, w, Float64[0.0]; reml = reml,
                            prior_variance = prior_variance, prior_sample_size = prior_sample_size,
                            optim_interval = optim_interval, decomp_scheme = decomp_scheme,
                            output_pvals = output_pvals, chisq_df = chisq_df, ctx = ctx)
    return pack((:L, :h2_null_list), L, h2, P, output_pvals, chisq_df)
end
bulkscan_null(Y, G, K; kw...) = bulkscan_null(Y, G, ones(size(Y, 1), 1), K; addIntercept = false, kw...)

function bulkscan(Y::Array{Float64, 2}, G::Array{Float64, 2}, Covar::Array{Float64, 2}, K::Array{Float64, 2};
                  method::String = "null-grid", h2_grid::Array{Float64, 1} = collect(0.0:0.1:0.9),
                  nb::Int64 = Threads.nthreads(), nt_blas::Int64 = 1,
                  weights::Union{Missing, Array{Float64, 1}} = missing, addIntercept::Bool = true,
                  prior_variance::Float64 = 1.0, prior_sample_size::Float64 = 0.0, reml::Bool = false,
                  optim_interval::Int64 = 1, decomp_scheme::String = "eigen", output_pvals::Bool = false,
                  chisq_df::Int64 = 1, ndev::Int64 = 1)
    # `nb` / `nt_blas` (CPU threading knobs of the reference) are accepted and unused; `ndev` (not in the reference)
    # is their GPU counterpart: the number of GPUs the traits are sharded over inside the library.
    kw = (weights = weights, addIntercept = addIntercept, prior_variance = prior_variance,
          prior_sample_size = prior_sample_size, reml = reml, decomp_scheme = decomp_scheme,
          output_pvals = output_pvals, chisq_df = chisq_df, ndev = ndev)
    if method == "null-exact"
        return bulkscan_null(Y, G, Covar, K; nb = nb, nt_blas = nt_blas, optim_interval = optim_interval, kw...)
    elseif method == "null-grid"
        return bulkscan_null_grid(Y, G, Covar, K, h2_grid; kw...)
    elseif method == "alt-grid"
        return bulkscan_alt_grid(Y, G, Covar, K, h2_grid; kw...)
    end
    throw(error("unknown method"))
end
bulkscan(Y::Array{Float64, 2}, G::Array{Float64, 2}, K::Array{Float64, 2}; kw...) =
    bulkscan(Y, G, ones(size(Y, 1), 1), K; addIntercept = false, kw...)

# Per-trait peaks of `bulkscan` (same keywords) without the p x m matrices (blmm_bulkscan_peaks): for every trait j,
# lod[j] = L[marker[j], j] at findmax(L[:, j]) (marker 1-based), h2[j] = h2_panel[marker[j], j] (alt-grid) or
# h2_null_list[j]; log10Pvals with output_pvals.
function bulkscan_peaks(Y::Array{Float64, 2}, G::Array{Float64, 2}, Covar::Array{Float64, 2}, K::Array{Float64, 2};
                        method::String = "null-grid", h2_grid::Array{Float64, 1} = collect(0.0:0.1:0.9),
                        nb::Int64 = Threads.nthreads(), nt_blas::Int64 = 1,
                        weights::Union{Missing, Array{Float64, 1}} = missing, addIntercept::Bool = true,
                        prior_variance::Float64 = 1.0, prior_sample_size::Float64 = 0.0, reml::Bool = false,
                        optim_interval::Int64 = 1, decomp_scheme::String = "eigen", output_pvals::Bool = false,
                        chisq_df::Int64 = 1, ndev::Int64 = 1)
    codes = Dict("null-grid" => METHOD_NULL_GRID, "alt-grid" => METHOD_ALT_GRID, "null-exact" => METHOD_NULL_EXACT)
    haskey(codes, method) || throw(error("unknown method"))
    ctx = context_for(ndev)
    Ys, Gs, Cs, Ks, w = prep(Y, G, Covar, K, weights, addIntercept; ctx = ctx)
    (n, m) = size(Ys); p = size(Gs, 2)
    U, lambda = decompose(Ks; decomp_scheme = decomp_scheme, ctx = ctx)
    grid = method == "null-exact" ? Float64[0.0] : h2_grid
    lod, marker, h2 = Array{Float64, 1}(undef, m), Array{Int64, 1}(undef, m), Array{Float64, 1}(undef, m)
    P = output_pvals ? Array{Float64, 1}(undef, m) : Array{Float64, 1}(undef, 0)
    prob = BlmmProblem(n, p, m, size(Cs, 2), pointer(Ys), pointer(Gs), pointer(Cs), pointer(U), pointer(lambda), wptr(w))
    opts = BlmmOpts(codes[method], reml, prior_variance, prior_sample_size, pointer(grid), length(grid), optim_interval,
                    H2PANEL_REFERENCE, BLMM_MEM_HOST, 0, output_pvals ? Int32(chisq_df) : Int32(0), Int32(0),
                    output_pvals ? pointer(P) : Ptr{Float64}(C_NULL))
    GC.@preserve Ys Gs Cs U lambda w grid lod marker h2 P check(ctx, ccall((:blmm_bulkscan_peaks, libblmm), Cint,
        (Ptr{Cvoid}, Ref{BlmmProblem}, Ref{BlmmOpts}, Ptr{Float64}, Ptr{Int64}, Ptr{Float64}), ctx.handle, prob, opts,
        lod, marker, h2))
    marker .+= 1
    return output_pvals ? (lod = lod, marker = marker, h2 = h2, log10Pvals = P) : (lod = lod, marker = marker, h2 = h2)
end
bulkscan_peaks(Y::Array{Float64, 2}, G::Array{Float64, 2}, K::Array{Float64, 2}; kw...) =
    bulkscan_peaks(Y, G, ones(size(Y, 1), 1), K; addIntercept = false, kw...)

# ---- scan with permutations (src/scan.jl:485-557) ------------------------------------------------------
# The shuffles are drawn HERE with the reference's own RNG and seed (src/transform_helpers.jl:94-102,
# src/util.jl:162-179) and cross the ABI as 0-based indices, so permuted inputs match the reference
# bit for bit whatever the Julia version's MersenneTwister stream is.
function permutation_indices(n::Int64, nperms::Int64, rndseed::Int64)
    rng = MersenneTwister(rndseed)
    idx = Array{Int32, 2}(undef, n, nperms)
    base = collect(1:n)
    for s in 1:nperms
        idx[:, s] = Int32.(shuffle(rng, base) .- 1)   # shuffle(rng, x) permutes positions identically for any x
    end
    return idx
end

function scan(y::Array{Float64, 2}, g::Array{Float64, 2}, covar::Array{Float64, 2}, K::Array{Float64, 2};
              weights::Union{Missing, Array{Float64, 1}} = missing, prior_variance::Float64 = 0.0,
              prior_sample_size::Float64 = 0.0, addIntercept::Bool = true, reml::Bool = false,
              assumption::String = "null", method::String = "qr", optim_interval::Int64 = 1,
              permutation_test::Bool = false, nperms::Int64 = 1024, rndseed::Int64 = 0,
              profileLL::Bool = false, markerID::Int = 0, h2_grid::Array{Float64, 1} = Array{Float64, 1}(undef, 1),
              decomp_scheme::String = "eigen", output_pvals::Bool = false, chisq_df::Int64 = 1,
              ndev::Int64 = 1, ctx::Context = context_for(ndev))
    # keyword surface of src/scan.jl:182-199; `method` ("qr"/"cholesky") selects the reference's CPU factorisation and
    # has no counterpart here (the device path uses closed-form c x c Gram solves); `ndev` / `ctx` are additions.
    assumption in ("null", "alt") || throw(error("Assumption keyword is not supported. Please enter null or alt."))
    (assumption == "alt" && permutation_test) &&
        throw(error("Permutation test option currently is not supported for the alternative assumption."))
    size(y, 2) == 1 || throw(error("Can only handle one trait."))
    ys, gs, cs, Ks, w = prep(y, g, covar, K, weights, addIntercept; ctx = ctx)
    (n, p) = size(gs)
    U, lambda = decompose(Ks; decomp_scheme = decomp_scheme, ctx = ctx)
    prob = BlmmProblem(n, p, 1, size(cs, 2), pointer(ys), pointer(gs), pointer(cs), pointer(U), pointer(lambda), wptr(w))
    df = output_pvals ? Int32(chisq_df) : Int32(0)
    local results
    if assumption == "alt"      # scan_alt, src/scan.jl:397-453: variance components re-estimated per marker
        lod = Array{Float64, 1}(undef, p); h2e = Array{Float64, 1}(undef, p)
        s2 = Ref{Float64}(0.0); h2 = Ref{Float64}(0.0)
        opts = BlmmOpts(METHOD_NULL_EXACT, reml, prior_variance, prior_sample_size, C_NULL, 0, optim_interval,
                        H2PANEL_REFERENCE, BLMM_MEM_HOST, 0)
        GC.@preserve ys gs cs U lambda w lod h2e check(ctx, ccall((:blmm_scan_alt, libblmm), Cint,
            (Ptr{Cvoid}, Ref{BlmmProblem}, Ref{BlmmOpts}, Ptr{Float64}, Ptr{Float64}, Ref{Float64}, Ref{Float64}),
            ctx.handle, prob, opts, lod, h2e, s2, h2))
        results = output_pvals ?
            (sigma2_e = s2[], h2_null = h2[], h2_each_marker = h2e, lod = lod, log10pvals = lod2log10p(lod, chisq_df; ctx = ctx)) :
            (sigma2_e = s2[], h2_null = h2[], h2_each_marker = h2e, lod = lod)
    elseif !permutation_test    # scan_null, src/scan.jl:310-360
        lod = Array{Float64, 2}(undef, p, 1); s2 = Ref{Float64}(0.0); h2 = Ref{Float64}(0.0)
        pv = output_pvals ? Array{Float64, 2}(undef, p, 1) : Array{Float64, 2}(undef, 0, 0)
        opts = BlmmOpts(METHOD_NULL_EXACT, reml, prior_variance, prior_sample_size, C_NULL, 0, optim_interval,
                        H2PANEL_REFERENCE, BLMM_MEM_HOST, 0, df, Int32(0), output_pvals ? pointer(pv) : Ptr{Float64}(C_NULL))
        GC.@preserve ys gs cs U lambda w lod pv check(ctx, ccall((:blmm_scan_null, libblmm), Cint,
            (Ptr{Cvoid}, Ref{BlmmProblem}, Ref{BlmmOpts}, Ptr{Float64}, Ref{Float64}, Ref{Float64}),
            ctx.handle, prob, opts, lod, s2, h2))
        results = output_pvals ? (sigma2_e = s2[], h2_null = h2[], lod = vec(lod), log10pvals = vec(pv)) :
                                 (sigma2_e = s2[], h2_null = h2[], lod = vec(lod))
    else                        # scan_perms_lite, src/scan.jl:485-557
        perm = permutation_indices(n, nperms, rndseed)
        lod = Array{Float64, 1}(undef, p); L_perms = Array{Float64, 2}(undef, p, nperms)
        maxlod = Array{Float64, 1}(undef, nperms); s2 = Ref{Float64}(0.0); h2 = Ref{Float64}(0.0)
        opts = BlmmOpts(METHOD_NULL_EXACT, reml, prior_variance, prior_sample_size, C_NULL, 0, optim_interval,
                        H2PANEL_REFERENCE, BLMM_MEM_HOST, 0)
        GC.@preserve ys gs cs U lambda w perm lod L_perms maxlod check(ctx, ccall((:blmm_scan_perms, libblmm), Cint,
            (Ptr{Cvoid}, Ref{BlmmProblem}, Ref{BlmmOpts}, Ptr{Int32}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Ref{Float64}, Ref{Float64}), ctx.handle, prob, opts, perm, nperms, lod, L_perms, maxlod, s2, h2))
        if output_pvals
            # The reference throws UndefVarError here (`log10pvals = pvals`, src/scan.jl:551, SURVEY B2) and never
            # forwards chisq_df to scan_perms_lite (df = 1 there).  The intended result is returned instead.
            results = (sigma2_e = s2[], h2_null = h2[], lod = lod, log10pvals = lod2log10p(lod, 1; ctx = ctx),
                       L_perms = L_perms, log10Pvals_perms = lod2log10p(L_perms, 1; ctx = ctx))
        else
            results = (sigma2_e = s2[], h2_null = h2[], lod = lod, L_perms = L_perms)
        end
    end
    if profileLL
        # profile_LL (src/analysis_helpers/single_trait_analysis.jl:46-73): the null and the marker-model log-likelihood
        # on h2_grid — two blmm_grid_loglik calls (covariates, covariates + marker `markerID`), no intercept added
        # (the reference rotates with addIntercept = false at this point, on the arrays as they stand after the
        # weights block)
        (1 <= markerID <= p) || throw(BoundsError(gs, (1:n, markerID)))
        if ismissing(weights)   # covar as passed: the reference adds no intercept here even when addIntercept = true
            yst = ys; cst = Array{Float64, 2}(covar); gcol = gs[:, markerID:markerID]
        else                    # the arrays of the recursive call: W*y, W*[1 covar], W*g (src/scan.jl:204-222)
            yst = ys .* w; cst = cs .* w; gcol = gs[:, markerID:markerID] .* w
        end
        ell_null = grid_loglik(yst, cst, U, lambda, h2_grid; reml = reml, prior_variance = prior_variance,
                               prior_sample_size = prior_sample_size, ctx = ctx)
        ell_alt = grid_loglik(yst, [cst gcol], U, lambda, h2_grid; reml = reml, prior_variance = prior_variance,
                              prior_sample_size = prior_sample_size, ctx = ctx)
        return (results, (ll_list_null = vec(ell_null), ll_list_alt = vec(ell_alt)))
    end
    return results
end
function scan(y::Array{Float64, 2}, g::Array{Float64, 2}, K::Array{Float64, 2}; addIntercept::Bool = true, kw...)
    addIntercept || throw(error("Intercept has to be added when no other covariate is given."))
    return scan(y, g, ones(size(y, 1), 1), K; addIntercept = false, kw...)
end
# vector-trait methods, src/scan.jl:94-148
scan(y::Array{Float64, 1}, g::Array{Float64, 2}, K::Array{Float64, 2}; kw...) = scan(reshape(y, :, 1), g, K; kw...)
scan(y::Array{Float64, 1}, g::Array{Float64, 2}, covar::Array{Float64, 2}, K::Array{Float64, 2}; kw...) =
    scan(reshape(y, :, 1), g, covar, K; kw...)

# wls_multivar(...).Ell over a grid for the columns of Y (src/bulkscan_helpers.jl:267-269): |grid| x m
function grid_loglik(Y::Array{Float64, 2}, C::Array{Float64, 2}, U::Array{Float64, 2}, lambda::Array{Float64, 1},
                     grid::Array{Float64, 1}; reml::Bool = false, prior_variance::Float64 = 0.0,
                     prior_sample_size::Float64 = 0.0, ctx::Context = default_context())
    (n, m) = size(Y)
    ell = Array{Float64, 2}(undef, length(grid), m)
    prob = BlmmProblem(n, 0, m, size(C, 2), pointer(Y), C_NULL, pointer(C), pointer(U), pointer(lambda), C_NULL)
    opts = BlmmOpts(METHOD_NULL_GRID, reml, prior_variance, prior_sample_size, pointer(grid), length(grid), 1,
                    H2PANEL_REFERENCE, BLMM_MEM_HOST, 0)
    GC.@preserve Y C U lambda grid ell check(ctx, ccall((:blmm_grid_loglik, libblmm), Cint,
        (Ptr{Cvoid}, Ref{BlmmProblem}, Ref{BlmmOpts}, Ptr{Float64}), ctx.handle, prob, opts, ell))
    return ell
end

# src/analysis_helpers/single_trait_analysis.jl:13-23: column maxima here, sort + type-7 quantiles on the device
function get_thresholds(L::Array{Float64, 2}, signif_level::Array{Float64, 1}; ctx::Context = default_context())
    return thresholds_from_max(vec(maximum(L, dims = 1)), signif_level; ctx = ctx)
end

# The same from the per-permutation maxima blmm_scan_perms already returns (no L_perms needed).
function thresholds_from_max(maxlod::Array{Float64, 1}, signif_level::Array{Float64, 1}; ctx::Context = default_context())
    thrs = Array{Float64, 1}(undef, length(signif_level))
    GC.@preserve maxlod signif_level thrs check(ctx, ccall((:blmm_thresholds, libblmm), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Ptr{Float64}, Cint, Ptr{Float64}, Cint),
        ctx.handle, maxlod, length(maxlod), signif_level, length(signif_level), thrs, BLMM_MEM_HOST))
    return (probs = 1 .- signif_level, thrs = thrs)
end

# src/util.jl:199-206.  The reference defines the scalar method and broadcasts it (`lod2log10p.(L, df)`); both the
# scalar and the whole-array form are provided, so `lod2log10p.(L, 1)` and `lod2log10p(L, 1)` agree.
lod2log10p(lod::Float64, df::Int64; ctx::Context = default_context()) = lod2log10p([lod], df; ctx = ctx)[1]
function lod2log10p(lod::Array{Float64}, df::Int64 = 1; ctx::Context = default_context())
    out = similar(lod)
    GC.@preserve lod out check(ctx, ccall((:blmm_lod2log10p, libblmm), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Int64, Int64, Cint, Ptr{Float64}, Cint),
        ctx.handle, lod, length(lod), 1, 0, 0, df, out, BLMM_MEM_HOST))
    return out
end

# ---- data ingest (src/readData.jl:85-96, 159-165): parsed by the library's host threads ----------------------
function read_csv_matrix(file::AbstractString; skip_rows::Int64 = 1, first_col::Int64 = 0, col_step::Int64 = 1,
                         drop_last_cols::Int64 = 0, dlm::AbstractChar = ',')
    rows = Ref{Int64}(0); cols = Ref{Int64}(0); data = Ref{Ptr{Float64}}(C_NULL)
    st = ccall((:blmm_read_csv, libblmm), Cint,
               (Cstring, Cchar, Int64, Int64, Int64, Int64, Cint, Ref{Int64}, Ref{Int64}, Ref{Ptr{Float64}}),
               file, Cchar(dlm), skip_rows, first_col, col_step, drop_last_cols, Cint(-1), rows, cols, data)
    st == 0 || throw(error(unsafe_string(ccall((:blmm_io_last_error, libblmm), Cstring, ()))))
    out = copy(unsafe_wrap(Array, data[], (rows[], cols[])))
    ccall((:blmm_free_matrix, libblmm), Cvoid, (Ptr{Float64}, Cint), data[], Cint(-1))
    return out
end
readBXDpheno(file::AbstractString) = read_csv_matrix(file; skip_rows = 1, first_col = 1, drop_last_cols = 1)
readBXDgeno(file::AbstractString; skipstart = 1) = read_csv_matrix(file; skip_rows = skipstart, first_col = 1, col_step = 2)
readGenoProb_ExcludeComplements(file::AbstractString; dlm::AbstractChar = ',') =
    read_csv_matrix(file; skip_rows = 1, first_col = 1, col_step = 2, dlm = dlm)

end # module
