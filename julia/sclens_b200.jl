# Reference-side binding of libsclens_b200.so: the `sclens(inp_df; device_="gpu")` method a
# maintainer of Mathbiomed/scLENS adds next to src/scLENS.jl:649.  It keeps the reference's
# signature and result Dict (:826-830) and replaces every CUDA.jl call on the path
# (:335-343, :365-369, :377, :505, :558, :561, :814-816) by one handle-based C-ABI session.
#
# NOT EXECUTED IN THIS REPOSITORY'S CI: the build image has no Julia.  The same call sequence is
# exercised from Python (sclens_b200/api.py) by the test-suite; keep the two in step.
module SclensB200

using DataFrames, SparseArrays

const LIB = get(ENV, "SCLENS_B200_LIB", "libsclens_b200.so")

# mirrors of the C structs in include/sclens_b200.h
struct SclConfig
    device::Int32; gram_mode::Int32; cta_group::Int32; verbose::Int32
    seed::UInt64
    subspace_extra::Int32; subspace_degree::Int32; exact_perturb::Int32
    gram_chunk_kb::Int32; gram_tc_diag::Int32; no_refine::Int32
    centering::Int32
    reserved::NTuple{3,Int32}
end
default_config(; verbose=0, seed=0, centering=0) =
    SclConfig(0, 0, 0, verbose, UInt64(seed), 0, 0, 0, 0, 0, 0, centering, ntuple(_ -> Int32(0), 3))
mutable struct SclSignalInfo
    N::Int32; M::Int32; nm::Int32; n_signal::Int32; n_Lmp::Int32; mp_iters::Int32; pass::Int32; gram_mode_used::Int32
    lambda_c::Float64; b_plus::Float64; b_minus::Float64; ks_static::Float64
    t_ingest_ms::Float64; t_normalize_ms::Float64; t_null_ms::Float64; t_gram_ms::Float64
    t_syevd_ms::Float64; t_fit_ms::Float64; t_backproject_ms::Float64
    SclSignalInfo() = new()
end
mutable struct SclRobustInfo
    n_search::Int32; n_perturb::Int32; min_pc::Int32; n_robust::Int32
    n_add::Int64
    p_sel::Float64; p_th::Float64
    t_baseline_ms::Float64; t_search_ms::Float64; t_search_syevd_ms::Float64
    t_perturb_ms::Float64; t_score_ms::Float64; t_outputs_ms::Float64
    n_subspace_fallbacks::Int32; reserved::Int32
    SclRobustInfo() = new()
end
struct SclUmapParams
    n_neighbors::Int32; n_components::Int32; n_epochs::Int32; metric::Int32
    init::Int32; neg_sample_rate::Int32; spectral_maxiter::Int32; reserved0::Int32
    min_dist::Float64; spread::Float64; learning_rate::Float64; repulsion_strength::Float64; local_connectivity::Float64
    seed::UInt64
    reserved::NTuple{4,Int32}
end
mutable struct SclUmapInfo
    a::Float64; b::Float64
    graph_nnz::Int64
    spectral_iters::Int32; init_fallback::Int32
    t_knn_ms::Float64; t_graph_ms::Float64; t_init_ms::Float64; t_layout_ms::Float64
    reserved::NTuple{4,Int32}
    SclUmapInfo() = new()
end
struct SclLeidenParams
    n_trials::Int32; max_iterations::Int32; max_sweeps::Int32; reserved0::Int32
    theta::Float64
    seed::UInt64
    reserved::NTuple{4,Int32}
end
mutable struct SclLeidenInfo
    max_levels::Int32; max_iterations::Int32; capped_levels::Int32; weight_shift::Int32
    copy_levels::Int64
    t_validate_ms::Float64; t_move_ms::Float64; t_refine_ms::Float64; t_aggregate_ms::Float64; t_labels_ms::Float64
    reserved::NTuple{4,Int32}
    SclLeidenInfo() = new()
end
struct SclClusterParams
    k_min::Int32; k_max::Int32; n_trials::Int32; max_rounds::Int32
    n_grid::Int32; max_widen::Int32; max_iterations::Int32; max_sweeps::Int32
    gamma_lo::Float64; gamma_hi::Float64; theta::Float64
    seed::UInt64
    reserved::NTuple{4,Int32}
end
mutable struct SclClusterInfo
    n_rounds::Int32; n_evaluated::Int32; n_found::Int32; weight_shift::Int32
    copy_levels::Int64
    t_validate_ms::Float64; t_leiden_ms::Float64; t_ecs_ms::Float64; t_total_ms::Float64
    reserved::NTuple{4,Int32}
    SclClusterInfo() = new()
end

function check(h, rc)
    rc == 0 && return
    msg = unsafe_string(ccall((:scl_last_error, LIB), Cstring, (Ptr{Cvoid},), h))
    error("libsclens_b200 error $rc: $msg")        # no CPU fallback: :379-381, :504-508, :741-745 become errors
end

"""
    sclens(inp_df; device_="gpu", th=60, p_step=0.001, n_perturb=20, centering="mean")

Drop-in for `scLENS.sclens` (src/scLENS.jl:649).  `df2sparr` is the reference's own (:90-120).
"""
function sclens(inp_df, df2sparr; device_="gpu", th=60, p_step=0.001, n_perturb=20, centering="mean", seed=0)
    device_ == "gpu" || error("sclens_b200 implements device_=\"gpu\" only")
    centering in ("mean", "median") || (println("Warning: The specified centering method is not supported in the current algorithm. scLENS will automatically use mean centering."); centering = "mean")   # :655-657
    println("Extracting matrices")
    X_ = df2sparr(inp_df)::SparseMatrixCSC{Float32,UInt32}
    N, M = size(X_)
    cfg = Ref(default_config(verbose=1, seed=seed, centering=(centering == "median" ? 1 : 0)))
    hr = Ref{Ptr{Cvoid}}(C_NULL)
    rc = ccall((:scl_create, LIB), Int32, (Ptr{Ptr{Cvoid}}, Ptr{SclConfig}), hr, cfg)
    rc == 0 || check(C_NULL, rc)
    h = hr[]
    try
        # Julia arrays are 1-based: index_base = 1; the library rebases on the device
        check(h, ccall((:scl_set_counts_csc, LIB), Int32,
                       (Ptr{Cvoid}, Int32, Int32, Int64, Ptr{UInt32}, Ptr{UInt32}, Ptr{Float32}, Int32),
                       h, N, M, nnz(X_), X_.colptr, X_.rowval, X_.nzval, 1))
        println("Extracting Signals...")
        si = SclSignalInfo()
        check(h, ccall((:scl_run_signal, LIB), Int32, (Ptr{Cvoid}, Ref{SclSignalInfo}), h, si))
        L = Vector{Float32}(undef, si.nm);  check(h, ccall((:scl_get_L, LIB), Int32, (Ptr{Cvoid}, Ptr{Float32}), h, L))
        L_mp = Vector{Float32}(undef, si.n_Lmp); check(h, ccall((:scl_get_Lmp, LIB), Int32, (Ptr{Cvoid}, Ptr{Float32}), h, L_mp))
        if si.n_signal == 0
            println("warning: There is no signal")
            return Dict(:L => L, :L_mp => L_mp, :λ => si.lambda_c, :cell_id => string.(inp_df.cell))
        end
        ri = SclRobustInfo()
        check(h, ccall((:scl_run_robustness, LIB), Int32, (Ptr{Cvoid}, Float64, Float64, Int32, Ref{SclRobustInfo}),
                       h, th, p_step, n_perturb, ri))
        k = Int(si.n_signal)
        nL = Vector{Float32}(undef, k);      check(h, ccall((:scl_get_signal_ev, LIB), Int32, (Ptr{Cvoid}, Ptr{Float32}), h, nL))
        nV = Matrix{Float32}(undef, N, k);   check(h, ccall((:scl_get_signal_evec, LIB), Int32, (Ptr{Cvoid}, Ptr{Float32}), h, nV))
        gmat = Matrix{Float32}(undef, k, M); check(h, ccall((:scl_get_gene_basis, LIB), Int32, (Ptr{Cvoid}, Ptr{Float32}), h, gmat))
        npairs = div(n_perturb * (n_perturb - 1), 2)
        b_ = Matrix{Float32}(undef, k, npairs); m_score = Vector{Float64}(undef, k); sd_score = Vector{Float64}(undef, k)
        check(h, ccall((:scl_get_scores, LIB), Int32, (Ptr{Cvoid}, Ptr{Float32}, Ptr{Float64}, Ptr{Float64}), h, b_, m_score, sd_score))
        sig0 = Vector{Int32}(undef, ri.n_robust)
        ri.n_robust > 0 && check(h, ccall((:scl_get_sig_id, LIB), Int32, (Ptr{Cvoid}, Ptr{Int32}), h, sig0))
        sig_id = Int.(sig0) .+ 1                                       # back to 1-based
        rec_vals = Dict{String,Union{VecOrMat{Float64}}}()
        if centering == "mean"                                         # the reference records them on the mean path only (:676-695)
            tgc = Vector{Float64}(undef, N); l2 = Vector{Float64}(undef, N)
            mn = Matrix{Float64}(undef, 1, M); sd = Matrix{Float64}(undef, 1, M); ct = Matrix{Float64}(undef, 1, M)
            check(h, ccall((:scl_get_rec_vals, LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                           h, tgc, mn, sd, l2, ct))
            rec_vals["TGC"] = tgc; rec_vals["mat2_mean"] = mn; rec_vals["mat2_std"] = sd
            rec_vals["norm_tgc"] = l2; rec_vals["cent_"] = ct
        end
        println("Reconstructing reduced data...")
        Xout0 = nV .* (sqrt.(nL))'                                      # :810
        Xout1 = nV[:, sig_id] .* sqrt.(nL[sig_id])'                     # :811
        df_X0 = DataFrame(Xout0, :auto); insertcols!(df_X0, 1, :cell => inp_df.cell)
        df_X1 = DataFrame(Xout1, :auto); insertcols!(df_X1, 1, :cell => inp_df.cell)
        return Dict(:pca => df_X0, :pca_n1 => df_X1, :sig_id => sig_id, :L => L, :L_mp => L_mp, :λ => si.lambda_c,
                    :robustness_scores => Dict(:b_ => b_, :rob_score => m_score, :m_scores => m_score, :sd_scores => sd_score),
                    :signal_evec => nV, :signal_ev => nL, :cell_id => inp_df.cell, :gene_id => names(inp_df)[2:end],
                    :gene_basis => gmat, :pass => si.pass != 0, :rec_vals => rec_vals)
    finally
        ccall((:scl_destroy, LIB), Int32, (Ptr{Cvoid},), h)
    end
end

"""
    get_denoised_df(inp_obj; out32=false)

Drop-in for scLENS.get_denoised_df(inp_obj; device_="gpu") (src/scLENS.jl:889-931) on a result Dict of `sclens`:
one fused device kernel behind `scl_op_denoise` instead of the cu()/mul! of :893-896 and the broadcasts of :921-927.
"""
function get_denoised_df(inp_obj; out32::Bool=false)
    g_mat = Matrix{Float32}(inp_obj[:gene_basis][inp_obj[:sig_id], :])              # r x M  (:890)
    Xout0 = Matrix{Float32}(inp_obj[:pca_n1][!, 2:end])                             # N x r  (:891)
    N, r = size(Xout0); M = size(g_mat, 2)
    rv = inp_obj[:rec_vals]
    f64(x) = Vector{Float64}(vec(x))
    out = out32 ? Matrix{Float32}(undef, N, M) : Matrix{Float64}(undef, N, M)
    hr = Ref{Ptr{Cvoid}}(C_NULL)
    cfg = Ref(default_config())
    rc = ccall((:scl_create, LIB), Int32, (Ptr{Ptr{Cvoid}}, Ptr{SclConfig}), hr, cfg)
    rc == 0 || check(C_NULL, rc)
    h = hr[]
    try
        check(h, ccall((:scl_op_denoise, LIB), Int32,
                       (Ptr{Cvoid}, Int32, Int32, Int32, Ptr{Float32}, Ptr{Float32}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                        Ptr{Float64}, Ptr{Float64}, Int32, Ptr{Cvoid}),
                       h, N, M, r, Xout0, g_mat, f64(rv["TGC"]), f64(rv["mat2_mean"]), f64(rv["mat2_std"]),
                       f64(rv["norm_tgc"]), f64(rv["cent_"]), out32 ? 1 : 0, out))
    finally
        ccall((:scl_destroy, LIB), Int32, (Ptr{Cvoid},), h)
    end
    odf = DataFrame(out, inp_obj[:gene_id])                                         # :928
    insertcols!(odf, 1, :cell => inp_obj[:cell_id])                                 # :929
    odf
end

# metric of apply_umap!: :cosine / :euclidean, or a Distances.jl CosineDist() / Euclidean() (matched by type name, so
# Distances.jl need not be loaded here)
function umap_metric(metric)
    name = metric isa Symbol ? String(metric) : lowercase(String(nameof(typeof(metric))))
    name in ("cosine", "cosinedist") && return Int32(1)
    name in ("euclidean",) && return Int32(0)
    error("apply_umap!: unsupported metric $(metric) (cosine or euclidean)")
end

"""
    apply_umap!(l_inp; k=15, nc=2, md=0.1, metric=CosineDist(), n_epochs=300, seed=0)

Drop-in for scLENS.apply_umap! (src/scLENS.jl:863-873) on the device: exact kNN, fuzzy graph, spectral start and a
deterministic synchronous layout (DESIGN.md).  Reads `:pca_n1` when it exists and has at least one signal column,
otherwise `:pca`.  Stores `:umap` (N x nc) and `:umap_obj` = (graph = SparseMatrixCSC, knns, dists) (k x N, 1-based
indices, UMAP.jl's layout) and returns `l_inp`.
"""
function apply_umap!(l_inp; k=15, nc=2, md=0.1, metric=:cosine, n_epochs=300, seed=0)
    src = haskey(l_inp, :pca_n1) && size(l_inp[:pca_n1], 2) > 1 ? l_inp[:pca_n1] : l_inp[:pca]
    X = Matrix{Float32}(src[!, 2:end])                                              # N x r, column-major
    N, d = size(X)
    p = Ref(SclUmapParams(k, nc, n_epochs, umap_metric(metric), 0, 5, 100, 0, md, 1.0, 1.0, 1.0, 1.0, UInt64(seed),
                          ntuple(_ -> Int32(0), 4)))
    info = Ref(SclUmapInfo())
    emb = Matrix{Float32}(undef, N, nc)
    hr = Ref{Ptr{Cvoid}}(C_NULL)
    cfg = Ref(default_config())
    rc = ccall((:scl_create, LIB), Int32, (Ptr{Ptr{Cvoid}}, Ptr{SclConfig}), hr, cfg)
    rc == 0 || check(C_NULL, rc)
    h = hr[]
    try
        check(h, ccall((:scl_op_umap, LIB), Int32,
                       (Ptr{Cvoid}, Int32, Int32, Ptr{Float32}, Ptr{SclUmapParams}, Ptr{Float32}, Ptr{Float32}, Ptr{SclUmapInfo}),
                       h, N, d, X, p, C_NULL, emb, info))
        nnz = Ref{Int64}(0)
        check(h, ccall((:scl_get_umap_graph, LIB), Int32, (Ptr{Cvoid}, Ptr{Int64}, Ptr{UInt32}, Ptr{UInt32}, Ptr{Float32}),
                       h, nnz, C_NULL, C_NULL, C_NULL))
        rowptr = Vector{UInt32}(undef, N + 1); colidx = Vector{UInt32}(undef, nnz[]); val = Vector{Float32}(undef, nnz[])
        check(h, ccall((:scl_get_umap_graph, LIB), Int32, (Ptr{Cvoid}, Ptr{Int64}, Ptr{UInt32}, Ptr{UInt32}, Ptr{Float32}),
                       h, nnz, rowptr, colidx, val))
        knns = Matrix{Int32}(undef, k, N); dists = Matrix{Float32}(undef, k, N)   # row-major N x k == column-major k x N
        check(h, ccall((:scl_get_umap_knn, LIB), Int32, (Ptr{Cvoid}, Ptr{Int32}, Ptr{Float32}), h, knns, dists))
        # the graph is symmetric: its CSR arrays are the CSC arrays of the same matrix
        graph = SparseMatrixCSC(N, N, Int.(rowptr) .+ 1, Int.(colidx) .+ 1, val)
        l_inp[:umap] = emb
        l_inp[:umap_obj] = (graph = graph, knns = knns .+ Int32(1), dists = dists)
    finally
        ccall((:scl_destroy, LIB), Int32, (Ptr{Cvoid},), h)
    end
    l_inp
end

"""
    clustering!(l_inp; k_min=2, k_max=20, n_trials=50, seed=0)

scICE-style clustering on the device from `l_inp[:umap_obj].graph` (run `apply_umap!` first): `n_trials` Leiden trials
per resolution, a resolution search for every cluster count in k_min:k_max and the inconsistency coefficient of each.
Stores `:graph`, `:n_cluster` (the counts found), `:ic` (aligned with `:n_cluster`), `:l_df` (DataFrame: `:cell` plus
one column `:k_<k>` per found count, labels 1..k by cluster size) and `:cluster_obj` (gamma, share, info).
"""
function clustering!(l_inp; k_min=2, k_max=20, n_trials=50, seed=0, max_rounds=12)
    graph = l_inp[:umap_obj].graph                      # symmetric: its CSC arrays are the CSR arrays
    N = size(graph, 1)
    rowptr = UInt32.(graph.colptr .- 1); colidx = UInt32.(graph.rowval .- 1); val = Float64.(graph.nzval)
    p = Ref(SclClusterParams(k_min, k_max, n_trials, max_rounds, 16, 4, 10, 64, 0.01, 10.0, 0.01, UInt64(seed),
                             ntuple(_ -> Int32(0), 4)))
    nk = k_max - k_min + 1
    found = Vector{Int32}(undef, nk); gam = Vector{Float64}(undef, nk); share = Vector{Float64}(undef, nk)
    ic = Vector{Float64}(undef, nk); labels = Matrix{Int32}(undef, N, nk)     # row-major nk x N == column-major N x nk
    info = Ref(SclClusterInfo())
    hr = Ref{Ptr{Cvoid}}(C_NULL)
    cfg = Ref(default_config())
    rc = ccall((:scl_create, LIB), Int32, (Ptr{Ptr{Cvoid}}, Ptr{SclConfig}), hr, cfg)
    rc == 0 || check(C_NULL, rc)
    h = hr[]
    try
        check(h, ccall((:scl_op_cluster, LIB), Int32,
                       (Ptr{Cvoid}, Int32, Int64, Ptr{UInt32}, Ptr{UInt32}, Ptr{Float64}, Ptr{SclClusterParams}, Ptr{Int32},
                        Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Int32, Ptr{Float64}, Ptr{Int32}, Ptr{SclClusterInfo}),
                       h, N, length(val), rowptr, colidx, val, p, found, gam, share, ic, labels, 0, C_NULL, C_NULL, info))
    finally
        ccall((:scl_destroy, LIB), Int32, (Ptr{Cvoid},), h)
    end
    ks = [k_min + i - 1 for i in 1:nk if found[i] != 0]
    sel = [i for i in 1:nk if found[i] != 0]
    l_df = DataFrame(:cell => l_inp[:cell_id])
    for (k, i) in zip(ks, sel)
        l_df[!, Symbol("k_$(k)")] = labels[:, i] .+ 1
    end
    l_inp[:graph] = graph
    l_inp[:n_cluster] = ks
    l_inp[:ic] = ic[sel]
    l_inp[:l_df] = l_df
    l_inp[:cluster_obj] = (gamma = gam[sel], share = share[sel], info = info[])
    l_inp
end

# a new handle for one call, destroyed afterwards
function with_handle(f)
    hr = Ref{Ptr{Cvoid}}(C_NULL)
    cfg = Ref(default_config())
    rc = ccall((:scl_create, LIB), Int32, (Ptr{Ptr{Cvoid}}, Ptr{SclConfig}), hr, cfg)
    rc == 0 || check(C_NULL, rc)
    h = hr[]
    try
        return f(h)
    finally
        ccall((:scl_destroy, LIB), Int32, (Ptr{Cvoid},), h)
    end
end

"""
    leiden(graph, resolutions; n_trials=50, seed=0, max_iterations=10, max_sweeps=64, theta=0.01)

Leiden trials on a symmetric SparseMatrixCSC: labels (N x T x R, ids 1..k by cluster size), cluster counts and
modularity (T x R each).
"""
function leiden(graph::SparseMatrixCSC, resolutions::Vector{Float64}; n_trials=50, seed=0, max_iterations=10, max_sweeps=64,
                theta=0.01)
    N = size(graph, 1); R = length(resolutions)
    rowptr = UInt32.(graph.colptr .- 1); colidx = UInt32.(graph.rowval .- 1); val = Float64.(graph.nzval)
    p = Ref(SclLeidenParams(n_trials, max_iterations, max_sweeps, 0, theta, UInt64(seed), ntuple(_ -> Int32(0), 4)))
    labels = Array{Int32}(undef, N, n_trials, R); ncl = Matrix{Int32}(undef, n_trials, R); q = Matrix{Float64}(undef, n_trials, R)
    info = Ref(SclLeidenInfo())
    with_handle() do h
        check(h, ccall((:scl_op_leiden, LIB), Int32,
                       (Ptr{Cvoid}, Int32, Int64, Ptr{UInt32}, Ptr{UInt32}, Ptr{Float64}, Int32, Ptr{Float64}, Ptr{SclLeidenParams},
                        Ptr{Int32}, Ptr{Int32}, Ptr{Float64}, Ptr{SclLeidenInfo}),
                       h, N, length(val), rowptr, colidx, val, R, resolutions, p, labels, ncl, q, info))
    end
    (labels = labels .+ Int32(1), n_clusters = ncl, modularity = q, info = info[])
end

"""
    label_ecs(labels)

T x T element-centric similarity of the columns of `labels` (N x T, ids 1..k per column).
"""
function label_ecs(labels::Matrix{<:Integer})
    N, T = size(labels)
    L = Int32.(labels .- 1)
    S = Matrix{Float64}(undef, T, T)
    with_handle() do h
        check(h, ccall((:scl_op_label_ecs, LIB), Int32, (Ptr{Cvoid}, Int32, Int32, Ptr{Int32}, Ptr{Float64}), h, T, N, L, S))
    end
    S
end

end # module
