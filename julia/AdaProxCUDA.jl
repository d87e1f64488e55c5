# AdaProxCUDA.jl -- Julia binding of libadaprox_cuda.so (include/adaprox.h).
#
# NOT EXECUTED: Julia is not installed in the build image.  This file is the
# reference-side stub a maintainer would add; the same C ABI is exercised here
# through Python ctypes (adaptive-proximal-algorithms_b200/core.py).
#
# Usage: `using AdaProxCUDA` next to `using AdaProx`; then
#   AdaProxCUDA.adaptive_proxgrad(x0; f = AdaProx.Counting(f), g, rule, tol, maxit, name)
# has the signature of AdaProx.adaptive_proxgrad (src/AdaProx.jl:418) and emits
# the same `@logmsg Record` lines (src/AdaProx.jl:351) from the returned records.
module AdaProxCUDA

using Logging
using LinearAlgebra
using SparseArrays
import AdaProx
import ProximalCore
import ProximalOperators

const lib = get(ENV, "ADAPROX_CUDA_LIB", "libadaprox_cuda.so")
const Handle = Ptr{Cvoid}
const Id = Int64

# ---- structs of include/adaprox.h (isbits, same field order) -----------------
struct CProx
    kind::Int32; conjugate::Int32
    lambda::Float64; lo::Float64; hi::Float64
    lo_vec::Id; hi_vec::Id; shift::Id
end
struct CProblem
    f_kind::Int32; f_ipar::Int32
    f_mat::Id; f_vec::Id; f_c::Float64
    g::CProx; h::CProx
    A_mat::Id; n::Int64; m_dual::Int64
end
struct COptions
    solver::Int32; rule::Int32
    gamma::Float64; t::Float64; norm_A::Float64; delta::Float64; Theta::Float64; xi::Float64; nu::Float64; r::Float64
    R::Float64; eta::Float64; shrink::Float64; sigma::Float64; muf::Float64; mug::Float64; theta::Float64
    gamma_max::Float64; phi::Float64; tol::Float64
    maxit::Int64
    want_objective::Int32; counting_f::Int32; counting_g::Int32; counting_h::Int32; counting_A::Int32
    max_records::Int64
end
struct CRecord
    it::Int64
    gamma::Float64; sigma::Float64; norm_res::Float64; f_x::Float64; g_x::Float64; h_Ax::Float64
    f_evals::Int64; grad_f_evals::Int64; prox_g_evals::Int64; prox_h_evals::Int64; A_evals::Int64; At_evals::Int64
end
mutable struct CResult
    iters::Int64; flags::UInt32; reserved::Int32
    f_evals::Int64; grad_f_evals::Int64; prox_g_evals::Int64; prox_h_evals::Int64; A_evals::Int64; At_evals::Int64
    n_records::Int64
    final_gamma::Float64; final_sigma::Float64; final_norm_res::Float64; solve_ms::Float64; kernel_launches::Int64; matrix_passes::Int64; collective::Int64
    CResult() = new(0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0.0, 0.0, 0.0, 0.0, 0, 0, 0)
end

# ---- handle -------------------------------------------------------------------
const _handle = Ref{Handle}(C_NULL)
function handle()
    if _handle[] == C_NULL
        h = Ref{Handle}(C_NULL)
        rc = ccall((:adaprox_create, lib), Cint, (Ref{Handle}, Cint), h, parse(Int, get(ENV, "LOCAL_RANK", "0")))
        rc == 0 || error("adaprox_create failed (status $rc): no usable CUDA device; there is no CPU fallback")
        _handle[] = h[]
    end
    return _handle[]
end
check(rc) = rc == 0 ? nothing :
    error("adaprox status $rc: " * unsafe_string(ccall((:adaprox_last_error, lib), Cstring, (Handle,), handle())))

# ---- device-resident data -------------------------------------------------------
function upload(A::Matrix{Float64})                       # Julia layout: column-major
    id = Ref{Id}(0)
    check(ccall((:adaprox_matrix_upload_colmajor, lib), Cint, (Handle, Ptr{Float64}, Int64, Int64, Int64, Ref{Id}),
                handle(), A, size(A, 1), size(A, 2), stride(A, 2), id))
    return id[]
end
function upload(A::SparseMatrixCSC{Float64})              # CSC(A) = CSR(A'), so transpose once on the host
    At = sparse(transpose(A))                             # CSC of A' == CSR of A
    rowptr = Int64.(At.colptr .- 1); colind = Int32.(At.rowval .- 1)
    id = Ref{Id}(0)
    check(ccall((:adaprox_matrix_upload_csr, lib), Cint,
                (Handle, Int64, Int64, Int64, Ptr{Int64}, Ptr{Int32}, Ptr{Float64}, Ref{Id}),
                handle(), size(A, 1), size(A, 2), nnz(A), rowptr, colind, At.nzval, id))
    return id[]
end
upload(A::AbstractMatrix) = upload(Matrix{Float64}(A))
function upload(v::AbstractVector)
    w = Vector{Float64}(v); id = Ref{Id}(0)
    check(ccall((:adaprox_vector_upload, lib), Cint, (Handle, Ptr{Float64}, Int64, Ref{Id}), handle(), w, length(w), id))
    return id[]
end

# ---- traits: one line per oracle struct of the experiment scripts ----------------
# A script opts in with e.g.  AdaProxCUDA.device_oracle(f::LinearLeastSquares) = AdaProxCUDA.least_squares(f.A, f.b)
unwrap(f) = f
unwrap(c::AdaProx.Counting) = c.f
iscounting(f) = f isa AdaProx.Counting
device_oracle(f) = error("eval_with_pullback not defined on the device for type $(typeof(f)) (no CPU fallback)")
device_oracle(::ProximalCore.Zero) = (kind = 0, ipar = 0, mat = 0, vec = 0, c = 0.0)
least_squares(A, b) = (kind = 1, ipar = 0, mat = upload(A), vec = upload(b), c = 0.0, n = size(A, 2))   # lasso/runme.jl:16-27
logistic(X, y) = (kind = 2, ipar = 0, mat = upload(X), vec = upload(y), c = 0.0)        # sparse_logreg/runme.jl:18-39
quadratic(Q, q) = (kind = 3, ipar = 0, mat = upload(Q), vec = upload(q), c = 0.0)       # dual_svm/runme.jl:19-28
quadratic_gram(Z, q) = (kind = 7, ipar = 0, mat = upload(Z), vec = upload(q), c = 0.0)  # Quadratic(Z*Z', q) by its factor: dual_svm/runme.jl:47-49 has Z = Dy*X
cubic(Q, q, c) = (kind = 4, ipar = 0, mat = upload(Q), vec = upload(q), c = Float64(c)) # cubic_sparse_logreg/runme.jl:20-32
worst_quadratic(k, L) = (kind = 5, ipar = Int(k), mat = 0, vec = 0, c = Float64(L))     # nesterov_worst_case/runme.jl:14-40

noprox() = CProx(0, 0, 1.0, 0.0, 0.0, 0, 0, 0)
device_prox(::ProximalCore.Zero) = CProx(0, 0, 1.0, 0.0, 0.0, 0, 0, 0)
device_prox(::ProximalCore.IndZero) = CProx(1, 0, 1.0, 0.0, 0.0, 0, 0, 0)
device_prox(g::ProximalOperators.NormL1) = CProx(2, 0, Float64(g.lambda), 0.0, 0.0, 0, 0, 0)
device_prox(g::ProximalOperators.NormL2) = CProx(3, 0, Float64(g.lambda), 0.0, 0.0, 0, 0, 0)
function device_prox(g::ProximalOperators.IndBox)
    (g.lb isa Real && g.ub isa Real) && return CProx(4, 0, 1.0, Float64(g.lb), Float64(g.ub), 0, 0, 0)
    n = max(length(g.lb), length(g.ub))
    return CProx(4, 0, 1.0, 0.0, 0.0, upload(fill(0.0, n) .+ g.lb), upload(fill(0.0, n) .+ g.ub), 0)
end
function device_prox(g::ProximalOperators.Translate)
    p = device_prox(g.f)
    return CProx(p.kind, 0, p.lambda, p.lo, p.hi, p.lo_vec, p.hi_vec, upload(g.b))
end
device_prox(c::AdaProx.Counting) = device_prox(c.f)
function device_prox(c::ProximalCore.ConvexConjugate)          # conjugate flag: Moreau on the device (src/AdaProx.jl:325 applies it to h)
    p = device_prox(c.f)
    return CProx(p.kind, 1, p.lambda, p.lo, p.hi, p.lo_vec, p.hi_vec, p.shift)
end

rule_fields(r::AdaProx.FixedStepsize) = (0, r.gamma, r.t, 0.0, 0.0, 1.2, 1.0, 1.0, 0.5)
rule_fields(r::AdaProx.MalitskyMishchenkoRule) = (1, r.gamma, r.t, 0.0, 0.0, 1.2, 1.0, 1.0, 0.5)
rule_fields(r::AdaProx.OurRule) = (2, r.gamma, r.t, r.norm_A, r.delta, r.Theta, 1.0, 1.0, 0.5)
rule_fields(r::AdaProx.OurRulePlus) = (3, r.gamma, 1.0, 0.0, 0.0, 1.2, r.xi, r.nu, r.r)

function options(solver; rule = (0, 0.0, 1.0, 0.0, 0.0, 1.2, 1.0, 1.0, 0.5), R = 0.95, eta = 1.0, shrink = 0.5, sigma = 0.0,
                 muf = 0.0, mug = 0.0, theta = -1.0, gamma_max = 1e6, phi = 1.5, tol, maxit, want, counting)
    (rk, gamma, t, norm_A, delta, Theta, xi, nu, r) = rule
    COptions(solver, rk, gamma, t, norm_A, delta, Theta, xi, nu, r, R, eta, shrink, sigma, muf, mug, theta, gamma_max, phi,
             tol, Int64(maxit), want, counting..., want == 1 ? Int64(maxit) : 0)
end

# ---- the generic call ---------------------------------------------------------------
function solve(solver, x0, y0; f, g, h = nothing, A = nothing, opts, name, pd)
    fo = device_oracle(unwrap(f))
    n = length(x0)
    Aid = pd ? upload(unwrap(A)) : 0
    md = pd ? size(unwrap(A), 1) : 0
    prob = CProblem(fo.kind, fo.ipar, fo.mat, fo.vec, fo.c, device_prox(g), pd ? device_prox(h) : noprox(), Aid, n, md)
    want = opts.want_objective
    recs = Vector{CRecord}(undef, max(want == 1 ? opts.maxit : 0, 1))
    res = CResult()
    x = Vector{Float64}(undef, n); y = Vector{Float64}(undef, max(md, 1))
    x0v = Vector{Float64}(x0); y0v = y0 === nothing ? Float64[] : Vector{Float64}(y0)
    GC.@preserve x0v y0v x y recs begin
        check(ccall((:adaprox_solve, lib), Cint,
                    (Handle, Ref{CProblem}, Ref{COptions}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                     Ptr{CRecord}, Ref{CResult}),
                    handle(), prob, opts, x0v, isempty(y0v) ? C_NULL : pointer(y0v), x, pd ? pointer(y) : C_NULL,
                    want == 1 ? pointer(recs) : C_NULL, res))
    end
    # src/counting.jl: the Counting wrappers accumulate exactly as the reference's do
    if iscounting(f); f.eval_count += res.f_evals; f.grad_count += res.grad_f_evals; end
    if iscounting(g); g.prox_count += res.prox_g_evals; end
    if pd && iscounting(h); h.prox_count += res.prox_h_evals; end
    if pd && iscounting(A); A.mul_count += res.A_evals; A.amul_count += res.At_evals; end
    for k in 1:res.n_records                                   # replay the records (src/AdaProx.jl:351)
        r = recs[k]
        @logmsg AdaProx.Record "" method=name it=r.it gamma=r.gamma sigma=r.sigma norm_res=r.norm_res objective=(r.f_x + r.g_x + r.h_Ax) grad_f_evals=(iscounting(f) ? r.grad_f_evals : nothing) prox_g_evals=(iscounting(g) ? r.prox_g_evals : nothing) f_evals=(iscounting(f) ? r.f_evals : nothing)
    end
    return x, y[1:md], Int(res.iters)
end

logging_active() = Logging.min_enabled_level(current_logger()) <= AdaProx.Record
cflags(f, g, h, A) = (Int32(iscounting(f)), Int32(iscounting(g)), Int32(h !== nothing && iscounting(h)), Int32(A !== nothing && iscounting(A)))

# ---- entry points with the reference's signatures -----------------------------------
function adaptive_primal_dual(x, y; f, g, h, A, rule, tol = 1e-5, maxit = 10_000, name = "AdaPDM")   # src/AdaProx.jl:312
    o = options(0; rule = rule_fields(rule), tol, maxit, want = Int32(logging_active()), counting = cflags(f, g, h, A))
    return solve(0, x, y; f, g, h, A, opts = o, name, pd = true)
end
function adaptive_proxgrad(x; f, g, rule, tol = 1e-5, maxit = 100_000, name = "AdaPGM")              # :418
    o = options(1; rule = rule_fields(rule), tol, maxit, want = Int32(logging_active()), counting = cflags(f, g, nothing, nothing))
    xs, _, it = solve(1, x, nothing; f, g, opts = o, name, pd = false)
    return xs, it
end
fixed_proxgrad(x; f, g, gamma, tol = 1e-5, maxit = 100_000, name = "Fixed stepsize PGM") =              # :457
    adaptive_proxgrad(x; f, g, rule = AdaProx.FixedStepsize(gamma, one(gamma)), tol, maxit, name)
function adaptive_linesearch_primal_dual(x, y; f, g, h, A, gamma = nothing, eta = 1.0, t = 1.0, delta = 1e-8, Theta = 1.2,
                                         r = 2, R = 0.95, tol = 1e-5, maxit = 10_000, name = "AdaPDM+")  # :463
    @assert eta > 0 "eta must be positive"
    @assert Theta > (delta + 1) "must be Theta > (delta + 1)"
    gamma === nothing && (gamma = 1 / (2 * Theta * t * eta))
    @assert gamma <= 1 / (2 * Theta * t * eta) "gamma is too large"
    o = options(2; rule = (0, gamma, t, 0.0, delta, Theta, 1.0, 1.0, Float64(r)), R, eta, tol, maxit,
                want = Int32(logging_active()), counting = cflags(f, g, h, A))
    return solve(2, x, y; f, g, h, A, opts = o, name, pd = true)
end
function backtracking_proxgrad(x0; f, g, gamma0, xi = 1.0, shrink = 0.5, tol = 1e-5, maxit = 100_000, name = "Backtracking PG")  # :50
    o = options(3; rule = (0, gamma0, 1.0, 0.0, 0.0, 1.2, xi, 1.0, 0.5), shrink, tol, maxit, want = Int32(logging_active()),
                counting = cflags(f, g, nothing, nothing))
    xs, _, it = solve(3, x0, nothing; f, g, opts = o, name, pd = false)
    return xs, it
end
function backtracking_nesterov(x0; f, g, gamma0, shrink = 0.5, tol = 1e-5, maxit = 100_000, name = "Backtracking Nesterov")     # :66
    o = options(4; rule = (0, gamma0, 1.0, 0.0, 0.0, 1.2, 1.0, 1.0, 0.5), shrink, tol, maxit, want = Int32(logging_active()),
                counting = cflags(f, g, nothing, nothing))
    xs, _, it = solve(4, x0, nothing; f, g, opts = o, name, pd = false)
    return xs, it
end


function fixed_nesterov(x0; f, g, Lf = nothing, muf = 0, mug = 0, gamma = nothing, theta = nothing, tol = 1e-5, maxit = 100_000,
                        name = "Fixed Nesterov")                                                                       # :91
    @assert (gamma === nothing) != (Lf === nothing)
    gamma === nothing && (gamma = 1 / Lf)
    o = options(5; rule = (0, gamma, 1.0, 0.0, 0.0, 1.2, 1.0, 1.0, 0.5), muf, mug, theta = theta === nothing ? -1.0 : theta, tol, maxit,
                want = Int32(logging_active()), counting = cflags(f, g, nothing, nothing))
    xs, _, it = solve(5, x0, nothing; f, g, opts = o, name, pd = false)
    return xs, it
end
function malitsky_pock(x, y; f, g, h, A, sigma, t = 1.0, tol = 1e-5, maxit = 10_000, name = "MP-ls")                    # :581
    o = options(6; rule = (0, 0.0, t, 0.0, 0.0, 1.2, 1.0, 1.0, 0.5), sigma, tol, maxit, want = Int32(logging_active()), counting = cflags(f, g, h, A))
    return solve(6, x, y; f, g, h, A, opts = o, name, pd = true)
end
function agraal(x1; f, g, x0 = nothing, gamma0 = nothing, gamma_max = 1e6, phi = 1.5, tol = 1e-5, maxit = 100_000, name = "aGRAAL")   # :150
    x0 === nothing && (x0 = x1 + randn(size(x1)))                                                                     # :162-164
    o = options(7; rule = (0, gamma0 === nothing ? 0.0 : gamma0, 1.0, 0.0, 0.0, 1.2, 1.0, 1.0, 0.5), gamma_max, phi, tol, maxit,
                want = Int32(logging_active()), counting = cflags(f, g, nothing, nothing))
    xs, _, it = solve(7, x1, x0; f, g, opts = o, name, pd = false)      # the second start point travels in the y0 slot
    return xs, it
end

# src/AdaProx.jl:423-455: the stepsize estimate is a handful of oracle calls (device calls through eval_f / prox_eval), the loop
# is the persistent kernel.  `gamma = nothing` cannot run in the reference (:431 calls prox without g) and is not offered.
function eval_with_gradient(f, x)
    fo = device_oracle(unwrap(f)); n = length(x)
    prob = CProblem(fo.kind, fo.ipar, fo.mat, fo.vec, fo.c, noprox(), noprox(), 0, n, 0)
    fx = Ref{Float64}(0.0); grad = Vector{Float64}(undef, n); xv = Vector{Float64}(x)
    check(ccall((:adaprox_eval_f, lib), Cint, (Handle, Ref{CProblem}, Ptr{Float64}, Ref{Float64}, Ptr{Float64}), handle(), prob, xv, fx, grad))
    return fx[], grad
end
function prox(g, x, gamma)
    y = Vector{Float64}(undef, length(x)); gy = Ref{Float64}(0.0); xv = Vector{Float64}(x)
    check(ccall((:adaprox_prox_eval, lib), Cint, (Handle, Ref{CProx}, Ptr{Float64}, Int64, Float64, Ptr{Float64}, Ref{Float64}),
                handle(), device_prox(g), xv, length(xv), Float64(gamma), y, gy))
    return y, gy[]
end
function auto_adaptive_proxgrad(x; f, g, gamma, tol = 1e-5, maxit = 100_000, name = "AutoAdaPGM")
    _, grad_x = eval_with_gradient(f, x)
    norm(grad_x) <= tol && return x, 0
    @assert gamma > 0
    x_prev, grad_x_prev, gamma_prev = x, grad_x, gamma
    x, _ = prox(g, x - gamma * grad_x, gamma)
    _, grad_x = eval_with_gradient(f, x)
    L = dot(grad_x - grad_x_prev, x - x_prev) / norm(x - x_prev)^2
    gamma = iszero(L) ? sqrt(2) * gamma : 1 / L
    if gamma_prev / gamma > 1e5
        x, _ = prox(g, x_prev - gamma * grad_x_prev, gamma)
        _, grad_x = eval_with_gradient(f, x)
        L = dot(grad_x - grad_x_prev, x - x_prev) / norm(x - x_prev)^2
        gamma = iszero(L) ? sqrt(2) * gamma : 1 / L
    end
    return adaptive_proxgrad(x_prev; f, g, rule = AdaProx.OurRule(; gamma, t = 1, norm_A = 0, delta = 0, Theta = 1.2), tol, maxit, name)
end

# cubic_sparse_logreg/runme.jl:34-45 on the device: (H, g) of the logistic loss at w, the setup of Cubic(H, g, lam)
function logistic_loss_grad_Hessian(X, y, w)
    n1 = size(X, 2) + 1
    H = Matrix{Float64}(undef, n1, n1); g = Vector{Float64}(undef, n1); wv = Vector{Float64}(w)
    check(ccall((:adaprox_logistic_grad_hessian, lib), Cint, (Handle, Id, Id, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                handle(), upload(X), upload(y), wv, H, g))
    return H, g
end

# ---- batched multi-lambda lasso path (include/adaprox.h: adaprox_solve_lambda_path) ---------------------------
# Column j of the result is what `adaptive_proxgrad(X0[:, j]; f, g = NormL1(lambdas[j]), rule, tol, maxit)` returns; the L
# columns advance together so that A*X and A'*R are FP64 tensor-core contractions.  NOT EXECUTED (no Julia in the build image).
function adaptive_proxgrad_path(X0::Union{Nothing,Matrix{Float64}}; f, lambdas::Vector{Float64}, rule, gamma0 = nothing,
                                tol = 1e-5, maxit = 100_000)
    L = length(lambdas)
    fo = device_oracle(unwrap(f))                              # same CProblem as solve(); g is ignored by the library
    n = X0 === nothing ? fo.n : size(X0, 1)                    # least_squares(A, b) records n = size(A, 2)
    prob = CProblem(fo.kind, fo.ipar, fo.mat, fo.vec, fo.c, device_prox(NormL1(1.0)), noprox(), 0, n, 0)
    o = options(1; rule = rule_fields(rule), tol, maxit, want = Int32(0), counting = cflags(f, nothing, nothing, nothing))
    X = Matrix{Float64}(undef, n, L)                          # column-major: column j contiguous = the library's [L][n] layout
    its = zeros(Int64, L); nres = zeros(L); gam = zeros(L); fx = zeros(L)
    res = CResult()
    x0ptr = X0 === nothing ? Ptr{Float64}(C_NULL) : pointer(X0)
    g0ptr = gamma0 === nothing ? Ptr{Float64}(C_NULL) : pointer(gamma0)
    GC.@preserve X0 gamma0 lambdas X its nres gam fx begin
        check(ccall((:adaprox_solve_lambda_path, lib), Cint,
                    (Handle, Ref{CProblem}, Ref{COptions}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                     Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int64, Ref{CResult}),
                    handle(), prob, o, L, lambdas, g0ptr, x0ptr, X, its, nres, gam, fx, C_NULL, 0, res))
    end
    return X, its, (norm_res = nres, gamma = gam, f_x = fx, solve_ms = res.solve_ms)
end

# ---- batched C path of the dual SVM (include/adaprox.h: adaprox_solve_box_path) ----------------------------------
# Column j of the result is what `adaptive_primal_dual(X0[:, j], [Y0[j]]; f, g = IndBox(lower, upper[j]), h = IndZero(), A,
# rule, tol, maxit)` returns; f is Quadratic(Q, q) or QuadraticGram(Z, q), A the 1 x n label row.  NOT EXECUTED (no Julia
# in the build image).
function adaptive_primal_dual_path(X0::Union{Nothing,Matrix{Float64}}, Y0::Union{Nothing,Vector{Float64}}; f, A,
                                   upper::Vector{Float64}, rule, lower = 0.0, gamma0 = nothing, tol = 1e-5, maxit = 10_000)
    L = length(upper)
    fo = device_oracle(unwrap(f))
    n = size(unwrap(A), 2)
    prob = CProblem(fo.kind, fo.ipar, fo.mat, fo.vec, fo.c, CProx(4, 0, 1.0, Float64(lower), Float64(lower), 0, 0, 0),
                    device_prox(ProximalCore.IndZero()), upload(unwrap(A)), n, 1)
    o = options(0; rule = rule_fields(rule), tol, maxit, want = Int32(0), counting = cflags(f, nothing, nothing, A))
    X = Matrix{Float64}(undef, n, L)                          # column-major: column j contiguous = the library's [L][n] layout
    Y = zeros(L); its = zeros(Int64, L); nres = zeros(L); gam = zeros(L); sig = zeros(L); fx = zeros(L)
    res = CResult()
    x0ptr = X0 === nothing ? Ptr{Float64}(C_NULL) : pointer(X0)
    y0ptr = Y0 === nothing ? Ptr{Float64}(C_NULL) : pointer(Y0)
    g0ptr = gamma0 === nothing ? Ptr{Float64}(C_NULL) : pointer(gamma0)
    GC.@preserve X0 Y0 gamma0 upper X Y its nres gam sig fx begin
        check(ccall((:adaprox_solve_box_path, lib), Cint,
                    (Handle, Ref{CProblem}, Ref{COptions}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                     Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                     Ptr{Float64}, Int64, Ref{CResult}),
                    handle(), prob, o, L, upper, g0ptr, x0ptr, y0ptr, X, Y, its, nres, gam, sig, fx, C_NULL, 0, res))
    end
    return X, Y, its, (norm_res = nres, gamma = gam, sigma = sig, f_x = fx, solve_ms = res.solve_ms)
end

# ---- batched lambda path of LAD and the square-root lasso (include/adaprox.h: adaprox_solve_pd_lambda_path) --------
# Column j of the result is what `adaptive_primal_dual(X0[:, j], Y0[:, j]; f = Zero(), g = NormL1(lambdas[j]), h, A, rule,
# tol, maxit)` returns; h is NormL1 / NormL2, optionally Translate'd, A a dense matrix.  NOT EXECUTED (no Julia in the
# build image).
function adaptive_primal_dual_lambda_path(X0::Union{Nothing,Matrix{Float64}}, Y0::Union{Nothing,Matrix{Float64}}; h, A,
                                          lambdas::Vector{Float64}, rule, gamma0 = nothing, tol = 1e-5, maxit = 10_000)
    L = length(lambdas)
    m, n = size(unwrap(A))
    prob = CProblem(0, 0, 0, 0, 0.0, CProx(2, 0, 1.0, 0.0, 0.0, 0, 0, 0), device_prox(unwrap(h)), upload(unwrap(A)), n, m)
    o = options(0; rule = rule_fields(rule), tol, maxit, want = Int32(0), counting = cflags(nothing, nothing, h, A))
    X = Matrix{Float64}(undef, n, L)                          # column-major: column j contiguous = the library's [L][n] layout
    Y = Matrix{Float64}(undef, m, L)
    its = zeros(Int64, L); nres = zeros(L); gam = zeros(L); sig = zeros(L)
    res = CResult()
    x0ptr = X0 === nothing ? Ptr{Float64}(C_NULL) : pointer(X0)
    y0ptr = Y0 === nothing ? Ptr{Float64}(C_NULL) : pointer(Y0)
    g0ptr = gamma0 === nothing ? Ptr{Float64}(C_NULL) : pointer(gamma0)
    GC.@preserve X0 Y0 gamma0 lambdas X Y its nres gam sig begin
        check(ccall((:adaprox_solve_pd_lambda_path, lib), Cint,
                    (Handle, Ref{CProblem}, Ref{COptions}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                     Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                     Ptr{Float64}, Int64, Ref{CResult}),
                    handle(), prob, o, L, lambdas, g0ptr, x0ptr, y0ptr, X, Y, its, nres, gam, sig, C_NULL, 0, res))
    end
    return X, Y, its, (norm_res = nres, gamma = gam, sigma = sig, solve_ms = res.solve_ms)
end

# ---- multi-GPU: peer exchange blocks for the all-reduce inside the kernels (adaprox_p2p_*) -----------------------
# `allgather` is supplied by the caller (e.g. MPI.Allgather on the 64-byte handles); rank order.  NOT EXECUTED.
function attach_p2p(n_max::Integer, nranks::Integer, rank::Integer, allgather::Function)
    mine = zeros(UInt8, 64)
    check(ccall((:adaprox_p2p_export, lib), Cint, (Handle, Int64, Ptr{UInt8}), handle(), n_max, mine))
    all = allgather(mine)::Vector{UInt8}                      # 64 * nranks bytes
    check(ccall((:adaprox_p2p_attach, lib), Cint, (Handle, Cint, Cint, Ptr{UInt8}), handle(), nranks, rank, all))
end

# after a sharded solve failed with status -4 (a peer did not arrive): every rank calls this, then a host barrier
p2p_reset() = check(ccall((:adaprox_p2p_reset, lib), Cint, (Handle,), handle()))

end # module
