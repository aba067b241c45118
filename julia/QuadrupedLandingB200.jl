# QuadrupedLandingB200.jl -- the reference-side binding of libqlnlp.so (include/qlnlp.h).
#
# ZERO-EDIT drop-in.  `include` this file after the reference's src/nlp.jl and src/moi.jl and call
#
#     QuadrupedLandingB200.install!(nlp)                      # or install!(nlp; sparse=true, pattern=:true)
#
# `install!` builds a GPU evaluator for THIS `HybridNLP` object (src/nlp.jl:13-84), remembers it in an IdDict and
# re-defines the seven `MOI.*(::HybridNLP, ...)` methods of src/moi.jl:1-33 so that they `ccall` the C ABI.  The
# reference's `solve(Z0, nlp; ...)` (src/moi.jl:46-103) then runs UNCHANGED: it is typed to `HybridNLP`, reads
# `num_primals(prob)`, `num_duals(prob)`, `prob.N`, `prob.lb`, `prob.ub` -- all still the reference's own -- and reaches
# the evaluator only through the MOI callbacks.  With `sparse=true` the structure handed to Ipopt is the column-major
# filter of the entries `jac_c!` assigns (32,161 pairs instead of the dense 1,327,995 of src/moi.jl:31-33, the reason
# the recorded run spends 575 s inside Ipopt, src/main.ipynb:724); the default `sparse=false` reports exactly the
# reference's dense structure.
#
# NOT EXECUTED in the build environment (no julia binary in the image).  tests/test_julia_shim.py checks every
# `ccall` below (symbol, arity, argument and return types) and both struct layouts against include/qlnlp.h; the
# executable twin with the same calls in the same order is quadruped_landing_b200/evaluator.py (ctypes).
module QuadrupedLandingB200

using MathOptInterface
const MOI = MathOptInterface

const LIBQLNLP = get(ENV, "LIBQLNLP", "libqlnlp.so")

# mirrors `qlnlp_model` / `qlnlp_problem_desc` / `qlnlp_batch_io` of include/qlnlp.h field for field
struct QlModel
    g::Cdouble; mb::Cdouble; mf::Cdouble; lb::Cdouble; l1::Cdouble; l2::Cdouble
end
struct QlProblemDesc
    N::Int64; k_trans::Int64; init_mode::Int64
    model::QlModel
    x0::NTuple{15,Cdouble}; xf::NTuple{15,Cdouble}
    Q::Ptr{Cdouble}; R::Ptr{Cdouble}; q::Ptr{Cdouble}; r::Ptr{Cdouble}; c::Ptr{Cdouble}
end
struct QlBatchIO
    Z::Ptr{Cdouble}; ldz::Int64
    x0::Ptr{Cdouble}; xf::Ptr{Cdouble}
    f::Ptr{Cdouble}
    grad::Ptr{Cdouble}; ldgrad::Int64
    g::Ptr{Cdouble}; ldg::Int64
    jac::Ptr{Cdouble}; ldjac::Int64
end

const JAC_SPARSE_BLOCK = Cint(0)
const JAC_DENSE = Cint(1)
const JAC_SPARSE_TRUE = Cint(2)

check(rc::Cint) = rc == 0 || error("qlnlp error $rc: " * unsafe_string(ccall((:qlnlp_last_error, LIBQLNLP), Cstring, ())))

mutable struct GpuEvaluator
    handle::Ptr{Cvoid}
    n_nlp::Int
    m_nlp::Int
    nnz::Int          # values per evaluation in the handle's structure (dense: m_nlp * n_nlp)
    nnz_batch::Int    # values per evaluation in batched calls (the handle's sparse pattern)
end

const HANDLES = IdDict{Any,GpuEvaluator}()

"""
    GpuEvaluator(nlp; sparse=false, pattern=:block, device=0, devices=nothing)

Build the GPU evaluator from the reference's `HybridNLP` (src/nlp.jl:13-84).  `sparse=false` reports the dense
m_nlp x n_nlp structure exactly like src/moi.jl:31-33; `sparse=true` reports SPARSE_BLOCK, the column-major filter of
the entries `jac_c!` assigns, or with `pattern=:true` only the 4,840 structurally non-zero entries.
`devices=[0,1,...]` spreads host batches over several GPUs (qlnlp_create_multi).
"""
function GpuEvaluator(nlp; sparse::Bool=false, pattern::Symbol=:block, device::Integer=0, devices=nothing)
    N = nlp.N
    Q = Matrix{Cdouble}(undef, 15, N); R = Matrix{Cdouble}(undef, 5, N)
    q = Matrix{Cdouble}(undef, 15, N); r = Matrix{Cdouble}(undef, 5, N); c = Vector{Cdouble}(undef, N)
    for k = 1:N                      # knot-major rows == column-major 15xN / 5xN in Julia
        o = nlp.obj[k]
        Q[:, k] .= o.Q.diag; R[:, k] .= o.R.diag; q[:, k] .= o.q; r[:, k] .= o.r; c[k] = o.c
    end
    m = nlp.model
    desc = Ref(QlProblemDesc(N, nlp.k_trans, nlp.init_mode, QlModel(m.g, m.mb, m.mf, m.lb, m.l1, m.l2),
                             Tuple(nlp.x0), Tuple(nlp.xf), pointer(Q), pointer(R), pointer(q), pointer(r), pointer(c)))
    mode = sparse ? (pattern == :true ? JAC_SPARSE_TRUE : JAC_SPARSE_BLOCK) : JAC_DENSE
    h = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve Q R q r c begin      # the descriptor's tables are copied during creation, not retained
        if devices === nothing
            check(ccall((:qlnlp_create, LIBQLNLP), Cint, (Ref{QlProblemDesc}, Cint, Cint, Ref{Ptr{Cvoid}}),
                        desc, device, mode, h))
        else
            devs = Vector{Cint}(devices)
            check(ccall((:qlnlp_create_multi, LIBQLNLP), Cint, (Ref{QlProblemDesc}, Ptr{Cint}, Cint, Cint, Ref{Ptr{Cvoid}}),
                        desc, devs, length(devs), mode, h))
        end
    end
    n = Ref{Int64}(0); mm = Ref{Int64}(0); nnz = Ref{Int64}(0); nb = Ref{Int64}(0)
    check(ccall((:qlnlp_dims, LIBQLNLP), Cint, (Ptr{Cvoid}, Ref{Int64}, Ref{Int64}, Ref{Int64}, Ref{Int64}), h[], n, mm, nnz, nb))
    ev = GpuEvaluator(h[], n[], mm[], nnz[], sparse ? nnz[] : nb[])
    finalizer(e -> ccall((:qlnlp_destroy, LIBQLNLP), Cint, (Ptr{Cvoid},), e.handle), ev)
    return ev
end

# ---- the callbacks, one `ccall` each -------------------------------------------------------------------------
function gpu_eval_objective(ev::GpuEvaluator, x)                              # moi.jl:1-3
    f = Ref{Cdouble}(0.0)
    check(ccall((:qlnlp_eval_objective, LIBQLNLP), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Ref{Cdouble}), ev.handle, x, f))
    return f[]
end
function gpu_eval_objective_gradient(ev::GpuEvaluator, grad_f, x)             # moi.jl:5-8
    check(ccall((:qlnlp_eval_objective_gradient, LIBQLNLP), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Ptr{Cdouble}), ev.handle, x, grad_f))
    return nothing
end
function gpu_eval_constraint(ev::GpuEvaluator, g, x)                          # moi.jl:10-13
    check(ccall((:qlnlp_eval_constraint, LIBQLNLP), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Ptr{Cdouble}), ev.handle, x, g))
    return nothing
end
function gpu_eval_constraint_jacobian(ev::GpuEvaluator, vec, x)               # moi.jl:15-24
    check(ccall((:qlnlp_eval_constraint_jacobian, LIBQLNLP), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Ptr{Cdouble}), ev.handle, x, vec))
    return nothing
end
function gpu_jacobian_structure(ev::GpuEvaluator)                             # moi.jl:31-33
    rows = Vector{Int64}(undef, ev.nnz); cols = Vector{Int64}(undef, ev.nnz)
    check(ccall((:qlnlp_jacobian_structure, LIBQLNLP), Cint, (Ptr{Cvoid}, Ptr{Int64}, Ptr{Int64}), ev.handle, rows, cols))
    return collect(zip(rows, cols))                                           # 1-based (row, col), value order
end
# f, grad f, g and the Jacobian values of one iterate with one launch (the callbacks above share that launch anyway:
# the library serves callbacks at an unchanged x from its last evaluation)
function gpu_eval_all!(ev::GpuEvaluator, x, grad_f, g, vec)
    f = Ref{Cdouble}(0.0)
    check(ccall((:qlnlp_eval_all, LIBQLNLP), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Ref{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}),
                ev.handle, x, f, grad_f, g, vec))
    return f[]
end

# Lagrangian Hessian (NOT in the reference: src/moi.jl:26-28 offers [:Grad, :Jac]); used when install!(...; hessian=true)
function gpu_hessian_lagrangian_structure(ev::GpuEvaluator)
    nnz = Ref{Int64}(0)
    check(ccall((:qlnlp_hessian_nnz, LIBQLNLP), Cint, (Ptr{Cvoid}, Ref{Int64}), ev.handle, nnz))
    rows = Vector{Int64}(undef, nnz[]); cols = Vector{Int64}(undef, nnz[])
    check(ccall((:qlnlp_hessian_structure, LIBQLNLP), Cint, (Ptr{Cvoid}, Ptr{Int64}, Ptr{Int64}), ev.handle, rows, cols))
    return collect(zip(rows, cols))                                           # lower triangle, 1-based
end
# matrix-free products (MOI :JacVec / :HessVec; NOT in the reference); used when install!(...; products=true)
function gpu_eval_constraint_jacobian_product(ev::GpuEvaluator, y, x, w)
    check(ccall((:qlnlp_eval_constraint_jacobian_product, LIBQLNLP), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}),
                ev.handle, x, w, y))
    return y
end
function gpu_eval_constraint_jacobian_transpose_product(ev::GpuEvaluator, y, x, w)
    check(ccall((:qlnlp_eval_constraint_jacobian_transpose_product, LIBQLNLP), Cint,
                (Ptr{Cvoid}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}), ev.handle, x, w, y))
    return y
end
function gpu_eval_hessian_lagrangian_product(ev::GpuEvaluator, h, x, v, sigma, mu)
    check(ccall((:qlnlp_eval_hessian_lagrangian_product, LIBQLNLP), Cint,
                (Ptr{Cvoid}, Ptr{Cdouble}, Ptr{Cdouble}, Cdouble, Ptr{Cdouble}, Ptr{Cdouble}), ev.handle, x, v, sigma, mu, h))
    return h
end
function gpu_eval_hessian_lagrangian(ev::GpuEvaluator, H, x, sigma, mu)
    check(ccall((:qlnlp_eval_hessian_lagrangian, LIBQLNLP), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Cdouble, Ptr{Cdouble}, Ptr{Cdouble}),
                ev.handle, x, sigma, mu, H))
    return nothing
end

# constraint / variable bounds as the library restates them (src/nlp.jl:66-69, src/moi.jl:51-67); solve() keeps using
# the reference's own prob.lb / prob.ub, these are for callers that build the bounds themselves
function constraint_bounds(ev::GpuEvaluator)
    lb = Vector{Cdouble}(undef, ev.m_nlp); ub = similar(lb)
    check(ccall((:qlnlp_constraint_bounds, LIBQLNLP), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Ptr{Cdouble}), ev.handle, lb, ub))
    return lb, ub
end
function variable_bounds(ev::GpuEvaluator)
    xl = Vector{Cdouble}(undef, ev.n_nlp); xu = similar(xl)
    check(ccall((:qlnlp_variable_bounds, LIBQLNLP), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Ptr{Cdouble}), ev.handle, xl, xu))
    return xl, xu
end

"""
    eval_batch_host!(ev, Z; f, grad, g, jac)

B decision vectors at once on host arrays: `Z` is `n_nlp x B` (one decision vector per COLUMN, i.e. the row-major
`[B][n_nlp]` layout of the C ABI), `f` a `B`-vector, `grad` `n_nlp x B`, `g` `m_nlp x B`, `jac` `nnz_batch x B`; pass
`nothing` to skip an output.  Multi-start guesses, line-search trial points and sweeps go through here.
"""
function eval_batch_host!(ev::GpuEvaluator, Z::Matrix{Cdouble}; f=nothing, grad=nothing, g=nothing, jac=nothing)
    B = size(Z, 2)
    p(a) = a === nothing ? Ptr{Cdouble}(C_NULL) : pointer(a)
    ld(a) = a === nothing ? Int64(0) : Int64(size(a, 1))
    io = Ref(QlBatchIO(pointer(Z), size(Z, 1), C_NULL, C_NULL, p(f), p(grad), ld(grad), p(g), ld(g), p(jac), ld(jac)))
    GC.@preserve Z f grad g jac check(ccall((:qlnlp_eval_batch_host, LIBQLNLP), Cint, (Ptr{Cvoid}, Int64, Ref{QlBatchIO}), ev.handle, B, io))
    return nothing
end

# a `jac` matrix that is reused for every batch: its structural zeros and +-1 entries are written once, later batches
# rewrite only the lines that change (like jac_c! relying on the caller's zeros, constraints.jl:212-291)
register_output!(ev::GpuEvaluator, jac::Matrix{Cdouble}) =
    check(ccall((:qlnlp_host_output_register, LIBQLNLP), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Int64, Int64), ev.handle, jac, size(jac, 1), size(jac, 2)))
unregister_output!(ev::GpuEvaluator, jac::Matrix{Cdouble}) =
    check(ccall((:qlnlp_host_output_unregister, LIBQLNLP), Cint, (Ptr{Cvoid}, Ptr{Cdouble}), ev.handle, jac))
# page-lock a Julia array so that the copies to and from the GPU are asynchronous
pin!(a::Array{Cdouble}) = check(ccall((:qlnlp_host_pin, LIBQLNLP), Cint, (Ptr{Cvoid}, Int64), a, sizeof(a)))
unpin!(a::Array{Cdouble}) = check(ccall((:qlnlp_host_unpin, LIBQLNLP), Cint, (Ptr{Cvoid},), a))

evaluator(nlp) = get(HANDLES, nlp) do
    error("no GPU evaluator installed for this HybridNLP: call QuadrupedLandingB200.install!(nlp) first")
end

"""
    install!(nlp; sparse=false, pattern=:block, device=0, devices=nothing, hessian=false, products=false, into=Main)

Make `nlp` (a `HybridNLP` of the reference) evaluate on the GPU.  Re-defines, in module `into` (where the reference's
src/nlp.jl and src/moi.jl were included), the seven MOI methods of src/moi.jl:1-33 for `::HybridNLP`; afterwards
`solve(Z0, nlp; c_tol=1e-3, tol=1e-3)` (src/main.ipynb:742-744, src/moi.jl:46-103) runs without any edit.
Every `HybridNLP` handed to MOI after this call needs its own `install!`.
`products=true` also defines the matrix-free MOI methods `eval_constraint_jacobian_product` and
`eval_constraint_jacobian_transpose_product` (`:JacVec`), and with `hessian=true` `eval_hessian_lagrangian_product`
(`:HessVec`); the summation order of every product is fixed (include/qlnlp.h).
"""
function install!(nlp; into::Module=Main, hessian::Bool=false, products::Bool=false, kwargs...)
    HANDLES[nlp] = GpuEvaluator(nlp; kwargs...)
    feats = hessian ? [:Grad, :Jac, :Hess] : [:Grad, :Jac]
    products && append!(feats, hessian ? [:JacVec, :HessVec] : [:JacVec])
    Core.eval(into, quote
        $MOI.eval_objective(prob::HybridNLP, x) =
            $gpu_eval_objective($evaluator(prob), x)                                          # moi.jl:1-3
        $MOI.eval_objective_gradient(prob::HybridNLP, grad_f, x) =
            $gpu_eval_objective_gradient($evaluator(prob), grad_f, x)                         # moi.jl:5-8
        $MOI.eval_constraint(prob::HybridNLP, g, x) =
            $gpu_eval_constraint($evaluator(prob), g, x)                                      # moi.jl:10-13
        $MOI.eval_constraint_jacobian(prob::HybridNLP, vec, x) =
            $gpu_eval_constraint_jacobian($evaluator(prob), vec, x)                           # moi.jl:15-24 (uses `prob`, not the global `nlp`)
        $MOI.features_available(prob::HybridNLP) = $feats                                     # moi.jl:26-28 (+ :Hess on request)
        $MOI.hessian_lagrangian_structure(prob::HybridNLP) = $gpu_hessian_lagrangian_structure($evaluator(prob))
        $MOI.eval_hessian_lagrangian(prob::HybridNLP, H, x, sigma, mu) =
            $gpu_eval_hessian_lagrangian($evaluator(prob), H, x, sigma, mu)
        $MOI.initialize(prob::HybridNLP, features) = nothing                                   # moi.jl:30
        $MOI.jacobian_structure(prob::HybridNLP) = $gpu_jacobian_structure($evaluator(prob))   # moi.jl:31-33
    end)
    products && Core.eval(into, quote
        $MOI.eval_constraint_jacobian_product(prob::HybridNLP, y, x, w) =
            $gpu_eval_constraint_jacobian_product($evaluator(prob), y, x, w)                  # y = J(x) w
        $MOI.eval_constraint_jacobian_transpose_product(prob::HybridNLP, y, x, w) =
            $gpu_eval_constraint_jacobian_transpose_product($evaluator(prob), y, x, w)        # y = J(x)' w
    end)
    products && hessian && Core.eval(into, quote
        $MOI.eval_hessian_lagrangian_product(prob::HybridNLP, h, x, v, sigma, mu) =
            $gpu_eval_hessian_lagrangian_product($evaluator(prob), h, x, v, sigma, mu)        # h = Hess L(x, sigma, mu) v
    end)
    return HANDLES[nlp]
end

uninstall!(nlp) = (delete!(HANDLES, nlp); nothing)

end # module
