# SetIntersectionProjectionB200.jl — ccall binding of libsipb200.so behind the reference's own entry points.
#
# STATUS: NEVER EXECUTED.  Julia is installed neither in the build image nor on the GPU box (probed: `julia`, ~/.julia,
# the offline wheelhouse), so this file has not been run, not even parsed by a Julia front end.  It is written call for
# call after the TESTED Python/ctypes host (setintersectionprojection.jl_b200/{constraints,precompute,solver}.py, which
# the GPU parity suite exercises through the same C ABI) and is the code a maintainer of
# slimgroup/SetIntersectionProjection.jl would start from; INTEGRATION.md lists, per function, what it replaces and
# what remains to be verified on a machine with Julia.  Struct layouts must match include/sipb200.h field for field
# (the Python mirror is checked against gcc's layout in tests/test_host_index_work.py).
#
# Entry points (same names, argument order and return tuples as the reference):
#   setup_constraints(constraint, comp_grid, TF)                         setup_constraints.jl:17-102
#   PARSDMM_precompute_distribute(TD_OP, set_Prop, comp_grid, options)   PARSDMM_precompute_distribute.jl:6-77
#   PARSDMM_precompute_distribute_Minkowski(...)                         PARSDMM_precompute_distribute_Minkowski.jl:3-157
#   PARSDMM(m, AtA, TD_OP, set_Prop, P_sub, comp_grid, options[, x, l, y])   PARSDMM.jl:25-258
#   init_slabs(rank, world, uid)                                         replaces options.parallel (one process per GPU)
module SIPB200

using SparseArrays
import SetIntersectionProjection            # types, get_TD_operator, mat2CDS, convert_options! of the reference
const SIP = SetIntersectionProjection

const lib = joinpath(@__DIR__, "libsipb200.so")

# ---------------------------------------------------------------------------------------------------------------
# structs of include/sipb200.h
# ---------------------------------------------------------------------------------------------------------------
struct SparseOp           # sipb_sparse: custom_TD_OP[1] as CSR (of A) and CSC (colptr/rowval/nzval .- 1), host arrays
    rows::Int64; cols::Int64; nnz::Int64
    rowptr::Ptr{Int64}; colidx::Ptr{Int32}; val::Ptr{Cvoid}
    colptr::Ptr{Int64}; rowidx::Ptr{Int32}; valt::Ptr{Cvoid}
end

struct SetDesc            # sipb_set_desc
    set_kind::Int32; op_kind::Int32; block_mode::Int32; ncvx::Int32
    min::Float64; max::Float64; k::Int64
    min_vec::Ptr{Cvoid}; max_vec::Ptr{Cvoid}
    fiber_axis::Int32; reserved::Int32; td_n::NTuple{3,Int64}
    sparse::Ptr{SparseOp}
end

struct Options            # sipb_options
    maxit::Int32; rho_update_frequency::Int32; adjust_rho::Int32; adjust_gamma::Int32
    adjust_feasibility_rho::Int32; zero_ini_guess::Int32; n_rho_ini::Int32; profile_kernels::Int32
    evol_rel_tol::Float64; feas_tol::Float64; obj_tol::Float64; gamma_ini::Float64
    rho_ini::Ptr{Float64}
    fixed_iterations::Int32; return_ly::Int32; resident_io::Int32; warm_resident::Int32
end

mutable struct Log        # sipb_log (arrays are caller-allocated, maxit rows, row-major)
    iters::Int32; feas_rows::Int32; stopped_feasible::Int32; p::Int32; pp::Int32
    set_feasibility::Ptr{Float64}; r_dual::Ptr{Float64}; r_pri::Ptr{Float64}
    r_dual_total::Ptr{Float64}; r_pri_total::Ptr{Float64}; obj::Ptr{Float64}; evol_x::Ptr{Float64}
    rho::Ptr{Float64}; gamma::Ptr{Float64}; cg_it::Ptr{Int32}; cg_relres::Ptr{Float64}
    phase_seconds::NTuple{7,Float64}; solve_seconds::Float64; device_seconds::Float64
    kernel_launches::NTuple{24,Int64}; kernel_ms::NTuple{24,Float64}; kernel_bytes::NTuple{24,Float64}
    total_launches::Int64; h2d_bytes::Int64; d2h_bytes::Int64
end

check(rc) = rc == 0 || error(unsafe_string(ccall((:sipb_last_error, lib), Cstring, ())))

# set kinds / operator kinds / block modes (include/sipb200.h)
const SET = Dict("bounds"=>0, "bounds_vector"=>1, "l1"=>2, "l2"=>3, "annulus"=>4, "cardinality"=>5, "prox_l1"=>6,
                 "distance"=>7, "bounds_fiber"=>8, "cardinality_fiber"=>9, "cardinality_slice"=>10, "histogram"=>11)
const OPK = Dict("identity"=>0, "D_x"=>1, "D_y"=>2, "D_z"=>3, "TV"=>4, "D2D"=>4, "D3D"=>4, "D_xz"=>5, "custom"=>6)
const BLOCK_PLAIN, BLOCK_LEFT, BLOCK_RIGHT, BLOCK_BOTH = Int32(0), Int32(1), Int32(2), Int32(3)
const PHASES = ("initialization", "form rhs for linear system", "argmin x", "argmin y and l update",
                "stopping conditions check", "adjust rho and gamma", "Q-update")     # PARSDMM.jl:40,100,105,113,152,163,229

# ---------------------------------------------------------------------------------------------------------------
# context (one process drives one GPU) and slabs
# ---------------------------------------------------------------------------------------------------------------
const ctx = Ref{Ptr{Cvoid}}(C_NULL)
function context(device::Integer = parse(Int, get(ENV, "LOCAL_RANK", "0")))
    ctx[] == C_NULL && check(ccall((:sipb_ctx_create, lib), Cint, (Cint, Ptr{Ptr{Cvoid}}), device, ctx))
    ctx[]
end

"128-byte NCCL unique id, created on rank 0 and sent to every worker over Julia's own transport (Distributed)."
function comm_unique_id()
    uid = zeros(UInt8, 128)
    check(ccall((:sipb_comm_unique_id, lib), Cint, (Ptr{UInt8},), uid))
    uid
end
"""
    init_slabs(rank, world, uid)

z-slab decomposition over `world` processes (one GPU each); replaces `options.parallel = true` (one Julia worker per
constraint set, update_y_l_parallel.jl).  With Distributed:

    uid = SIPB200.comm_unique_id()                                  # on the master
    @sync for (r, w) in enumerate(workers())
        @spawnat w SIPB200.init_slabs(r - 1, nworkers(), uid)
    end

Afterwards every worker calls the same setup_constraints / PARSDMM_precompute_distribute / PARSDMM sequence with the
GLOBAL grid; `PARSDMM` takes and returns this rank's planes of m and x (sipb_slab_range) and of l, y.
"""
function init_slabs(rank::Integer, world::Integer, uid::Vector{UInt8})
    check(ccall((:sipb_comm_init, lib), Cint, (Ptr{Cvoid}, Cint, Cint, Ptr{UInt8}), context(rank), rank, world, uid))
end
function slab_range(n_last::Integer, rank::Integer, world::Integer)
    k0 = Ref{Int64}(0); k1 = Ref{Int64}(0)
    check(ccall((:sipb_slab_range, lib), Cint, (Int64, Cint, Cint, Ptr{Int64}, Ptr{Int64}), n_last, rank, world, k0, k1))
    k0[], k1[]
end

# ---------------------------------------------------------------------------------------------------------------
# setup_constraints: functor structs instead of closures (the reference's closures capture constraint.min / max,
# get_projector.jl:10,33,41,90; the wrapper must see them)
# ---------------------------------------------------------------------------------------------------------------
"TD_OP[i]: descriptor of a banded operator of get_TD_operator.jl (applied matrix-free on the device) or an explicit
sparse custom_TD_OP (setup_constraints.jl:70-72)."
struct DeviceOperator{TF}
    kind::String                         # "identity","D_x","D_y","D_z","TV","D_xz","custom"
    n::NTuple{3,Int64}; ndim::Int
    h::NTuple{3,Float64}                 # TF(comp_grid.d[i]) widened
    block_mode::Int32                    # Minkowski placement [A 0] / [0 A] / [A A]
    A::Union{Nothing,SparseMatrixCSC{TF,Int64}}      # the matrix itself (always for "custom"; on demand otherwise)
end
Base.size(op::DeviceOperator, d) = d == 1 ? rows(op) : prod(op.n[1:op.ndim]) * (op.block_mode == BLOCK_PLAIN ? 1 : 2)
function rows(op::DeviceOperator)
    op.kind == "custom" && return size(op.A, 1)
    r = Ref{Int64}(0); n = Int64[op.n...]
    check(ccall((:sipb_op_rows, lib), Cint, (Cint, Ptr{Int64}, Cint, Ptr{Int64}), op.ndim, n, OPK[op.kind], r))
    r[]
end

struct DeviceProjector{TF}               # callable on a host vector like the reference's P_sub[i]: P(v) -> sipb_project
    set_kind::Int32
    min::Union{TF,Vector{TF}}; max::Union{TF,Vector{TF}}; k::Int64
    fiber_axis::Int32; td_n::NTuple{3,Int64}
end
function (P::DeviceProjector{TF})(v::Vector{TF}) where TF
    d = SetDesc(P.set_kind, 0, 0, 0, P.min isa Real ? P.min : 0.0, P.max isa Real ? P.max : 0.0, P.k,
                P.min isa Vector ? pointer(P.min) : C_NULL, P.max isa Vector ? pointer(P.max) : C_NULL,
                P.fiber_axis, 0, P.td_n, C_NULL)
    GC.@preserve P v check(ccall((:sipb_project, lib), Cint, (Ptr{Cvoid}, Cint, Ref{SetDesc}, Int64, Ptr{Cvoid}, Ptr{Cvoid}),
                                 context(), TF == Float32 ? 0 : 1, d, length(v), v, C_NULL))
    v
end

pad3(t) = ntuple(i -> i <= length(t) ? Int64(t[i]) : Int64(1), 3)

function get_projector(c, TD_n, ::Type{TF}) where TF          # get_projector.jl:3-103, device sets only
    st = c.set_type; mode = c.app_mode
    st in ("rank", "nuclear", "subspace") && error("set type $st is outside the device hot path (no CPU fallback)")
    if !(mode[1] in ("matrix", "tensor"))
        axis = Dict("x"=>0, "y"=>1, "z"=> (length(TD_n) == 2 ? 1 : 2))[mode[2]]
        st == "bounds" && mode[1] == "fiber" && return DeviceProjector{TF}(SET["bounds_fiber"], TF.(c.min), TF.(c.max), 0, axis, pad3(TD_n))
        st == "cardinality" && mode[1] == "fiber" && return DeviceProjector{TF}(SET["cardinality_fiber"], TF(0), TF(0), Int64(c.max), axis, pad3(TD_n))
        st == "cardinality" && mode[1] == "slice" && return DeviceProjector{TF}(SET["cardinality_slice"], TF(0), TF(0), Int64(c.max), axis, pad3(TD_n))
        error("only the fiber modes of bounds / cardinality and the slice mode of cardinality are on the device path")
    end
    z = (Int32(0), (Int64(0), Int64(0), Int64(0)))
    st == "bounds"      && return c.min isa Real ? DeviceProjector{TF}(SET["bounds"], TF(c.min), TF(c.max), 0, z...) :
                                                   DeviceProjector{TF}(SET["bounds_vector"], TF.(c.min), TF.(c.max), 0, z...)
    st == "histogram"   && return DeviceProjector{TF}(SET["histogram"], TF.(c.min), TF.(c.max), 0, z...)
    st == "prox_l1"     && return DeviceProjector{TF}(SET["prox_l1"], TF(0), TF(c.max), 0, z...)
    st == "l1"          && return DeviceProjector{TF}(SET["l1"], TF(0), TF(c.max), 0, z...)
    st == "l2"          && return DeviceProjector{TF}(SET["l2"], TF(0), TF(c.max), 0, z...)
    st == "annulus"     && return DeviceProjector{TF}(SET["annulus"], TF(c.min), TF(c.max), 0, z...)
    st == "cardinality" && return DeviceProjector{TF}(SET["cardinality"], TF(0), TF(0), Int64(c.max), z...)
    error("unknown set type $st")
end

function setup_constraints(constraint, comp_grid, ::Type{TF}) where TF
    nd = (length(comp_grid.n) == 3 && comp_grid.n[3] > 1) ? 3 : 2
    P_sub = Vector{Any}(undef, length(constraint)); TD_OP = Vector{Any}(undef, length(constraint))
    set_Prop = SIP.set_properties(fill(false, length(constraint)), fill(false, length(constraint)), fill(false, length(constraint)),
                                  Vector{Tuple}(undef, length(constraint)), Vector{Tuple{String,String,String,String}}(undef, length(constraint)),
                                  fill(false, length(constraint)), Vector{Vector{Int}}(undef, length(constraint)))
    for (i, c) in enumerate(constraint)
        c.TD_OP in ("DFT", "DCT", "wavelet", "curvelet") && error("JOLI transforms are outside the device CDS path")
        (c.set_type in ("l1", "l2") && c.app_mode[1] in ("slice", "fiber")) &&
            error("l1 and l2 constraints only available for matrix or tensor mode, currently")          # :65-67
        # structure flags and TD_n from the reference's own get_TD_operator on a 3-point surrogate grid would do; the
        # real one is cheap enough for the flags: (A, AtA_diag, dense, TD_n, banded)
        (_, AtA_diag, dense, TD_n, banded) = SIP.get_TD_operator(comp_grid, c.TD_OP, TF)                  # :69
        custom = c.custom_TD_OP[1]
        if c.set_type != "subspace" && !isempty(custom)                                                    # :70-72
            TD_OP[i] = DeviceOperator{TF}("custom", pad3(comp_grid.n[1:nd]), nd, ntuple(a -> a <= nd ? Float64(TF(comp_grid.d[a])) : 1.0, 3),
                                          BLOCK_PLAIN, SparseMatrixCSC{TF,Int64}(custom))
        else
            TD_OP[i] = DeviceOperator{TF}(c.TD_OP in ("D2D", "D3D") ? "TV" : c.TD_OP, pad3(comp_grid.n[1:nd]), nd,
                                          ntuple(a -> a <= nd ? Float64(TF(comp_grid.d[a])) : 1.0, 3), BLOCK_PLAIN, nothing)
        end
        P_sub[i] = get_projector(c, TD_n, TF)                                                              # :74
        set_Prop.AtA_diag[i] = AtA_diag; set_Prop.dense[i] = dense; set_Prop.TD_n[i] = TD_n; set_Prop.banded[i] = banded
        set_Prop.tag[i] = (c.set_type, c.TD_OP, c.app_mode[1], c.app_mode[2])                              # :86
        set_Prop.ncvx[i] = c.set_type in ("rank", "cardinality") ||
                           (c.set_type in ("bounds", "histogram") && c.TD_OP != "identity" && TF(maximum(c.min)) > TF(0))   # :89-97
    end
    return P_sub, TD_OP, set_Prop
end

# ---------------------------------------------------------------------------------------------------------------
# PARSDMM_precompute_distribute: the device keeps ONE ROW PER STENCIL CLASS of every A'A (sipb_problem_set_ata_classes).
# The table is read off mat2CDS(A'A) of the SAME operator on a 3 x 3 (x 3) grid, built with the reference's own
# get_TD_operator / mat2CDS: there, row index and class coincide.
# ---------------------------------------------------------------------------------------------------------------
struct ClassTable{TF}
    tab::Matrix{TF}            # nd x 54 (column-major == the C layout [54][nd])
    offsets::Vector{Int64}
end

function class_table(op::DeviceOperator{TF}, comp_grid) where TF
    nd = op.ndim
    small = deepcopy(comp_grid); small.n = ntuple(_ -> 3, nd)
    (A, _, _, _, _) = SIP.get_TD_operator(small, op.kind, TF)
    ns = 3^nd
    B = sparse(A' * A)
    B = op.block_mode == BLOCK_PLAIN ? B : op.block_mode == BLOCK_LEFT ? blockdiag(B, spzeros(TF, ns, ns)) :
        op.block_mode == BLOCK_RIGHT ? blockdiag(spzeros(TF, ns, ns), B) : [B B; B B]
    (R, offs_s) = SIP.mat2CDS(B)
    strides_s = vcat([1, 3, 9][1:nd], ns); strides = vcat([1, op.n[1], op.n[1] * op.n[2]][1:nd], prod(op.n[1:nd]))
    offs = map(offs_s) do o                         # balanced-ternary digits of the small offset -> real offset
        rest, real = o, 0
        for q in length(strides_s):-1:1
            d = round(Int, rest / strides_s[q]); rest -= d * strides_s[q]; real += d * strides[q]
        end
        real
    end
    order = sortperm(offs)
    tab = zeros(TF, length(offs), 54)
    for half in 0:(op.block_mode == BLOCK_PLAIN ? 0 : 1), c in 0:ns-1
        ci, cj = c % 3, (c ÷ 3) % 3; ck = nd == 3 ? (c ÷ 9) % 3 : 0
        cls = nd == 2 ? ((half * 3 + 0) * 3 + cj) * 3 + ci : ((half * 3 + ck) * 3 + cj) * 3 + ci
        tab[:, cls + 1] = R[half * ns + c + 1, order]
    end
    ClassTable{TF}(tab, Int64.(offs[order]))
end

function PARSDMM_precompute_distribute(TD_OP, set_Prop, comp_grid, options)
    options.parallel && error("options.parallel=true is replaced by slab decomposition on the device path (init_slabs)")
    TF = typeof(TD_OP[1]).parameters[1]
    nd = TD_OP[1].ndim
    if !options.feasibility_only                                                                       # :17-26
        push!(TD_OP, DeviceOperator{TF}("identity", TD_OP[1].n, nd, TD_OP[1].h, BLOCK_PLAIN, nothing))
        push!(set_Prop.TD_n, comp_grid.n); push!(set_Prop.AtA_offsets, [0]); push!(set_Prop.banded, true)
        push!(set_Prop.AtA_diag, true); push!(set_Prop.ncvx, false); push!(set_Prop.dense, false)
        push!(set_Prop.tag, ("distance squared", "identity", "matrix", ""))
    end
    p = length(TD_OP)
    AtA = Vector{Any}(undef, p)
    for i in 1:p
        if TD_OP[i].kind == "custom"              # explicit matrix: the CDS array itself (PARSDMM_precompute_distribute.jl:44-55)
            (AtA[i], set_Prop.AtA_offsets[i]) = SIP.mat2CDS(TD_OP[i].A' * TD_OP[i].A)
        else
            AtA[i] = class_table(TD_OP[i], comp_grid)
            set_Prop.AtA_offsets[i] = AtA[i].offsets
        end
    end
    y = [zeros(TF, size(TD_OP[i], 1)) for i in 1:p]; l = deepcopy(y)
    return TD_OP, AtA, l, y
end

with_block(op::DeviceOperator{TF}, mode) where TF = DeviceOperator{TF}(op.kind, op.n, op.ndim, op.h, mode, op.A)

function PARSDMM_precompute_distribute_Minkowski(TD_OP_c1, TD_OP_c2, TD_OP_sum, set_Prop_c1, set_Prop_c2, set_Prop_sum,
                                                 comp_grid, options)                                   # :3-157
    TF = typeof(TD_OP_c1[1]).parameters[1]
    TD_OP_c1 .= with_block.(TD_OP_c1, BLOCK_LEFT); TD_OP_c2 .= with_block.(TD_OP_c2, BLOCK_RIGHT)
    TD_OP_sum .= with_block.(TD_OP_sum, BLOCK_BOTH)
    if !options.feasibility_only
        push!(TD_OP_sum, DeviceOperator{TF}("identity", TD_OP_c1[1].n, TD_OP_c1[1].ndim, TD_OP_c1[1].h, BLOCK_BOTH, nothing))
        push!(set_Prop_sum.TD_n, comp_grid.n); push!(set_Prop_sum.AtA_offsets, [0]); push!(set_Prop_sum.banded, true)
        push!(set_Prop_sum.AtA_diag, false); push!(set_Prop_sum.dense, false); push!(set_Prop_sum.ncvx, false)
        push!(set_Prop_sum.tag, ("distance squared", "identity", "matrix", ""))
    end
    set_Prop = deepcopy(set_Prop_c1)
    for other in (set_Prop_c2, set_Prop_sum), f in (:AtA_diag, :AtA_offsets, :TD_n, :banded, :dense, :ncvx, :tag)
        append!(getfield(set_Prop, f), deepcopy(getfield(other, f)))
    end
    TD_OP = vcat(TD_OP_c1, TD_OP_c2, TD_OP_sum)
    if any(op -> op.kind == "custom", TD_OP)
        # a custom operator has no class table: CDS arrays for every set, mat2CDS of the 2N x 2N block matrices of
        # A'A formed like the reference (PARSDMM_precompute_distribute_Minkowski.jl:32-74,91-101,123-131)
        N = prod(TD_OP[1].n[1:TD_OP[1].ndim])
        Z = spzeros(TF, N, N)
        AtA = Vector{Any}(undef, length(TD_OP))
        for (i, op) in enumerate(TD_OP)
            if op.kind == "custom"
                B = op.A' * op.A
            elseif op.kind == "identity"
                B = spdiagm(0 => ones(TF, N))
            else
                A = SIP.get_TD_operator(comp_grid, op.kind, TF)[1]
                B = A' * A
            end
            M = op.block_mode == BLOCK_LEFT ? [B Z; Z Z] : (op.block_mode == BLOCK_RIGHT ? [Z Z; Z B] : [B B; B B])
            (AtA[i], set_Prop.AtA_offsets[i]) = SIP.mat2CDS(M)
        end
    else
        AtA = Any[class_table(op, comp_grid) for op in TD_OP]
    end
    for i in eachindex(TD_OP); AtA[i] isa ClassTable && (set_Prop.AtA_offsets[i] = AtA[i].offsets); end
    y = [zeros(TF, size(op, 1)) for op in TD_OP]; l = deepcopy(y)
    return TD_OP, set_Prop, AtA, l, y
end

# ---------------------------------------------------------------------------------------------------------------
# device problems: built once per AtA object, destroyed with it
# ---------------------------------------------------------------------------------------------------------------
mutable struct ProblemHandle
    ptr::Ptr{Cvoid}
    keep::Vector{Any}          # host arrays the descriptors pointed at during construction
    function ProblemHandle(ptr, keep)
        h = new(ptr, keep)
        finalizer(x -> (x.ptr != C_NULL && ccall((:sipb_problem_destroy, lib), Cint, (Ptr{Cvoid},), x.ptr); x.ptr = C_NULL), h)
        h
    end
end
const PROBLEMS = WeakKeyDict{Any,ProblemHandle}()       # keyed by the AtA vector returned by PARSDMM_precompute_distribute

function sparse_desc(A::SparseMatrixCSC{TF,Int64}, keep) where TF
    At = sparse(A')                                       # CSC of A' == CSR of A
    rowptr = At.colptr .- 1; colidx = Int32.(At.rowval .- 1); val = At.nzval
    colptr = A.colptr .- 1; rowidx = Int32.(A.rowval .- 1); valt = A.nzval
    append!(keep, (rowptr, colidx, val, colptr, rowidx, valt))
    r = Ref(SparseOp(size(A, 1), size(A, 2), nnz(A), pointer(rowptr), pointer(colidx), pointer(val), pointer(colptr),
                     pointer(rowidx), pointer(valt)))
    push!(keep, r)
    r
end

function device_problem(::Type{TF}, AtA, TD_OP, set_Prop, P_sub, comp_grid, options) where TF
    pb = Ref{Ptr{Cvoid}}(C_NULL)
    op1 = TD_OP[1]
    n = Int64[op1.n...]; h = Float64[op1.h...]
    check(ccall((:sipb_problem_create, lib), Cint,
                (Ptr{Cvoid}, Cint, Cint, Ptr{Int64}, Ptr{Float64}, Cint, Cint, Ptr{Ptr{Cvoid}}),
                context(), TF == Float32 ? 0 : 1, op1.ndim, n, h, options.Minkowski, options.feasibility_only, pb))
    keep = Any[]
    p = length(TD_OP); pp = options.feasibility_only ? p : p - 1
    for i in 1:p
        op = TD_OP[i]
        sp = op.kind == "custom" ? Base.unsafe_convert(Ptr{SparseOp}, sparse_desc(op.A, keep)) : Ptr{SparseOp}(C_NULL)
        if i <= pp
            P = P_sub[i]
            P.min isa Vector && push!(keep, P.min); P.max isa Vector && push!(keep, P.max)
            d = SetDesc(P.set_kind, OPK[op.kind], op.block_mode, set_Prop.ncvx[i],
                        P.min isa Real ? P.min : 0.0, P.max isa Real ? P.max : 0.0, P.k,
                        P.min isa Vector ? pointer(P.min) : C_NULL, P.max isa Vector ? pointer(P.max) : C_NULL,
                        P.fiber_axis, 0, P.td_n, sp)
        else
            d = SetDesc(SET["distance"], OPK[op.kind], op.block_mode, 0, 0.0, 0.0, 0, C_NULL, C_NULL, 0, 0, (0, 0, 0), sp)
        end
        GC.@preserve keep check(ccall((:sipb_problem_add_set, lib), Cint, (Ptr{Cvoid}, Ref{SetDesc}), pb[], d))
        off = Int64.(set_Prop.AtA_offsets[i])
        if AtA[i] isa ClassTable            # all sets of a problem come as tables, or all as arrays
            T = AtA[i].tab
            GC.@preserve T off check(ccall((:sipb_problem_set_ata_classes, lib), Cint,
                    (Ptr{Cvoid}, Cint, Ptr{Cvoid}, Ptr{Int64}, Cint), pb[], i - 1, T, off, length(off)))
        else
            R = AtA[i]::Matrix{TF}          # exactly what mat2CDS returned
            GC.@preserve R off check(ccall((:sipb_problem_set_ata, lib), Cint,
                    (Ptr{Cvoid}, Cint, Ptr{Cvoid}, Int64, Ptr{Int64}, Cint), pb[], i - 1, R, size(R, 1), off, length(off)))
        end
    end
    check(ccall((:sipb_problem_finalize, lib), Cint, (Ptr{Cvoid},), pb[]))
    ProblemHandle(pb[], keep)
end

# a problem with a custom operator needs CDS ARRAYS for every set: form them with the reference's own functions
function arrays_for_all!(AtA, TD_OP, comp_grid, ::Type{TF}) where TF
    any(a -> a isa Matrix, AtA) || return AtA
    for i in eachindex(AtA)
        AtA[i] isa ClassTable || continue
        (A, _, _, _, _) = SIP.get_TD_operator(comp_grid, TD_OP[i].kind, TF)
        (AtA[i], _) = SIP.mat2CDS(A' * A)
    end
    AtA
end

# ---------------------------------------------------------------------------------------------------------------
# PARSDMM
# ---------------------------------------------------------------------------------------------------------------
function PARSDMM(m::Vector{TF}, AtA, TD_OP, set_Prop, P_sub, comp_grid, options,
                 x = zeros(TF, length(m)), l = [], y = []) where {TF<:Real}
    SIP.convert_options!(options, TF)                                           # PARSDMM.jl:43
    options.parallel && error("options.parallel=true is rejected on the device path (use init_slabs)")
    arrays_for_all!(AtA, TD_OP, comp_grid, TF)
    pbh = get!(() -> device_problem(TF, AtA, TD_OP, set_Prop, P_sub, comp_grid, options), PROBLEMS, AtA)
    p = length(TD_OP); pp = options.feasibility_only ? p : p - 1; maxit = options.maxit
    N = options.Minkowski ? 2length(m) : length(m)
    length(x) == N || (x = [x; zeros(TF, N - length(x))])                       # PARSDMM.jl:85-89
    isempty(l) && (l = [zeros(TF, size(TD_OP[i], 1)) for i in 1:p]; y = deepcopy(l))
    rho = Float64.(options.rho_ini)
    o = Options(maxit, options.rho_update_frequency, options.adjust_rho, options.adjust_gamma,
                options.adjust_feasibility_rho, options.zero_ini_guess, length(rho), 0,
                options.evol_rel_tol, options.feas_tol, options.obj_tol, options.gamma_ini, pointer(rho), 0, 1, 0, 0)
    # row-major [maxit][p] of the C side == column-major (p, maxit) here
    A = Dict(k => zeros(Float64, k == :set_feasibility ? (max(pp, 1), maxit + 2) : (k in (:r_dual, :r_pri, :rho, :gamma) ? (p, maxit) : (maxit,)))
             for k in (:set_feasibility, :r_dual, :r_pri, :r_dual_total, :r_pri_total, :obj, :evol_x, :rho, :gamma, :cg_relres))
    cg_it = zeros(Int32, maxit)
    lg = Log(0, 0, 0, 0, 0, pointer(A[:set_feasibility]), pointer(A[:r_dual]), pointer(A[:r_pri]), pointer(A[:r_dual_total]),
             pointer(A[:r_pri_total]), pointer(A[:obj]), pointer(A[:evol_x]), pointer(A[:rho]), pointer(A[:gamma]),
             pointer(cg_it), pointer(A[:cg_relres]), ntuple(_ -> 0.0, 7), 0.0, 0.0, ntuple(_ -> 0, 24), ntuple(_ -> 0.0, 24),
             ntuple(_ -> 0.0, 24), 0, 0, 0)
    lp = Ptr{Cvoid}[pointer(v) for v in l]; yp = Ptr{Cvoid}[pointer(v) for v in y]
    GC.@preserve m x l y rho A cg_it lp yp pbh check(ccall((:sipb_solve, lib), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Ptr{Cvoid}}, Ptr{Ptr{Cvoid}}, Ref{Options}, Ref{Log}),
        pbh.ptr, m, x, lp, yp, o, lg))
    it = max(lg.iters, 1); c = lg.feas_rows
    if lg.stopped_feasible != 0 && options.zero_ini_guess          # feasible input: zero l, y (PARSDMM_initialize.jl:304-313)
        foreach(v -> fill!(v, 0), l); foreach(v -> fill!(v, 0), y)
    end
    # the seven TimerOutputs sections of PARSDMM.jl as device times (CUDA events close every phase): TimerOutputs has no
    # public way to inject measured times, so the log carries a Dict with the section names as keys
    timing = Dict(PHASES[q] => lg.phase_seconds[q] for q in 1:7)
    timing["device_seconds"] = lg.device_seconds; timing["solve_seconds"] = lg.solve_seconds
    log_PARSDMM = SIP.log_type_PARSDMM(permutedims(A[:set_feasibility][1:pp, 1:c]), permutedims(A[:r_dual][:, 1:it]),
        permutedims(A[:r_pri][:, 1:it]), A[:r_dual_total][1:it], A[:r_pri_total][1:it], A[:obj][1:it], A[:evol_x][1:it],
        permutedims(A[:rho][:, 1:it]), permutedims(A[:gamma][:, 1:it]), cg_it[1:it], A[:cg_relres][1:it], timing)
    return x, log_PARSDMM, l, y
end

end # module
