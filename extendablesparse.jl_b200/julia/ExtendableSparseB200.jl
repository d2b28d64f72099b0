# ExtendableSparseB200.jl -- Julia-side binding of libxsparse_b200.so.
#
# Plugs the CUDA library into ExtendableSparse.jl through the package's own extension
# interface (src/matrix/abstractsparsematrixextension.jl:1-19): `SparseMatrixB200` is an
# `AbstractSparseMatrixExtension`, and the user-facing matrix types are obtained exactly like
# the package's own aliases (src/ExtendableSparse.jl:35-39):
#
#     const B200ExtendableSparseMatrixCSC{Tv,Ti} =
#         GenericMTExtendableSparseMatrixCSC{SparseMatrixB200{Tv,Ti},Tv,Ti}
#
# NOTE: no Julia runtime exists in the build container of this repository, so this file has
# been written against the reference sources but NOT executed.  The call sequence it makes
# (xsb_set_csc -> xsb_insert_triplets per partition and flavour run -> xsb_flush -> xsb_fetch_csc, ONE
# device handle) is mirrored line by line by extendablesparse.jl_b200/dropin.py, which the GPU tests
# (tests/test_gpu_dropin.py) and the end-to-end leg of bench.py execute through ctypes.
#
# Per-entry calls are appended to a per-partition HOST buffer of 16-byte triplets (`XsbTriplet` =
# `xsb_triplet` of include/xsparse_b200.h: one 16-byte store per call, no ccall per entry) and stay
# there until `flush!`: like the reference's own buffers (SparseMatrixLNK / SparseMatrixDILNKC live in
# host memory until `flush!` merges them, extendable.jl:248-255) nothing touches the device before the
# flush.  16 bytes per insertion cross PCIe, once.

module ExtendableSparseB200

using SparseArrays
using ExtendableSparse
import ExtendableSparse: AbstractSparseMatrixExtension, rawupdateindex!, updateindex!, flush!, reset!

const libxsb = get(ENV, "XSPARSE_B200_LIB", "libxsparse_b200.so")

# status codes / enums of include/xsparse_b200.h
const XSB_OK, XSB_EBOUNDS, XSB_ESIZE, XSB_EILLEGAL = Int32(0), Int32(1), Int32(2), Int32(3)
const XSB_F64, XSB_I32, XSB_I64 = Int32(0), Int32(0), Int32(1)
const XSB_UPDATE, XSB_RAW, XSB_ASSIGN = Int32(0), Int32(1), Int32(2)
const XSB_DETERMINISTIC, XSB_FAST = Int32(0), Int32(1)
const XSB_COMBINE_SEED, XSB_COMBINE_ADD = Int32(0), Int32(1)
const XSB_OP_ADD, XSB_OP_SUB = Int32(0), Int32(1)

const CHUNK = 1 << 16

function check(h::Ptr{Cvoid}, rc::Int32)
    rc == XSB_OK && return nothing
    msg = unsafe_string(ccall((:xsb_last_error, libxsb), Cstring, (Ptr{Cvoid},), h))
    rc == XSB_EBOUNDS && throw(BoundsError())                    # sparsematrixcsc.jl:8-10
    rc == XSB_ESIZE && throw(AssertionError(msg))                # sparsematrixlnk.jl:296-297
    error("libxsparse_b200: [$rc] $msg")                        # genericmt...:67,80
end

"`xsb_triplet`: what one updateindex!/rawupdateindex!/setindex! call appends (1-based row/col)."
struct XsbTriplet
    row::UInt32
    col::UInt32
    val::Float64
end

idxcode(::Type{Int64}) = XSB_I64
idxcode(::Type{Int32}) = XSB_I32

"""
    SparseMatrixB200{Tv,Ti}(m, n)

Insert buffer of one partition: the calls since the last `flush!`, in call order, as 16-byte triplets in
host memory, plus the runs of equal flavour (update / rawupdate / assign).  Constructor signature
`T_ext(m,n)` as required by abstractsparsematrixextension.jl:10.  No device resource is held here; tasks
that insert with distinct `tid` touch distinct objects (test/femtools.jl:88-105), so no lock is needed.
"""
mutable struct SparseMatrixB200{Tv, Ti <: Integer} <: AbstractSparseMatrixExtension{Tv, Ti}
    m::Ti
    n::Ti
    T::Vector{XsbTriplet}
    fill::Int
    runs::Vector{Tuple{Int, Int32}}   # (index of the first triplet, flavour) of every run

    function SparseMatrixB200{Tv, Ti}(m, n) where {Tv, Ti <: Integer}
        Tv === Float64 || error("libxsparse_b200 implements Float64 values")
        (m < 2^32 && n < 2^32) || error("triplet buffers carry 32-bit indices")
        new{Tv, Ti}(m, n, Vector{XsbTriplet}(undef, CHUNK), 0, Tuple{Int, Int32}[])
    end
end

Base.size(x::SparseMatrixB200) = (x.m, x.n)
# upper bound of the distinct new entries, enough for `nnz(ext)>0` in flush!
# (genericextendablesparsematrixcsc.jl:31-37)
SparseArrays.nnz(x::SparseMatrixB200) = x.fill

@inline function push_entry!(x::SparseMatrixB200{Tv, Ti}, flavour::Int32, v, i, j) where {Tv, Ti}
    (1 <= i <= x.m && 1 <= j <= x.n) || throw(BoundsError(x, (i, j)))
    x.fill == length(x.T) && resize!(x.T, 2 * length(x.T))
    k = (x.fill += 1)
    (isempty(x.runs) || x.runs[end][2] != flavour) && push!(x.runs, (k, flavour))
    @inbounds x.T[k] = XsbTriplet(i % UInt32, j % UInt32, v)
    x
end

signed(op, v) = op === (+) ? v : op === (-) ? -v :
    error("libxsparse_b200 implements op in {+,-}; use the CPU buffers for other ops")

# the calls the generic wrappers forward to (genericmt...:87-114, genericextendable...:44-92)
rawupdateindex!(x::SparseMatrixB200, op, v, i, j) = push_entry!(x, XSB_RAW, signed(op, v), i, j)
rawupdateindex!(x::SparseMatrixB200, op, v, i, j, tid) = rawupdateindex!(x, op, v, i, j)
updateindex!(x::SparseMatrixB200, op, v, i, j) = push_entry!(x, XSB_UPDATE, signed(op, v), i, j)
Base.setindex!(x::SparseMatrixB200, v, i::Integer, j::Integer) = push_entry!(x, XSB_ASSIGN, v, i, j)
function Base.getindex(x::SparseMatrixB200{Tv}, i::Integer, j::Integer) where {Tv}
    # entries still in the buffer are not visible before flush! (same contract as the MT wrapper,
    # genericmt...:71-82); the single-buffer wrapper reaches here only on a CSC miss.
    nnz(x) == 0 ? zero(Tv) : error("flush! before reading unflushed entries of a B200 matrix")
end

# One device handle per (index type, size, partitions): created at the first flush!, reused by the following
# ones (its staging buffers and kernels stay warm), destroyed at exit.  flush! is called from one task
# (test/femtools.jl:109); the lock only guards the table.
const HANDLES = Dict{Tuple{DataType, Int, Int, Int}, Ptr{Cvoid}}()
const HANDLES_LOCK = ReentrantLock()
function device_handle(::Type{Ti}, m, n, nparts; device = 0) where {Ti}
    lock(HANDLES_LOCK) do
        get!(HANDLES, (Ti, Int(m), Int(n), nparts)) do
            h = Ref{Ptr{Cvoid}}(C_NULL)
            rc = ccall((:xsb_create, libxsb), Int32,
                       (Int64, Int64, Int32, Int32, Int32, Int32, Int32, Ref{Ptr{Cvoid}}),
                       m, n, XSB_F64, idxcode(Ti), 1, nparts, device, h)
            check(Ptr{Cvoid}(C_NULL), rc)
            h[]
        end
    end
end
function __init__()
    atexit() do
        lock(HANDLES_LOCK) do
            foreach(h -> ccall((:xsb_destroy, libxsb), Int32, (Ptr{Cvoid},), h), values(HANDLES))
            empty!(HANDLES)
        end
    end
end

"""
    Base.sum(exts::Vector{SparseMatrixB200}, csc) -> SparseMatrixCSC

The flush of the plug-in contract (abstractsparsematrixextension.jl:13): partitions are summed in vector
order like sparsematrixdilnkc.jl:416-426.  ONE device handle with one staging buffer per partition:

    xsb_set_csc(h, csc)                                   old CSC -> HBM  (16 B per old entry, once)
    xsb_insert_triplets(h, t-1, run, count, flavour)      every partition's calls, run by run, in call order
    xsb_flush(h, mode, &nnz, &changed)                    merge on the GPU
    xsb_fetch_csc(h, colptr, rowval, nzval)               new CSC -> Julia-owned arrays
"""
function Base.sum(exts::Vector{SparseMatrixB200{Tv, Ti}}, csc::SparseMatrixCSC{Tv, Ti};
                  mode = XSB_DETERMINISTIC) where {Tv, Ti}
    sum(nnz, exts) == 0 && return csc
    h = device_handle(Ti, csc.m, csc.n, length(exts))
    check(h, ccall((:xsb_set_csc, libxsb), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}),
                   h, csc.colptr, csc.rowval, csc.nzval))
    for (t, e) in enumerate(exts)
        for (r, (first, flavour)) in enumerate(e.runs)
            last = r < length(e.runs) ? e.runs[r + 1][1] - 1 : e.fill
            GC.@preserve e begin
                check(h, ccall((:xsb_insert_triplets, libxsb), Int32,
                               (Ptr{Cvoid}, Int32, Ptr{XsbTriplet}, Int64, Int32),
                               h, t - 1, pointer(e.T, first), last - first + 1, flavour))
            end
        end
    end
    nnz_new = Ref{Int64}(0); changed = Ref{Int32}(0)
    check(h, ccall((:xsb_flush, libxsb), Int32, (Ptr{Cvoid}, Int32, Ref{Int64}, Ref{Int32}), h, mode, nnz_new, changed))
    colptr = Vector{Ti}(undef, csc.n + 1)
    rowval = Vector{Ti}(undef, nnz_new[])
    nzval = Vector{Tv}(undef, nnz_new[])
    check(h, ccall((:xsb_fetch_csc, libxsb), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}),
                   h, colptr, rowval, nzval))
    SparseMatrixCSC{Tv, Ti}(csc.m, csc.n, colptr, rowval, nzval)
end

Base.:+(x::SparseMatrixB200, csc::SparseMatrixCSC) = sum([x], csc)

# ---------------------------------------------------------------------------------------
# B200Assembler: the device matrix proper (resident CSC + per-partition staging buffers).
# Users who can afford to keep the matrix on the GPU between flushes should use this type
# directly; the AbstractSparseMatrixExtension path above round-trips the CSC every flush!.
# ---------------------------------------------------------------------------------------
mutable struct B200Assembler{Tv, Ti <: Integer}
    m::Int
    n::Int
    handle::Ptr{Cvoid}
    nranks::Int # slab assemblers: ranks and own rank (0, 0: a whole matrix)
    rank::Int
    slab::Any # device buffers of a stream frozen across column slabs (freeze_slab!), or nothing
    function B200Assembler{Tv, Ti}(m, n, nparts = 1; device = 0) where {Tv, Ti}
        h = Ref{Ptr{Cvoid}}(C_NULL)
        rc = ccall((:xsb_create, libxsb), Int32,
                   (Int64, Int64, Int32, Int32, Int32, Int32, Int32, Ref{Ptr{Cvoid}}),
                   m, n, XSB_F64, idxcode(Ti), 1, nparts, device, h)
        check(Ptr{Cvoid}(C_NULL), rc)
        x = new{Tv, Ti}(m, n, h[], 0, 0, nothing)
        finalizer(y -> (free_slab_buffers!(y); y.handle == C_NULL || ccall((:xsb_destroy, libxsb), Int32, (Ptr{Cvoid},), y.handle);
                        y.handle = C_NULL), x)
        x
    end
    # column slab of a matrix sharded over `nranks` processes: rank r owns columns col_splits[r+1]+1 : col_splits[r+2]
    # (col_splits 0-based, nranks + 1 entries); insertions carry GLOBAL indices, the CSC is the slab's
    function B200Assembler{Tv, Ti}(m, n, nranks::Integer, rank::Integer, col_splits::Vector{Int64}; device = 0) where {Tv, Ti}
        h = Ref{Ptr{Cvoid}}(C_NULL)
        rc = ccall((:xsb_create_slab, libxsb), Int32,
                   (Int64, Int64, Int32, Int32, Ptr{Int64}, Int32, Int32, Int32, Int32, Ref{Ptr{Cvoid}}),
                   m, n, nranks, rank, col_splits, XSB_F64, idxcode(Ti), 1, device, h)
        check(Ptr{Cvoid}(C_NULL), rc)
        x = new{Tv, Ti}(m, n, h[], nranks, rank, nothing)
        finalizer(y -> (free_slab_buffers!(y); y.handle == C_NULL || ccall((:xsb_destroy, libxsb), Int32, (Ptr{Cvoid},), y.handle);
                        y.handle = C_NULL), x)
        x
    end
    # takes ownership of a plain handle the library returned (the result of + and -)
    function B200Assembler{Tv, Ti}(m, n, handle::Ptr{Cvoid}) where {Tv, Ti}
        x = new{Tv, Ti}(m, n, handle, 0, 0, nothing)
        finalizer(y -> (y.handle == C_NULL || ccall((:xsb_destroy, libxsb), Int32, (Ptr{Cvoid},), y.handle);
                        y.handle = C_NULL), x)
        x
    end
end

function set_csc!(a::B200Assembler{Tv, Ti}, csc::SparseMatrixCSC{Tv, Ti}) where {Tv, Ti}
    check(a.handle, ccall((:xsb_set_csc, libxsb), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}),
                          a.handle, csc.colptr, csc.rowval, csc.nzval))
end

"bulk insertion: k-th element == k-th updateindex!/rawupdateindex!/setindex! call"
function insert!(a::B200Assembler{Tv, Ti}, I::Vector{Ti}, J::Vector{Ti}, V::Vector{Tv};
                 flavour = XSB_UPDATE, tid = 0) where {Tv, Ti}
    check(a.handle, ccall((:xsb_insert_batch, libxsb), Int32,
                          (Ptr{Cvoid}, Int32, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Int64, Int32),
                          a.handle, tid, I, J, V, length(V), flavour))
end

"""
    insert_elements!(a, dofs, Aloc; flavour = XSB_RAW, tid = 0)

Element loop of test/femtools.jl:45-72 in one call: for every cell `c`, `for jl, for il`,
`rawupdateindex!(A, +, Aloc[il, jl, c], dofs[il, c], dofs[jl, c])` (or the `flavour`'s call), in that order.
`dofs` is `cellnodes` (k x ncells), `Aloc` the k x k x ncells element matrices.
"""
function insert_elements!(a::B200Assembler{Tv, Ti}, dofs::Matrix{Ti}, Aloc::Array{Tv, 3};
                          flavour = XSB_RAW, tid = 0) where {Tv, Ti}
    k = size(dofs, 1)
    size(Aloc) == (k, k, size(dofs, 2)) || throw(DimensionMismatch("size(Aloc) must be (k, k, size(dofs, 2))"))
    check(a.handle, ccall((:xsb_insert_elements, libxsb), Int32,
                          (Ptr{Cvoid}, Int32, Int32, Int64, Ptr{Cvoid}, Ptr{Cvoid}, Int32),
                          a.handle, tid, k, size(dofs, 2), dofs, Aloc, flavour))
end

"""
    insert_elements!(a, rowdofs, coldofs, Aloc; flavour = XSB_RAW, tid = 0)

The element loop whose rows and columns come from different connectivities (coupling blocks, rectangular
operators): for every cell `c`, `for jl, for il`, `rawupdateindex!(A, +, Aloc[il, jl, c], rowdofs[il, c],
coldofs[jl, c])`.  `rowdofs` is kr x ncells, `coldofs` kc x ncells, `Aloc` kr x kc x ncells.
"""
function insert_elements!(a::B200Assembler{Tv, Ti}, rowdofs::Matrix{Ti}, coldofs::Matrix{Ti}, Aloc::Array{Tv, 3};
                          flavour = XSB_RAW, tid = 0) where {Tv, Ti}
    kr, kc, ncells = size(rowdofs, 1), size(coldofs, 1), size(rowdofs, 2)
    size(coldofs, 2) == ncells || throw(DimensionMismatch("rowdofs and coldofs must have the same number of cells"))
    size(Aloc) == (kr, kc, ncells) || throw(DimensionMismatch("size(Aloc) must be (kr, kc, ncells)"))
    check(a.handle, ccall((:xsb_insert_elements_rect, libxsb), Int32,
                          (Ptr{Cvoid}, Int32, Int32, Int32, Int64, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Int32),
                          a.handle, tid, kr, kc, ncells, rowdofs, coldofs, Aloc, flavour))
end

"flush! + sparse(A): two-phase -- query nnz, allocate Julia arrays, fetch (ownership stays with Julia)"
function fetch!(a::B200Assembler{Tv, Ti}, mode = XSB_DETERMINISTIC) where {Tv, Ti}
    nnz = Ref{Int64}(0); changed = Ref{Int32}(0)
    check(a.handle, ccall((:xsb_flush, libxsb), Int32, (Ptr{Cvoid}, Int32, Ref{Int64}, Ref{Int32}),
                          a.handle, mode, nnz, changed))
    colptr = Vector{Ti}(undef, a.n + 1)
    rowval = Vector{Ti}(undef, nnz[])
    nzval = Vector{Tv}(undef, nnz[])
    check(a.handle, ccall((:xsb_fetch_csc, libxsb), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}),
                          a.handle, colptr, rowval, nzval))
    SparseMatrixCSC{Tv, Ti}(a.m, a.n, colptr, rowval, nzval)
end

"values-only Newton/transient loop: freeze the stream's positions once, then push values"
function freeze!(a::B200Assembler{Tv, Ti}, I::Vector{Ti}, J::Vector{Ti}) where {Tv, Ti}
    check(a.handle, ccall((:xsb_freeze_pattern, libxsb), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Int64),
                          a.handle, I, J, length(I)))
end
"freeze! for the element loop of insert_elements!: then `reassemble!(a, vec(Aloc))` each step"
function freeze_elements!(a::B200Assembler{Tv, Ti}, dofs::Matrix{Ti}) where {Tv, Ti}
    check(a.handle, ccall((:xsb_freeze_elements, libxsb), Int32, (Ptr{Cvoid}, Int32, Int64, Ptr{Cvoid}),
                          a.handle, size(dofs, 1), size(dofs, 2), dofs))
end
"freeze! for the element loop of insert_elements!(a, rowdofs, coldofs, Aloc)"
function freeze_elements!(a::B200Assembler{Tv, Ti}, rowdofs::Matrix{Ti}, coldofs::Matrix{Ti}) where {Tv, Ti}
    size(coldofs, 2) == size(rowdofs, 2) || throw(DimensionMismatch("rowdofs and coldofs must have the same number of cells"))
    check(a.handle, ccall((:xsb_freeze_elements_rect, libxsb), Int32, (Ptr{Cvoid}, Int32, Int32, Int64, Ptr{Cvoid}, Ptr{Cvoid}),
                          a.handle, size(rowdofs, 1), size(coldofs, 1), size(rowdofs, 2), rowdofs, coldofs))
end
function reassemble!(a::B200Assembler{Tv}, V::Vector{Tv}; mode = XSB_DETERMINISTIC, zero = true) where {Tv}
    # zero = true: nonzeros(A) .= 0 and the re-assembly as ONE pass over nzval (xsb_reassemble_values_zeroed)
    f = zero ? :xsb_reassemble_values_zeroed : :xsb_reassemble_values
    check(a.handle, ccall((f, libxsb), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Int64, Int32),
                          a.handle, V, length(V), mode))
end

"""
    pointblock(a::B200Assembler, blocksize) -> (colptr, rowval, blocks)

Device version of `pointblock` (src/matrix/extendable.jl:292-318): the block pattern is assembled on
the GPU from the resident CSC; `blocks[:, :, k]` is the k-th stored `blocksize x blocksize` block
(column-major, the memory layout of `SMatrix{bs,bs}`), so
`reinterpret(SMatrix{bs,bs,Tv,bs*bs}, vec(blocks))` is the `nzval` of the reference's result.
"""
function pointblock(a::B200Assembler{Tv, Ti}, blocksize::Integer) where {Tv, Ti}
    hb = Ref{Ptr{Cvoid}}(C_NULL)
    check(a.handle, ccall((:xsb_pointblock, libxsb), Int32, (Ptr{Cvoid}, Int32, Ref{Ptr{Cvoid}}),
                          a.handle, blocksize, hb))
    try
        nnzb = Ref{Int64}(0)
        check(hb[], ccall((:xsb_nnz, libxsb), Int32, (Ptr{Cvoid}, Ref{Int64}), hb[], nnzb))
        nb = a.n ÷ blocksize
        colptr = Vector{Ti}(undef, nb + 1)
        rowval = Vector{Ti}(undef, nnzb[])
        blocks = Array{Tv, 3}(undef, blocksize, blocksize, nnzb[])
        check(hb[], ccall((:xsb_fetch_csc, libxsb), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}),
                          hb[], colptr, rowval, C_NULL))
        check(hb[], ccall((:xsb_fetch_blocks, libxsb), Int32, (Ptr{Cvoid}, Ptr{Cvoid}), hb[], blocks))
        return colptr, rowval, blocks
    finally
        ccall((:xsb_destroy, libxsb), Int32, (Ptr{Cvoid},), hb[])
    end
end

"""
    a + b, a - b -> B200Assembler

SparseArrays' `+` / `-` of the two flushed matrices (src/matrix/abstractextendablesparsematrixcsc.jl: flush
both, then `map(+/-, A, B)`), computed on the device: entries equal to zero are not stored.  The result is a
new assembler on `a`'s device with its own handle: insert!, fetch!, freeze! and mul work on it.
"""
function add_sub(a::B200Assembler{Tv, Ti}, b::B200Assembler{Tv, Ti}, op) where {Tv, Ti}
    hc = Ref{Ptr{Cvoid}}(C_NULL)
    check(a.handle, ccall((:xsb_add, libxsb), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Int32, Ref{Ptr{Cvoid}}),
                          a.handle, b.handle, op, hc))
    B200Assembler{Tv, Ti}(a.m, a.n, hc[])
end
Base.:+(a::B200Assembler{Tv, Ti}, b::B200Assembler{Tv, Ti}) where {Tv, Ti} = add_sub(a, b, XSB_OP_ADD)
Base.:-(a::B200Assembler{Tv, Ti}, b::B200Assembler{Tv, Ti}) where {Tv, Ti} = add_sub(a, b, XSB_OP_SUB)

"""
    a * b -> B200Assembler

SparseArrays' `*` of the two flushed matrices (src/matrix/abstractextendablesparsematrixcsc.jl: flush both, then
`spmatmul`), computed on the device: the structural pattern, each entry the left fold in ascending k of the products.
The result is a new `a.m × b.n` assembler on `a`'s device with its own handle: insert!, fetch!, freeze! and mul work
on it.
"""
function Base.:*(a::B200Assembler{Tv, Ti}, b::B200Assembler{Tv, Ti}) where {Tv, Ti}
    hc = Ref{Ptr{Cvoid}}(C_NULL)
    check(a.handle, ccall((:xsb_matmul, libxsb), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ref{Ptr{Cvoid}}), a.handle, b.handle, hc))
    B200Assembler{Tv, Ti}(a.m, b.n, hc[])
end

"dropzeros!(a): the stored +-0.0 of the flushed matrix removed in place on the device (a slab: its own columns)"
function SparseArrays.dropzeros!(a::B200Assembler)
    nnz = Ref{Int64}(0); changed = Ref{Int32}(0)
    check(a.handle, ccall((:xsb_dropzeros, libxsb), Int32, (Ptr{Cvoid}, Ref{Int64}, Ref{Int32}), a.handle, nnz, changed))
    a
end

# the drop-in aliases, mirroring src/ExtendableSparse.jl:35-39
const B200ExtendableSparseMatrixCSC{Tv, Ti} =
    ExtendableSparse.GenericMTExtendableSparseMatrixCSC{SparseMatrixB200{Tv, Ti}, Tv, Ti}
const STB200ExtendableSparseMatrixCSC{Tv, Ti} =
    ExtendableSparse.GenericExtendableSparseMatrixCSC{SparseMatrixB200{Tv, Ti}, Tv, Ti}

"pattern_equal(a, b) on the device (sparsematrixcsc.jl:77-85)"
function pattern_equal(a::B200Assembler, b::B200Assembler)
    eq = Ref{Int32}(0)
    check(a.handle, ccall((:xsb_pattern_equal, libxsb), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ref{Int32}), a.handle, b.handle, eq))
    eq[] != 0
end

# ---- multi-GPU: one Julia process (MPI rank) per GPU, column slabs, peer exchange over NVLink (INTEGRATION.md §4) ----
"""
    peer_exchange!(a, caps_in, allgather)

Collective over the ranks of one node.  `caps_in[src+1]` = record slots this rank offers to rank `src` (0: the two
ranks exchange nothing); `allgather(v::Vector)` concatenates every rank's `v` in rank order (e.g.
`v -> MPI.Allgather(v, comm)`).  Afterwards every assembly step is `route_step!(a)`; `flush` follows as usual.
"""
function peer_exchange!(a::B200Assembler, caps_in::Vector{Int64}, allgather)
    caps = allgather(caps_in)                       # caps[dst * n + src + 1]
    handle = Vector{UInt8}(undef, 64)
    check(a.handle, ccall((:xsb_peer_exchange_create, libxsb), Int32, (Ptr{Cvoid}, Ptr{Int64}, Ptr{UInt8}),
                          a.handle, caps, handle))
    handles = allgather(handle)
    check(a.handle, ccall((:xsb_peer_exchange_connect, libxsb), Int32, (Ptr{Cvoid}, Ptr{UInt8}), a.handle, handles))
    a
end

"what other ranks own leaves for their mailboxes, what they sent is taken (both stream-ordered, no host round trip)"
function route_step!(a::B200Assembler)
    check(a.handle, ccall((:xsb_route_pack_peer, libxsb), Int32, (Ptr{Cvoid},), a.handle))
    check(a.handle, ccall((:xsb_route_unpack_peer, libxsb), Int32, (Ptr{Cvoid},), a.handle))
    a
end

"teardown: every rank disconnects, `barrier()`, every rank frees its mailbox"
function peer_exchange_close!(a::B200Assembler, barrier)
    check(a.handle, ccall((:xsb_peer_exchange_disconnect, libxsb), Int32, (Ptr{Cvoid},), a.handle))
    barrier()
    check(a.handle, ccall((:xsb_peer_exchange_destroy, libxsb), Int32, (Ptr{Cvoid},), a.handle))
    a
end

# ---- values-only re-assembly of a stream of GLOBAL positions frozen across the column slabs (INTEGRATION.md §4) ----
# `alltoallv(sendbuf::Ptr, sendcounts::Vector{Int64}, recvbuf::Ptr, recvcounts::Vector{Int64}, itembytes)` is the
# caller's all-to-all-v over the ranks (e.g. CUDA-aware `MPI.Alltoallv!`): item counts per rank, own rank 0; the
# buffers are host memory for the counts and device memory for positions and values.
const libcudart = get(ENV, "XSPARSE_B200_CUDART", "libcudart.so")
function device_alloc(bytes)
    p = Ref{Ptr{Cvoid}}(C_NULL)
    ccall((:cudaMalloc, libcudart), Int32, (Ref{Ptr{Cvoid}}, Csize_t), p, max(bytes, 16)) == 0 ||
        throw(OutOfMemoryError())
    p[]
end
function free_slab_buffers!(a::B200Assembler)
    if a.slab !== nothing
        for p in (a.slab.send, a.slab.recv)
            ccall((:cudaFree, libcudart), Int32, (Ptr{Cvoid},), p)
        end
        a.slab = nothing
    end
    a
end

function freeze_slab_exchange!(a::B200Assembler, send_counts::Vector{Int64}, alltoallv)
    nranks, rank = a.nranks, a.rank
    off = [r == rank ? 0 : send_counts[r + 1] for r in 0:nranks-1]
    recv_counts = zeros(Int64, nranks)
    ones_ = [r == rank ? 0 : 1 for r in 0:nranks-1]
    alltoallv(pointer(off), ones_, pointer(recv_counts), ones_, 8)
    send = device_alloc(8 * sum(off))
    recv = device_alloc(8 * sum(recv_counts))
    try
        check(a.handle, ccall((:xsb_freeze_slab_prepare, libxsb), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Int64),
                              a.handle, send, sum(off)))
        alltoallv(send, off, recv, recv_counts, 8)
        check(a.handle, ccall((:xsb_freeze_slab_finish, libxsb), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Int64}),
                              a.handle, recv, recv_counts))
    catch
        ccall((:cudaFree, libcudart), Int32, (Ptr{Cvoid},), send)
        ccall((:cudaFree, libcudart), Int32, (Ptr{Cvoid},), recv)
        rethrow()
    end
    ccall((:cudaFree, libcudart), Int32, (Ptr{Cvoid},), send)
    ccall((:cudaFree, libcudart), Int32, (Ptr{Cvoid},), recv)
    # the per-step value buffers: sizes fixed since the freeze
    a.slab = (send = device_alloc(8 * sum(off)), recv = device_alloc(8 * sum(recv_counts)), off = off,
              recv_counts = recv_counts)
    a
end

"""
    freeze_slab!(a, I, J, alltoallv)

Collective over the ranks: freezes this rank's stream of GLOBAL positions (any owner) on the slab assembler `a`;
afterwards every step is `reassemble_slab!(a, V, alltoallv)`.  A rank whose freeze fails throws; the caller
must make the other ranks give up too (e.g. an all-reduce of the status), every handle is then left unfrozen.
"""
function freeze_slab!(a::B200Assembler{Tv, Ti}, I::Vector{Ti}, J::Vector{Ti}, alltoallv) where {Tv, Ti}
    free_slab_buffers!(a)
    counts = zeros(Int64, a.nranks)
    check(a.handle, ccall((:xsb_freeze_slab, libxsb), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Int64, Ptr{Int64}),
                          a.handle, I, J, length(I), counts))
    freeze_slab_exchange!(a, counts, alltoallv)
end

"freeze_slab! for the element loop of insert_elements!: then `reassemble_slab!(a, vec(Aloc), alltoallv)` each step"
function freeze_slab_elements!(a::B200Assembler{Tv, Ti}, dofs::Matrix{Ti}, alltoallv) where {Tv, Ti}
    free_slab_buffers!(a)
    counts = zeros(Int64, a.nranks)
    check(a.handle, ccall((:xsb_freeze_slab_elements, libxsb), Int32, (Ptr{Cvoid}, Int32, Int64, Ptr{Cvoid}, Ptr{Int64}),
                          a.handle, size(dofs, 1), size(dofs, 2), dofs, counts))
    freeze_slab_exchange!(a, counts, alltoallv)
end

"freeze_slab! for the element loop of insert_elements!(a, rowdofs, coldofs, Aloc)"
function freeze_slab_elements!(a::B200Assembler{Tv, Ti}, rowdofs::Matrix{Ti}, coldofs::Matrix{Ti}, alltoallv) where {Tv, Ti}
    size(coldofs, 2) == size(rowdofs, 2) || throw(DimensionMismatch("rowdofs and coldofs must have the same number of cells"))
    free_slab_buffers!(a)
    counts = zeros(Int64, a.nranks)
    check(a.handle, ccall((:xsb_freeze_slab_elements_rect, libxsb), Int32,
                          (Ptr{Cvoid}, Int32, Int32, Int64, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Int64}),
                          a.handle, size(rowdofs, 1), size(coldofs, 1), size(rowdofs, 2), rowdofs, coldofs, counts))
    freeze_slab_exchange!(a, counts, alltoallv)
end

"""
    reassemble_slab!(a, V, alltoallv; mode = XSB_DETERMINISTIC, zero = true)

One values-only step of a stream frozen with `freeze_slab!`: the values of positions other ranks own leave through
`alltoallv` with the sizes of the freeze, and every slab entry folds its resident value (+0.0 with `zero`) followed
by the values of rank 0, 1, ... in each rank's stream order.
"""
function reassemble_slab!(a::B200Assembler{Tv}, V::Vector{Tv}, alltoallv; mode = XSB_DETERMINISTIC, zero = true) where {Tv}
    s = a.slab
    s === nothing && error("no frozen slab stream: freeze_slab! first")
    check(a.handle, ccall((:xsb_reassemble_slab_pack, libxsb), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Int64, Ptr{Cvoid}),
                          a.handle, V, length(V), s.send))
    ccall((:xsb_synchronize, libxsb), Int32, (Ptr{Cvoid},), a.handle)
    alltoallv(s.send, s.off, s.recv, s.recv_counts, 8)
    check(a.handle, ccall((:xsb_reassemble_slab_values, libxsb), Int32,
                          (Ptr{Cvoid}, Ptr{Cvoid}, Int64, Ptr{Cvoid}, Int32, Int32),
                          a.handle, V, length(V), s.recv, mode, zero ? 1 : 0))
    a
end

export freeze_slab!, freeze_slab_elements!, reassemble_slab!

export peer_exchange!, route_step!, peer_exchange_close!
export SparseMatrixB200, B200Assembler, pattern_equal, B200ExtendableSparseMatrixCSC, STB200ExtendableSparseMatrixCSC,
       set_csc!, insert!, insert_elements!, fetch!, freeze!, freeze_elements!, reassemble!, pointblock, XsbTriplet

end # module
