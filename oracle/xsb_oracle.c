/*
 * xsb_oracle.c -- CPU ORACLE (test infrastructure, NOT product code).
 *
 * A plain-C, single-threaded restatement of the assembly hot path of
 * ExtendableSparse.jl v1.5.1, written from the algorithm's description in the
 * reference sources (paths relative to /root/reference):
 *
 *   src/matrix/sparsematrixlnk.jl      SparseMatrixLNK (linked-list buffer), lnk + csc flush
 *   src/matrix/sparsematrixcsc.jl      findindex (binary search in a CSC column)
 *   src/matrix/extendable.jl           ExtendableSparseMatrixCSC router + flush!
 *   src/matrix/sparsematrixdilnkc.jl   SparseMatrixDILNKC + Base.sum(Vector, csc)
 *   src/matrix/genericmtextendablesparsematrixcsc.jl   per-partition buffers
 *   src/matrix/sprand.jl               fdrand! insertion stream
 *   test/femtools.jl                   P1 FEM insertion stream
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl
 * reference legs may load this library.  The product (libxsparse_b200.so) never
 * links, loads or calls it.
 *
 * PARITY PINNING.  The reference is pure Julia; no Julia runtime exists in the
 * build container and the reference's tests hold no stored golden vectors
 * (SURVEY.md section 4, 8c).  The oracle is therefore pinned against the
 * reference's own KNOWN-ANSWER tests, restated in tests/test_oracle_kat.py:
 *   test/test_updates.jl:10-25      nnz sequence 0,2,3,(2),3,(3) - zero semantics
 *   test/test_assembly.jl:6-35      exact equality with sequential accumulation,
 *                                   sorted columns, multi-splice flush
 *   test/test_operations.jl:8-13    csc + LNK(csc) == 2*csc
 *   test/test_constructors.jl:26-31 CSC -> LNK -> CSC round trip exact
 *   test/test_fdrand.jl:22-53       fdrand(rand=()->1) analytic matrix
 *   README.md:15-27                 10x10 tridiagonal example
 *   SURVEY.md 8(c')                 hand-stepped 3x3 micro vector
 * It has NOT been compared with outputs of the Julia package itself.
 *
 * The one third-party algorithm on the multi-partition path is the Julia
 * stdlib SparseArrays.sparse!(I,J,V,m,n,+) (un-vendored, version = the running
 * Julia's; Project.toml:38 julia = "1.9").  Its published semantics are restated in
 * ora_mt_flush below: rows sorted per column, duplicates combined in input
 * order with the first occurrence copied, explicit zeros kept.
 *
 * All indices crossing this API are 1-based like Julia's.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <math.h>
#include <pthread.h>

typedef int64_t i64;

#define ORA_OK 0
#define ORA_EBOUNDS 1
#define ORA_ESIZE 2
#define ORA_EILLEGAL 3

/* insertion flavours (same numbering as include/xsparse_b200.h) */
#define ORA_UPDATE 0 /* updateindex!(A,+,v,i,j)     : no new entry if v==0 */
#define ORA_RAW 1    /* rawupdateindex!(A,+,v,i,j)  : always creates       */
#define ORA_ASSIGN 2 /* A[i,j]=v (setindex!)        : creates only if v!=0 */

/* ------------------------------------------------------------------ */
/* growable arrays                                                     */
/* ------------------------------------------------------------------ */
static void *xrealloc(void *p, size_t bytes)
{
    void *q = realloc(p, bytes ? bytes : 1);
    if (!q)
        abort();
    return q;
}

/* ------------------------------------------------------------------ */
/* SparseMatrixCSC (1-based colptr/rowval like Julia)                  */
/* ------------------------------------------------------------------ */
typedef struct
{
    i64 m, n;
    i64 *colptr; /* n+1 */
    i64 *rowval; /* nnz */
    double *nzval;
} ora_csc;

static ora_csc *csc_alloc(i64 m, i64 n, i64 cap)
{
    ora_csc *c = (ora_csc *)calloc(1, sizeof(ora_csc));
    c->m = m;
    c->n = n;
    c->colptr = (i64 *)xrealloc(NULL, sizeof(i64) * (size_t)(n + 1));
    for (i64 j = 0; j <= n; j++)
        c->colptr[j] = 1; /* spzeros */
    c->rowval = (i64 *)xrealloc(NULL, sizeof(i64) * (size_t)cap);
    c->nzval = (double *)xrealloc(NULL, sizeof(double) * (size_t)cap);
    return c;
}

static void csc_free(ora_csc *c)
{
    if (!c)
        return;
    free(c->colptr);
    free(c->rowval);
    free(c->nzval);
    free(c);
}

static i64 csc_nnz(const ora_csc *c) { return c->colptr[c->n] - 1; }

/* findindex(csc,i,j): src/matrix/sparsematrixcsc.jl:7-23.
 * Returns the 1-based nz index, 0 when absent, -1 on a bounds error. */
static i64 csc_findindex(const ora_csc *c, i64 i, i64 j)
{
    if (!(1 <= i && i <= c->m && 1 <= j && j <= c->n))
        return -1;
    i64 r1 = c->colptr[j - 1];
    i64 r2 = c->colptr[j] - 1;
    if (r1 > r2)
        return 0;
    /* searchsortedfirst(rowval, i, r1, r2) */
    i64 lo = r1 - 1, hi = r2 + 1;
    while (lo < hi - 1)
    {
        i64 mid = lo + ((hi - lo) >> 1);
        if (c->rowval[mid - 1] < i)
            lo = mid;
        else
            hi = mid;
    }
    r1 = hi;
    if (r1 > r2 || c->rowval[r1 - 1] != i)
        return 0;
    return r1;
}

/* ------------------------------------------------------------------ */
/* SparseMatrixLNK: src/matrix/sparsematrixlnk.jl:21-68                */
/* Arrays are 1-based in the reference; slot k lives at [k-1] here.    */
/* ------------------------------------------------------------------ */
typedef struct
{
    i64 m, n, nnz, nentries, len;
    i64 *colptr;
    i64 *rowval;
    double *nzval;
} ora_lnk;

/* ctor: sparsematrixlnk.jl:75-77 */
ora_lnk *ora_lnk_create(i64 m, i64 n)
{
    ora_lnk *l = (ora_lnk *)calloc(1, sizeof(ora_lnk));
    l->m = m;
    l->n = n;
    l->nnz = 0;
    l->nentries = n;
    l->len = n;
    l->colptr = (i64 *)calloc((size_t)(n ? n : 1), sizeof(i64));
    l->rowval = (i64 *)calloc((size_t)(n ? n : 1), sizeof(i64));
    l->nzval = (double *)calloc((size_t)(n ? n : 1), sizeof(double));
    return l;
}

void ora_lnk_destroy(ora_lnk *l)
{
    if (!l)
        return;
    free(l->colptr);
    free(l->rowval);
    free(l->nzval);
    free(l);
}

i64 ora_lnk_nnz(const ora_lnk *l) { return l->nnz; }

/* findindex(lnk,i,j): sparsematrixlnk.jl:120-135. *k0 receives the list tail. */
static i64 lnk_findindex(const ora_lnk *l, i64 i, i64 j, i64 *k0out)
{
    i64 k = j, k0 = j;
    while (k > 0)
    {
        if (l->rowval[k - 1] == i)
        {
            *k0out = 0;
            return k;
        }
        k0 = k;
        k = l->colptr[k - 1];
    }
    *k0out = k0;
    return 0;
}

/* addentry!: sparsematrixlnk.jl:151-171 (growth factor 5/4, :154-159) */
static i64 lnk_addentry(ora_lnk *l, i64 i, i64 k0)
{
    l->nentries += 1;
    if (l->len < l->nentries)
    {
        i64 newsize = (i64)ceil(5.0 * (double)l->nentries / 4.0);
        l->nzval = (double *)xrealloc(l->nzval, sizeof(double) * (size_t)newsize);
        l->rowval = (i64 *)xrealloc(l->rowval, sizeof(i64) * (size_t)newsize);
        l->colptr = (i64 *)xrealloc(l->colptr, sizeof(i64) * (size_t)newsize);
        l->len = newsize;
    }
    l->rowval[l->nentries - 1] = i;
    l->colptr[l->nentries - 1] = 0;
    l->colptr[k0 - 1] = l->nentries;
    l->nnz += 1;
    return l->nentries;
}

static int lnk_inbounds(const ora_lnk *l, i64 i, i64 j)
{
    return (1 <= i && i <= l->m) && (1 <= j && j <= l->n);
}

/* setindex!(lnk,v,i,j): sparsematrixlnk.jl:178-201 */
int ora_lnk_setindex(ora_lnk *l, double v, i64 i, i64 j)
{
    if (!lnk_inbounds(l, i, j))
        return ORA_EBOUNDS;
    if (l->rowval[j - 1] == 0 && v != 0.0)
    {
        l->rowval[j - 1] = i;
        l->nzval[j - 1] = v;
        l->nnz += 1;
        return ORA_OK;
    }
    i64 k0;
    i64 k = lnk_findindex(l, i, j, &k0);
    if (k > 0)
    {
        l->nzval[k - 1] = v;
        return ORA_OK;
    }
    if (v != 0.0)
    {
        k = lnk_addentry(l, i, k0);
        l->nzval[k - 1] = v;
    }
    return ORA_OK;
}

/* updateindex!(lnk,+,v,i,j): sparsematrixlnk.jl:210-228 */
int ora_lnk_updateindex(ora_lnk *l, double v, i64 i, i64 j)
{
    if (!lnk_inbounds(l, i, j)) /* the public path checks in findindex(csc) first */
        return ORA_EBOUNDS;
    if (l->rowval[j - 1] == 0 && v != 0.0)
    {
        l->rowval[j - 1] = i;
        l->nzval[j - 1] = l->nzval[j - 1] + v;
        l->nnz += 1;
        return ORA_OK;
    }
    i64 k0;
    i64 k = lnk_findindex(l, i, j, &k0);
    if (k > 0)
    {
        l->nzval[k - 1] = l->nzval[k - 1] + v;
        return ORA_OK;
    }
    if (v != 0.0)
    {
        k = lnk_addentry(l, i, k0);
        l->nzval[k - 1] = 0.0 + v; /* op(zero(Tv), v), :225 */
    }
    return ORA_OK;
}

/* rawupdateindex!(lnk,+,v,i,j): sparsematrixlnk.jl:237-253 */
int ora_lnk_rawupdateindex(ora_lnk *l, double v, i64 i, i64 j)
{
    if (!lnk_inbounds(l, i, j))
        return ORA_EBOUNDS;
    if (l->rowval[j - 1] == 0)
    {
        l->rowval[j - 1] = i;
        l->nzval[j - 1] = l->nzval[j - 1] + v;
        l->nnz += 1;
        return ORA_OK;
    }
    i64 k0;
    i64 k = lnk_findindex(l, i, j, &k0);
    if (k > 0)
    {
        l->nzval[k - 1] = l->nzval[k - 1] + v;
    }
    else
    {
        k = lnk_addentry(l, i, k0);
        l->nzval[k - 1] = 0.0 + v;
    }
    return ORA_OK;
}

/* getindex(lnk,i,j): sparsematrixlnk.jl:142-149 */
int ora_lnk_getindex(const ora_lnk *l, i64 i, i64 j, double *out)
{
    if (!lnk_inbounds(l, i, j))
        return ORA_EBOUNDS;
    i64 k0;
    i64 k = lnk_findindex(l, i, j, &k0);
    *out = k ? l->nzval[k - 1] : 0.0;
    return ORA_OK;
}

typedef struct
{
    i64 rowval;
    double nzval;
} colentry;

static int colentry_less(const void *a, const void *b)
{
    i64 ra = ((const colentry *)a)->rowval, rb = ((const colentry *)b)->rowval;
    return (ra > rb) - (ra < rb);
}

/* Base.:+(lnk,csc): sparsematrixlnk.jl:294-383.  Rows inside one LNK column are
 * unique, so the (unstable) QuickSort of :339 has a unique result. */
static ora_csc *lnk_plus_csc(const ora_lnk *l, const ora_csc *c)
{
    i64 n = c->n;
    i64 cnnz = csc_nnz(c);
    i64 xnnz = cnnz + l->nnz;
    ora_csc *r = csc_alloc(c->m, n, xnnz);
    i64 maxcol = 0;
    for (i64 j = 1; j <= n; j++)
    { /* :307-316 */
        i64 lcol = 0, k = j;
        while (k > 0)
        {
            lcol++;
            k = l->colptr[k - 1];
        }
        if (lcol > maxcol)
            maxcol = lcol;
    }
    colentry *col = (colentry *)xrealloc(NULL, sizeof(colentry) * (size_t)(maxcol + 1));
    i64 inz = 1;
    for (i64 j = 1; j <= n; j++)
    { /* :328-377 */
        i64 k = j, lc = 0;
        while (k > 0)
        {
            if (l->rowval[k - 1] > 0)
            {
                col[lc].rowval = l->rowval[k - 1];
                col[lc].nzval = l->nzval[k - 1];
                lc++;
            }
            k = l->colptr[k - 1];
        }
        qsort(col, (size_t)lc, sizeof(colentry), colentry_less);
        r->colptr[j - 1] = inz;
        i64 jl = 0;
        i64 jc = c->colptr[j - 1];
        for (;;)
        {
            int in_c = (cnnz > 0) && (jc < c->colptr[j]);
            int in_l = jl < lc;
            if (in_c && ((in_l && c->rowval[jc - 1] < col[jl].rowval) || !in_l))
            {
                r->rowval[inz - 1] = c->rowval[jc - 1];
                r->nzval[inz - 1] = c->nzval[jc - 1];
                jc++;
                inz++;
            }
            else if (in_c && in_l && c->rowval[jc - 1] == col[jl].rowval)
            {
                r->rowval[inz - 1] = c->rowval[jc - 1];
                r->nzval[inz - 1] = c->nzval[jc - 1] + col[jl].nzval; /* :363 */
                jc++;
                inz++;
                jl++;
            }
            else if (in_l)
            {
                r->rowval[inz - 1] = col[jl].rowval;
                r->nzval[inz - 1] = col[jl].nzval;
                jl++;
                inz++;
            }
            else
                break;
        }
    }
    r->colptr[n] = inz;
    free(col);
    return r;
}

/* Stand-alone `lnk + csc` on caller-provided CSC arrays (test_operations.jl:8-13).
 * Outputs must hold nnz(csc)+nnz(lnk) entries; returns the result nnz or <0. */
i64 ora_lnk_plus_csc(const ora_lnk *l, i64 m, i64 n, const i64 *colptr, const i64 *rowval,
                     const double *nzval, i64 *colptr_out, i64 *rowval_out, double *nzval_out)
{
    if (m != l->m || n != l->n)
        return -ORA_ESIZE; /* @assert :296-297 */
    ora_csc c;
    c.m = m;
    c.n = n;
    c.colptr = (i64 *)colptr;
    c.rowval = (i64 *)rowval;
    c.nzval = (double *)nzval;
    ora_csc *r = lnk_plus_csc(l, &c);
    i64 nnz = csc_nnz(r);
    memcpy(colptr_out, r->colptr, sizeof(i64) * (size_t)(n + 1));
    memcpy(rowval_out, r->rowval, sizeof(i64) * (size_t)nnz);
    memcpy(nzval_out, r->nzval, sizeof(double) * (size_t)nnz);
    csc_free(r);
    return nnz;
}

/* ------------------------------------------------------------------ */
/* ExtendableSparseMatrixCSC: src/matrix/extendable.jl                 */
/* ------------------------------------------------------------------ */
typedef struct
{
    ora_csc *csc;
    ora_lnk *lnk; /* NULL == nothing */
    i64 nflush;   /* number of flushes that merged something (phash recomputations, :252) */
} ora_ext;

ora_ext *ora_ext_create(i64 m, i64 n)
{
    ora_ext *e = (ora_ext *)calloc(1, sizeof(ora_ext));
    e->csc = csc_alloc(m, n, 0);
    e->lnk = NULL;
    return e;
}

void ora_ext_destroy(ora_ext *e)
{
    if (!e)
        return;
    csc_free(e->csc);
    ora_lnk_destroy(e->lnk);
    free(e);
}

/* reset!: extendable.jl:269-272 */
void ora_ext_reset(ora_ext *e)
{
    i64 m = e->csc->m, n = e->csc->n;
    csc_free(e->csc);
    ora_lnk_destroy(e->lnk);
    e->csc = csc_alloc(m, n, 0);
    e->lnk = NULL;
}

/* ctor from CSC: extendable.jl:61-67 */
void ora_ext_set_csc(ora_ext *e, const i64 *colptr, const i64 *rowval, const double *nzval)
{
    i64 m = e->csc->m, n = e->csc->n;
    i64 nnz = colptr[n] - 1;
    csc_free(e->csc);
    ora_lnk_destroy(e->lnk);
    e->lnk = NULL;
    e->csc = csc_alloc(m, n, nnz);
    memcpy(e->csc->colptr, colptr, sizeof(i64) * (size_t)(n + 1));
    memcpy(e->csc->rowval, rowval, sizeof(i64) * (size_t)nnz);
    memcpy(e->csc->nzval, nzval, sizeof(double) * (size_t)nnz);
}

static void ext_need_lnk(ora_ext *e)
{
    if (!e->lnk)
        e->lnk = ora_lnk_create(e->csc->m, e->csc->n); /* :168-170 */
}

/* updateindex!(ext,+,v,i,j): extendable.jl:159-174 */
int ora_ext_updateindex(ora_ext *e, double v, i64 i, i64 j)
{
    i64 k = csc_findindex(e->csc, i, j);
    if (k < 0)
        return ORA_EBOUNDS;
    if (k > 0)
    {
        e->csc->nzval[k - 1] = e->csc->nzval[k - 1] + v;
        return ORA_OK;
    }
    ext_need_lnk(e);
    return ora_lnk_updateindex(e->lnk, v, i, j);
}

/* rawupdateindex!(ext,+,v,i,j): extendable.jl:181-197 */
int ora_ext_rawupdateindex(ora_ext *e, double v, i64 i, i64 j)
{
    i64 k = csc_findindex(e->csc, i, j);
    if (k < 0)
        return ORA_EBOUNDS;
    if (k > 0)
    {
        e->csc->nzval[k - 1] = e->csc->nzval[k - 1] + v;
        return ORA_OK;
    }
    ext_need_lnk(e);
    return ora_lnk_rawupdateindex(e->lnk, v, i, j);
}

/* setindex!(ext,v,i,j): extendable.jl:205-218 */
int ora_ext_setindex(ora_ext *e, double v, i64 i, i64 j)
{
    i64 k = csc_findindex(e->csc, i, j);
    if (k < 0)
        return ORA_EBOUNDS;
    if (k > 0)
    {
        e->csc->nzval[k - 1] = v;
        return ORA_OK;
    }
    ext_need_lnk(e);
    return ora_lnk_setindex(e->lnk, v, i, j);
}

/* getindex(ext,i,j): extendable.jl:226-238 */
int ora_ext_getindex(const ora_ext *e, i64 i, i64 j, double *out)
{
    i64 k = csc_findindex(e->csc, i, j);
    if (k < 0)
        return ORA_EBOUNDS;
    if (k > 0)
    {
        *out = e->csc->nzval[k - 1];
        return ORA_OK;
    }
    if (!e->lnk)
    {
        *out = 0.0;
        return ORA_OK;
    }
    return ora_lnk_getindex(e->lnk, i, j, out);
}

/* flush!(ext): extendable.jl:248-255 */
void ora_ext_flush(ora_ext *e)
{
    if (e->lnk && e->lnk->nnz > 0)
    {
        ora_csc *r = lnk_plus_csc(e->lnk, e->csc);
        csc_free(e->csc);
        e->csc = r;
        ora_lnk_destroy(e->lnk);
        e->lnk = NULL;
        e->nflush += 1;
    }
}

i64 ora_ext_nflush(const ora_ext *e) { return e->nflush; }

/* nnz(ext) flushes first: abstractextendablesparsematrixcsc.jl:24 */
i64 ora_ext_nnz(ora_ext *e)
{
    ora_ext_flush(e);
    return csc_nnz(e->csc);
}

i64 ora_ext_nnz_csc(const ora_ext *e) { return csc_nnz(e->csc); }
i64 ora_ext_nnz_lnk(const ora_ext *e) { return e->lnk ? e->lnk->nnz : 0; }

/* copy of the current CSC part (no flush); 1-based */
void ora_ext_get_csc(const ora_ext *e, i64 *colptr, i64 *rowval, double *nzval)
{
    i64 n = e->csc->n, nnz = csc_nnz(e->csc);
    memcpy(colptr, e->csc->colptr, sizeof(i64) * (size_t)(n + 1));
    if (rowval)
        memcpy(rowval, e->csc->rowval, sizeof(i64) * (size_t)nnz);
    if (nzval)
        memcpy(nzval, e->csc->nzval, sizeof(double) * (size_t)nnz);
}

/* nonzeros(A) .= 0 (sprand.jl:80-85, test_parallel.jl:55) */
void ora_ext_zero_values(ora_ext *e)
{
    i64 nnz = csc_nnz(e->csc);
    for (i64 k = 0; k < nnz; k++)
        e->csc->nzval[k] = 0.0;
    if (e->lnk)
        for (i64 k = 0; k < e->lnk->len; k++)
            e->lnk->nzval[k] = 0.0;
}

/* The per-entry call loop a user runs; returns the index of the first failing
 * entry + 1 (as a negative number) on a bounds error, else 0. */
i64 ora_ext_insert_batch(ora_ext *e, const i64 *I, const i64 *J, const double *V, i64 count,
                         int flavour)
{
    for (i64 k = 0; k < count; k++)
    {
        int rc;
        if (flavour == ORA_UPDATE)
            rc = ora_ext_updateindex(e, V[k], I[k], J[k]);
        else if (flavour == ORA_RAW)
            rc = ora_ext_rawupdateindex(e, V[k], I[k], J[k]);
        else
            rc = ora_ext_setindex(e, V[k], I[k], J[k]);
        if (rc)
            return -(k + 1);
    }
    return 0;
}

/* ------------------------------------------------------------------ */
/* Dirichlet helpers on the flushed CSC: sparsematrixcsc.jl:97-148     */
/* ------------------------------------------------------------------ */
void ora_ext_mark_dirichlet(ora_ext *e, double penalty, uint8_t *marker)
{
    ora_ext_flush(e);
    const ora_csc *c = e->csc;
    for (i64 i = 1; i <= c->n; i++)
    {
        marker[i - 1] = 0;
        for (i64 j = c->colptr[i - 1]; j < c->colptr[i]; j++)
            if (c->rowval[j - 1] == i && c->nzval[j - 1] >= penalty)
                marker[i - 1] = 1;
    }
}

void ora_ext_eliminate_dirichlet(ora_ext *e, const uint8_t *marker)
{
    ora_ext_flush(e);
    ora_csc *c = e->csc;
    for (i64 i = 1; i <= c->n; i++)
    {
        if (marker[i - 1])
            for (i64 j = c->colptr[i - 1]; j < c->colptr[i]; j++)
                c->nzval[j - 1] = (c->rowval[j - 1] == i) ? 1.0 : 0.0;
        for (i64 j = c->colptr[i - 1]; j < c->colptr[i]; j++)
            if (c->rowval[j - 1] != i && marker[c->rowval[j - 1] - 1])
                c->nzval[j - 1] = 0.0;
    }
}

/* pointblock(A0, blocksize): src/matrix/extendable.jl:292-318.
 * A = SparseMatrixCSC(A0) (flushes), nblock = n / blocksize, Ab = ExtendableSparseMatrixCSC of
 * nblock x nblock SMatrix{bs,bs} blocks.  The loop visits column i, entries k, row j = rowval[k]:
 *   iblock = (i-1)/bs+1 (from the COLUMN), jblock = (j-1)/bs+1 (from the ROW), ii, jj likewise;
 *   block[ii,jj] = nzval[k]; rawupdateindex!(Ab, +, block, iblock, jblock); block[ii,jj] = 0
 * then flush!(Ab).  Restated with the scalar machinery above: the PATTERN of Ab is what the same
 * rawupdateindex! calls build in a scalar matrix (a block-valued LNK buffer links the same slots in
 * the same order); the VALUES are the block sums in call order, zero(Tb) + block for the call that
 * creates the entry (sparsematrixlnk.jl:242,251), acc + block after that (:247), all bs*bs
 * components each time.  Blocks are column-major (SMatrix layout), in CSC order of Ab.
 * colptr_out[nblock+1]; rowval_out / blocks_out sized for nnz(A) entries / nnz(A)*bs*bs values.
 * Returns nnz(Ab), or -(k+1) when entry k of A falls outside the block matrix (BoundsError). */
i64 ora_ext_pointblock(ora_ext *e, i64 bs, i64 *colptr_out, i64 *rowval_out, double *blocks_out)
{
    ora_ext_flush(e);
    const ora_csc *A = e->csc;
    const i64 n = A->n, nb = n / bs;
    if (bs < 1 || nb < 1)
        return -1;
    ora_ext *P = ora_ext_create(nb, nb);
    i64 k0 = 0;
    for (i64 i = 1; i <= n; i++)
        for (i64 k = A->colptr[i - 1]; k < A->colptr[i]; k++, k0++)
        {
            i64 j = A->rowval[k - 1];
            i64 iblock = (i - 1) / bs + 1, jblock = (j - 1) / bs + 1;
            if (ora_ext_rawupdateindex(P, 0.0, iblock, jblock))
            {
                ora_ext_destroy(P);
                return -(k0 + 1);
            }
        }
    ora_ext_flush(P);
    const i64 nnzb = csc_nnz(P->csc);
    memcpy(colptr_out, P->csc->colptr, sizeof(i64) * (size_t)(nb + 1));
    memcpy(rowval_out, P->csc->rowval, sizeof(i64) * (size_t)nnzb);
    unsigned char *created = (unsigned char *)calloc((size_t)(nnzb ? nnzb : 1), 1);
    double *block = (double *)calloc((size_t)(bs * bs), sizeof(double));
    for (i64 i = 1; i <= n; i++)
        for (i64 k = A->colptr[i - 1]; k < A->colptr[i]; k++)
        {
            i64 j = A->rowval[k - 1];
            i64 iblock = (i - 1) / bs + 1, jblock = (j - 1) / bs + 1;
            i64 ii = (i - 1) % bs + 1, jj = (j - 1) % bs + 1;
            block[(ii - 1) + (jj - 1) * bs] = A->nzval[k - 1];
            i64 pos = csc_findindex(P->csc, iblock, jblock); /* 1-based slot of Ab[iblock,jblock] */
            double *acc = blocks_out + (size_t)(pos - 1) * (size_t)(bs * bs);
            for (i64 c = 0; c < bs * bs; c++)
                acc[c] = (created[pos - 1] ? acc[c] : 0.0) + block[c];
            created[pos - 1] = 1;
            block[(ii - 1) + (jj - 1) * bs] = 0.0;
        }
    free(created);
    free(block);
    ora_ext_destroy(P);
    return nnzb;
}

/* ------------------------------------------------------------------ */
/* Multi-partition path: GenericMTExtendableSparseMatrixCSC with        */
/* SparseMatrixDILNKC buffers (src/ExtendableSparse.jl:35-39).          */
/* ------------------------------------------------------------------ */
typedef struct
{
    i64 m, n, nnz, nentries, len;
    i64 jlo, jhi;  /* 1-based range of columns that have a list (the Dict's keys lie inside it) */
    i64 *colstart; /* Dict{Ti,Ti} of the reference, restated as a dense map (0 = absent) */
    i64 *colptr;
    i64 *rowval;
    double *nzval;
} ora_dilnkc;

/* ctor: sparsematrixdilnkc.jl:61-63 (initial capacity 10) */
static ora_dilnkc *dilnkc_create(i64 m, i64 n)
{
    /* own cache lines: partitions are filled by concurrent threads (ora_mt_insert_partitioned) */
    ora_dilnkc *l = (ora_dilnkc *)aligned_alloc(128, (sizeof(ora_dilnkc) + 127) / 128 * 128);
    memset(l, 0, sizeof(ora_dilnkc));
    l->m = m;
    l->n = n;
    l->len = 10;
    l->colstart = (i64 *)calloc((size_t)(n ? n : 1), sizeof(i64));
    l->colptr = (i64 *)calloc(10, sizeof(i64));
    l->rowval = (i64 *)calloc(10, sizeof(i64));
    l->nzval = (double *)calloc(10, sizeof(double));
    return l;
}

static void dilnkc_destroy(ora_dilnkc *l)
{
    if (!l)
        return;
    free(l->colstart);
    free(l->colptr);
    free(l->rowval);
    free(l->nzval);
    free(l);
}

/* findindex: sparsematrixdilnkc.jl:111-129 */
static i64 dilnkc_findindex(const ora_dilnkc *l, i64 i, i64 j, i64 *k0out)
{
    i64 k = l->colstart[j - 1];
    if (k == 0)
    {
        *k0out = 0;
        return 0;
    }
    i64 k0 = k;
    while (k > 0)
    {
        if (l->rowval[k - 1] == i)
        {
            *k0out = 0;
            return k;
        }
        k0 = k;
        k = l->colptr[k - 1];
    }
    *k0out = k0;
    return 0;
}

/* addentry!: sparsematrixdilnkc.jl:150-177 */
static i64 dilnkc_addentry(ora_dilnkc *l, i64 i, i64 j, i64 k0)
{
    l->nentries += 1;
    if (l->len < l->nentries)
    {
        i64 newsize = (i64)ceil(5.0 * (double)l->nentries / 4.0);
        l->nzval = (double *)xrealloc(l->nzval, sizeof(double) * (size_t)newsize);
        l->rowval = (i64 *)xrealloc(l->rowval, sizeof(i64) * (size_t)newsize);
        l->colptr = (i64 *)xrealloc(l->colptr, sizeof(i64) * (size_t)newsize);
        l->len = newsize;
    }
    if (k0 == 0)
    {
        l->colstart[j - 1] = l->nentries;
        if (l->jhi == 0 || j < l->jlo)
            l->jlo = j;
        if (j > l->jhi)
            l->jhi = j;
    }
    l->rowval[l->nentries - 1] = i;
    l->colptr[l->nentries - 1] = 0;
    if (k0 > 0)
        l->colptr[k0 - 1] = l->nentries;
    l->nnz += 1;
    return l->nentries;
}

/* updateindex!/rawupdateindex!: sparsematrixdilnkc.jl:208-237 */
static void dilnkc_update(ora_dilnkc *l, double v, i64 i, i64 j, int raw)
{
    i64 k0;
    i64 k = dilnkc_findindex(l, i, j, &k0);
    if (k > 0)
    {
        l->nzval[k - 1] = l->nzval[k - 1] + v;
        return;
    }
    if (raw || v != 0.0)
    {
        k = dilnkc_addentry(l, i, j, k0);
        l->nzval[k - 1] = 0.0 + v;
    }
}

typedef struct
{
    ora_csc *csc;
    i64 np;
    ora_dilnkc **x;
} ora_mt;

/* ctor: genericmtextendablesparsematrixcsc.jl:16-22 */
ora_mt *ora_mt_create(i64 m, i64 n, i64 np)
{
    ora_mt *e = (ora_mt *)calloc(1, sizeof(ora_mt));
    e->csc = csc_alloc(m, n, 0);
    e->np = np;
    e->x = (ora_dilnkc **)calloc((size_t)np, sizeof(ora_dilnkc *));
    for (i64 p = 0; p < np; p++)
        e->x[p] = dilnkc_create(m, n);
    return e;
}

void ora_mt_destroy(ora_mt *e)
{
    if (!e)
        return;
    csc_free(e->csc);
    for (i64 p = 0; p < e->np; p++)
        dilnkc_destroy(e->x[p]);
    free(e->x);
    free(e);
}

/* rawupdateindex!/updateindex!(ext,+,v,i,j,tid): genericmt...:87-114, setindex!: :63-68; tid is 1-based */
int ora_mt_update(ora_mt *e, double v, i64 i, i64 j, i64 tid, int flavour)
{
    i64 k = csc_findindex(e->csc, i, j);
    if (k < 0 || tid < 1 || tid > e->np)
        return ORA_EBOUNDS;
    if (k > 0)
    { /* setindex! of a stored entry overwrites it */
        e->csc->nzval[k - 1] = flavour == ORA_ASSIGN ? v : e->csc->nzval[k - 1] + v;
        return ORA_OK;
    }
    if (flavour == ORA_ASSIGN)
        return ORA_EILLEGAL; /* setindex! of a new entry is an error, :63-68 */
    dilnkc_update(e->x[tid - 1], v, i, j, flavour == ORA_RAW);
    return ORA_OK;
}

i64 ora_mt_insert_batch(ora_mt *e, const i64 *I, const i64 *J, const double *V, i64 count,
                        i64 tid, int flavour)
{
    for (i64 k = 0; k < count; k++)
        if (ora_mt_update(e, V[k], I[k], J[k], tid, flavour))
            return -(k + 1);
    return 0;
}

/* Partitioned parallel insertion, the loop of test/femtools.jl:75-110 (testassemble_parallel!):
 * `for color in pcolors(grid)` runs the colours one after the other; inside a colour the partitions
 * are independent tasks (`@tasks for part in pcolor_partitions(grid, color)`), each inserting its own
 * cells with its own tid = part into xmatrices[part] (genericmt...:87-114).  Here partition p
 * (tid p+1) is the slice [part_begin[p], part_begin[p+1]) of a pre-generated stream, colours are
 * the parities of p (neighbouring slabs never run together), and `nthreads` POSIX threads pull the
 * partitions of the running colour from a shared counter.  A partition is inserted by exactly one
 * thread in stream order, so the result equals the serial tid-wise insertion bit for bit. */
typedef struct
{
    ora_mt *e;
    const i64 *I, *J, *part_begin;
    const double *V;
    i64 colour, ncolours;
    int flavour;
    i64 next; /* next partition index of this colour (atomic) */
    i64 err;
} mt_colour_job;

static void *mt_colour_worker(void *arg)
{
    mt_colour_job *job = (mt_colour_job *)arg;
    for (;;)
    {
        i64 k = __atomic_fetch_add(&job->next, 1, __ATOMIC_RELAXED);
        i64 p = job->colour + k * job->ncolours;
        if (p >= job->e->np)
            break;
        for (i64 r = job->part_begin[p]; r < job->part_begin[p + 1]; r++)
            if (ora_mt_update(job->e, job->V[r], job->I[r], job->J[r], p + 1, job->flavour))
            {
                i64 zero = 0;
                __atomic_compare_exchange_n(&job->err, &zero, -(r + 1), 0, __ATOMIC_RELAXED, __ATOMIC_RELAXED);
                return NULL;
            }
    }
    return NULL;
}

i64 ora_mt_insert_partitioned(ora_mt *e, const i64 *I, const i64 *J, const double *V, const i64 *part_begin,
                              i64 nthreads, int flavour)
{
    if (nthreads < 1)
        nthreads = 1;
    pthread_t *th = (pthread_t *)calloc((size_t)nthreads, sizeof(pthread_t));
    mt_colour_job job = {e, I, J, part_begin, V, 0, 2, flavour, 0, 0};
    for (i64 colour = 0; colour < 2 && job.err == 0; colour++)
    {
        job.colour = colour;
        job.next = 0;
        i64 started = 0;
        for (i64 t = 0; t < nthreads; t++, started++)
            if (pthread_create(&th[t], NULL, mt_colour_worker, &job))
                break;
        if (started == 0)
            mt_colour_worker(&job);
        for (i64 t = 0; t < started; t++)
            pthread_join(th[t], NULL);
    }
    free(th);
    return job.err;
}

typedef struct
{
    i64 row;
    i64 seq;
    double v;
} coo_ent;

static int coo_less(const void *a, const void *b)
{
    const coo_ent *x = (const coo_ent *)a, *y = (const coo_ent *)b;
    if (x->row != y->row)
        return (x->row > y->row) - (x->row < y->row);
    return (x->seq > y->seq) - (x->seq < y->seq);
}

/* flush!: genericmt...:45-51 -> Base.sum(Vector{DILNKC},csc) sparsematrixdilnkc.jl:397-435.
 * COO = [csc entries in column order] ++ [partition 1 lists] ++ [partition 2 lists] ...
 * then stdlib sparse!(I,J,V,m,n,+): sorted rows per column, duplicates combined
 * in input order (first occurrence copied, the rest added), zeros kept.
 * Every (i,j) occurs at most once per partition, so the Dict iteration order of
 * :417 cannot influence the result. */
void ora_mt_flush(ora_mt *e)
{
    i64 lnew = 0;
    for (i64 p = 0; p < e->np; p++)
        lnew += e->x[p]->nnz;
    i64 m = e->csc->m, n = e->csc->n;
    if (lnew > 0)
    {
        i64 total = lnew + csc_nnz(e->csc);
        i64 *cnt = (i64 *)calloc((size_t)(n + 2), sizeof(i64));
        /* counting sort by column keeps input order inside a column */
        for (i64 j = 1; j <= n; j++)
            cnt[j] += e->csc->colptr[j] - e->csc->colptr[j - 1];
        for (i64 p = 0; p < e->np; p++)
            for (i64 j = e->x[p]->jlo; j <= e->x[p]->jhi && j >= 1; j++)
                for (i64 k = e->x[p]->colstart[j - 1]; k > 0; k = e->x[p]->colptr[k - 1])
                    cnt[j] += 1;
        i64 *start = (i64 *)calloc((size_t)(n + 2), sizeof(i64));
        for (i64 j = 1; j <= n; j++)
            start[j + 1] = start[j] + cnt[j];
        coo_ent *buf = (coo_ent *)xrealloc(NULL, sizeof(coo_ent) * (size_t)total);
        i64 *fill = (i64 *)calloc((size_t)(n + 2), sizeof(i64));
        i64 seq = 0;
        for (i64 j = 1; j <= n; j++)
            for (i64 k = e->csc->colptr[j - 1]; k < e->csc->colptr[j]; k++)
            {
                coo_ent *t = &buf[start[j] + fill[j]++];
                t->row = e->csc->rowval[k - 1];
                t->v = e->csc->nzval[k - 1];
                t->seq = seq++;
            }
        for (i64 p = 0; p < e->np; p++)
            for (i64 j = e->x[p]->jlo; j <= e->x[p]->jhi && j >= 1; j++)
                for (i64 k = e->x[p]->colstart[j - 1]; k > 0; k = e->x[p]->colptr[k - 1])
                {
                    coo_ent *t = &buf[start[j] + fill[j]++];
                    t->row = e->x[p]->rowval[k - 1];
                    t->v = e->x[p]->nzval[k - 1];
                    t->seq = seq++;
                }
        ora_csc *r = csc_alloc(m, n, total);
        i64 inz = 1;
        for (i64 j = 1; j <= n; j++)
        {
            r->colptr[j - 1] = inz;
            coo_ent *c = buf + start[j];
            i64 len = cnt[j];
            if (len <= 64)
            { /* stable insertion sort by row: input order (seq) survives among equal rows */
                for (i64 a = 1; a < len; a++)
                {
                    coo_ent x = c[a];
                    i64 b = a;
                    while (b > 0 && c[b - 1].row > x.row)
                    {
                        c[b] = c[b - 1];
                        b--;
                    }
                    c[b] = x;
                }
            }
            else
                qsort(c, (size_t)len, sizeof(coo_ent), coo_less);
            for (i64 t = 0; t < len; t++)
            {
                if (t > 0 && c[t].row == c[t - 1].row)
                    r->nzval[inz - 2] = r->nzval[inz - 2] + c[t].v;
                else
                {
                    r->rowval[inz - 1] = c[t].row;
                    r->nzval[inz - 1] = c[t].v;
                    inz++;
                }
            }
        }
        r->colptr[n] = inz;
        free(cnt);
        free(start);
        free(fill);
        free(buf);
        csc_free(e->csc);
        e->csc = r;
    }
    for (i64 p = 0; p < e->np; p++)
    { /* fresh buffers: genericmt...:47-49 */
        dilnkc_destroy(e->x[p]);
        e->x[p] = dilnkc_create(m, n);
    }
}

i64 ora_mt_nnz(ora_mt *e)
{
    ora_mt_flush(e);
    return csc_nnz(e->csc);
}

i64 ora_mt_nnznew(const ora_mt *e)
{ /* nnznew: genericmt...:84 */
    i64 s = 0;
    for (i64 p = 0; p < e->np; p++)
        s += e->x[p]->nnz;
    return s;
}

void ora_mt_get_csc(const ora_mt *e, i64 *colptr, i64 *rowval, double *nzval)
{
    i64 n = e->csc->n, nnz = csc_nnz(e->csc);
    memcpy(colptr, e->csc->colptr, sizeof(i64) * (size_t)(n + 1));
    if (rowval)
        memcpy(rowval, e->csc->rowval, sizeof(i64) * (size_t)nnz);
    if (nzval)
        memcpy(nzval, e->csc->nzval, sizeof(double) * (size_t)nnz);
}

void ora_mt_zero_values(ora_mt *e)
{
    i64 nnz = csc_nnz(e->csc);
    for (i64 k = 0; k < nnz; k++)
        e->csc->nzval[k] = 0.0;
}
