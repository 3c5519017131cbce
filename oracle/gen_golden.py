"""Generate tests/golden/*.pt by running the UNMODIFIED reference (rusty1s/pytorch_sparse @ 91feaa5), from a
read-only checkout ($TSB200_REFERENCE, else `reference` beside this repository; see oracle/build_ref.py):

  * its 12 CPU operator libraries compiled from its csrc/ (oracle/build_ref.build_full, into a build cache
    in the system's temporary directory, nothing copied into the repo),
  * its Python package imported from a scratch copy of its torch_sparse/ (the package loads its .so files
    from its own directory, torch_sparse/__init__.py:8-21),
  * `torch_scatter` provided by oracle/torch_scatter_standin (third-party, absent, unpinned; only the
    coalesce VALUE reductions and nothing else on the fixtures below go through it),
  * SpSpMM arithmetic by torch.sparse.mm of the installed PyTorch (third-party; torch 2.11.0+cu128).

    python oracle/gen_golden.py            # rewrites tests/golden/

The fixtures hold inputs AND the reference's outputs (no file over 1 MB: the larger ones keep a seeded sample of
rows), so the tests check both the oracle and the CUDA path against the reference itself without it.
"""
from __future__ import annotations

import atexit
import shutil
import sys
import tempfile
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
GOLD = ROOT / "tests" / "golden"


def import_reference():
    from oracle import build_ref
    if not build_ref.sources_available():
        raise SystemExit(f"no readable checkout of the reference in {build_ref.REF} (set TSB200_REFERENCE)")
    ref = build_ref.REF
    full = Path(tempfile.gettempdir()) / "tsb200_ref_full"   # reused: libraries newer than their sources are kept
    build_ref.build_full(full)
    scratch = Path(tempfile.mkdtemp(prefix="tsb200_refpkg_"))
    atexit.register(shutil.rmtree, scratch, ignore_errors=True)
    shutil.copytree(ref / "torch_sparse", scratch / "torch_sparse")
    for so in full.glob("*.so"):
        shutil.copy(so, scratch / "torch_sparse" / so.name)
    sys.path.insert(0, str(scratch))
    sys.path.insert(0, str(ROOT / "oracle" / "torch_scatter_standin"))
    import torch_sparse  # the reference package, unmodified
    assert torch_sparse.__version__ == "0.6.18"
    return torch_sparse


def random_structure(M, N, avg_deg, seed, empty_rows=(), long_rows=()):
    g = torch.Generator().manual_seed(seed)
    deg = torch.poisson(torch.full((M,), float(avg_deg)), generator=g).long().clamp_(max=N)
    for r in empty_rows:
        deg[r] = 0
    for r, d in long_rows:
        deg[r] = min(d, N)
    rows, cols = [], []
    for m in range(M):
        d = int(deg[m])
        if d:
            rows.append(torch.full((d,), m, dtype=torch.long))
            cols.append(torch.randperm(N, generator=g)[:d].sort().values)
    return torch.cat(rows), torch.cat(cols)


def main():
    ts = import_reference()
    from torch_sparse import SparseTensor
    from torch_sparse.matmul import matmul
    GOLD.mkdir(parents=True, exist_ok=True)
    meta = {"reference": "rusty1s/pytorch_sparse 0.6.18 @ 91feaa5e", "torch": torch.__version__}

    # ---- (a) the reference's own SpMM test recipe (test/test_matmul.py:12-51), fwd + both grads ----
    cases = {}
    for dtype in (torch.float32, torch.float64, torch.float16, torch.bfloat16):
        for reduce in ("sum", "mean", "min", "max"):
            torch.manual_seed(12345)
            src = torch.randn((10, 8), dtype=dtype)
            src[2:4, :] = 0
            src[:, 2:4] = 0
            src = SparseTensor.from_dense(src).requires_grad_()
            row, col, value = src.coo()
            other = torch.randn((2, 8, 2), dtype=dtype, requires_grad=True)
            grad_out = torch.randn((2, 10, 2), dtype=dtype)
            out = matmul(src, other, reduce)
            out.backward(grad_out)
            c = dict(row=row.clone(), col=col.clone(), value=value.detach().clone(), other=other.detach().clone(),
                     grad_out=grad_out, out=out.detach().clone(), grad_value=value.grad.clone(),
                     grad_other=other.grad.clone())
            if reduce in ("min", "max"):
                rowptr, col2, val2 = src.csr()
                fn = torch.ops.torch_sparse.spmm_min if reduce == "min" else torch.ops.torch_sparse.spmm_max
                c["arg_out"] = fn(rowptr, col2, val2.detach(), other.detach())[1]
            cases[f"{str(dtype).split('.')[-1]}_{reduce}"] = c
    torch.save({"meta": meta, "cases": cases}, GOLD / "spmm_reference_recipe.pt")

    # ---- (b) medium random SpMM incl. empty rows and rows longer than the kernel's segment length ----
    cases = {}
    M, N = 96, 300
    row, col = random_structure(M, N, 9, seed=7, empty_rows=(0, 17, 95), long_rows=[(5, 290), (6, 256), (7, 257)])
    rowptr = torch.ops.torch_sparse.ind2ptr(row, M)
    g = torch.Generator().manual_seed(8)
    for dtype, K in ((torch.float32, 32), (torch.float32, 128), (torch.bfloat16, 128), (torch.float16, 64),
                     (torch.float64, 6), (torch.int64, 5)):
        if dtype.is_floating_point:
            value = torch.randn(col.numel(), generator=g).to(dtype)
            mat = torch.randn(N, K, generator=g).to(dtype)
        else:
            value = torch.randint(-4, 5, (col.numel(),), generator=g)
            mat = torch.randint(-4, 5, (N, K), generator=g)
        c = dict(rowptr=rowptr, row=row, col=col, value=value, mat=mat)
        for has_value in (True, False):
            v = value if has_value else None
            tag = "v" if has_value else "nv"
            c[f"sum_{tag}"] = torch.ops.torch_sparse.spmm_sum(None, rowptr, col, v, None, None, mat)
            c[f"mean_{tag}"] = torch.ops.torch_sparse.spmm_mean(None, rowptr, col, v, None, None, None, mat)
            c[f"min_{tag}"], c[f"argmin_{tag}"] = torch.ops.torch_sparse.spmm_min(rowptr, col, v, mat)
            c[f"max_{tag}"], c[f"argmax_{tag}"] = torch.ops.torch_sparse.spmm_max(rowptr, col, v, mat)
        cases[f"{str(dtype).split('.')[-1]}_K{K}"] = c
    # stored: the special rows (empty, longer than a segment) and a seeded sample of the others
    keep = keep_rows(M, (0, 5, 6, 7, 17, 95), 16, seed=9)
    cases = {k: sample_spmm_rows(c, keep) for k, c in cases.items()}
    torch.save({"meta": dict(meta, rows=f"{keep.numel()} of {M} rows"), "cases": cases}, GOLD / "spmm_medium.pt")

    # ---- (c) storage views: sort-on-construct, rowptr, csr2csc, colptr (storage.py:149-162, 369-429) ----
    g = torch.Generator().manual_seed(21)
    M, N, E = 50, 40, 400
    row = torch.randint(M, (E,), generator=g)
    col = torch.randint(N, (E,), generator=g)
    key = torch.unique(row * N + col)
    key = key[torch.randperm(key.numel(), generator=g)]       # unique keys, shuffled => sort is well defined
    row, col = key // N, key % N
    value = torch.randn(row.numel(), generator=g)
    st = ts.SparseStorage(row=row, col=col, value=value, sparse_sizes=(M, N))
    st.fill_cache_()
    torch.save({"meta": meta, "in": dict(row=row, col=col, value=value, M=M, N=N),
                "out": dict(row=st.row(), col=st.col(), value=st.value(), rowptr=st.rowptr(), rowcount=st.rowcount(),
                            colptr=st.colptr(), colcount=st.colcount(), csr2csc=st.csr2csc(), csc2csr=st.csc2csr())},
               GOLD / "storage_views.pt")

    # ---- (d) coalesce (coalesce.py:5-25). Indices come from the reference's own code; duplicate VALUE
    #      reductions come from the torch_scatter stand-in (parity unpinned at the last ulp for float add) ----
    g = torch.Generator().manual_seed(31)
    M, N, E0 = 60, 50, 500
    row = torch.randint(M, (E0,), generator=g)
    col = torch.randint(N, (E0,), generator=g)
    reps = torch.randint(1, 4, (E0,), generator=g)
    row, col = row.repeat_interleave(reps), col.repeat_interleave(reps)
    perm = torch.randperm(row.numel(), generator=g)
    row, col = row[perm], col[perm]
    index = torch.stack([row, col])
    vi = torch.randint(-9, 10, (row.numel(), 2), generator=g)       # integer values: order independent
    vf = torch.randn(row.numel(), generator=g, dtype=torch.float64)
    outs = {}
    for op in ("add", "mean", "min", "max"):
        if op != "mean":
            oi, ov = ts.coalesce(index, vi, M, N, op=op)
            outs[f"int_{op}"] = dict(index=oi, value=ov)
        oi, ov = ts.coalesce(index, vf, M, N, op=op)
        outs[f"f64_{op}"] = dict(index=oi, value=ov)
    oi, _ = ts.coalesce(index, None, M, N)
    outs["none"] = dict(index=oi)
    torch.save({"meta": meta, "in": dict(index=index, vi=vi, vf=vf, M=M, N=N), "out": outs}, GOLD / "coalesce.pt")

    # ---- (e) transpose (transpose.py:39-62) ----
    ti, tv = ts.transpose(index, vf, M, N)
    torch.save({"meta": meta, "in": dict(index=index, value=vf, M=M, N=N), "out": dict(index=ti, value=tv)},
               GOLD / "transpose.pt")

    # ---- (f) SpSpMM through the reference's functional API (spspmm.py:6-33 -> torch.sparse.mm) ----
    cases = {}
    for name, (M, Kd, N, da, db, dtype) in {"small_f32": (40, 30, 35, 4, 5, torch.float32),
                                            "wide_f64": (25, 60, 3000, 6, 40, torch.float64)}.items():
        ra, ca = random_structure(M, Kd, da, seed=41, empty_rows=(0,))
        rb, cb = random_structure(Kd, N, db, seed=42, empty_rows=(1,))
        g = torch.Generator().manual_seed(43)
        va = torch.randn(ra.numel(), generator=g).to(dtype)
        vb = torch.randn(rb.numel(), generator=g).to(dtype)
        ic, vc = ts.spspmm(torch.stack([ra, ca]), va, torch.stack([rb, cb]), vb, M, Kd, N)
        cases[name] = dict(indexA=torch.stack([ra, ca]), valueA=va, indexB=torch.stack([rb, cb]), valueB=vb,
                           M=M, K=Kd, N=N, indexC=ic, valueC=vc)
    # cancellation -> explicit zero kept
    iA = torch.tensor([[0, 0], [0, 1]]); vA = torch.tensor([1.0, -1.0])
    iB = torch.tensor([[0, 1], [0, 0]]); vB = torch.tensor([2.0, 2.0])
    ic, vc = ts.spspmm(iA, vA, iB, vB, 1, 2, 1)
    cases["cancel"] = dict(indexA=iA, valueA=vA, indexB=iB, valueB=vB, M=1, K=2, N=1, indexC=ic, valueC=vc)
    torch.save({"meta": meta, "cases": cases}, GOLD / "spspmm.pt")

    # ---- (g) ind2ptr / ptr2ind (convert.cpp) ----
    g = torch.Generator().manual_seed(51)
    ind = torch.randint(1000, (5000,), generator=g).sort().values
    ptr = torch.ops.torch_sparse.ind2ptr(ind, 1200)
    back = torch.ops.torch_sparse.ptr2ind(ptr, ind.numel())
    torch.save({"meta": meta, "ind": ind, "M": 1200, "ptr": ptr, "ind_back": back}, GOLD / "convert.pt")

    # ---- (h) SURVEY §8(f) "next" rows: reductions (reduce.py), sparse add (add.py / spadd.py), narrow (narrow.py) ----
    import torch_sparse as tsr
    g = torch.Generator().manual_seed(61)
    M, N = 40, 30
    ra, ca = random_structure(M, N, 5, seed=62, empty_rows=(0, 7))
    rb, cb = random_structure(M, N, 4, seed=63, empty_rows=(3,))
    va = torch.randn(ra.numel(), generator=g, dtype=torch.float64)
    vb = torch.randn(rb.numel(), generator=g, dtype=torch.float64)
    va2 = torch.randn(ra.numel(), 3, generator=g, dtype=torch.float64)
    A = SparseTensor(row=ra, col=ca, value=va, sparse_sizes=(M, N))
    A2 = SparseTensor(row=ra, col=ca, value=va2, sparse_sizes=(M, N))
    A0 = SparseTensor(row=ra, col=ca, sparse_sizes=(M, N))
    Bm = SparseTensor(row=rb, col=cb, value=vb, sparse_sizes=(M, N))
    red = {}
    for name, T in (("v", A), ("v2", A2), ("nv", A0)):
        for op in ("sum", "mean", "min", "max"):
            for dim in (None, 0, 1, -1):
                if name == "nv" and dim == -1:
                    dim_eff = 1
                else:
                    dim_eff = dim
                try:
                    red[f"{name}_{op}_{dim}"] = getattr(tsr, op)(T, dim_eff)
                except Exception as e:  # shape/dtype corner the reference itself rejects
                    red[f"{name}_{op}_{dim}"] = None
    C = A.add(Bm) if hasattr(A, "add") else tsr.add(A, Bm)
    si, sv = tsr.spadd(torch.stack([ra, ca]), va, torch.stack([rb, cb]), vb, M, N)
    dr = torch.randn(M, 1, generator=g, dtype=torch.float64)
    dc = torch.randn(1, N, generator=g, dtype=torch.float64)
    mr, mc = tsr.mul(A, dr), tsr.mul(A, dc)
    n0 = tsr.narrow(A, 0, 5, 20)
    n1 = tsr.narrow(A, 1, 4, 15)
    torch.save({"meta": meta,
                "in": dict(ra=ra, ca=ca, va=va, va2=va2, rb=rb, cb=cb, vb=vb, M=M, N=N),
                "reduce": red,
                "add": dict(row=C.storage.row(), col=C.storage.col(), value=C.storage.value()),
                "spadd": dict(index=si, value=sv),
                "mul": dict(dr=dr, dc=dc, row_scaled=mr.storage.value(), col_scaled=mc.storage.value()),
                "narrow0": dict(rowptr=n0.storage.rowptr(), col=n0.storage.col(), value=n0.storage.value(), sizes=n0.sparse_sizes()),
                "narrow1": dict(row=n1.storage.row(), col=n1.storage.col(), value=n1.storage.value(), sizes=n1.sparse_sizes())},
               GOLD / "next_rows.pt")

    gen_next_rows2(ts, meta)
    gen_spspmm2(ts, meta)
    gen_grads(ts, meta)
    gen_reference_ops(meta)

    sizes = {p.name: p.stat().st_size for p in sorted(GOLD.glob("*.pt"))}
    print("wrote", sizes, "total", sum(sizes.values()))


def gen_next_rows2(ts, meta):
    """SURVEY §8(f) ranks 2 and 4: to_symmetric (tensor.py:404-438), index_select / index_select_nnz
    (index_select.py:9-99) run through the unmodified reference."""
    from torch_sparse import SparseTensor
    g = torch.Generator().manual_seed(71)
    out = {"meta": meta, "cases": {}}
    for name, (M, N, deg) in {"rect": (37, 29, 4), "square": (33, 33, 5)}.items():
        r, c = random_structure(M, N, deg, seed=72 + M, empty_rows=(0, 5))
        v = torch.randn(r.numel(), generator=g, dtype=torch.float64)
        v2 = torch.randn(r.numel(), 2, generator=g, dtype=torch.float64)
        A = SparseTensor(row=r, col=c, value=v, sparse_sizes=(M, N))
        A2 = SparseTensor(row=r, col=c, value=v2, sparse_sizes=(M, N))
        A0 = SparseTensor(row=r, col=c, sparse_sizes=(M, N))
        idx0 = torch.randint(M, (25,), generator=g)          # unsorted, with repeats
        idx1 = torch.randint(N, (19,), generator=g)
        idxe = torch.randperm(r.numel(), generator=g)[: r.numel() // 2].sort().values
        case = {"in": dict(row=r, col=c, v=v, v2=v2, M=M, N=N, idx0=idx0, idx1=idx1, idxe=idxe)}
        for tag, T in (("v", A), ("v2", A2), ("nv", A0)):
            s0 = T.index_select(0, idx0)
            s1 = T.index_select(1, idx1)
            case[f"sel0_{tag}"] = dict(rowptr=s0.storage.rowptr(), row=s0.storage.row(), col=s0.storage.col(),
                                       value=s0.storage.value(), sizes=s0.sparse_sizes())
            case[f"sel1_{tag}"] = dict(row=s1.storage.row(), col=s1.storage.col(), value=s1.storage.value(),
                                       colptr=s1.storage.colptr(), sizes=s1.sparse_sizes())
            for lay in ("coo", "csc"):
                sn = T.index_select_nnz(idxe, lay)
                case[f"selnnz_{lay}_{tag}"] = dict(row=sn.storage.row(), col=sn.storage.col(), value=sn.storage.value())
            for red in ("sum", "mean", "min", "max"):
                if tag == "nv" and red != "sum":
                    continue
                sy = T.to_symmetric(red)
                case[f"sym_{red}_{tag}"] = dict(row=sy.storage.row(), col=sy.storage.col(), value=sy.storage.value(),
                                                sizes=sy.sparse_sizes())
        out["cases"][name] = case
    torch.save(out, GOLD / "next_rows2.pt")


def gen_spspmm2(ts, meta):
    """SpSpMM shapes on the limits of the CUDA kernel's row classes (flat rows hold <= 2048 products and <= 128 A
    entries; one bitmap window is 2^18 columns), through the reference's functional API (spspmm.py:6-33)."""
    cases = {}
    shapes = {"p2048_f32": (24, 64, 9000, 45, 45, torch.float32),      # products per row straddle 2048
              "na128_f64": (20, 500, 3000, 140, 6, torch.float64),     # A entries per row straddle 128
              "window_edge_f32": (30, 300, 262_145, 10, 40, torch.float32),  # one column past a 2^18 window
              "dups_f64": (48, 64, 96, 28, 28, torch.float64)}         # >= 3 products per output column
    for name, (M, Kd, N, da, db, dtype) in shapes.items():
        ra, ca = random_structure(M, Kd, da, seed=81, empty_rows=(0,))
        rb, cb = random_structure(Kd, N, db, seed=82, empty_rows=(1,))
        g = torch.Generator().manual_seed(83)
        va = torch.randn(ra.numel(), generator=g).to(dtype)
        vb = torch.randn(rb.numel(), generator=g).to(dtype)
        ic, vc = ts.spspmm(torch.stack([ra, ca]), va, torch.stack([rb, cb]), vb, M, Kd, N)
        c = dict(indexA=torch.stack([ra, ca]), valueA=va, indexB=torch.stack([rb, cb]), valueB=vb,
                 M=M, K=Kd, N=N, indexC=ic, valueC=vc)
        cases[name] = sample_spspmm_rows(c, spspmm_keep_rows(c))
    torch.save({"meta": dict(meta, rows="a quarter of the rows of A (and C)"), "cases": cases}, GOLD / "spspmm2.pt")


# ---- row samples: every fixture file stays under 1 MB ---------------------------------------------------------
def keep_rows(M, must, n, seed):
    """`must` plus a seeded sample of the other rows, n rows in all, ascending."""
    must = torch.tensor(sorted(set(must)), dtype=torch.long)
    rest = torch.ones(M, dtype=torch.bool)
    rest[must] = False
    rest = rest.nonzero().flatten()
    g = torch.Generator().manual_seed(seed)
    extra = rest[torch.randperm(rest.numel(), generator=g)[:max(n - must.numel(), 0)]]
    return torch.cat([must, extra]).sort().values


def _csr_rows(rowptr, rows):
    """Entry positions of `rows` (in order) and the rowptr of the CSR made of those rows."""
    deg = rowptr[rows + 1] - rowptr[rows]
    new_ptr = torch.zeros(rows.numel() + 1, dtype=torch.long)
    new_ptr[1:] = torch.cumsum(deg, 0)
    pos = torch.cat([torch.arange(int(rowptr[r]), int(rowptr[r + 1])) for r in rows.tolist()] +
                    [torch.empty(0, dtype=torch.long)])
    return pos, new_ptr


def sample_spmm_rows(c, rows):
    """An spmm_medium case restricted to `rows` of the sparse matrix. Every output row depends on its own entries and
    `mat` only, so the reference's outputs of those rows are exactly the outputs for the smaller matrix; arg_out
    positions are renumbered to the smaller entry list (the empty-row sentinel E becomes the new E)."""
    pos, rowptr = _csr_rows(c["rowptr"], rows)
    E, E2 = c["col"].numel(), pos.numel()
    shift = (rowptr[:-1] - c["rowptr"][rows]).view(-1, *([1] * (c["mat"].dim() - 1)))
    out = dict(rowptr=rowptr, row=torch.repeat_interleave(torch.arange(rows.numel()), rowptr.diff()),
               col=c["col"][pos], value=c["value"][pos], mat=c["mat"])
    for k, t in c.items():
        if k in out:
            continue
        t = t[rows]
        if k.startswith("arg"):
            t = torch.where(t == E, torch.full_like(t, E2), t + shift)
        out[k] = t
    return out


def spspmm_keep_rows(c):
    """Row 0 (empty), the rows with the fewest / most A entries and products, and a seeded sample: M / 4 rows."""
    (ra, ca), (rb, _) = c["indexA"], c["indexB"]
    M = c["M"]
    deg_a = torch.bincount(ra, minlength=M)
    prods = torch.zeros(M, dtype=torch.long).index_add_(0, ra, torch.bincount(rb, minlength=c["K"])[ca])
    big = torch.iinfo(torch.long).max
    must = [0]
    for m in (deg_a, prods):
        must += [int(m.argmax()), int(torch.where(m > 0, m, big).argmin())]
    return keep_rows(M, must, M // 4, seed=84)


def sample_spspmm_rows(c, rows):
    """A SpSpMM case restricted to `rows` of A, renumbered 0..len(rows)-1: row i of C = row i of A times B, so the
    reference's C restricted to the same rows is the product of the smaller A with B."""
    new = torch.full((c["M"],), -1, dtype=torch.long)
    new[rows] = torch.arange(rows.numel())
    ka, kc = new[c["indexA"][0]] >= 0, new[c["indexC"][0]] >= 0
    ia, ic = c["indexA"][:, ka].clone(), c["indexC"][:, kc].clone()
    ia[0], ic[0] = new[ia[0]], new[ic[0]]
    return dict(c, indexA=ia, valueA=c["valueA"][ka], M=rows.numel(), indexC=ic, valueC=c["valueC"][kc])


def gen_grads(ts, meta):
    """Gradients w.r.t. the stored values through every value-carrying op that rides on coalesce / segment reduce,
    taken from the unmodified reference's autograd (torch_scatter stand-in = plain differentiable torch ops):
    coalesce (coalesce.py:5-25 -> storage.py:436-466), transpose (transpose.py:39-62), spadd (spadd.py:5-18),
    add (add.py:38-56), to_symmetric (tensor.py:404-438), sum/mean/min/max over dim 0/1 (reduce.py:36-54), and a
    GCN-normalisation flow (deg = A.sum(1); D^-1/2 A D^-1/2 @ x). Random float64 values: no ties inside a run."""
    import torch_sparse as tsr
    from torch_sparse import SparseTensor
    g = torch.Generator().manual_seed(91)
    out = {"meta": meta}

    # duplicated, shuffled COO entries (same recipe as coalesce.pt)
    M, N, E0 = 45, 38, 300
    row = torch.randint(M, (E0,), generator=g)
    col = torch.randint(N, (E0,), generator=g)
    reps = torch.randint(1, 4, (E0,), generator=g)
    row, col = row.repeat_interleave(reps), col.repeat_interleave(reps)
    perm = torch.randperm(row.numel(), generator=g)
    index = torch.stack([row[perm], col[perm]])
    E = index.size(1)
    v1 = torch.randn(E, generator=g, dtype=torch.float64)
    v2 = torch.randn(E, 3, generator=g, dtype=torch.float64)
    co = {"in": dict(index=index, v1=v1, v2=v2, M=M, N=N)}
    for tag, v in (("v1", v1), ("v2", v2)):
        for op in ("add", "mean", "min", "max"):
            vv = v.clone().requires_grad_()
            oi, ov = tsr.coalesce(index, vv, M, N, op=op)
            go = torch.randn(ov.shape, generator=g, dtype=torch.float64)
            ov.backward(go)
            co[f"{tag}_{op}"] = dict(index=oi, value=ov.detach(), grad_out=go, grad_value=vv.grad.clone())
    vv = v1.clone().requires_grad_()
    ti, tv = tsr.transpose(index, vv, M, N)
    go = torch.randn(tv.shape, generator=g, dtype=torch.float64)
    tv.backward(go)
    co["transpose"] = dict(index=ti, value=tv.detach(), grad_out=go, grad_value=vv.grad.clone())
    out["coalesce"] = co

    # coalesced operands: spadd / add / to_symmetric / reductions
    M, N = 36, 36
    ra, ca = random_structure(M, N, 5, seed=92, empty_rows=(0, 9))
    rb, cb = random_structure(M, N, 4, seed=93, empty_rows=(4,))
    va = torch.randn(ra.numel(), generator=g, dtype=torch.float64)
    vb = torch.randn(rb.numel(), generator=g, dtype=torch.float64)
    va2 = torch.randn(ra.numel(), 2, generator=g, dtype=torch.float64)
    ops = {"in": dict(ra=ra, ca=ca, va=va, va2=va2, rb=rb, cb=cb, vb=vb, M=M, N=N)}

    a, b = va.clone().requires_grad_(), vb.clone().requires_grad_()
    si, sv = tsr.spadd(torch.stack([ra, ca]), a, torch.stack([rb, cb]), b, M, N)
    go = torch.randn(sv.shape, generator=g, dtype=torch.float64)
    sv.backward(go)
    ops["spadd"] = dict(index=si, value=sv.detach(), grad_out=go, grad_a=a.grad.clone(), grad_b=b.grad.clone())

    a, b = va.clone().requires_grad_(), vb.clone().requires_grad_()
    C = tsr.add(SparseTensor(row=ra, col=ca, value=a, sparse_sizes=(M, N)),
                SparseTensor(row=rb, col=cb, value=b, sparse_sizes=(M, N)))
    cv = C.storage.value()
    go = torch.randn(cv.shape, generator=g, dtype=torch.float64)
    cv.backward(go)
    ops["add"] = dict(row=C.storage.row(), col=C.storage.col(), value=cv.detach(), grad_out=go,
                      grad_a=a.grad.clone(), grad_b=b.grad.clone())

    for tag, v in (("v", va), ("v2", va2)):
        for red in ("sum", "mean", "min", "max"):
            a = v.clone().requires_grad_()
            S = SparseTensor(row=ra, col=ca, value=a, sparse_sizes=(M, N)).to_symmetric(red)
            sv = S.storage.value()
            go = torch.randn(sv.shape, generator=g, dtype=torch.float64)
            sv.backward(go)
            ops[f"sym_{red}_{tag}"] = dict(row=S.storage.row(), col=S.storage.col(), value=sv.detach(), grad_out=go,
                                           grad_value=a.grad.clone())
            for dim in (0, 1):
                a = v.clone().requires_grad_()
                r = getattr(tsr, red)(SparseTensor(row=ra, col=ca, value=a, sparse_sizes=(M, N)), dim)
                go = torch.randn(r.shape, generator=g, dtype=torch.float64)
                r.backward(go)
                ops[f"reduce_{red}_{dim}_{tag}"] = dict(out=r.detach(), grad_out=go, grad_value=a.grad.clone())
    out["ops"] = ops

    # GCN normalisation: deg = A.sum(1); A_hat = D^-1/2 A D^-1/2; y = A_hat @ x  (learnable edge weights)
    a = va.abs().add(0.1).requires_grad_()
    x = torch.randn(N, 5, generator=g, dtype=torch.float64, requires_grad=True)
    A = SparseTensor(row=ra, col=ca, value=a, sparse_sizes=(M, N))
    deg = tsr.sum(A, dim=1)
    dis = deg.pow(-0.5)
    dis = dis.masked_fill(dis == float("inf"), 0.0)
    Ah = tsr.mul(tsr.mul(A, dis.view(-1, 1)), dis.view(1, -1))
    y = Ah @ x
    go = torch.randn(y.shape, generator=g, dtype=torch.float64)
    y.backward(go)
    out["gcn"] = dict(value=a.detach().clone(), x=x.detach().clone(), y=y.detach(), grad_out=go,
                      grad_value=a.grad.clone(), grad_x=x.grad.clone())
    torch.save(out, GOLD / "grads.pt")
    print("grads.pt", (GOLD / "grads.pt").stat().st_size)


def gen_reference_ops(meta):
    """The reference's compiled CPU operators (ind2ptr / ptr2ind, spmm_sum / mean / min / max over a batched dense
    operand) for five dtypes, registered as torch.ops.torch_sparse.* by import_reference() or build_ref.load()."""
    g = torch.Generator().manual_seed(0)
    M, N, K = 160, 96, 4
    deg = torch.randint(0, 12, (M,), generator=g)
    row = torch.repeat_interleave(torch.arange(M), deg)
    col = torch.randint(N, (row.numel(),), generator=g)
    rowptr = torch.ops.torch_sparse.ind2ptr(row, M)
    out = {"meta": meta, "in": dict(row=row, col=col, M=M), "rowptr": rowptr,
           "row_back": torch.ops.torch_sparse.ptr2ind(rowptr, row.numel()), "cases": {}}
    for dt in (torch.float32, torch.float64, torch.bfloat16, torch.float16, torch.int64):
        if dt.is_floating_point:
            v = torch.randn(col.numel(), generator=g).to(dt); x = torch.randn(2, N, K, generator=g).to(dt)
        else:
            v = torch.randint(-5, 6, (col.numel(),), generator=g); x = torch.randint(-5, 6, (2, N, K), generator=g)
        c = dict(value=v, mat=x, sum=torch.ops.torch_sparse.spmm_sum(None, rowptr, col, v, None, None, x),
                 mean=torch.ops.torch_sparse.spmm_mean(None, rowptr, col, v, None, None, None, x))
        c["min"], c["argmin"] = torch.ops.torch_sparse.spmm_min(rowptr, col, v, x)
        c["max"], c["argmax"] = torch.ops.torch_sparse.spmm_max(rowptr, col, v, x)
        out["cases"][str(dt).split(".")[-1]] = c
    torch.save(out, GOLD / "reference_ops.pt")


if __name__ == "__main__":
    _meta = {"reference": "rusty1s/pytorch_sparse 0.6.18 @ 91feaa5e", "torch": torch.__version__}
    if len(sys.argv) > 1 and sys.argv[1] == "spspmm2":
        gen_spspmm2(import_reference(), _meta)
    elif len(sys.argv) > 1 and sys.argv[1] == "next_rows2":
        gen_next_rows2(import_reference(), {"reference": "rusty1s/pytorch_sparse 0.6.18 @ 91feaa5e", "torch": torch.__version__})
    elif len(sys.argv) > 1 and sys.argv[1] == "grads":
        gen_grads(import_reference(), _meta)
    elif len(sys.argv) > 1 and sys.argv[1] == "reference_ops":   # needs only the operators build_ref.build() makes
        from oracle import build_ref
        build_ref.build()
        build_ref.load()
        gen_reference_ops(_meta)
    else:
        main()
