"""Fixed SMPL mesh hierarchy: loading, Laplacians, operator composition, ELL packing.

Host-side counterpart of the reference's topology prep:
  - `laplacian`, `rescale_L`  : lib/mesh_sampling.py:10-38 (same names, same arithmetic in fp32)
  - `load_graph_mtx`          : lib/load_data.py:7-32 (same return convention) -- reads the pickle-free
                                copy of data/transform_matrices/** under tests/golden/ (made by
                                cape_b200/pack_topology.py from a checkout of the reference)
The reference turns every scipy matrix into a tf.SparseTensor and runs one SpMM per Chebyshev order and
per pool/unpool (lib/models.py:74-96,141-149).  Here the operators are constants, so they are composed
offline:  op_k = D . T_k(L~) . U  -- one sparse "row-gather" per polynomial order with pooling (row
selection) and unpooling (3-tap barycentric) folded in -- and packed as ELL tables for the CUDA kernels.
"""
import os

import numpy as np
import scipy.sparse as sp

DATA_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
# the fixtures are split in parts so that no single file grows past 1 MB
DATA_PARTS = ("for_demo", "ds2", "assets")
_cache = {}


def data_files(directory=DATA_DIR):
    return [os.path.join(directory, "smpl_topology.%s.npz" % part) for part in DATA_PARTS]


def laplacian(W, normalized=True):
    """Normalised graph Laplacian I - D^-1/2 W D^-1/2 (lib/mesh_sampling.py:10-29)."""
    W = sp.csr_matrix(W)
    d = np.asarray(W.sum(axis=0)).reshape(-1).astype(W.dtype)
    if not normalized:
        return sp.csr_matrix(sp.diags(d, 0) - W)
    d = d + np.spacing(np.array(0, W.dtype))
    d = (1 / np.sqrt(d)).astype(W.dtype)
    Dm = sp.diags(d, 0)
    I = sp.identity(d.size, dtype=W.dtype)
    return sp.csr_matrix(I - Dm * W * Dm)


def rescale_L(L, lmax=2):
    """L/(lmax/2) - I on a copy (lib/mesh_sampling.py:31-38; chebyshev5 copies first, models.py:74)."""
    L = sp.csr_matrix(L, copy=True)
    I = sp.identity(L.shape[0], format="csr", dtype=L.dtype)
    L /= lmax / 2        # in place, as the reference does: keeps fp32 (scipy's out-of-place "/" upcasts to fp64)
    L -= I
    return sp.csr_matrix(L)


def _npz():
    if "npz" not in _cache:
        z = {}
        for fn in data_files():
            with np.load(fn) as part:
                z.update((k, part[k]) for k in part.files)
        _cache["npz"] = z
    return _cache["npz"]


def _mats(kind, name, dtype):
    z = _npz()
    out = []
    for i in range(int(z["%s.%s.count" % (kind, name)])):
        k = "%s.%s.%d" % (kind, name, i)
        m = sp.csr_matrix((z[k + ".data"], z[k + ".indices"], z[k + ".indptr"]), shape=tuple(z[k + ".shape"]))
        out.append(m.astype(dtype))
    return out


def load_graph_mtx(project_dir=None, load_for_demo=False):
    """Same contract as lib/load_data.py:7-32: returns L_ds2, D_ds2, U_ds2 or, with load_for_demo,
    L, D, U, p, L_ds2, D_ds2, U_ds2 (all fp32; L = normalised Laplacians of the adjacency fixtures).
    `project_dir` is accepted for signature compatibility and ignored (the fixtures are read from DATA_DIR)."""
    A_ds2, D_ds2, U_ds2 = (_mats("ds2", n, np.float32) for n in "ADU")
    L_ds2 = [laplacian(a, normalized=True) for a in A_ds2]
    if not load_for_demo:
        return L_ds2, D_ds2, U_ds2
    A, D, U = (_mats("for_demo", n, np.float32) for n in "ADU")
    p = [a.shape[0] for a in A]
    L = [laplacian(a, normalized=True) for a in A]
    return L, D, U, p, L_ds2, D_ds2, U_ds2


def smpl_edges():
    """[20664, 2] int32 vertex pairs (data/edges_smpl.npy of the reference = upper triangle of A[0])."""
    return _npz()["edges"]


def trainset_stats():
    z = _npz()
    return z["stats.mean"], z["stats.std"]


def clothing_verts_idx():
    return _npz()["clothing_verts_idx"]


def template_mesh():
    """(vertices [6890, 3] float64, faces [13776, 3] int32) of data/template_mesh.obj (demos.py:352-353)."""
    z = _npz()
    return z["template.v"], z["template.f"]


def demo_pose_params():
    """(rot [6, 216], pose [6, 72]) of data/demo_data/demo_pose_params.npz (demos.py:355-356)."""
    z = _npz()
    return z["demo.rot"], z["demo.pose"]


# ---------------------------------------------------------------------------------------------------
# operator algebra
# ---------------------------------------------------------------------------------------------------
def is_identity(S, tol=1e-9):
    S = sp.csr_matrix(S)
    if S.shape[0] != S.shape[1]:
        return False
    d = S - sp.identity(S.shape[0], dtype=S.dtype, format="csr")
    return d.nnz == 0 or float(np.abs(d.data).max()) <= tol


def is_selection(S):
    """True if S has exactly one entry, equal to 1, in every row (a pure row selection, like the reference's
    down-sampling matrices D).  Only then does pooling commute with a pointwise bias/activation."""
    S = sp.csr_matrix(S, copy=True)
    S.eliminate_zeros()
    return bool(S.nnz == S.shape[0] and np.all(np.diff(S.indptr) == 1) and np.all(S.data == 1))


def cheb_polynomials(L, K):
    """[T_0(L~) .. T_{K-1}(L~)] as float64 CSR (sparse; intended for small K)."""
    Lt = rescale_L(sp.csr_matrix(L), lmax=2).astype(np.float64)
    Lt.eliminate_zeros()
    M = Lt.shape[0]
    T = [sp.identity(M, format="csr", dtype=np.float64)]
    if K > 1:
        T.append(Lt)
    for _ in range(2, K):
        T.append(sp.csr_matrix(2 * Lt @ T[-1] - T[-2]))
    return T


def compose(D, T, U):
    """D . T . U with None = identity; float64 CSR, explicit zeros removed."""
    m = sp.csr_matrix(T, dtype=np.float64)
    if U is not None:
        m = m @ sp.csr_matrix(U, dtype=np.float64)
    if D is not None:
        m = sp.csr_matrix(D, dtype=np.float64) @ m
    m = sp.csr_matrix(m)
    m.sum_duplicates()
    m.eliminate_zeros()
    m.sort_indices()
    return m


def to_ell(m):
    """CSR -> (idx int32 [rows, width], w fp32 [rows, width]); empty slots idx=-1, w=0, left-packed."""
    m = sp.csr_matrix(m)
    m.sort_indices()
    rows = m.shape[0]
    counts = np.diff(m.indptr)
    width = max(int(counts.max()) if rows else 1, 1)
    idx = np.full((rows, width), -1, np.int32)
    w = np.zeros((rows, width), np.float32)
    slot = np.arange(m.nnz) - np.repeat(m.indptr[:-1], counts)
    rr = np.repeat(np.arange(rows), counts)
    idx[rr, slot] = m.indices
    w[rr, slot] = m.data.astype(np.float32)
    return idx, w


# ---------------------------------------------------------------------------------------------------
# internal vertex order (data layout only: results do not depend on it)
# ---------------------------------------------------------------------------------------------------
def _fiedler_halves(A, nodes):
    """Split `nodes` into two halves along the Fiedler vector of the induced subgraph."""
    import scipy.sparse.csgraph as csg
    import scipy.sparse.linalg as sla
    n = len(nodes)
    sub = A[nodes][:, nodes].tocsr()
    nc, lab = csg.connected_components(sub, directed=False)
    if nc > 1:                                   # keep components together
        sizes = np.bincount(lab)
        left, na, nb = [], 0, 0
        for c in np.argsort(-sizes, kind="stable"):
            if na <= nb:
                left.append(c)
                na += sizes[c]
            else:
                nb += sizes[c]
        m = np.isin(lab, left)
        return nodes[m], nodes[~m]
    lap = (sp.diags(np.asarray(sub.sum(1)).ravel()) - sub).astype(np.float64)
    f = None
    if n >= 64:
        try:
            v0 = np.cos(np.arange(n) * 0.7) + 1.5          # fixed start vector: the order is reproducible
            w, v = sla.eigsh(lap.tocsc(), k=2, sigma=-1e-3, which="LM", tol=1e-7, v0=v0)
            f = v[:, np.argsort(w)[1]]
        except Exception:
            f = None
    if f is None:
        f = np.linalg.eigh(lap.toarray())[1][:, 1]
    nz = np.flatnonzero(np.abs(f) > 1e-12)
    if len(nz) and f[nz[0]] < 0:
        f = -f
    o = np.argsort(f, kind="stable")
    return nodes[o[:n // 2]], nodes[o[n // 2:]]


def patch_order(L, leaf=8):
    """Vertex order in which consecutive vertices form compact surface patches at every scale (recursive spectral
    bisection of the mesh graph): order[new] = old.  The CUDA kernels process 128 consecutive rows per tile and
    gather each row's one-ring, so this decides how often a neighbour row is already in L1 (1.55 distinct source
    rows per output row for the SMPL level-0 Laplacian instead of 2.4 in SMPL's own numbering)."""
    A = sp.csr_matrix(L, copy=True).astype(np.float64)
    A.setdiag(0)
    A.eliminate_zeros()
    A.data[:] = 1.0
    key = ("order", A.shape[0], A.nnz, hash(A.indices.tobytes()), hash(A.indptr.tobytes()), leaf)
    if key in _cache:
        return _cache[key]
    out, stack = [], [np.arange(A.shape[0])]
    while stack:
        nodes = stack.pop()
        if len(nodes) <= leaf:
            out.extend(sorted(nodes.tolist()))
            continue
        a, b = _fiedler_halves(A, nodes)
        stack.append(b)
        stack.append(a)
    order = np.asarray(out, dtype=np.int64)
    assert len(order) == A.shape[0] and len(np.unique(order)) == A.shape[0]
    _cache[key] = order
    return order


def induce_order(order_fine, D):
    """Order of the next-coarser level: its vertices are a subset of the finer level's (D is a row selection),
    keep them in the order the finer level visits them.  Identity D (factor-1 levels): same order."""
    D = sp.csr_matrix(D)
    if D.shape[0] == D.shape[1]:
        return order_fine
    assert D.nnz == D.shape[0], "down-sampling matrix must select one fine vertex per coarse vertex"
    pos = np.empty(len(order_fine), np.int64)
    pos[order_fine] = np.arange(len(order_fine))
    return np.argsort(pos[D.indices], kind="stable")


def level_orders(L0, Ds):
    """Orders of every level of a hierarchy, level 0 first."""
    orders = [patch_order(L0)]
    for D in Ds:
        orders.append(induce_order(orders[-1], D))
    return orders


def permute(m, order_out=None, order_in=None):
    """m[order_out][:, order_in]: the operator acting between re-ordered levels (None = reference order)."""
    m = sp.csr_matrix(m)
    if order_out is not None:
        m = m[order_out]
    if order_in is not None:
        m = sp.csr_matrix(sp.csc_matrix(m)[:, order_in])
    m.sort_indices()
    return m


def inverse_order(order):
    inv = np.empty(len(order), np.int64)
    inv[order] = np.arange(len(order))
    return inv


def adjacency_ell(L):
    """Neighbour table of a level (off-diagonal pattern of its Laplacian), for the edge loss."""
    A = sp.csr_matrix(L, copy=True)
    A.setdiag(0)
    A.eliminate_zeros()
    A.data[:] = 1.0
    return to_ell(A)


def window_split(m, tile=128, halo=32):
    """Classify the taps of a same-level operator for window staging (DESIGN.md section 7): for the rows of each
    `tile`-row tile, the taps whose source row lies in [tile_start - halo, tile_start + tile + halo) can be served
    from one contiguous window of the source staged in shared memory (a single TMA box), the rest are "far" taps.
    Returns (idx, w, n_in): ELL tables like `to_ell` but with the window taps packed first in every row (by source
    row), far taps after them, and n_in[r] = number of window taps of row r."""
    m = sp.csr_matrix(m)
    assert m.shape[0] == m.shape[1], "window staging is for same-level operators"
    idx, w = to_ell(m)
    rows, width = idx.shape
    start = (np.arange(rows) // tile) * tile - halo
    local = idx - start[:, None]
    inside = (idx >= 0) & (local >= 0) & (local < tile + 2 * halo)
    # stable sort key: window taps (0) < far taps (1) < padding (2); ties keep the source-row order of to_ell
    key = np.where(idx < 0, 2, np.where(inside, 0, 1))
    order = np.argsort(key, axis=1, kind="stable")
    take = lambda a: np.take_along_axis(a, order, axis=1)
    return take(idx), take(w), inside.sum(1).astype(np.int32)
