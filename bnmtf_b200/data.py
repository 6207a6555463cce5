"""Data path around the models (SURVEY.md section 8f #4): the reference's text loaders and toy generators, and the
upload of a host (R, M) pair into the device layout the kernels read.  Host code; the on-disk formats are the
reference's.

  load_gdsc / negate_gdsc / store_gdsc   data_drug_sensitivity/gdsc/load_data.py:15-86
  load_ccle                              data_drug_sensitivity/ccle/load_data.py:16-28
  generate_dataset / add_noise / try_generate_M    data_toy/bnmf/generate_bnmf.py:27-66 (two factors),
  generate_dataset_nmtf                            data_toy/bnmtf/generate_bnmtf.py:28-44 (three factors)
  load_matrix_pair                       the `numpy.loadtxt(R.txt), numpy.loadtxt(M.txt)` idiom of every experiment script
  upload                                 (R, M) -> engine.Dataset: R and R^T zero-padded, the mask as bit words in both
                                         orientations (the digit planes are built on first use)

The reference's data files are not shipped with this package: the loaders take the file location (the reference's
default paths inside its own checkout are what `location=None` meant there).  The generators consume numpy's global
random stream in the reference's order (U row-major, V row-major, then the noise row-major), so a seeded call
reproduces the reference's matrices.
"""
import numpy as np

from . import mask as _mask


# ---- GDSC (Sanger) drug sensitivity -------------------------------------------------------------------------
def load_gdsc(location, standardised=False, sep=","):
    """-> (X, X_min, M, drug_names, cell_lines, cancer_types, tissues).  First line: three header cells then the drug
    names; then one line per cell line: name, cancer type, tissue, values ('' = missing).  X has 0 at missing entries;
    X_min = X - (min(X) - 1) on the observed entries (so the smallest observed value becomes 1), 0 elsewhere.
    `standardised` only selected another default file in the reference; it is accepted and ignored."""
    assert location, "load_gdsc: give the location of the GDSC text file (the reference's data is not shipped)."
    with open(location, 'r') as fin:
        lines = [line.split("\n")[0].split("\r")[0].split(sep) for line in fin.readlines()]
    drug_names = lines[0][3:]
    cell_lines, cancer_types, tissues, X, M = [], [], [], [], []
    for line in lines[1:]:
        cell_lines.append(line[0])
        cancer_types.append(line[1])
        tissues.append(line[2])
        X.append([float(v) if v != '' else 0.0 for v in line[3:]])
        M.append([1.0 if v != '' else 0.0 for v in line[3:]])
    X, M = np.array(X, dtype=float), np.array(M, dtype=float)
    minimum = X.min() - 1
    X_min = np.where(M != 0, X - minimum, 0.0)
    return (X, X_min, M, drug_names, cell_lines, cancer_types, tissues)


def negate_gdsc(X, M):
    """-X shifted so that its smallest value (over ALL entries, like the reference) maps to 0; 0 at missing entries."""
    X = -np.asarray(X, dtype=float)
    minimum = X.min()
    return np.where(np.asarray(M) != 0, X - minimum, 0.0)


def store_gdsc(location, X, M, drug_names, cell_lines, cancer_types, tissues):
    """Tab-separated, same columns as load_gdsc reads (with sep='\\t'); nothing is written for a missing value."""
    with open(location, 'w') as fout:
        fout.write("Cell Line\tCancer Type\tTissue\t" + "\t".join(drug_names) + "\n")
        for i, (cell_line, cancer_type, tissue, row) in enumerate(zip(cell_lines, cancer_types, tissues, X)):
            data = [str(val) if M[i][j] else "" for (j, val) in enumerate(row)]
            fout.write(cell_line + "\t" + cancer_type + "\t" + tissue + "\t" + "\t".join(data) + "\n")


# ---- CCLE ------------------------------------------------------------------------------------------------------
def load_ccle(location, delim='\t'):
    """-> (X, M): a bare delimiter-separated matrix, empty / nan cells are missing (X = 0, M = 0 there)."""
    assert location, "load_ccle: give the location of ic50.txt / ec50.txt (the reference's data is not shipped)."
    data = np.genfromtxt(location, delimiter=delim, missing_values=[np.nan])
    data = np.atleast_2d(data)
    known = ~np.isnan(data)
    return np.where(known, data, 0.0), known.astype(float)


def load_matrix_pair(location_R, location_M):
    """The whitespace-separated R.txt / M.txt pair of data_toy/ (numpy.loadtxt on both)."""
    R, M = np.loadtxt(location_R), np.loadtxt(location_M)
    assert R.shape == M.shape, "R and M have different shapes: %s and %s." % (R.shape, M.shape)
    return R, M


# ---- toy generators -------------------------------------------------------------------------------------------
def add_noise(true_R, tau):
    """R_ij ~ N(true_R_ij, 1/tau); tau = inf: a copy."""
    true_R = np.asarray(true_R, dtype=float)
    if np.isinf(tau):
        return np.copy(true_R)
    return np.random.normal(loc=true_R, scale=1.0 / np.sqrt(tau))


def generate_dataset(I, J, K, lambdaU, lambdaV, tau):
    """-> (U, V, tau, true_R, R) with U_ik ~ Exp(lambdaU_ik), V_jk ~ Exp(lambdaV_jk), R = U V^T + noise."""
    U = np.random.exponential(scale=1.0 / np.asarray(lambdaU, dtype=float)[:I, :K])
    V = np.random.exponential(scale=1.0 / np.asarray(lambdaV, dtype=float)[:J, :K])
    true_R = np.dot(U, V.T)
    return (U, V, tau, true_R, add_noise(true_R, tau))


def generate_dataset_nmtf(I, J, K, L, lambdaF, lambdaS, lambdaG, tau):
    """-> (F, S, G, tau, true_R, R) with R = F S G^T + noise."""
    F = np.random.exponential(scale=1.0 / np.asarray(lambdaF, dtype=float)[:I, :K])
    S = np.random.exponential(scale=1.0 / np.asarray(lambdaS, dtype=float)[:K, :L])
    G = np.random.exponential(scale=1.0 / np.asarray(lambdaG, dtype=float)[:J, :L])
    true_R = np.dot(F, np.dot(S, G.T))
    return (F, S, G, tau, true_R, add_noise(true_R, tau))


def try_generate_M(I, J, fraction_unknown, attempts):
    """A random mask with no empty row or column (mask.generate_M, python `random`), or an Exception after `attempts`."""
    for attempt in range(1, attempts + 1):
        M = _mask.generate_M(I, J, fraction_unknown)
        if (M.sum(axis=0) != 0).all() and (M.sum(axis=1) != 0).all():
            return M
    raise Exception("Tried to generate M %s times, with I=%s, J=%s, fraction=%s, but failed." % (attempts, I, J, fraction_unknown))


# ---- host -> device ---------------------------------------------------------------------------------------------
def upload(R, M, device=None, distributed=False):
    """(R, M) host arrays -> engine.Dataset on `device` (default: the current CUDA device): fp64 R and R^T, padded,
    with the float mask packed into bit words (256 MiB instead of 16 GiB at 65536 x 32768).  distributed=True keeps
    only this rank's row shards of R and R^T (an initialised torch.distributed group is required).  The result can be
    passed to `Model.from_dataset(ds, K, priors)` so that several models share one resident copy of the matrix."""
    from .engine import Dataset, require_cuda
    dev = require_cuda(device)
    world, rank = 1, 0
    if distributed:
        import torch.distributed as dist
        world, rank = dist.get_world_size(), dist.get_rank()
    return Dataset.from_host(np.array(R, dtype=float), np.array(M, dtype=float), dev, world, rank)


# ---- sparse input ------------------------------------------------------------------------------------------------
def _entries(A, name):
    """(rows, cols, values) of every stored entry of a scipy.sparse matrix / array, explicit zeros and duplicates included."""
    import scipy.sparse as sp
    if not sp.issparse(A):
        raise ValueError("%s must be a scipy.sparse matrix or array, not %s" % (name, type(A).__name__))
    if A.ndim != 2:
        raise ValueError("%s must be two-dimensional" % name)
    C = A.tocoo()
    return np.asarray(C.row, dtype=np.int64), np.asarray(C.col, dtype=np.int64), np.asarray(C.data, dtype=np.float64)


def canonical_csr(R):
    """The stored entries of a scipy.sparse R (any format) as a canonical CSR: float64 values, indices sorted within each
    row, explicit zeros KEPT (a stored zero is a known entry).  Duplicate (i, j) entries raise ValueError: summing them
    would change the data."""
    import scipy.sparse as sp
    if not sp.issparse(R):
        raise ValueError("R must be a scipy.sparse matrix or array, not %s" % type(R).__name__)
    I, J = R.shape
    if R.format == "csr" and R.has_canonical_format:          # sorted and duplicate-free already: no sort needed
        return sp.csr_matrix((np.array(R.data, dtype=np.float64), np.array(R.indices, dtype=np.int32),
                              np.array(R.indptr, dtype=np.int64)), shape=(I, J))
    rows, cols, vals = _entries(R, "R")
    order = np.lexsort((cols, rows))
    rows, cols, vals = rows[order], cols[order], vals[order]
    if rows.size > 1:
        dup = (rows[1:] == rows[:-1]) & (cols[1:] == cols[:-1])
        if dup.any():
            k = int(np.argmax(dup))
            raise ValueError("R has more than one stored entry at (%d, %d)" % (rows[k], cols[k]))
    indptr = np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=I))]).astype(np.int64)
    return sp.csr_matrix((vals, cols.astype(np.int32), indptr), shape=(I, J))


def sparse_selection(Rc, M, name="M"):
    """Boolean per stored entry of the canonical CSR Rc: True where the scipy.sparse M has a non-zero entry.  Every such
    entry must be a stored entry of Rc (ValueError otherwise)."""
    rows, cols, vals = _entries(M, name)
    if tuple(M.shape) != tuple(Rc.shape):
        raise ValueError("%s has shape %s, R has %s" % (name, tuple(M.shape), tuple(Rc.shape)))
    nz = vals != 0
    J = Rc.shape[1]
    key = np.unique(rows[nz] * J + cols[nz])
    rkey = np.repeat(np.arange(Rc.shape[0], dtype=np.int64), np.diff(Rc.indptr)) * J + Rc.indices.astype(np.int64)
    pos = np.searchsorted(rkey, key)
    inside = pos < rkey.size
    inside[inside] = rkey[pos[inside]] == key[inside]
    if not inside.all():
        k = key[np.argmin(inside)]
        raise ValueError("%s selects (%d, %d), which is not a stored entry of R" % (name, k // J, k % J))
    sel = np.zeros(rkey.size, dtype=bool)
    sel[pos] = True
    return sel


def training_csr(Rc, train):
    """The training entries of the canonical CSR Rc as a canonical CSR (train: bool per stored entry, or None: all)."""
    import scipy.sparse as sp
    if train is None or bool(np.all(train)):
        return Rc
    I = Rc.shape[0]
    rows = np.repeat(np.arange(I, dtype=np.int64), np.diff(Rc.indptr))[train]
    indptr = np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=I))]).astype(np.int64)
    return sp.csr_matrix((Rc.data[train], Rc.indices[train], indptr), shape=Rc.shape)


def validate_sparse(R, M=None):
    """Host-side checks and canonical form of sparse input (no GPU call): -> (R as canonical CSR, M as CSR of ones on the
    training entries, bool per stored entry of R: training or not).  M None: every stored entry of R is a training
    entry.  Raises the reference's AssertionError texts for a shape mismatch and an unobserved row / column, ValueError
    for duplicate entries in R and for an M entry outside R's pattern."""
    import scipy.sparse as sp
    if M is not None:
        if not sp.issparse(M):
            raise ValueError("with sparse R, M must be None or a scipy.sparse matrix, not %s" % type(M).__name__)
        assert tuple(R.shape) == tuple(M.shape), "Input matrix R is not of the same size as " \
            "the indicator matrix M: %s and %s respectively." % (tuple(R.shape), tuple(M.shape))
    Rc = canonical_csr(R)
    I, J = Rc.shape
    train = np.ones(Rc.nnz, dtype=bool) if M is None else sparse_selection(Rc, M)
    rows = np.repeat(np.arange(I, dtype=np.int64), np.diff(Rc.indptr))
    sums_rows = np.bincount(rows[train], minlength=I)
    sums_columns = np.bincount(Rc.indices[train], minlength=J)
    for i, c in enumerate(sums_rows):
        assert c != 0, "Fully unobserved row in R, row %s." % i
    for j, c in enumerate(sums_columns):
        assert c != 0, "Fully unobserved column in R, column %s." % j
    indptr = np.concatenate([[0], np.cumsum(sums_rows)]).astype(np.int64)
    Mc = sp.csr_matrix((np.ones(int(train.sum())), Rc.indices[train], indptr), shape=(I, J))
    return Rc, Mc, train


def upload_sparse(R, M=None, device=None):
    """Sparse (R, M) -> engine.SparseDataset on `device` (default: the current CUDA device): the training entries in
    CSR form for the row phase and for the column phase, with the static work plan of the statistics kernel.  R and M
    as the model constructors take them (validate_sparse).  The result can be passed to `Model.from_dataset(ds, K,
    priors)` of the two-factor models so that several models share one resident copy of the matrix."""
    from .engine import SparseDataset, require_cuda
    Rc, _, train = validate_sparse(R, M)
    return SparseDataset(Rc, train, require_cuda(device))
