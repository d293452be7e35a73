"""Readers for the on-disk inputs either side of the hot path (SURVEY.md 8f row 4), no R needed.

  * tab/space-separated genotype text with a header row and a sample-id column, the format the reference's scripts
    feed to read.table / read.delim (paper_materials/Real Data Analysis/Full_Test/dataprep.R:3-4,
    paper_materials/Timing Tests/test_time_Gaus.R:13-19) -> int8 matrix (genotype codes) ready for the device;
  * two-column phenotype text (sample id, value), pheno_left.txt;
  * .rda / .RDS (R's XDR serialisation; the package's bundled BASIS.rda, y.rda, ...), via pareben_b200.rdata;
  * .npy / .npz for convenience.
`load_problem` applies the row selection of the published workflow (rows of the genotype table whose sample id occurs
in the phenotype table, in phenotype order: SL_filter.R:14 `genotype[pheno[,1],]`); `load_problem_multi` does the same
for several phenotype files of one design."""
from __future__ import annotations

import io as _io
import os
import zipfile

import numpy as np

from . import rdata


def _open_text(path: str, member: str | None = None):
    if path.endswith(".zip"):
        z = zipfile.ZipFile(path)
        name = member or z.namelist()[0]
        return z.open(name)
    return open(path, "rb")


def read_genotype_text(path: str, member: str | None = None, dtype=np.int8):
    """-> (sample_ids [n], marker_names [k], matrix [n, k]).  First row = header (first field names the id column),
    first field of every other row = sample id, the rest numeric codes.  Values are parsed as numbers and stored as
    `dtype` (int8 for genotype codes; pass np.float64 for real-valued designs); a non-integer value with an integer
    dtype raises."""
    with _open_text(path, member) as f:
        header = f.readline().decode().rstrip("\r\n")
        sep = "\t" if "\t" in header else None
        names = header.split(sep)[1:]
        ids, rows = [], []
        for raw in f:
            line = raw.decode().rstrip("\r\n")
            if not line:
                continue
            first, _, rest = line.partition("\t") if sep else line.partition(" ")
            v = np.fromstring(rest, dtype=np.float64, sep="\t" if sep else " ")
            if v.size != len(names):
                raise ValueError(f"{path}: row '{first}' has {v.size} values, header has {len(names)}")
            if np.issubdtype(dtype, np.integer):
                w = v.astype(dtype)
                if not np.array_equal(w, v):
                    raise ValueError(f"{path}: row '{first}' holds values that are not {np.dtype(dtype).name} codes")
                v = w
            ids.append(first.strip('"'))
            rows.append(v)
    return np.array(ids), np.array([n.strip('"') for n in names]), np.vstack(rows) if rows else np.zeros((0, len(names)), dtype)


def read_phenotype_text(path: str):
    """-> (sample_ids [n], values [n]) from a headerless two-column table; a single-column file gives ids = None."""
    ids, vals = [], []
    with _open_text(path) as f:
        for raw in f:
            parts = raw.decode().split()
            if not parts:
                continue
            if len(parts) == 1:
                vals.append(float(parts[0]))
            else:
                ids.append(parts[0].strip('"')); vals.append(float(parts[1]))
    return (np.array(ids) if ids else None), np.array(vals)


def read_matrix(path: str, name: str | None = None):
    """A numeric matrix or vector from .rda / .RDS / .npy / .npz / delimited text.  For containers with several objects
    `name` picks one (default: the only one, or the one named like the file)."""
    ext = os.path.splitext(path)[1].lower()
    if ext == ".rda" or ext == ".rdata":
        objs = rdata.read_rda(path)
        key = name or (next(iter(objs)) if len(objs) == 1 else os.path.splitext(os.path.basename(path))[0])
        return np.asarray(objs[key], dtype=np.float64)
    if ext == ".rds":
        return np.asarray(rdata.read_rds(path), dtype=np.float64)
    if ext == ".npy":
        return np.load(path)
    if ext == ".npz":
        z = np.load(path)
        return z[name or z.files[0]]
    ids, _names, M = read_genotype_text(path, dtype=np.float64)
    return M


def _text_like(p: str) -> bool:
    return os.path.splitext(p)[1].lower() in (".txt", ".tsv", ".zip", ".tab", "")


def _genotype_rows(basis_path: str, pid):
    """Rows of the genotype text in the order of the phenotype ids `pid` (None: as stored)."""
    ids, _names, X = read_genotype_text(basis_path)
    if pid is not None:
        pos = {s: i for i, s in enumerate(ids)}
        missing = [s for s in pid if s not in pos]
        if missing:
            raise ValueError(f"{len(missing)} phenotype ids are absent from the genotype table (first: {missing[0]})")
        X = X[[pos[s] for s in pid]]
    return X


def read_targets(paths, name: str | None = None):
    """-> (sample_ids [n] or None, Targets [n, T]) from several response files, one response each (phenotype text or a
    vector file), or from ONE .npy / .npz holding an n x T matrix.  Phenotype texts are joined on the sample id in the
    order of the first file and must all list the same ids; files without ids are taken row for row."""
    paths = list(paths)
    if not paths:
        raise ValueError("no response file given")
    if len(paths) == 1 and os.path.splitext(paths[0])[1].lower() in (".npy", ".npz"):
        Y = np.asarray(read_matrix(paths[0], name), dtype=np.float64)
        return None, Y.reshape(-1, 1) if Y.ndim == 1 else Y
    first_ids, cols = None, []
    for j, p in enumerate(paths):
        ids, v = read_phenotype_text(p) if _text_like(p) else (None, np.asarray(read_matrix(p, name), dtype=np.float64).ravel())
        if j == 0:
            first_ids = ids
        elif (ids is None) != (first_ids is None):
            raise ValueError(f"{p}: either every response file lists sample ids or none does ({paths[0]} differs)")
        elif ids is not None:
            pos = {s: i for i, s in enumerate(ids)}
            if len(pos) != ids.size or ids.size != first_ids.size or set(pos) != set(first_ids.tolist()):
                raise ValueError(f"{p}: sample ids differ from those of {paths[0]}")
            v = v[[pos[s] for s in first_ids]]
        elif v.size != cols[0].size:
            raise ValueError(f"{p}: {v.size} values, {paths[0]} has {cols[0].size}")
        cols.append(np.asarray(v, dtype=np.float64))
    return first_ids, np.column_stack(cols)


def load_problem_multi(basis_path: str, target_paths, basis_name: str | None = None, target_name: str | None = None):
    """(BASIS [n, k], Targets [n, T]) for several responses of one design (read_targets).  With genotype text and
    phenotype texts the genotype rows follow the ids of the first phenotype file, as in load_problem."""
    pid, Y = read_targets(target_paths, target_name)
    X = _genotype_rows(basis_path, pid) if _text_like(basis_path) and pid is not None else read_matrix(basis_path, basis_name)
    return X, Y


def load_problem(basis_path: str, target_path: str, basis_name: str | None = None, target_name: str | None = None):
    """(BASIS [n, k], Target [n]) from a pair of files.  Genotype text + two-column phenotype text are joined on the
    sample id (rows in phenotype order, SL_filter.R:14); everything else is taken row for row."""
    text_like = _text_like
    if text_like(basis_path) and text_like(target_path):
        pid, y = read_phenotype_text(target_path)
        return _genotype_rows(basis_path, pid), y
    X = read_matrix(basis_path, basis_name)
    y = read_matrix(target_path, target_name) if not text_like(target_path) else read_phenotype_text(target_path)[1]
    return X, np.asarray(y, dtype=np.float64).ravel()
