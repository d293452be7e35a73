"""Generates tests/golden/{BASIS,y,BASISbinomial,yBinomial}.rda: the package's bundled inputs as R data files, the input
of the .rda reader's test (pareben_b200/rdata.py through pareben_b200/io.py).  Run:   python tests/golden/make_rda_golden.py

The values are tests/golden/inputs_bundled.npz.  The bytes are laid out as `save(<name>, file = "<name>.rda",
version = 2, compress = ...)` writes them (R's serialize.c, XDR format 2): the header "RDX2\\n" "X\\n", format version 2,
the writer's and the oldest reader's R versions, then a pairlist with one tagged entry holding a double vector and, for
a matrix, its "dim" attribute.  The two matrices are xz-compressed (compress = "xz", which keeps them small), the two
vectors gzip-compressed (R's default), so both container formats are read.  Written here with struct only,
independently of the reader under test.
"""
from __future__ import annotations

import gzip
import lzma
import os
import struct

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

LISTSXP, SYMSXP, CHARSXP, INTSXP, REALSXP, NILVALUE_SXP = 2, 1, 9, 13, 14, 254
HAS_ATTR, HAS_TAG, ASCII = 0x200, 0x400, 64 << 12      # flag bits; ASCII_MASK sits in the gp field (bits 12..27)


def _i(v: int) -> bytes:
    return struct.pack(">i", v)


def _symbol(name: str) -> bytes:
    b = name.encode("ascii")
    return _i(SYMSXP) + _i(CHARSXP | ASCII) + _i(len(b)) + b


def _doubles(a: np.ndarray) -> bytes:
    v = np.asarray(a, dtype=np.float64)
    out = _i(REALSXP | (HAS_ATTR if v.ndim == 2 else 0)) + _i(v.size) + v.ravel(order="F").astype(">f8").tobytes()
    if v.ndim == 2:                                   # attributes: pairlist (dim = c(nrow, ncol))
        out += _i(LISTSXP | HAS_TAG) + _symbol("dim") + _i(INTSXP) + _i(2) + _i(v.shape[0]) + _i(v.shape[1])
        out += _i(NILVALUE_SXP)
    return out


def rda_bytes(name: str, a: np.ndarray) -> bytes:
    body = b"RDX2\n" + b"X\n" + _i(2) + _i(0x030402) + _i(0x020300)     # format 2, written by R 3.4.2, readable by R >= 2.3.0
    body += _i(LISTSXP | HAS_TAG) + _symbol(name) + _doubles(a) + _i(NILVALUE_SXP)
    if np.ndim(a) == 2:
        return lzma.compress(body, format=lzma.FORMAT_XZ, preset=9)
    return gzip.compress(body, compresslevel=6, mtime=0)


def main():
    g = np.load(os.path.join(HERE, "inputs_bundled.npz"))
    for name in ("BASIS", "y", "BASISbinomial", "yBinomial"):
        path = os.path.join(HERE, name + ".rda")
        with open(path, "wb") as f:
            f.write(rda_bytes(name, g[name]))
        print(path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
