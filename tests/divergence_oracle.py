"""CPU oracles for the divergence between populations (d_xy, d_a, Hudson's F_ST)  --  TEST INFRASTRUCTURE ONLY.

The divergence statistics are beyond the reference, so their oracles live with their tests rather than next to the pinned
restatement of the reference in oracle/.  They are built on that restatement's column counts (every character is an allele,
PolyFastA.py:256-258):

    Dxy_site(p) = n_x n_y - sum_a c_{X,a}(p) c_{Y,a}(p)      D_xy = sum_p Dxy_site(p)

and the float formulas below in the operation order of pfa_div_finalize.  `divergence_c` is the C + OpenMP twin of
`divergence` for shapes the pure-Python loop cannot finish in seconds; it is compiled into a temporary directory on first use."""
import ctypes
import math
import os
import shutil
import subprocess
import tempfile

import numpy as np

from oracle import polyfasta_oracle as orc

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def divergence(rows_x, rows_y, L, per_site=False):
    """rows_x, rows_y: upper-cased sequences (str) of the two populations -> D_xy, or (D_xy, [Dxy_site per column])"""
    nx, ny = len(rows_x), len(rows_y)
    ds = []
    for p in range(L):
        cx, cy = orc.column_counts(rows_x, p), orc.column_counts(rows_y, p)
        ds.append(nx * ny - sum(c * cy.get(a, 0) for a, c in cx.items()))
    return (sum(ds), ds) if per_site else sum(ds)


def pi_site(rows, L, jc):
    """pi_site of K5 for one population: 0 when the population has no variable column"""
    st = orc.site_stats(rows, L, want_sfs=False)
    return orc.finalize(st["n"], st["S"], st["H"], L, jc)[1]


def finalize(n_x, n_y, D, seqlen, pi_x, pi_y, jc):
    """-> (dxy, da, fst | "NA"); ("NA", "NA", "NA") when n_x n_y == 0 or seqlen <= 0"""
    if n_x * n_y == 0 or seqlen <= 0:
        return "NA", "NA", "NA"
    dxy = (D / (n_x * n_y)) / seqlen
    if jc:
        x = 1 - (4. / 3.) * dxy
        if x > 0:
            dxy = -0.75 * math.log(x)
    hw = 0.5 * (pi_x + pi_y)
    da = dxy - hw
    fst = 1 - hw / dxy if dxy != 0 else "NA"
    return dxy, da, fst


def pairs(k):
    return [(x, y) for x in range(k) for y in range(x + 1, k)]


def divergence_rows(seqs, pops, jc):
    """seqs: upper-cased sequences of the alignment; pops: row-index lists -> [(D, dxy, da, fst)] per pair in pair order"""
    L = len(seqs[0]) if seqs else 0
    rows = [[seqs[i] for i in p] for p in pops]
    pis = [pi_site(r, L, jc) for r in rows]
    out = []
    for x, y in pairs(len(pops)):
        D = divergence(rows[x], rows[y], L)
        out.append((D,) + finalize(len(rows[x]), len(rows[y]), D, L, pis[x], pis[y], jc))
    return out


def _build():
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else (shutil.which("cc") or "gcc")
    out = os.path.join(tempfile.mkdtemp(prefix="pfa_div_oracle_"), "libdivergence_oracle.so")
    subprocess.check_call([cc, "-O2", "-fopenmp", "-fPIC", "-shared", "-o", out, os.path.join(_HERE, "divergence_oracle.c")])
    return out


def _c():
    global _lib
    if _lib is None:
        L = ctypes.CDLL(_build())
        p, i64 = ctypes.c_void_p, ctypes.c_int64
        L.orc_divergence.argtypes = [p, i64, i64, p, i64, p, i64, p]
        L.orc_divergence.restype = i64
        _lib = L
    return _lib


def divergence_c(mat, rows_x, rows_y, per_site=False):
    """C twin of divergence: mat = upper-cased uint8 [n][L] -> D_xy, or (D_xy, int64 [L] Dxy_site)"""
    mat = np.ascontiguousarray(mat, dtype=np.uint8)
    L = mat.shape[1]
    ld = max(L, 1)
    rx = np.ascontiguousarray(rows_x, dtype=np.int32)
    ry = np.ascontiguousarray(rows_y, dtype=np.int32)
    ds = np.zeros(max(L, 1), dtype=np.int64) if per_site else None
    D = _c().orc_divergence(mat.ctypes.data, ld, L, rx.ctypes.data, len(rx), ry.ctypes.data, len(ry),
                            ds.ctypes.data if per_site else None)
    return (int(D), ds[:L]) if per_site else int(D)
