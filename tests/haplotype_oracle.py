"""CPU oracle for the haplotype statistics (number of haplotypes h, haplotype diversity Hd and its variance)  --  TEST
INFRASTRUCTURE ONLY.

The statistics are beyond the reference, so the oracle lives with its tests.  It states the definitions literally:

- two rows are one haplotype iff their upper-cased sequence strings are equal (PolyFastA.py:236/:245, oracle.parse_fasta),
  over the whole alignment or over a window's columns;
- rep(r) = the smallest row index of r's class, over all rows whatever the populations;
- for a population of n rows whose classes have c_1 .. c_h rows inside it: h, s2 = sum c^2, s3 = sum c^3;
- Hd = (n^2 - s2) / (n (n - 1)), ONE fp64 division of two integers;
- Hd_var = Nei (1987) eq. 8.12, V = 2 / (n (n - 1)) [2 (n - 2) (sum p^3 - (sum p^2)^2) + sum p^2 - (sum p^2)^2], p = c / n, as an
  exact Fraction;
- n = 1: h = 1, Hd and Hd_var are "NA"."""
from fractions import Fraction


def upper(rows):
    return [r.upper() for r in rows]


def rep(rows):
    """rows: sequences (str) -> rep list: the smallest index with the same upper-cased string"""
    first = {}
    out = []
    for i, r in enumerate(upper(rows)):
        out.append(first.setdefault(r, i))
    return out


def pop_stats(rows, members):
    """rows: all sequences; members: the population's row indices -> dict(n, h, s2, s3, Hd, Hd_var) with Hd a float (one
    division) and Hd_var an exact Fraction ("NA" for both when n = 1)"""
    r = rep(rows)
    counts = {}
    for i in members:
        counts[r[i]] = counts.get(r[i], 0) + 1
    n = len(members)
    c = list(counts.values())
    s2, s3 = sum(x * x for x in c), sum(x ** 3 for x in c)
    res = {"n": n, "h": len(c), "s2": s2, "s3": s3, "Hd": "NA", "Hd_var": "NA"}
    if n > 1:
        res["Hd"] = float(n * n - s2) / float(n * (n - 1))
        p2 = sum(Fraction(x, n) ** 2 for x in c)
        p3 = sum(Fraction(x, n) ** 3 for x in c)
        res["Hd_var"] = Fraction(2, n * (n - 1)) * (2 * (n - 2) * (p3 - p2 * p2) + p2 - p2 * p2)
    return res


def window_rows(rows, start, end):
    """the rows cut to the columns [start, end)"""
    return [r[start:end] for r in rows]


def differing_pairs(rows, members):
    """the literal pair loop: unordered pairs of the population whose upper-cased strings differ"""
    u = upper(rows)
    m = list(members)
    return sum(1 for a in range(len(m)) for b in range(a + 1, len(m)) if u[m[a]] != u[m[b]])
