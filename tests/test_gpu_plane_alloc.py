"""Where the planes live (PFA_PLANE_ALLOC = pool | vmm | compressible) must not change a bit of what is computed: the planes
themselves, the site scan (K2), the codon scan (K4) and the pairwise sums (K3), clean or gapped, with the validity plane
forced, with several populations, and through the hybrid host ingest.  Then the one-range cache of the context: a freed
range is reused by the next alignment that fits, replaced by a larger one, and released by trim."""
import ctypes

import numpy as np
import pytest

import polyfasta_b200 as pf
from polyfasta_b200 import _lib

KINDS = ("pool", "vmm", "compressible")


def test_plane_alloc_symbol_is_exported():
    assert "pfa_aln_plane_alloc" in _lib.EXPORTS
    assert hasattr(_lib.lib(), "pfa_aln_plane_alloc")


def _compression_supported():
    try:
        cu = ctypes.CDLL("libcuda.so.1")
        dev, attr = ctypes.c_int(), ctypes.c_int(0)
        if cu.cuInit(0) or cu.cuDeviceGet(ctypes.byref(dev), 0):
            return False
        return cu.cuDeviceGetAttribute(ctypes.byref(attr), 107, dev) == 0 and attr.value == 1  # GENERIC_COMPRESSION_SUPPORTED
    except OSError:
        return False


@pytest.fixture(scope="module")
def ctx():
    return pf.default_context(0)


def _check_kind(want, got):
    if want == "compressible" and not _compression_supported():
        assert got in ("pool", "vmm")
    else:
        assert got == want


def _everything(a, pops):
    a.set_pops(pops)
    site, cds, pw = a.site_stats(want_isvar=True), a.cds_stats(want_labels=True), a.pairwise()
    return [a.plane(i) for i in range(3)], site, cds, pw


def _same(x, y):
    (px, sx, cx, wx), (py, sy, cy, wy) = x, y
    for a, b in zip(px, py):
        assert np.array_equal(a, b)
    assert len(sx) == len(sy) and len(cx) == len(cy)
    for a, b in zip(sx, sy):
        assert (a["S"], a["H"], a["sfs"]) == (b["S"], b["H"], b["sfs"]) and np.array_equal(a["isvar"], b["isvar"])
    for a, b in zip(cx, cy):
        assert np.array_equal(a["raw"], b["raw"]) and np.array_equal(a["labels"], b["labels"])
    assert list(wx) == list(wy)


@pytest.mark.gpu
@pytest.mark.parametrize("n,L,gaps,force,k", [(1000, 30_000, 0, False, 1), (1000, 30_000, 0, True, 2), (2000, 9_000, 200, False, 3),
                                              (300, 40_001, 50, True, 2), (10_000, 3_000, 0, False, 1)])
def test_kinds_compute_the_same(ctx, monkeypatch, n, L, gaps, force, k):
    monkeypatch.setenv("PFA_PLANE_ALLOC_MIN_BYTES", "0")
    pops = [list(range(n)), list(range(0, n, 2)), list(range(n // 3, n // 2))][:k]
    res = {}
    for kind in KINDS:
        monkeypatch.setenv("PFA_PLANE_ALLOC", kind)
        a = pf.Alignment.synthetic(ctx, n, L, 11 + n)
        _check_kind(kind, a.plane_alloc)
        if gaps:
            a.poke_gaps(11 + n, gaps)
        a.force_validity(force)
        res[kind] = _everything(a, pops)
        assert ("planes=" + a.plane_alloc) in ctx.last_kernel
        a.free()
    _same(res["pool"], res["vmm"])
    _same(res["pool"], res["compressible"])


@pytest.mark.gpu
@pytest.mark.parametrize("pinned", [False, True])
def test_hybrid_ingest_into_each_kind(ctx, monkeypatch, pinned):
    import torch
    rng = np.random.default_rng(5)
    n, L = 700, 50_000
    text = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, (n, L))]
    text[rng.integers(0, n, 60), rng.integers(0, L, 60)] = np.frombuffer(b"-NR?", dtype=np.uint8)[rng.integers(0, 4, 60)]
    monkeypatch.setenv("PFA_PLANE_ALLOC_MIN_BYTES", "0")
    monkeypatch.setenv("PFA_INGEST_CHUNK_MB", "1")
    monkeypatch.setenv("PFA_INGEST_HYBRID", "1")
    host = torch.from_numpy(text).pin_memory() if pinned else None
    pops = [list(range(n)), list(range(1, n, 3))]
    res = {}
    for kind in KINDS:
        monkeypatch.setenv("PFA_PLANE_ALLOC", kind)
        a = pf.Alignment.from_host_ptr(ctx, host.data_ptr(), n, L, L) if pinned else pf.Alignment.from_rows(ctx, text)
        _check_kind(kind, a.plane_alloc)
        res[kind] = _everything(a, pops)
        a.free()
    _same(res["pool"], res["vmm"])
    _same(res["pool"], res["compressible"])


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["vmm", "compressible"])
def test_range_cache_reuse_grow_trim(ctx, monkeypatch, kind):
    """device memory in use, from cudaMemGetInfo: a range is 1.5-2.3 GB here, far above anything else this test allocates"""
    import torch
    monkeypatch.setenv("PFA_PLANE_ALLOC", kind)
    monkeypatch.delenv("PFA_PLANE_ALLOC_MIN_BYTES", raising=False)
    gb = 1 << 30
    ctx.trim()
    used = lambda: torch.cuda.mem_get_info(0)[1] - torch.cuda.mem_get_info(0)[0]  # noqa: E731
    u0 = used()
    a = pf.Alignment.synthetic(ctx, 1000, 4_000_000, 3)          # 3 x 512 MB of planes
    got = a.plane_alloc
    if got == "pool":
        pytest.skip("the device granted no VMM range")
    S = a.site_stats()[0]["S"]
    a.free()
    u1 = used()
    assert u1 - u0 > 1.2 * gb                                    # the freed range stays mapped
    b = pf.Alignment.synthetic(ctx, 1000, 2_000_000, 3)          # fits: takes the cached range over
    assert b.plane_alloc == got and abs(used() - u1) < 0.3 * gb
    assert b.site_stats()[0]["S"] > 0
    b.free()
    c = pf.Alignment.synthetic(ctx, 1000, 6_000_000, 3)          # does not fit: the cached range goes, a larger one comes
    assert c.plane_alloc == got and abs(used() - u0 - 2.25 * gb) < 0.3 * gb
    c.free()
    d = pf.Alignment.synthetic(ctx, 1000, 4_000_000, 3)          # the same alignment as `a` in the larger range
    assert d.site_stats()[0]["S"] == S
    d.free()
    ctx.trim()
    assert abs(used() - u0) < 0.3 * gb                           # trim released it
