"""The launch plan of the site scan (K2) and the codon scan (K4) is a function of the shape alone: kernel, template arguments,
grid, passes per slot and validity records per slot, as reported by ctx.last_kernel.  The table covers the shape boundaries
of the kernel choice (records of 3 / 4 / 10 / 11 chunks, 20,480 and 12,288 rows), one and two populations, flagged-site
densities on each side of the validity-area thresholds (1/64, 1/16, 1/4 of the sites), a forced validity plane, the
PFA_VDIV / PFA_VCOMPACT / PFA_*_TMA_M overrides, and codon shards shorter than one codon column.  The grids depend on the
number of SMs, so the strings hold for a B200 with 148 SMs only."""
import numpy as np
import pytest

import polyfasta_b200 as pf

pytestmark = pytest.mark.gpu

SMS = 148

# (case id, rows, sites, populations, a gap in every k-th site (0: none), force_validity, environment)
CASES = [
    ("n300", 300, 3000, 1, 0, False, {}),
    ("n384", 384, 3000, 1, 0, False, {}),
    ("n385", 385, 3000, 1, 0, False, {}),
    ("n1000", 1000, 3000, 1, 0, False, {}),
    ("n1280", 1280, 3000, 1, 0, False, {}),
    ("n1281", 1281, 3000, 1, 0, False, {}),
    ("n2000", 2000, 3000, 1, 0, False, {}),
    ("n10000", 10000, 900, 1, 0, False, {}),
    ("n13000", 13000, 303, 1, 0, False, {}),
    ("n21000", 21000, 240, 1, 0, False, {}),
    ("n300_k2", 300, 3000, 2, 0, False, {}),
    ("n385_k2", 385, 3000, 2, 0, False, {}),
    ("n1280_k2", 1280, 3000, 2, 0, False, {}),
    ("n1281_k2", 1281, 3000, 2, 0, False, {}),
    ("n2000_k2", 2000, 3000, 2, 0, False, {}),
    ("n10000_k2", 10000, 900, 2, 0, False, {}),
    ("n13000_k2", 13000, 303, 2, 0, False, {}),
    ("n21000_k2", 21000, 240, 2, 0, False, {}),
    ("n2000_gap1in70", 2000, 6720, 1, 70, False, {}),
    ("n2000_gap1in60", 2000, 6720, 1, 60, False, {}),
    ("n2000_gap1in17", 2000, 6720, 1, 17, False, {}),
    ("n2000_gap1in15", 2000, 6720, 1, 15, False, {}),
    ("n2000_gap1in5", 2000, 6720, 1, 5, False, {}),
    ("n2000_gap1in3", 2000, 6720, 1, 3, False, {}),
    ("n2000_gap1in70_k2", 2000, 6720, 2, 70, False, {}),
    ("n2000_gap1in3_k2", 2000, 6720, 2, 3, False, {}),
    ("n10000_gap1in20", 10000, 1200, 1, 20, False, {}),
    ("n10000_gap1in20_k2", 10000, 1200, 2, 20, False, {}),
    ("n300_gap1in20", 300, 3000, 1, 20, False, {}),
    ("n1000_gap1in20", 1000, 3000, 1, 20, False, {}),
    ("n300_force", 300, 3000, 1, 0, True, {}),
    ("n1000_force", 1000, 3000, 1, 0, True, {}),
    ("n2000_force", 2000, 3000, 1, 0, True, {}),
    ("n10000_force_k2", 10000, 900, 2, 0, True, {}),
    ("n2000_gap1in70_vdiv2", 2000, 6720, 1, 70, False, {"PFA_VDIV": "2"}),
    ("n2000_gap1in70_vcompact0", 2000, 6720, 1, 70, False, {"PFA_VCOMPACT": "0"}),
    ("n2000_m3", 2000, 3000, 1, 0, False, {"PFA_SITE_TMA_M": "3", "PFA_CDS_TMA_M": "3"}),
    ("n2000_gap1in70_m3", 2000, 6720, 1, 70, False, {"PFA_SITE_TMA_M": "3", "PFA_CDS_TMA_M": "3"}),
    ("n300_L1", 300, 1, 1, 0, False, {}),
    ("n300_L2_k2", 300, 2, 2, 0, False, {}),
    ("n2000_L1", 2000, 1, 1, 0, False, {}),
    ("n2000_L2", 2000, 2, 1, 0, False, {}),
    ("n2000_L2_gap", 2000, 2, 1, 1, False, {}),
]

EXPECTED = {
    'n300': (
        'pfa_site_scan_tma_kernel<LPS=1,ITER=3,HAS_V=0,MULTI=0> grid=2 block=512 passes_per_slot=3 v_records_per_slot=0 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=2,ITER=2,HAS_V=0,MULTI=0,NT=512> grid=2 passes_per_slot=3 v_records_per_slot=0 planes=pool'),
    'n384': (
        'pfa_site_scan_tma_kernel<LPS=1,ITER=3,HAS_V=0,MULTI=0> grid=2 block=512 passes_per_slot=3 v_records_per_slot=0 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=2,ITER=2,HAS_V=0,MULTI=0,NT=512> grid=2 passes_per_slot=3 v_records_per_slot=0 planes=pool'),
    'n385': (
        'pfa_site_scan_reg_kernel<LPS=1,ITER=4,HAS_V=0,MULTI=0> grid=12 block=256 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=2,ITER=2,HAS_V=0,MULTI=0,NT=512> grid=2 passes_per_slot=2 v_records_per_slot=0 planes=pool'),
    'n1000': (
        'pfa_site_scan_reg_kernel<LPS=2,ITER=4,HAS_V=0,MULTI=0> grid=24 block=256 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=4,ITER=2,HAS_V=0,MULTI=0,NT=512> grid=4 passes_per_slot=2 v_records_per_slot=0 planes=pool'),
    'n1280': (
        'pfa_site_scan_reg_kernel<LPS=2,ITER=5,HAS_V=0,MULTI=0> grid=24 block=256 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=8,ITER=2,HAS_V=0,MULTI=0,NT=512> grid=6 passes_per_slot=3 v_records_per_slot=0 planes=pool'),
    'n1281': (
        'pfa_site_scan_tma_kernel<LPS=4,ITER=3,HAS_V=0,MULTI=0> grid=8 block=512 passes_per_slot=3 v_records_per_slot=0 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=8,ITER=2,HAS_V=0,MULTI=0,NT=512> grid=6 passes_per_slot=3 v_records_per_slot=0 planes=pool'),
    'n2000': (
        'pfa_site_scan_tma_kernel<LPS=4,ITER=4,HAS_V=0,MULTI=0> grid=12 block=512 passes_per_slot=2 v_records_per_slot=0 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=8,ITER=2,HAS_V=0,MULTI=0,NT=512> grid=8 passes_per_slot=2 v_records_per_slot=0 planes=pool'),
    'n10000': (
        'pfa_site_scan_tma_kernel<LPS=16,ITER=5,HAS_V=0,MULTI=0> grid=29 block=512 passes_per_slot=1 v_records_per_slot=0 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=32,ITER=3,HAS_V=0,MULTI=0,NT=256> grid=19 passes_per_slot=2 v_records_per_slot=0 planes=pool'),
    'n13000': (
        'pfa_site_scan_tma_kernel<LPS=32,ITER=4,HAS_V=0,MULTI=0> grid=7 block=512 passes_per_slot=3 v_records_per_slot=0 planes=pool',
        'pfa_cds_scan_kernel<LPS=32,ITER=4,HAS_V=0,MULTI=0> grid=13 block=256 planes=pool'),
    'n21000': (
        'pfa_site_scan_kernel<LPS=32,ITER=6,HAS_V=0,MULTI=0> grid=30 block=256 planes=pool',
        'pfa_cds_scan_kernel<LPS=32,ITER=6,HAS_V=0,MULTI=0> grid=10 block=256 planes=pool'),
    'n300_k2': (
        'pfa_site_scan_tma_kernel<LPS=1,ITER=3,HAS_V=0,MULTI=1> grid=2 block=512 passes_per_slot=3 v_records_per_slot=0 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=2,ITER=2,HAS_V=0,MULTI=1,NT=512> grid=2 passes_per_slot=3 v_records_per_slot=0 planes=pool'),
    'n385_k2': (
        'pfa_site_scan_reg_kernel<LPS=1,ITER=4,HAS_V=0,MULTI=1> grid=12 block=256 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=2,ITER=2,HAS_V=0,MULTI=1,NT=512> grid=2 passes_per_slot=2 v_records_per_slot=0 planes=pool'),
    'n1280_k2': (
        'pfa_site_scan_reg_kernel<LPS=2,ITER=5,HAS_V=0,MULTI=1> grid=24 block=256 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=8,ITER=2,HAS_V=0,MULTI=1,NT=512> grid=6 passes_per_slot=3 v_records_per_slot=0 planes=pool'),
    'n1281_k2': (
        'pfa_site_scan_tma_kernel<LPS=4,ITER=3,HAS_V=0,MULTI=1> grid=8 block=512 passes_per_slot=3 v_records_per_slot=0 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=8,ITER=2,HAS_V=0,MULTI=1,NT=512> grid=6 passes_per_slot=3 v_records_per_slot=0 planes=pool'),
    'n2000_k2': (
        'pfa_site_scan_tma_kernel<LPS=4,ITER=4,HAS_V=0,MULTI=1> grid=12 block=512 passes_per_slot=2 v_records_per_slot=0 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=8,ITER=2,HAS_V=0,MULTI=1,NT=512> grid=8 passes_per_slot=2 v_records_per_slot=0 planes=pool'),
    'n10000_k2': (
        'pfa_site_scan_tma_kernel<LPS=16,ITER=5,HAS_V=0,MULTI=1> grid=29 block=512 passes_per_slot=1 v_records_per_slot=0 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=32,ITER=3,HAS_V=0,MULTI=1,NT=256> grid=19 passes_per_slot=2 v_records_per_slot=0 planes=pool'),
    'n13000_k2': (
        'pfa_site_scan_tma_kernel<LPS=32,ITER=4,HAS_V=0,MULTI=1> grid=7 block=512 passes_per_slot=3 v_records_per_slot=0 planes=pool',
        'pfa_cds_scan_kernel<LPS=32,ITER=4,HAS_V=0,MULTI=1> grid=13 block=256 planes=pool'),
    'n21000_k2': (
        'pfa_site_scan_kernel<LPS=32,ITER=6,HAS_V=0,MULTI=1> grid=30 block=256 planes=pool',
        'pfa_cds_scan_kernel<LPS=32,ITER=6,HAS_V=0,MULTI=1> grid=10 block=256 planes=pool'),
    'n2000_gap1in70': (
        'pfa_site_scan_tma_kernel<LPS=4,ITER=4,HAS_V=1,MULTI=0> grid=18 block=512 passes_per_slot=3 v_records_per_slot=6 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=8,ITER=2,HAS_V=1,MULTI=0,NT=512> grid=18 passes_per_slot=2 v_records_per_slot=3 planes=pool'),
    'n2000_gap1in60': (
        'pfa_site_scan_tma_kernel<LPS=4,ITER=4,HAS_V=1,MULTI=0> grid=18 block=512 passes_per_slot=3 v_records_per_slot=6 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=8,ITER=2,HAS_V=1,MULTI=0,NT=512> grid=35 passes_per_slot=1 v_records_per_slot=3 planes=pool'),
    'n2000_gap1in17': (
        'pfa_site_scan_tma_kernel<LPS=4,ITER=4,HAS_V=1,MULTI=0> grid=18 block=512 passes_per_slot=3 v_records_per_slot=6 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=8,ITER=2,HAS_V=1,MULTI=0,NT=512> grid=35 passes_per_slot=1 v_records_per_slot=3 planes=pool'),
    'n2000_gap1in15': (
        'pfa_site_scan_tma_kernel<LPS=4,ITER=4,HAS_V=1,MULTI=0> grid=27 block=512 passes_per_slot=2 v_records_per_slot=8 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=8,ITER=2,HAS_V=1,MULTI=0,NT=512> grid=35 passes_per_slot=1 v_records_per_slot=6 planes=pool'),
    'n2000_gap1in5': (
        'pfa_site_scan_tma_kernel<LPS=4,ITER=4,HAS_V=1,MULTI=0> grid=27 block=512 passes_per_slot=2 v_records_per_slot=8 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=8,ITER=2,HAS_V=1,MULTI=0,NT=512> grid=35 passes_per_slot=1 v_records_per_slot=6 planes=pool'),
    'n2000_gap1in3': (
        'pfa_site_scan_tma_kernel<LPS=4,ITER=4,HAS_V=1,MULTI=0> grid=27 block=512 passes_per_slot=2 v_records_per_slot=16 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=8,ITER=2,HAS_V=1,MULTI=0,NT=512> grid=35 passes_per_slot=1 v_records_per_slot=12 planes=pool'),
    'n2000_gap1in70_k2': (
        'pfa_site_scan_tma_kernel<LPS=4,ITER=4,HAS_V=1,MULTI=1> grid=18 block=512 passes_per_slot=3 v_records_per_slot=6 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=8,ITER=2,HAS_V=1,MULTI=1,NT=512> grid=18 passes_per_slot=2 v_records_per_slot=3 planes=pool'),
    'n2000_gap1in3_k2': (
        'pfa_site_scan_tma_kernel<LPS=4,ITER=4,HAS_V=1,MULTI=1> grid=27 block=512 passes_per_slot=2 v_records_per_slot=16 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=8,ITER=2,HAS_V=1,MULTI=1,NT=512> grid=35 passes_per_slot=1 v_records_per_slot=12 planes=pool'),
    'n10000_gap1in20': (
        'pfa_site_scan_tma_kernel<LPS=16,ITER=5,HAS_V=1,MULTI=0> grid=19 block=512 passes_per_slot=2 v_records_per_slot=1 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=32,ITER=3,HAS_V=1,MULTI=0,NT=256> grid=17 passes_per_slot=3 v_records_per_slot=3 planes=pool'),
    'n10000_gap1in20_k2': (
        'pfa_site_scan_tma_kernel<LPS=16,ITER=5,HAS_V=1,MULTI=1> grid=19 block=512 passes_per_slot=2 v_records_per_slot=1 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=32,ITER=3,HAS_V=1,MULTI=1,NT=256> grid=17 passes_per_slot=3 v_records_per_slot=3 planes=pool'),
    'n300_gap1in20': (
        'pfa_site_scan_tma_kernel<LPS=1,ITER=3,HAS_V=1,MULTI=0> grid=2 block=512 passes_per_slot=3 v_records_per_slot=96 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=2,ITER=2,HAS_V=1,MULTI=0,NT=512> grid=2 passes_per_slot=2 v_records_per_slot=96 planes=pool'),
    'n1000_gap1in20': (
        'pfa_site_scan_reg_kernel<LPS=2,ITER=4,HAS_V=1,MULTI=0> grid=24 block=256 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=4,ITER=2,HAS_V=1,MULTI=0,NT=512> grid=8 passes_per_slot=1 v_records_per_slot=6 planes=pool'),
    'n300_force': (
        'pfa_site_scan_tma_kernel<LPS=1,ITER=3,HAS_V=1,MULTI=0> grid=2 block=512 passes_per_slot=3 v_records_per_slot=96 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=2,ITER=2,HAS_V=1,MULTI=0,NT=512> grid=2 passes_per_slot=2 v_records_per_slot=96 planes=pool'),
    'n1000_force': (
        'pfa_site_scan_reg_kernel<LPS=2,ITER=4,HAS_V=1,MULTI=0> grid=24 block=256 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=4,ITER=2,HAS_V=1,MULTI=0,NT=512> grid=8 passes_per_slot=1 v_records_per_slot=24 planes=pool'),
    'n2000_force': (
        'pfa_site_scan_tma_kernel<LPS=4,ITER=4,HAS_V=1,MULTI=0> grid=12 block=512 passes_per_slot=2 v_records_per_slot=16 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=8,ITER=2,HAS_V=1,MULTI=0,NT=512> grid=16 passes_per_slot=1 v_records_per_slot=12 planes=pool'),
    'n10000_force_k2': (
        'pfa_site_scan_tma_kernel<LPS=16,ITER=5,HAS_V=1,MULTI=1> grid=29 block=512 passes_per_slot=1 v_records_per_slot=2 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=32,ITER=3,HAS_V=1,MULTI=1,NT=256> grid=19 passes_per_slot=2 v_records_per_slot=6 planes=pool'),
    'n2000_gap1in70_vdiv2': (
        'pfa_site_scan_tma_kernel<LPS=4,ITER=4,HAS_V=1,MULTI=0> grid=27 block=512 passes_per_slot=2 v_records_per_slot=8 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=8,ITER=2,HAS_V=1,MULTI=0,NT=512> grid=35 passes_per_slot=1 v_records_per_slot=6 planes=pool'),
    'n2000_gap1in70_vcompact0': (
        'pfa_site_scan_tma_kernel<LPS=4,ITER=4,HAS_V=1,MULTI=0> grid=27 block=512 passes_per_slot=2 v_records_per_slot=16 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=8,ITER=2,HAS_V=1,MULTI=0,NT=512> grid=35 passes_per_slot=1 v_records_per_slot=12 planes=pool'),
    'n2000_m3': (
        'pfa_site_scan_tma_kernel<LPS=4,ITER=4,HAS_V=0,MULTI=0> grid=8 block=512 passes_per_slot=3 v_records_per_slot=0 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=8,ITER=2,HAS_V=0,MULTI=0,NT=512> grid=8 passes_per_slot=2 v_records_per_slot=0 planes=pool'),
    'n2000_gap1in70_m3': (
        'pfa_site_scan_tma_kernel<LPS=4,ITER=4,HAS_V=1,MULTI=0> grid=18 block=512 passes_per_slot=3 v_records_per_slot=6 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=8,ITER=2,HAS_V=1,MULTI=0,NT=512> grid=18 passes_per_slot=2 v_records_per_slot=3 planes=pool'),
    'n300_L1': (
        'pfa_site_scan_tma_kernel<LPS=1,ITER=3,HAS_V=0,MULTI=0> grid=1 block=512 passes_per_slot=3 v_records_per_slot=0 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=2,ITER=2,HAS_V=0,MULTI=0,NT=512> grid=1 passes_per_slot=3 v_records_per_slot=0 planes=pool'),
    'n300_L2_k2': (
        'pfa_site_scan_tma_kernel<LPS=1,ITER=3,HAS_V=0,MULTI=1> grid=1 block=512 passes_per_slot=3 v_records_per_slot=0 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=2,ITER=2,HAS_V=0,MULTI=1,NT=512> grid=1 passes_per_slot=3 v_records_per_slot=0 planes=pool'),
    'n2000_L1': (
        'pfa_site_scan_tma_kernel<LPS=4,ITER=4,HAS_V=0,MULTI=0> grid=1 block=512 passes_per_slot=2 v_records_per_slot=0 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=8,ITER=2,HAS_V=0,MULTI=0,NT=512> grid=1 passes_per_slot=2 v_records_per_slot=0 planes=pool'),
    'n2000_L2': (
        'pfa_site_scan_tma_kernel<LPS=4,ITER=4,HAS_V=0,MULTI=0> grid=1 block=512 passes_per_slot=2 v_records_per_slot=0 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=8,ITER=2,HAS_V=0,MULTI=0,NT=512> grid=1 passes_per_slot=2 v_records_per_slot=0 planes=pool'),
    'n2000_L2_gap': (
        'pfa_site_scan_tma_kernel<LPS=4,ITER=4,HAS_V=1,MULTI=0> grid=1 block=512 passes_per_slot=2 v_records_per_slot=16 planes=pool',
        'pfa_cds_scan_tma_kernel<LPS=8,ITER=2,HAS_V=1,MULTI=0,NT=512> grid=1 passes_per_slot=1 v_records_per_slot=12 planes=pool'),
}


def kernels(ctx, n, L, npops, gap_every, force):
    """(ctx.last_kernel after site_stats, after cds_stats) of one seeded alignment"""
    rng = np.random.default_rng(n * 7919 + L)
    text = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, (n, L))]
    if gap_every:
        text[rng.integers(0, n, (L + gap_every - 1) // gap_every), np.arange(0, L, gap_every)] = ord("-")
    aln = pf.Alignment.from_rows(ctx, text)
    try:
        aln.set_pops([list(range(n)), list(range(0, n, 2))][:npops])
        if force:
            aln.force_validity()
        aln.site_stats()
        site = ctx.last_kernel
        aln.cds_stats()
        return site, ctx.last_kernel
    finally:
        aln.free()


@pytest.fixture(scope="module")
def ctx():
    import torch
    if torch.cuda.get_device_properties(0).multi_processor_count != SMS:
        pytest.skip("the recorded grids are for a GPU with %d SMs" % SMS)
    return pf.default_context(0)


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_launch_plan(ctx, monkeypatch, case):
    cid, n, L, npops, gap_every, force, env = case
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    assert kernels(ctx, n, L, npops, gap_every, force) == EXPECTED[cid]
