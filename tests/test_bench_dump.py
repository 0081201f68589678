"""bench.py --dump-outputs on the GPU: the arrays the timed path computed in its last step, written as float64 .npy files,
equal the generator's closed form / the C oracle on the same seeded inputs and do not depend on the number of steps;
--steps sets the number of timed steps."""
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from conftest import ROOT
from oracle import c_oracle as co
from polyfasta_b200 import api, synth

pytestmark = pytest.mark.gpu


def _bench(out, *argv):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--warmup", "1", "--no-cpu", "--no-e2e",
                        "--dump-outputs", str(out)] + list(argv), capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-3000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    files = {f[:-len(".npy")]: np.load(out / f) for f in os.listdir(out)}
    assert all(a.dtype == np.float64 for a in files.values())
    return json.loads(lines[0]), files


def test_c4_dump_and_steps(tmp_path):
    n, L = 300, 40_000
    runs = {k: _bench(tmp_path / ("steps%d" % k), "--n", str(n), "--sites", str(L), "--steps", str(k)) for k in (2, 5)}
    want = synth.expected_site_stats(bench.SEED, n, L, bench.P_SEG_PPM, bench.TRI_PPM)
    for k, (d, files) in runs.items():
        assert d["steps"] == k and sorted(files) == ["site_stats"]
        assert files["site_stats"].tolist() == [want["S"], want["H"]] + want["sfs"]
    # the timed region holds exactly --steps steps: the same launches per step for 2 and 5 steps
    l2, l5 = runs[2][0]["gpu_launches"], runs[5][0]["gpu_launches"]
    assert l2 > 0 and l2 % 2 == 0 and l5 == l2 // 2 * 5


def test_c3_dump(tmp_path):
    n, L = 200, 3000
    _, files = _bench(tmp_path / "c3", "--workload", "c3", "--n", str(n), "--sites", str(L), "--steps", "2")
    text = co.synth_text(bench.C3_SEED, n, L, bench.P_SEG_PPM, bench.TRI_PPM)
    pops = [list(range(n // 2)), list(range(n // 2, n))]
    want_site, want_cds = [], []
    for rows in pops:
        s, c = co.site_stats(text, rows), co.cds_stats(text, rows)
        want_site += [s["S"], s["H"]] + s["sfs"]
        row = [c[k] for k in ("nstops", "missing", "S_s", "H_s", "S_n", "H_n")] + [0] * 65
        for length, v in c["sum3_by_len"].items():
            row[6 + length] = v
        want_cds.append(row)
    assert files["site_stats"].tolist() == want_site
    assert files["cds_stats"].shape == (2, api.PFA_CDS_LEN) and files["cds_stats"].tolist() == want_cds


def test_c5_dump(tmp_path):
    n, L, loci = 20, 300, 30
    _, files = _bench(tmp_path / "c5", "--workload", "c5", "--n", str(n), "--sites", str(L), "--loci", str(loci), "--steps", "2")
    assert files["locus"].tolist() == list(range(loci)) and files["sfs"].shape == (loci, n // 2)
    for i in range(loci):
        want = synth.expected_site_stats(bench.C5_SEED + i, n, L, bench.P_SEG_PPM, bench.TRI_PPM)
        assert (files["S"][i], files["H"][i], files["sfs"][i].tolist()) == (want["S"], want["H"], want["sfs"]), i
        _, pi, theta, D = co.finalize(n, want["S"], want["H"], L, True)
        assert math.isclose(files["pi_site"][i], pi, rel_tol=1e-12) and math.isclose(files["theta_site"][i], theta, rel_tol=1e-12)
        assert math.isnan(files["tajimas_d"][i]) if D == "NA" else math.isclose(files["tajimas_d"][i], D, rel_tol=1e-9, abs_tol=1e-12)
