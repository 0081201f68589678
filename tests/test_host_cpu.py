"""CPU-only checks of the product's host side: the C-ABI library loads and exports every declared symbol, the
FASTA parser follows the reference's readfasta on the golden corner cases, and compute fails loudly without a GPU."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import polyfasta_b200 as pf
from polyfasta_b200 import _lib
from conftest import GOLDEN, ROOT, load_golden


def test_library_exports_every_declared_symbol():
    L = _lib.lib()
    with open(os.path.join(ROOT, "include", "polyfasta_b200.h")) as f:
        header = f.read()
    declared = set(re.findall(r"\b(pfa_[a-z0-9_]+)\s*\(", header))
    declared -= {"pfa_final_in", "pfa_final_out"}
    assert declared == set(_lib.EXPORTS)
    for name in sorted(declared):
        assert hasattr(L, name), name
    assert L.pfa_version() >= 100


def test_ingest_cases_match_reference():
    for name, rec in load_golden("ingest_cases.json").items():
        if "ret" in rec:
            with pytest.raises(pf.NotFasta):
                pf.Fasta.from_bytes(rec["text"])
            continue
        f = pf.Fasta.from_bytes(rec["text"])
        assert f.headers == rec["keys"], name
        assert [f.row(i) for i in range(f.nseq)] == rec["seqs"], name
        lens = {len(s) for s in rec["seqs"]}
        assert f.seqlen == (lens.pop() if len(lens) == 1 else -1), name
        f.close()


def test_readfasta_mirror(tmp_path, capsys):
    p = tmp_path / "x.fa"
    p.write_text(">a\nacgt\n>b\nAC-N\n")
    assert pf.readfasta(str(p), False) == {"a": "ACGT", "b": "AC-N"}
    q = tmp_path / "bad.fa"
    q.write_text("no header here\n")
    assert pf.readfasta(str(q), False) == 1
    assert capsys.readouterr().out == f"# file {q} is not FASTA!\n"


def test_example_files_parse():
    kat = load_golden("kat_examples.json")
    for fn, entry in kat.items():
        f = pf.Fasta.from_file(os.path.join(GOLDEN, "example_theta_0.01", fn))
        assert f.headers == entry["headers"] and f.seqlen == entry["seqlen"] and f.nseq == 20


def test_non_ascii_sequence_rejected():
    with pytest.raises(ValueError):
        pf.Fasta.from_bytes(">a\nAC\xc3\xa9T\n".encode("latin-1"))


def test_codon_tables_match_reference():
    """the product's own classifier tables (host side of K4) against the reference's exhaustive vectors"""
    L = _lib.lib()
    g = load_golden("codon_classifier.json")
    bases = "ACGT"
    idx = lambda c: 16 * bases.index(c[0]) + 4 * bases.index(c[1]) + bases.index(c[2])  # noqa: E731
    for c, v in g["syn3"].items():
        assert L.pfa_codon_syn3(idx(c)) == v, c
    stops = {"TAA", "TAG", "TGA"}
    for key, (S, N) in g["pairs"].items():
        a, b = key[:3], key[3:]
        lab = L.pfa_codon_pair_labels(idx(a), idx(b))
        if a in stops or b in stops:
            continue
        got_s = [i for i in range(3) if (lab >> (2 * i)) & 3 == 1]
        got_n = [i for i in range(3) if (lab >> (2 * i)) & 3 == 2]
        assert (got_s, got_n) == (S, N), key
    for cods, S, N in g["multi"]:
        m = 0
        for c in cods:
            if c not in stops:
                m |= 1 << idx(c)
        lab = L.pfa_codon_set_labels(m)
        got_s = [i for i in range(3) if (lab >> (2 * i)) & 3 == 1]
        got_n = [i for i in range(3) if (lab >> (2 * i)) & 3 == 2]
        assert (got_s, got_n) == (S, N), cods


def test_compute_fails_loudly_without_gpu():
    if _lib.lib().pfa_device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(pf.PolyFastaError):
        pf.Context(0)
    with pytest.raises(pf.PolyFastaError):
        pf.getvarsites({"a": "ACGT", "b": "ACGA"}, 4)


def test_cli_argument_errors():
    env = dict(os.environ, PYTHONPATH=ROOT)
    cmd = [sys.executable, os.path.join(ROOT, "PolyFastA.py")]
    p = subprocess.run(cmd + ["-f", "a.fa", "-d", "somedir"], capture_output=True, text=True, env=env)
    assert p.returncode == 2 and "Run with either --file/-f or --dir/-d, but not both" in p.stderr
    p = subprocess.run(cmd + ["-h"], capture_output=True, text=True, env=env)
    assert p.returncode == 0
    for flag in ("--file", "--dir", "--pops", "--out", "--pipe", "--cds", "--silent", "--name", "--jc"):
        assert flag in p.stdout
    p = subprocess.run(cmd, input="n\n", capture_output=True, text=True, env=env)
    assert p.returncode == 2 and "Both --file/-f and --dir/-d were not found." in p.stdout


def test_synth_twin_closed_form_small():
    """numpy twin: the closed-form counts equal a brute-force recount of the generated text (oracle)"""
    from oracle import c_oracle as co
    from polyfasta_b200 import synth
    for n, L in [(2, 200), (3, 500), (20, 3000), (101, 2000), (257, 700)]:
        mat = synth.text_matrix(11, n, L, 200000, 100000)
        want = co.site_stats(mat)
        got = synth.expected_site_stats(11, n, L, 200000, 100000)
        assert (got["S"], got["H"], got["sfs"]) == (want["S"], want["H"], want["sfs"]), (n, L)


def _pack_ref(row):
    lut = np.full(256, 255, np.uint8)
    for i, ch in enumerate(b"ACTG"):
        lut[ch] = i
        lut[ch | 32] = i
    c = lut[row]
    dirty = bool((c == 255).any())
    c = np.concatenate([c & 3, np.zeros((-len(c)) % 4, np.uint8)]).reshape(-1, 4)
    return (c[:, 0] | (c[:, 1] << 2) | (c[:, 2] << 4) | (c[:, 3] << 6)).astype(np.uint8), dirty


def test_host_packer_variants_agree_with_numpy():
    """the ingest's host packer (4 bases per byte, A0 C1 T2 G3, either case; anything else marks the row dirty):
    scalar, AVX2 and AVX-512 variants against a numpy restatement, all tail lengths"""
    from polyfasta_b200 import _lib
    L = _lib.lib()
    rng = np.random.default_rng(3)
    txt = np.frombuffer(b"ACGTacgt", dtype=np.uint8)[rng.integers(0, 8, 1500)].copy()
    ran = 0
    for variant in (0, 1, 2, 3):
        for cols in list(range(0, 140)) + [255, 256, 257, 1000, 1499]:
            dst = np.full(cols // 4 + 2, 0xEE, np.uint8)
            r = L.pfa_host_pack2(txt.ctypes.data, cols, dst.ctypes.data, variant)
            if r == -2:
                break  # this CPU lacks the instruction set
            want, _ = _pack_ref(txt[:cols])
            assert r == 0 and np.array_equal(dst[: (cols + 3) // 4], want), (variant, cols)
            assert dst[(cols + 3) // 4] == 0xEE                      # nothing written past the row
        else:
            ran += 1
            for pos in (0, 3, 63, 64, 65, 127, 128, 200, 299):
                for bad in b"N-nRr?.* \x00\x01\xc1\xe1!@[`{":
                    t = txt[:300].copy()
                    t[pos] = bad
                    dst = np.zeros(80, np.uint8)
                    assert L.pfa_host_pack2(t.ctypes.data, 300, dst.ctypes.data, variant) == 1, (variant, pos, bad)
    assert ran >= 2  # the scalar variant and the dispatcher always run


def test_host_packer_matrix_threads():
    from polyfasta_b200 import _lib
    L = _lib.lib()
    rng = np.random.default_rng(4)
    n, cols, ld = 37, 1001, 1100
    txt = np.frombuffer(b"ACGTacgt", dtype=np.uint8)[rng.integers(0, 8, (n, ld))].copy()
    txt[5, 1000] = ord("N")   # inside the packed range: one dirty row
    txt[7, 1001] = ord("N")   # outside it: ignored
    ldp = 256
    dst = np.zeros((n, ldp), np.uint8)
    for threads in (1, 3, 0):
        assert L.pfa_host_pack2_rows(txt.ctypes.data, n, cols, ld, dst.ctypes.data, ldp, threads) == 1
        for r in range(n):
            want, dirty = _pack_ref(txt[r, :cols])
            assert dirty == (r == 5)
            assert np.array_equal(dst[r, : (cols + 3) // 4], want)


def _fasta_dump(f):
    return f.headers, [f.row(i) for i in range(f.nseq)], f.seqlen


@pytest.mark.parametrize("segments", [2, 3, 5, 16])
def test_segmented_parse_equals_sequential(tmp_path, monkeypatch, segments):
    """large FASTA files are scanned in segments by several threads and compacted in place (no copy into a matrix); the
    result must be what the sequential scan gives: the golden ingest cases of the reference plus a random torture set
    (wrapped lines, duplicate and empty headers, text before the first header, blank lines, trailing blanks, CRLF)"""
    rng = np.random.default_rng(segments)
    cases = {k: v["text"] for k, v in load_golden("ingest_cases.json").items()}
    for i in range(60):
        parts = []
        if rng.random() < 0.3:
            parts.append("junk before\n")
        for r in range(int(rng.integers(1, 9))):
            name = ["a", "b", "c", "", "a b", "dup"][int(rng.integers(0, 6))]
            parts.append(">" + name + ["", " ", "\t"][int(rng.integers(0, 3))] + "\n")
            for _ in range(int(rng.integers(0, 5))):
                line = "".join("ACGTacgtN-"[int(x)] for x in rng.integers(0, 10, int(rng.integers(0, 30))))
                parts.append(line + ["", "  ", "\n"][int(rng.integers(0, 3))] + "\n")
        text = "".join(parts)
        if rng.random() < 0.2:
            text = text.replace("\n", "\r\n")
        cases["rand%d" % i] = text
    # regularly wrapped records (what a mapped file keeps as (first byte, line width, gap) and gathers on access)
    for i, (w, nl) in enumerate(((60, "\n"), (7, "\n"), (13, "\r\n"), (1, "\n"), (80, " \n"))):
        rows = ["".join("ACGTN-acgt"[int(x)] for x in rng.integers(0, 10, 157 + 3 * r)) for r in range(5)]
        cases["wrap%d" % i] = "".join(">r%d%s" % (r, nl) + "".join(row[o:o + w] + nl for o in range(0, len(row), w)) for r, row in enumerate(rows))
    for name, text in cases.items():
        monkeypatch.delenv("PFA_PARSE_SEGMENTS", raising=False)
        monkeypatch.delenv("PFA_BIG_FILE_MIN", raising=False)
        try:
            want = _fasta_dump(pf.Fasta.from_bytes(text))
        except pf.NotFasta:
            want = "not fasta"
        monkeypatch.setenv("PFA_PARSE_SEGMENTS", str(segments))
        try:
            got = _fasta_dump(pf.Fasta.from_bytes(text))
        except pf.NotFasta:
            got = "not fasta"
        assert got == want, name
        # the same through the big-file path: parallel read, segmented scan, rows compacted inside the file buffer
        p = tmp_path / "case.fa"
        p.write_bytes(text.encode("utf-8", "surrogateescape") if isinstance(text, str) else text)
        monkeypatch.setenv("PFA_BIG_FILE_MIN", "1")
        for mapped in ("1", "0"):   # private file mapping (copy-on-write), or a buffer filled with pread
            monkeypatch.setenv("PFA_PARSE_MMAP", mapped)
            try:
                got = _fasta_dump(pf.Fasta.from_file(str(p)))
            except pf.NotFasta:
                got = "not fasta"
            assert got == want, (name, mapped)


def test_host_packer_with_validity_bitmap():
    """gaps, N and ? are packed too (codes A0 C1 G2 T3 / '-'0 'N'1 '?'2 + one validity bit per base); any other byte marks
    the row dirty.  Scalar and AVX-512 VBMI variants against a numpy restatement."""
    L = _lib.lib()
    rng = np.random.default_rng(12)
    code = {65: 0, 67: 1, 71: 2, 84: 3, 97: 0, 99: 1, 103: 2, 116: 3, 45: 0, 78: 1, 110: 1, 63: 2}
    ok = {65, 67, 71, 84, 97, 99, 103, 116}
    alpha = np.frombuffer(b"ACGTacgtNn-?", dtype=np.uint8)
    ran = 0
    for variant in (0, 1, 4):
        for cols in list(range(0, 150)) + [511, 512, 1000]:
            for kind in range(3):
                row = alpha[rng.integers(0, 8 if kind == 0 else 12, cols)].copy()
                if kind == 2 and cols:
                    row[rng.integers(0, cols)] = rng.choice([82, 0x80, 0xC1, 32, 42, 0])
                c = np.array([code.get(int(x), 3) for x in row], np.uint8)
                v = np.array([int(x) in ok for x in row], np.uint8)
                flags = (0 if v.all() else 1) | (0 if all(int(x) in code for x in row) else 2)
                cp = np.concatenate([c, np.zeros((-cols) % 4, np.uint8)]).reshape(-1, 4)
                vp = np.concatenate([v, np.zeros((-cols) % 8, np.uint8)]).reshape(-1, 8)
                wc = (cp[:, 0] | (cp[:, 1] << 2) | (cp[:, 2] << 4) | (cp[:, 3] << 6)).astype(np.uint8)
                wv = np.packbits(vp, axis=1, bitorder="little").reshape(-1)
                codes = np.full(cols // 4 + 2, 0xEE, np.uint8)
                valid = np.full(cols // 8 + 2, 0xEE, np.uint8)
                r = L.pfa_host_pack3(row.ctypes.data, cols, codes.ctypes.data, valid.ctypes.data, variant)
                if r == -2:
                    break
                assert r == flags, (variant, cols, kind)
                if not flags & 2:
                    assert np.array_equal(codes[: (cols + 3) // 4], wc) and np.array_equal(valid[: (cols + 7) // 8], wv), (variant, cols)
                assert codes[(cols + 3) // 4] == 0xEE and valid[(cols + 7) // 8] == 0xEE
            else:
                continue
            break
        else:
            ran += 1
    assert ran >= 2


def test_bench_reference_arm_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours) prints ONE JSON line with the contract's keys;
    tiny sizes here so that it runs in seconds"""
    import json
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                        "--n", "200", "--sites", "20000", "--cpu-sample-sites", "2000"], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "bases/s" and d["higher_is_better"] is True and d["steps"] == 2
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["gpu_launches"] == 0
    assert "workload" in d["config"]


def test_bench_dump_outputs_helpers(tmp_path, monkeypatch):
    """--dump-outputs: float64 files, integers only where float64 holds them exactly, and for c5 every locus in locus order
    or, beyond the size limit, the same seeded sample of loci on every run"""
    import types
    import bench

    class FakeBatch:
        def __init__(self, ids):
            self.ids = ids

        def result(self, j, pop, want_sfs=False):
            i = self.ids[j]
            return {"S": i, "H": 3 * i, "sfs": [i % 7] * 10, "poly": (0, 0, 0, "NA") if i % 5 == 0 else (i, 0.5 * i, 0.25 * i, -1.5)}

    args, env = types.SimpleNamespace(n=20, loci=25), types.SimpleNamespace(world=1, rank=0)
    batches = [(FakeBatch(list(range(10))), list(range(10))), (FakeBatch(list(range(10, 25))), list(range(10, 25)))]
    out = bench.c5_outputs(args, env, batches)
    assert out["locus"].tolist() == list(range(25)) and out["sfs"].shape == (25, 10) and out["H"].tolist() == [3 * i for i in range(25)]
    assert np.isnan(out["tajimas_d"][[0, 5]]).all() and out["tajimas_d"][1] == -1.5
    bench.dump_outputs(str(tmp_path / "d"), out)
    for name, a in out.items():
        got = np.load(tmp_path / "d" / (name + ".npy"))
        assert got.dtype == np.float64 and np.array_equal(got, a, equal_nan=True)
    with pytest.raises(SystemExit):
        bench.dump_outputs(str(tmp_path / "e"), {"x": np.array([2 ** 53 + 1])})
    monkeypatch.setattr(bench, "DUMP_LIMIT", 8 * (6 + 10) * 7)   # room for 7 of the 25 loci
    picks = [bench.c5_outputs(args, env, batches)["locus"].tolist() for _ in range(2)]
    assert picks[0] == picks[1] and len(picks[0]) == 7 and picks[0] == sorted(picks[0])
    with pytest.raises(SystemExit):
        bench.dump_outputs(str(tmp_path / "f"), out)


@pytest.mark.parametrize("mapped", ["1", "0"])
def test_big_file_path_refuses_non_ascii_sequence_bytes(tmp_path, monkeypatch, mapped):
    """bytes >= 0x80 in SEQUENCE lines are refused on every parse path (headers may hold them)"""
    monkeypatch.setenv("PFA_BIG_FILE_MIN", "1")
    monkeypatch.setenv("PFA_PARSE_MMAP", mapped)
    ok = tmp_path / "ok.fa"
    ok.write_bytes(b">caf\xc3\xa9\nACGT\nACGT\n>b\nACGT\nACGT\n")
    f = pf.Fasta.from_file(str(ok))
    assert f.nseq == 2 and f.seqlen == 8 and f.row(0) == "ACGTACGT"
    for body in (b">a\nAC\xc3\xa9T\n>b\nACGGT\n", b">a\nACGT\nAC\xe9T\nAC\n>b\nACGT\nACGT\nAC\n"):
        bad = tmp_path / "bad.fa"
        bad.write_bytes(body)
        with pytest.raises(ValueError):
            pf.Fasta.from_file(str(bad))


def test_layout_export_import(tmp_path, monkeypatch):
    """column-sharded runs parse a large file ONCE: the rank that parsed exports where the rows are, the others map the file and
    adopt that layout without scanning it (pfa_fasta_export_layout / pfa_fasta_import_layout).  Rows on one line and rows
    wrapped at a fixed width, headers of different lengths; a small file (not mapped in place) has no layout to export."""
    import numpy as np
    from polyfasta_b200 import api
    rng = np.random.default_rng(5)
    n, L = 37, 5000
    rows = ["".join(rng.choice(list("ACGTacgtN-"), L)) for _ in range(n)]
    for wrap in (0, 60):
        path = tmp_path / ("big%d.fa" % wrap)
        with open(path, "w") as f:
            for i, r in enumerate(rows):
                f.write(">pop%d_row%d%s\n" % (i % 2, i, "x" * (i % 5)))
                if wrap:
                    f.write("\n".join(r[o:o + wrap] for o in range(0, L, wrap)) + "\n")
                else:
                    f.write(r + "\n")
        small = api.Fasta.from_file(str(path))
        assert small.export_layout() is None
        monkeypatch.setenv("PFA_BIG_FILE_MIN", "1")
        big = api.Fasta.from_file(str(path))
        blob = big.export_layout()
        assert blob is not None and len(blob) < 40 * n + sum(len(h) for h in big.headers) + 100
        twin = api.Fasta.from_layout(str(path), blob)
        monkeypatch.delenv("PFA_BIG_FILE_MIN")
        assert twin.headers == big.headers == small.headers and (twin.nseq, twin.seqlen) == (n, L)
        for i in (0, 1, n // 2, n - 1):
            assert twin.row(i) == small.row(i) == rows[i].upper()
        with pytest.raises((OSError, Exception)):
            api.Fasta.from_layout(str(path) + ".missing", blob)
        for x in (small, big, twin):
            x.close()


@pytest.mark.parametrize("workload,sample", [("c4", "500"), ("c3", "600"), ("c5", "4")])
def test_bench_reference_arm_prints_one_json_line(workload, sample):
    """`bench.py --impl reference` (the CPU arm the driver times beside the GPU arm) for every workload: one JSON line with the
    contract's keys, no GPU needed"""
    import json
    import subprocess
    import sys
    from conftest import ROOT
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", workload, "--steps", "1", "--warmup", "0",
                        "--cpu-sample-sites", sample], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr
    lines = [ln for ln in p.stdout.strip().split("\n") if ln]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["value"] > 0 and d["unit"] == "bases/s" and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "port" and d["e2e"]["h2d_bytes_per_step"] == 0 and "workload" in d["config"]
