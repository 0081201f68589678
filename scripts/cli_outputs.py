"""Print the drop-in CLI's output for a fixed list of commands: every mode (default, --cds, --window, --cds --window, --dxy,
--dxy --window), each with -f, -d, --pipe and --out, on tests/golden/example_theta_0.01 and the edge-case fixtures.  Two
checkouts that compute the same thing print byte-identical text; compare them with cmp.
usage: python scripts/cli_outputs.py OUT_FILE"""
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# paths as the CLI sees them: it runs in a scratch directory that links the fixtures as ./golden, so that the printed paths are
# the same for every checkout
LOCI = "golden/example_theta_0.01"
FILES = [LOCI + "/file1.fa", LOCI + "/file7.fa"] + ["golden/edge/" + f for f in sorted(os.listdir(os.path.join(ROOT, "tests", "golden", "edge")))]
WIN = ["--window", "300", "--step", "150"]   # multiples of 3 (--cds --window); the loci have 1,000 columns
MODES = [[], ["--cds"], WIN, ["--cds"] + WIN, ["--dxy"], ["--dxy"] + WIN]
POPS = [["-p", "indiv1,nobody,indiv2", "--jc"], []]


def commands():
    for mode in MODES:
        for pops in POPS:
            if "--dxy" in mode and not pops:
                continue   # --dxy needs -p
            yield ["-f"] + FILES + mode + pops, None
            yield ["-d", LOCI] + mode + pops, None
            yield ["--pipe"] + mode + pops, LOCI + "/file1.fa"
            yield ["-d", LOCI, "--out", "out.csv"] + mode + pops, None


def main(path):
    env = dict(os.environ, PYTHONPATH=ROOT)
    with open(path, "w") as log, tempfile.TemporaryDirectory() as tmp:
        os.symlink(os.path.join(ROOT, "tests", "golden"), os.path.join(tmp, "golden"))
        out = os.path.join(tmp, "out.csv")
        for argv, stdin in commands():
            data = open(os.path.join(tmp, stdin), "rb").read() if stdin else b""
            p = subprocess.run([sys.executable, "-m", "polyfasta_b200.cli"] + argv, input=data, capture_output=True, cwd=tmp, env=env)
            log.write("### %s\nexit %d\n%s" % (" ".join(argv), p.returncode, p.stdout.decode("utf-8", "replace")))
            if os.path.exists(out):
                log.write("--- out.csv\n" + open(out).read())
                os.remove(out)
    print("wrote", path)


if __name__ == "__main__":
    main(sys.argv[1])
