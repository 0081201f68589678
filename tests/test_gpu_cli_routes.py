"""The column-sharded route of the CLI on one GPU: two ranks share device 0 and sum their shards' vectors on the host (gloo),
so every statistic's sharded path runs where only one GPU is present.  Rank 0 must print exactly what one process prints."""
import io
import os
import socket
from contextlib import redirect_stdout

import numpy as np
import pytest

from test_gpu_parity import _random_text

pytestmark = pytest.mark.gpu

W, STEP = "900", "600"   # multiples of 3 (--cds --window); the window at 14,400 straddles the shard boundary at 15,000


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, port, argv_list, q):
    os.environ.update({"RANK": str(rank), "WORLD_SIZE": "2", "LOCAL_RANK": "0", "MASTER_ADDR": "127.0.0.1",
                       "MASTER_PORT": str(port), "POLYFASTA_HOST_ALLREDUCE": "1"})
    from polyfasta_b200 import cli
    cli.SHARD_MIN_BYTES = 1_000_000
    outs = []
    for argv in argv_list:
        buf = io.StringIO()
        with redirect_stdout(buf):
            cli.main(argv)
        outs.append(buf.getvalue())
    q.put((rank, outs))


@pytest.fixture(scope="module")
def big_fasta(tmp_path_factory):
    """60 rows of 30,001 columns (not a multiple of 3) in three populations, about 1.8 MB: column-sharded over two ranks"""
    rng = np.random.default_rng(31)
    n, L = 60, 30001
    text = _random_text(rng, n, L, p_junk=0.002)
    path = tmp_path_factory.mktemp("routes") / "big.fa"
    with open(path, "wb") as f:
        for i in range(n):
            f.write((">pop%d_%d\n" % (i % 3, i)).encode() + text[i].tobytes() + b"\n")
    return str(path)


def test_sharded_rows_equal_one_process(big_fasta):
    import torch.multiprocessing as mp
    from polyfasta_b200 import cli
    base = ["-f", big_fasta, "-p", "pop0,nobody,pop1,pop2", "--jc"]
    argvs = [base, base + ["--cds"], base + ["--window", W, "--step", STEP], base + ["--cds", "--window", W, "--step", STEP],
             base + ["--dxy"], base + ["--dxy", "--window", W, "--step", STEP]]
    want = []
    for argv in argvs:
        buf = io.StringIO()
        with redirect_stdout(buf):
            cli.main(argv)
        want.append(buf.getvalue())
    for out in want:
        assert "# Pop nobody string was not found" in out
    assert want[0].count("\n") == 5 and want[4].count("\n") == 5   # header, note, three populations / three pairs
    mpc = mp.get_context("spawn")
    q = mpc.Queue()
    port = _free_port()
    procs = [mpc.Process(target=_worker, args=(r, port, argvs, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=600) for _ in range(2))
    for p in procs:
        p.join(60)
    for argv, w, g in zip(argvs, want, got[0]):
        assert g == w, argv
    assert all(o == "" for o in got[1])
