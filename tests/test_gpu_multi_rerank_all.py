"""The sharded `rerank_all` on two GPUs (tests/dist_rerank_all_check.py under torchrun; skipped below two GPUs; the
same sequencing is covered on CPU by tests/test_dist_rerank_all_gloo.py), and the leaf-partitioned index on one GPU."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def test_sharded_rerank_all_on_two_gpus():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "dist_rerank_all_check.py")],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0 and "DIST RERANK_ALL CHECK OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_rerank_all_on_a_doc_ids_index_equals_the_plain_index(gauss):
    """Rows stored in a permuted order with their document ids in `doc_ids` (a leaf-partitioned shard's layout): the
    same CSR as the plain index, bit for bit - ids mapped before the sort, so ties are ordered by document id."""
    from gpu_util import dev
    from mevi_b200.rerank import ClusterIndex, ClusterReranker

    dec = gauss.load("beam100_labels.npy")
    perm = np.random.RandomState(3).permutation(gauss.n)
    X = gauss.X[perm].copy()
    X[: gauss.n // 10] = gauss.X[perm[gauss.n // 10 : 2 * (gauss.n // 10)]]  # duplicated rows: ties between documents
    Xo = gauss.X.copy()
    Xo[perm[: gauss.n // 10]] = X[: gauss.n // 10]
    off, ids, sc = ClusterReranker(dev(Xo), ClusterIndex.from_codes(gauss.codes, gauss.K), mode="stream").rerank_all(gauss.Q, dec)
    part = ClusterIndex.from_codes(gauss.codes[perm], gauss.K, doc_ids=torch.from_numpy(perm))
    off2, ids2, sc2 = ClusterReranker(dev(X), part, mode="stream").rerank_all(gauss.Q, dec)
    assert torch.equal(off, off2) and torch.equal(ids, ids2) and torch.equal(sc.view(torch.int32), sc2.view(torch.int32))
    assert int(off[-1]) > 0
