"""GPU parity of the PCM outlier rejection (osb_pcm: pairwise consistency + FMC::maxCliqueHeu) against oracle/pcm_ref.py, and
against the clique the REFERENCE's own maxCliqueHeu finds on the oracle's consistency graph (tests/golden/ref_fmc.npz, written
by tests/golden/make_ref_fmc.py from the library oracle/ref_build compiles from its sources)."""
import os

import numpy as np
import pytest

from conftest import GOLDEN
from omniswarm_b200 import synth, host
from oracle import pcm_ref as pr

pytestmark = pytest.mark.gpu
THRES, POS, ANG = 15.0, 1e-4, 1e-5
REF_FMC = np.load(os.path.join(GOLDEN, "ref_fmc.npz"))


@pytest.mark.parametrize("n,out,seed", [(60, 0.3, 0), (150, 0.5, 1), (33, 0.0, 2), (1, 0.0, 3)])
def test_pcm_matches_oracle(gpu, n, out, seed):
    edges = synth.pcm_edges(n, out, seed, other_pair=3 if n > 1 else 0)
    clique, adj, smd = host.pcm_outlier_rejection(edges, THRES, POS, ANG, want_matrices=True)
    radj, rsmd = pr.consistency_matrix(edges, THRES, POS, ANG)
    fin = np.isfinite(rsmd)
    assert np.array_equal(np.isfinite(smd), fin)
    assert np.allclose(smd[fin], rsmd[fin], rtol=1e-9, atol=1e-12)
    margin = np.abs(rsmd[fin] - THRES).min() if fin.any() else 1.0
    assert margin > 1e-6, "test data has a pair on the threshold"
    assert np.array_equal(adj, radj)                                  # consistency graph bit-exact
    rclique, rsize = pr.max_clique_heu(radj)
    assert clique.tolist() == rclique                                 # same vertices in maxCliqueHeu's order
    assert clique.tolist() == REF_FMC[f"pcm_{n}_{seed}"].tolist()     # ... and in the order of the REFERENCE's own library
    if n > 30:
        assert all(edges[i]["inlier"] for i in clique) and len(clique) >= 0.4 * sum(e["inlier"] for e in edges)


def test_pcm_large_graph_bitmatrix_in_global_memory(gpu):
    """1500 loops: the bit matrix (1500 x 47 words = 282 KB) no longer fits shared memory, the clique kernel reads it
    from L2.  The oracle's O(n^2) Python consistency loop is too slow here, so: a random sample of pairs against the oracle,
    symmetry / zero diagonal as properties, and the clique against the oracle heuristic run on the DEVICE adjacency."""
    n = 1500
    edges = synth.pcm_edges(n, 0.4, 5)
    clique, adj, smd = host.pcm_outlier_rejection(edges, THRES, POS, ANG, want_matrices=True)
    assert np.array_equal(adj, adj.T) and adj.diagonal().sum() == 0
    rng = np.random.default_rng(0)
    for _ in range(300):
        i, j = sorted(rng.choice(n, 2, replace=False))[::-1]
        s = pr.pair_smd(edges[i], edges[j], POS, ANG)
        assert np.isclose(smd[i, j], s, rtol=1e-9) and np.isclose(smd[j, i], s, rtol=1e-9)
        assert adj[i, j] == (s < THRES)
    rclique, _ = pr.max_clique_heu(adj)
    assert clique.tolist() == rclique
    assert clique.tolist() == REF_FMC[f"pcm_{n}_5"].tolist()          # the reference's library on the oracle's graph
    assert all(edges[i]["inlier"] for i in clique) and len(clique) > 100


def test_pcm_argument_errors(gpu):
    with pytest.raises(host._l.OsbError):
        host.pcm_outlier_rejection(synth.pcm_edges(2, 0.0, 0) * 2100, THRES, POS, ANG)       # > 4096 edges
