"""Golden vectors from the REFERENCE's own max-clique finder: `FMC::maxCliqueHeu` (third_party/fast_max-clique_finder of
swarm_outlier_rejection), compiled from its sources in place by oracle/ref_build/Makefile into oracle/_ref/libfmc_ref.so and
called through oracle/fmc_ref.py.  Stores the graphs and the clique (vertex list in the library's order, and the size it
returns) the library finds on each, as tests/golden/ref_fmc.npz:

  * pin_*   the 423 graphs of tests/test_oracle_pins.py::test_max_clique_restatement_equals_the_references_own_library --
            degenerate ones, random ones of every density, PCM-shaped ones -- each as the packed upper triangle of its
            adjacency matrix;
  * pcm_<n>_<seed>   the clique on the oracle's consistency graph of every synth.pcm_edges case of tests/test_gpu_pcm.py.

    python tests/golden/make_ref_fmc.py            (needs the reference tree to build the library; the .npz travels without it)
    python tests/golden/make_ref_fmc.py --check    compare the committed fixture with the library instead of writing it
"""
import multiprocessing as mp
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from omniswarm_b200 import synth                     # noqa: E402
from oracle import fmc_ref                           # noqa: E402
from oracle import pcm_ref as pr                     # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_fmc.npz")
THRES, POS, ANG = 15.0, 1e-4, 1e-5                   # tests/test_gpu_pcm.py
PCM_CASES = [(60, 0.3, 0, 3), (150, 0.5, 1, 3), (33, 0.0, 2, 3), (1, 0.0, 3, 0), (1500, 0.4, 5, 0)]   # n, outliers, seed, other


def pin_graphs():
    rng = np.random.default_rng(1)
    graphs = [np.zeros((1, 1), np.uint8), np.zeros((7, 7), np.uint8), (1 - np.eye(9, dtype=np.uint8))]
    for _ in range(400):
        n = int(rng.integers(2, 60))
        a = np.triu(rng.uniform(size=(n, n)) < rng.uniform(0.02, 0.95), 1)
        graphs.append((a | a.T).astype(np.uint8))
    # PCM-shaped graphs: a big consistent block plus scattered false links
    for _ in range(20):
        n = int(rng.integers(30, 120)); k = int(0.5 * n)
        a = np.zeros((n, n), bool)
        idx = rng.choice(n, k, replace=False)
        a[np.ix_(idx, idx)] = True
        a |= np.triu(rng.uniform(size=(n, n)) < 0.05, 1); a = np.triu(a, 1); a = a | a.T
        graphs.append(a.astype(np.uint8))
    return graphs


def _smd_rows(args):
    edges, rows = args
    out = []
    for i in rows:
        row = np.full(len(edges), np.inf)
        for j in range(i):
            s = pr.pair_smd(edges[i], edges[j], POS, ANG)
            if s is not None:
                row[j] = s
        out.append(row)
    return out


def consistency_matrix(edges, pool):
    """pcm_ref.consistency_matrix, rows spread over processes (the 1500-edge case takes minutes on one core)"""
    n = len(edges)
    chunks = [list(range(r, n, 64)) for r in range(64)]
    smd = np.full((n, n), np.inf)
    for rows, res in zip(chunks, pool.map(_smd_rows, [(edges, c) for c in chunks])):
        for i, row in zip(rows, res):
            smd[i, :i] = row[:i]
    smd = np.minimum(smd, smd.T)
    return (smd < THRES).astype(np.uint8), smd


def generate():
    assert fmc_ref.build(), "oracle/_ref/libfmc_ref.so could not be built (the reference tree is needed)"
    graphs = pin_graphs()
    out = {"pin_n": np.array([a.shape[0] for a in graphs], np.int32)}
    tri, cliques, sizes = [], [], []
    for a in graphs:
        tri.append(np.packbits(a[np.triu_indices(a.shape[0], 1)]))
        c, s = fmc_ref.max_clique_heu(a)
        cliques.append(np.array(c, np.int32)); sizes.append(s)
    out["pin_adj_bytes"] = np.array([len(t) for t in tri], np.int32)
    out["pin_adj"] = np.concatenate(tri)
    out["pin_clique_len"] = np.array([len(c) for c in cliques], np.int32)
    out["pin_clique"] = np.concatenate(cliques)
    out["pin_size"] = np.array(sizes, np.int32)
    with mp.Pool() as pool:
        for n, outl, seed, other in PCM_CASES:
            adj, smd = consistency_matrix(synth.pcm_edges(n, outl, seed, other_pair=other), pool)
            fin = np.isfinite(smd)
            assert not fin.any() or np.abs(smd[fin] - THRES).min() > 1e-6, "a pair lies on the threshold"
            out[f"pcm_{n}_{seed}"] = np.array(fmc_ref.max_clique_heu(adj)[0], np.int32)
    return out


def main(check=False):
    out = generate()
    if check:
        z = np.load(OUT)
        assert sorted(z.files) == sorted(out) and all(np.array_equal(z[k], v) for k, v in out.items()), \
            "tests/golden/ref_fmc.npz differs from the reference's library"
        print("ref_fmc.npz matches the reference's library")
        return
    np.savez_compressed(OUT, **out)
    print("wrote", OUT, {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main(check="--check" in sys.argv[1:])
