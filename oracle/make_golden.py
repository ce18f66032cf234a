"""Generate the committed fixtures under tests/golden/ (run in the build container).

    python -m oracle.make_golden           # everything (needs the reference)
    python -m oracle.make_golden layers    # layer_cases.npz only, from the stored graph

Two kinds of vectors:

* ``ref_*.npz`` -- outputs of the REFERENCE's own functions (``/root/reference/lib_new/graph.py``
  and ``coarsening.py`` imported unmodified through ``oracle/ref_loader.py``) on seeded inputs.
  They pin the oracle's restatement and the package's host code, and travel to the GPU box
  where the reference does not exist.
* ``layer_cases.npz`` -- outputs of the oracle (fp64 truth and fp32 as-run) for the layer
  variants, forward and backward; they pin the oracle against accidental change and give the
  GPU tests fixed known answers.  (The TF-executed layer results themselves are pinned by no
  reference artefact: parity unpinned at that boundary.)
"""
import contextlib
import hashlib
import io
import os

import numpy as np
import scipy.sparse as sp

from oracle import layers_np as O
from oracle import ref_loader

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def csr_dict(prefix, m):
    m = sp.csr_matrix(m)
    m.sort_indices()
    return {prefix + "_indptr": m.indptr.astype(np.int32), prefix + "_indices": m.indices.astype(np.int32),
            prefix + "_data": m.data, prefix + "_shape": np.array(m.shape, np.int64)}


def ref_graph(graph, coarsening, levels):
    """SURVEY 8(d) synthetic graph, built with the reference's functions only."""
    rng = np.random.RandomState(1234)
    z = rng.randn(360, 3).astype(np.float32)
    dist, idx = graph.distance_sklearn_metrics(z, k=8, metric="euclidean")
    A = graph.adjacency(dist, idx)
    np.random.seed(1234)
    A = graph.replace_random_edges(A, 0.01)
    with contextlib.redirect_stdout(io.StringIO()):
        graphs, perm = coarsening.coarsen(A, levels=levels, self_connections=False)
    L = [graph.laplacian(g, normalized=True) for g in graphs]
    return A, graphs, perm, L


def main():
    os.makedirs(OUT, exist_ok=True)
    graph, coarsening = ref_loader.load()

    # ---- A. graphs, permutation, Laplacians, rescaled Laplacians (reference) -------------------
    for levels in (1, 4):
        A, graphs, perm, L = ref_graph(graph, coarsening, levels)
        d = dict(perm=np.asarray(perm, np.int64), sizes=np.array([l.shape[0] for l in L], np.int64),
                 perm_sha1=np.array(hashlib.sha1(np.asarray(perm, np.int64).tobytes()).hexdigest()[:16]))
        d.update(csr_dict("A", A))
        for i, l in enumerate(L):
            d.update(csr_dict("L%d" % i, l))
            d.update(csr_dict("Lt%d" % i, graph.rescale_L(sp.csr_matrix(l, copy=True), lmax=2)))
        np.savez_compressed(os.path.join(OUT, "ref_graph_l%d.npz" % levels), **d)
        if levels == 4:
            L4, perm4 = L, perm

    # ---- B. the reference's own Chebyshev recursion (graph.chebyshev) --------------------------
    rng = np.random.RandomState(11)
    d = {}
    for name, lvl, ncol, K in (("a", 0, 24, 5), ("b", 0, 7, 2), ("c", 0, 5, 1), ("d", 2, 8, 25), ("e", 4, 33, 10)):
        Lt = graph.rescale_L(sp.csr_matrix(L4[lvl], copy=True), lmax=2)
        X = rng.randn(Lt.shape[0], ncol).astype(np.float32)
        d["X_" + name] = X
        d["meta_" + name] = np.array([lvl, K], np.int64)
        d["Xt_" + name] = graph.chebyshev(Lt, X, K)
    np.savez_compressed(os.path.join(OUT, "ref_chebyshev.npz"), **d)

    # ---- C. Fourier basis (graph.fourier) and D. perm_data_3d ----------------------------------
    lamb, U = graph.fourier(L4[2])
    x = np.random.RandomState(12).randn(3, 360, 4).astype(np.float32)
    np.savez_compressed(os.path.join(OUT, "ref_fourier_perm.npz"), lamb=lamb, U=U, x=x,
                        x_perm=coarsening.perm_data_3d(x, perm4),
                        kat_parents0=np.array([4, 1, 1, 2, 2, 3, 0, 0, 3]), kat_parents1=np.array([2, 1, 0, 1, 0]))

    layer_cases(L4)


def layer_cases(L4):
    """E. layer cases from the oracle.  Each case draws ``B`` windows and keeps the first ``nb`` of them (the draws, and so
    the stored vectors, are those of the full-batch cases the file first held; fewer windows keep it under 1 MB).  Only
    what the tests read is stored: the spectral cases' backward reference is recomputed from the stored basis, and the
    pre-activation of the pooling checks comes from the oracle at test time."""
    rng = np.random.RandomState(7)
    cases = {}

    def add(name, lvl, B, nb, Fin, Fout, K, p, filt, brelu):
        L = L4[lvl]
        M = L.shape[0]
        x = rng.randn(B, M, Fin).astype(np.float32)[:nb]
        if filt == "fourier":
            W = (rng.randn(M, Fout, Fin) * 0.2).astype(np.float32)
        else:
            W = (rng.randn(Fin * K, Fout) * 0.2).astype(np.float32)
        b = (0.2 + 0.1 * rng.randn(*((M, Fout) if brelu == "b2relu" else (Fout,)))).astype(np.float32)
        dy = rng.randn(B, -(-M // p), Fout).astype(np.float32)[:nb]
        pr = [dict(W=W, b=b, K=K, p=p)]
        c = dict(x=x, W=W, b=b, dy=dy, meta=np.array([lvl, nb, Fin, Fout, K, p], np.int64),
                 kind=np.array(filt + "/" + brelu))
        for tag, dt in (("64", np.float64), ("32", np.float32)):
            y, tr = O.conv_stack(x, [L], pr, filter=filt, brelu=brelu, dtype=dt, keep=True)
            if tag == "32":  # the as-run fp32 oracle only documents the noise floor
                c.update(y32=y)
            elif filt == "fourier":
                c.update(y64=y, Ut=O.fourier_basis(L, np.float32))
            else:
                dx, g = O.conv_stack_bwd(tr, [L], pr, dy, filter=filt, brelu=brelu, dtype=dt, first_needs_dx=True)
                c.update(y64=y, dx64=dx, dW64=g[0]["dW"], db64=g[0]["db"], argmax=tr[0]["argmax"])
        for k, v in c.items():
            cases[name + "." + k] = v

    add("cheb_l2_k5_p4_b1", 2, 4, 2, 32, 32, 5, 4, "chebyshev5", "b1relu")
    add("cheb_l0_k5_p4_b1", 0, 2, 1, 15, 32, 5, 4, "chebyshev5", "b1relu")
    add("cheb_l0_k3_p1_b2", 0, 2, 1, 15, 32, 3, 1, "chebyshev5", "b2relu")
    add("cheb_l3_k1_p2_b1", 3, 3, 3, 5, 8, 1, 2, "chebyshev5", "b1relu")
    add("cheb_l2_k2_p2_b2", 2, 3, 3, 6, 16, 2, 2, "chebyshev2", "b2relu")
    add("cheb_l4_k20_p1_b1", 4, 2, 2, 3, 7, 20, 1, "chebyshev5", "b1relu")
    add("four_l2_p4_b1", 2, 3, 3, 8, 16, 0, 4, "fourier", "b1relu")
    add("four_l3_p1_b2", 3, 2, 2, 5, 6, 0, 1, "fourier", "b2relu")
    np.savez_compressed(os.path.join(OUT, "layer_cases.npz"), **cases)
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


def stored_laplacians():
    """The Laplacians of ``ref_graph_l4.npz`` (section A's output), so that the layer cases can be rebuilt without the
    reference."""
    z = np.load(os.path.join(OUT, "ref_graph_l4.npz"))
    return [sp.csr_matrix((z["L%d_data" % i], z["L%d_indices" % i], z["L%d_indptr" % i]), shape=tuple(z["L%d_shape" % i]))
            for i in range(len(z["sizes"]))]


if __name__ == "__main__":
    import sys

    if sys.argv[1:] == ["layers"]:
        layer_cases(stored_laplacians())
    else:
        main()
