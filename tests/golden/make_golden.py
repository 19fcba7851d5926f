"""Generate the golden fixtures under tests/golden/ from the reference's own checkpoints.

usage: python tests/golden/make_golden.py <checkout of BGU-CS-VIL/DPMMSubClusters.jl>
The outputs are committed, so that the tests need no copy of the reference.

Sources (data files only, no reference source code is copied):
  examples/save_load_model/2d1ksample.npy + checkpoint__50.jld2   (NIW, D=2, K=5)
  test/save_load_test/mnm_data.npy       + checkpoint_20.jld2     (multinomial, D=100, K=2)

The JLD2 checkpoints store `group.labels`, `group.labels_subcluster` (Int64, uncompressed) and,
inside every local_cluster, the cluster / left / right sufficient statistics that the reference
computed with create_suff_stats_dict_worker (src/local_clusters_actions.jl:149-169,
src/priors/niw.jl:42-51, src/priors/multinomial_prior.jl:27-32).  We locate the stored statistics
by value (they sit uncompressed in the file) and save the STORED bytes as the golden answer.
"""
import os
import sys
import numpy as np

REF = sys.argv[1] if len(sys.argv) > 1 else None
OUT = os.path.dirname(os.path.abspath(__file__))


def _find_f64(blob, value, rtol=1e-9):
    """Return (offset, stored_value) of the stored float64 closest to `value` (any byte alignment)."""
    best = None
    for a in range(8):
        n = (len(blob) - a) // 8
        v = np.frombuffer(blob, dtype="<f8", count=n, offset=a)
        with np.errstate(all="ignore"):
            err = np.abs(v - value) / max(abs(value), 1e-300)
        err = np.where(np.isfinite(err), err, np.inf)
        i = int(np.argmin(err))
        if err[i] <= rtol and (best is None or err[i] < best[2]):
            best = (a + 8 * i, float(v[i]), float(err[i]))
    if best is None:
        raise RuntimeError(f"value {value!r} not found in checkpoint")
    return best[0], best[1]


def _find_f32_vector(blob, vec):
    pat = np.asarray(vec, dtype="<f4").tobytes()
    off = blob.find(pat)
    if off < 0:
        raise RuntimeError("float32 vector not found byte-exact in checkpoint")
    return off


def make_niw():
    x = np.load(f"{REF}/examples/save_load_model/2d1ksample.npy")  # (1000, 2) f64, N x D
    blob = open(f"{REF}/examples/save_load_model/checkpoint__50.jld2", "rb").read()
    labels = np.frombuffer(blob, dtype="<i8", count=1000, offset=5957).copy()
    sub = np.frombuffer(blob, dtype="<i8", count=1000, offset=14015).copy()
    assert labels.min() == 1 and labels.max() == 5 and set(np.unique(sub)) == {1, 2}
    # The stored statistics of THIS checkpoint reproduce from the Float64 npy values (it was written
    # by a reference version that had not yet rounded the points to Float32), accumulated in
    # Float64 (niw.jl:46-49).  The fixture therefore keeps x in Float64, D x N (utils.jl:5-14);
    # a Float32 consumer (the GPU path) agrees to ~1e-7 relative, inside the 1e-4 tolerance.
    pts = np.ascontiguousarray(x.T)  # D x N, float64
    K, D = 5, 2
    counts = np.zeros((K, 3), np.int64)
    sum_x = np.zeros((K, 3, D))
    sum_xx = np.zeros((K, 3, D, D))
    offsets = []
    for k in range(K):
        for s, mask in enumerate([labels == k + 1,
                                  (labels == k + 1) & (sub == 1),
                                  (labels == k + 1) & (sub == 2)]):
            p = pts[:, mask].astype(np.float64)
            counts[k, s] = p.shape[1]
            sx = p.sum(axis=1)
            S = p @ p.T
            S = 0.5 * (S + S.T)
            for d in range(D):
                off, val = _find_f64(blob, sx[d])
                sum_x[k, s, d] = val
                offsets.append(off)
            for i in range(D):
                for j in range(D):
                    off, val = _find_f64(blob, S[i, j])
                    sum_xx[k, s, i, j] = val
                    offsets.append(off)
    # The checkpoint also stores every cluster's POSTERIOR hyper-parameters (cluster_parameters.posterior_hyperparams,
    # ds.jl:13-18) next to the statistics: m' and psi' of calc_posterior (niw.jl:20-31) under the example's prior
    # niw_hyperparams(1.0, [0,0], 5.0, I) (examples/save_load_model/params_2d.jl).  Located by value like the
    # statistics; the STORED bytes are the golden answer for calc_posterior.
    post_m = np.zeros((K, 3, D))
    post_psi = np.zeros((K, 3, D, D))
    kappa0, nu0 = 1.0, 5.0
    for k in range(K):
        for s in range(3):
            N = float(counts[k, s])
            kp, nup = kappa0 + N, nu0 + N
            m = sum_x[k, s] / kp
            psi = (nu0 * np.eye(D) - kp * np.outer(m, m) + sum_xx[k, s]) / nup
            for d in range(D):
                post_m[k, s, d] = _find_f64(blob, m[d], rtol=1e-11)[1]
            for i in range(D):
                for j in range(D):
                    post_psi[k, s, i, j] = _find_f64(blob, psi[i, j], rtol=1e-11)[1]
    np.savez_compressed(f"{OUT}/niw_2d1k_checkpoint50.npz", x=pts, labels=labels, sublabels=sub,
                        counts=counts, sum_x=sum_x, sum_xx=sum_xx, post_m=post_m, post_psi=post_psi,
                        prior=np.array([kappa0, nu0]), found_offsets=np.asarray(offsets, np.int64))
    print("niw: counts\n", counts)


def make_mnm():
    m = np.load(f"{REF}/test/save_load_test/mnm_data.npy")  # (1000, 100) f32
    blob = open(f"{REF}/test/save_load_test/checkpoint_20.jld2", "rb").read()
    labels = np.frombuffer(blob, dtype="<i8", count=1000, offset=6150).copy()
    sub = np.frombuffer(blob, dtype="<i8", count=1000, offset=14208).copy()
    pts = m.astype(np.float32).T.copy()  # D x N
    K, D = 2, 100
    counts = np.zeros((K, 3), np.int64)
    sum_x = np.zeros((K, 3, D), np.float32)
    offsets = []
    for k in range(K):
        for s, mask in enumerate([labels == k + 1,
                                  (labels == k + 1) & (sub == 1),
                                  (labels == k + 1) & (sub == 2)]):
            p = pts[:, mask]
            counts[k, s] = p.shape[1]
            sx = p.sum(axis=1, dtype=np.float32)
            off = _find_f32_vector(blob, sx)
            offsets.append(off)
            sum_x[k, s] = np.frombuffer(blob, dtype="<f4", count=D, offset=off)
    # posterior alpha' = alpha + sum x (multinomial_prior.jl:16-21) under multinomial_hyper(ones(Float32,100))
    # (test/save_load_test/multinomial_params.jl): stored as Float32 vectors, found byte-exact
    post_alpha = np.zeros((K, 3, D), np.float32)
    for k in range(K):
        for s in range(3):
            off = _find_f32_vector(blob, np.ones(D, np.float32) + sum_x[k, s])
            post_alpha[k, s] = np.frombuffer(blob, dtype="<f4", count=D, offset=off)
    # generate_mnmm_data invariants of the reference's own data file (data_generators.jl:59-72): integral counts,
    # every point is `trials` draws
    assert np.array_equal(m, np.round(m)) and m.min() >= 0
    np.savez_compressed(f"{OUT}/mnm_1k_checkpoint20.npz", x=pts, labels=labels, sublabels=sub,
                        counts=counts, sum_x=sum_x, post_alpha=post_alpha, row_sums=m.sum(axis=1).astype(np.float32),
                        found_offsets=np.asarray(offsets, np.int64))
    print("mnm: counts\n", counts, "\noffsets", offsets)


if __name__ == "__main__":
    if REF is None or not os.path.isdir(REF):
        sys.exit("usage: make_golden.py <checkout of BGU-CS-VIL/DPMMSubClusters.jl>")
    make_niw()
    make_mnm()
