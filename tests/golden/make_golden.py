"""Generate the committed golden fixtures from the UNMODIFIED reference (oracle/_ref).

Run in the build container only (needs /root/reference to have been built by oracle/build_ref.sh):

    python tests/golden/make_golden.py

MLPG-family vectors come from the reference itself (nnmnkwii.paramgen / nnmnkwii.autograd /
nnmnkwii.metrics / nnmnkwii.util.linalg imported from oracle/_ref).  DTW vectors CANNOT come from
the reference (fastdtw is not installable here - "parity unpinned"); they come from the literal
pure-Python restatement oracle/fastdtw_py.py with the reference's own ``melcd`` as ``dist`` and are
labelled ``restated`` in the file name.
"""
import os
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
HERE = os.path.dirname(os.path.abspath(__file__))

import oracle  # noqa: E402
from oracle import fastdtw_py  # noqa: E402


def windows_set():
    # tests/test_paramgen.py:4-28 of the reference
    return [
        [(0, 0, np.array([1.0]))],
        [(0, 0, np.array([1.0])), (1, 1, np.array([-0.5, 0.0, 0.5]))],
        [(0, 0, np.array([1.0])), (1, 1, np.array([-0.5, 0.0, 0.5])), (1, 1, np.array([1.0, -2.0, 1.0]))],
        [(0, 0, np.array([1.0])), (2, 2, np.array([1.0, -8.0, 0.0, 8.0, -1.0]) / 12.0),
         (2, 2, np.array([-1.0, 16.0, -30.0, 16.0, -1.0]) / 12.0)],
    ]


def main():
    oracle.import_reference()
    import torch
    from nnmnkwii import autograd as AF
    from nnmnkwii import paramgen as G
    from nnmnkwii.metrics import melcd
    from nnmnkwii.paramgen._bandmat import linalg as bla
    from nnmnkwii.util.linalg import cholesky_inv_banded

    out = {}
    rng = np.random.default_rng(20260923)
    for wi, ws in enumerate(windows_set()):
        nw = len(ws)
        for dt in (np.float32, np.float64):
            for T in (1, 2, 5, 12):
                sd = 2
                key = "w%d_%s_T%d" % (wi, np.dtype(dt).name, T)
                m = rng.random((T, sd * nw)).astype(dt)
                v = (rng.random((T, sd * nw)) + 0.05).astype(dt)
                go = rng.standard_normal((T, sd)).astype(np.float32)
                out[key + "_means"] = m
                out[key + "_vars"] = v
                out[key + "_go"] = go
                out[key + "_y"] = G.mlpg(m, v, ws)
                out[key + "_y1d"] = G.mlpg(m, v[0].copy(), ws)
                out[key + "_grad"] = G.mlpg_grad(m, v, ws, go)
        for T in (3, 10):
            out["w%d_R_T%d" % (wi, T)] = G.unit_variance_mlpg_matrix(ws, T)
    ws = windows_set()[2]
    out["w2_R_T40"] = G.unit_variance_mlpg_matrix(ws, 40)

    # config 1 of BASELINE.json: T=100, static_dim=59, 3 windows, diag variance (inputs re-derived
    # from the seed in the tests; only the reference outputs are stored).
    r1 = np.random.default_rng(1234)
    m = r1.random((100, 177)).astype(np.float32)
    v = (r1.random((100, 177)) + 0.1).astype(np.float32)
    out["cfg1_y"] = G.mlpg(m, v, ws)
    out["cfg1_y_unitvar"] = G.mlpg(m, np.ones(177, dtype=np.float32), ws)

    # autograd: UnitVarianceMLPG fwd + bwd (T=16, sd=3, B=2) through the reference's Function
    T, sd, B = 16, 3, 2
    R = torch.from_numpy(G.unit_variance_mlpg_matrix(ws, T))
    mu = torch.from_numpy(rng.standard_normal((B, T, sd * 3)).astype(np.float32)).requires_grad_(True)
    y = AF.unit_variance_mlpg(R, mu)
    wgt = torch.from_numpy(rng.standard_normal((B, T, sd)).astype(np.float32))
    (y * wgt).sum().backward()
    out["uv_means"] = mu.detach().numpy()
    out["uv_wgt"] = wgt.numpy()
    out["uv_y"] = y.detach().numpy()
    out["uv_grad"] = mu.grad.numpy()
    # autograd.MLPG fwd + bwd
    mu2 = torch.from_numpy(rng.random((T, sd * 3)).astype(np.float32)).requires_grad_(True)
    var2 = torch.from_numpy((rng.random((T, sd * 3)) + 0.1).astype(np.float32))
    y2 = AF.mlpg(mu2, var2, ws)
    w2 = torch.from_numpy(rng.standard_normal((T, sd)).astype(np.float32))
    (y2 * w2).sum().backward()
    out["ag_means"], out["ag_vars"], out["ag_wgt"] = mu2.detach().numpy(), var2.numpy(), w2.numpy()
    out["ag_y"], out["ag_grad"] = y2.detach().numpy(), mu2.grad.numpy()

    # bandmat known answers (reference tests/bandmat/test_linalg.py:100-114): lower band storage
    ab = np.array([[4.0, 4.0, 4.0, 4.0], [1.0, 0.5, 0.2, -1.0]])
    out["chol4_ab"] = ab
    out["chol4_c"] = bla._cholesky_banded(ab.copy(), lower=True)
    # cholesky_inv_banded (tests/test_util.py:62-81)
    P = G.build_win_mats(ws, 10)
    import scipy.linalg
    from nnmnkwii.paramgen import _bandmat as bm
    Pb = bm.zeros(2, 2, 10)
    for wm in P:
        bm.dot_mm_plus_equals(wm.T, wm, target_bm=Pb)
    L = scipy.linalg.cholesky(Pb.full(), lower=True)
    out["cib_L"] = L
    out["cib_Pinv"] = cholesky_inv_banded(L, width=3)

    # melcd known values
    xs = rng.standard_normal((6, 25))
    ys = rng.standard_normal((6, 25))
    out["melcd_x"], out["melcd_y"] = xs, ys
    out["melcd_rows"] = np.array([melcd(a, b) for a, b in zip(xs, ys)])
    out["melcd_2d"] = np.array(melcd(xs, ys))
    out["melcd_len"] = np.array(melcd(xs[None], ys[None], lengths=[4]))
    # delta_features (SURVEY 8f row 2), straight from the reference
    from nnmnkwii.preprocessing import delta_features
    for wi, ws in enumerate(windows_set()):
        for dt in (np.float32, np.float64):
            x = rng.standard_normal((9, 3)).astype(dt)
            out["delta_w%d_%s_x" % (wi, np.dtype(dt).name)] = x
            out["delta_w%d_%s_y" % (wi, np.dtype(dt).name)] = delta_features(x, ws)
    # length-masked metrics (SURVEY 8f row 4), straight from the reference
    from nnmnkwii import metrics as M
    mr = np.random.default_rng(2024)
    for dt in (np.float32, np.float64):
        n = np.dtype(dt).name
        X = mr.standard_normal((6, 37, 25)).astype(dt)
        Y = (X + 0.3 * mr.standard_normal((6, 37, 25))).astype(dt)
        lens = [37, 20, 1, 33, 0, 12]
        f0a = (5.0 + 0.3 * mr.standard_normal((6, 37))).astype(dt)
        f0b = (5.0 + 0.3 * mr.standard_normal((6, 37))).astype(dt)
        va = (mr.random((6, 37)) > 0.3).astype(dt)
        vb = (mr.random((6, 37)) > 0.3).astype(dt)
        out["met_%s_X" % n], out["met_%s_Y" % n], out["met_lens"] = X, Y, np.array(lens)
        out["met_%s_f0a" % n], out["met_%s_f0b" % n], out["met_%s_va" % n], out["met_%s_vb" % n] = f0a, f0b, va, vb
        out["met_%s_vals" % n] = np.array([
            M.melcd(X, Y), M.melcd(X, Y, lens), M.melcd(X[0], Y[0]), M.melcd(X[0, 0], Y[0, 0]),
            M.mean_squared_error(X, Y), M.mean_squared_error(X, Y, lens), M.mean_squared_error(X[0, 0], Y[0, 0]),
            M.lf0_mean_squared_error(f0a, va, f0b, vb), M.lf0_mean_squared_error(f0a, va, f0b, vb, lens),
            M.lf0_mean_squared_error(f0a, va, f0b, vb, lens, linear_domain=True),
            M.lf0_mean_squared_error(f0a[0], va[0], f0b[0], vb[0], linear_domain=True),
            M.lf0_mean_squared_error(f0a[:, :, None], va[:, :, None], f0b[:, :, None], vb[:, :, None], lens),
            M.vuv_error(va, vb), M.vuv_error(va, vb, lens), M.vuv_error(va[:, :, None], vb[:, :, None], lens),
            M.melcd(f0a, f0b, lens), M.mean_squared_error(f0a, f0b, lens),
        ], dtype=np.float64)
    # GMM-based conversion (SURVEY 8f row 1): baseline.gmm.MLPG / MLPGBase on a fitted joint GMM
    from sklearn.mixture import GaussianMixture
    from nnmnkwii.baseline.gmm import MLPG as RefGMMMLPG
    from nnmnkwii.baseline.gmm import MLPGBase as RefMLPGBase
    gr = np.random.default_rng(99)
    dim = 12  # = 2 windows x 6 static dims = 3 windows x 4 static dims
    base = gr.standard_normal((400, dim))
    joint = np.concatenate([base + 0.3 * gr.standard_normal((400, dim)),
                            0.7 * base + 0.5 + 0.3 * gr.standard_normal((400, dim))], axis=-1)
    gmm = GaussianMixture(n_components=4, covariance_type="full", random_state=0).fit(joint)
    src = base[:50] + 0.1 * gr.standard_normal((50, dim))
    out["gmm_means"], out["gmm_covars"], out["gmm_weights"], out["gmm_src"] = gmm.means_, gmm.covariances_, gmm.weights_, src
    out["gmm_default"] = RefGMMMLPG(gmm).transform(src)
    out["gmm_w3"] = RefGMMMLPG(gmm, windows=windows_set()[2]).transform(src)
    out["gmm_w3_diff"] = RefGMMMLPG(gmm, windows=windows_set()[2], diff=True).transform(src)
    out["gmm_w3_swap"] = RefGMMMLPG(gmm, windows=windows_set()[2], swap=True).transform(src)
    out["gmm_static"] = RefGMMMLPG(gmm, windows=[(0, 0, np.array([1.0]))]).transform(src)
    out["gmm_static_f32"] = RefGMMMLPG(gmm, windows=[(0, 0, np.array([1.0]))]).transform(src.astype(np.float32))
    out["gmm_base_2d"] = RefMLPGBase(gmm, diff=True).transform(src)
    out["gmm_base_1d"] = RefMLPGBase(gmm).transform(src[3])
    np.savez_compressed(os.path.join(HERE, "mlpg_reference_golden.npz"), **out)

    # DTW (restated oracle; see module docstring)
    d = {}
    for case, (Tx, Ty, D, radius) in enumerate([(23, 31, 5, 1), (40, 37, 25, 1), (64, 50, 3, 2), (9, 2, 4, 1), (1, 7, 2, 1)]):
        r = np.random.default_rng(100 + case)
        x = (np.cumsum(r.standard_normal((Tx, D)), 0) * 0.3).astype(np.float32)
        y = (np.cumsum(r.standard_normal((Ty, D)), 0) * 0.3).astype(np.float32)
        dist, path, cells = fastdtw_py.fastdtw(x, y, radius=radius, dist=melcd, return_cells=True)
        de, pe, ce = fastdtw_py.dtw(x, y, dist=melcd, return_cells=True)
        d["c%d_x" % case], d["c%d_y" % case] = x, y
        d["c%d_radius" % case] = np.array(radius)
        d["c%d_fast_dist" % case], d["c%d_fast_path" % case], d["c%d_fast_cells" % case] = (
            np.array(dist), np.array(path, dtype=np.int32), np.array(cells))
        d["c%d_exact_dist" % case], d["c%d_exact_path" % case] = np.array(de), np.array(pe, dtype=np.int32)
    np.savez_compressed(os.path.join(HERE, "dtw_restated_golden.npz"), **d)
    reference_parity()
    print("wrote", os.listdir(HERE))


def reference_parity():
    """What tests/test_oracle_golden.py::test_oracle_vs_live_reference and
    tests/test_host_logic_cpu.py::test_gmm_parameter_split_matches_reference compare against: the
    reference's outputs on their inputs (same seeds and draw order), inputs stored beside them."""
    oracle.import_reference()
    from nnmnkwii import paramgen as G
    from nnmnkwii.baseline.gmm import MLPGBase as RefMLPGBase
    out = {}
    rng = np.random.default_rng(7)
    for wi, ws in enumerate(windows_set()):
        for dt in (np.float32, np.float64):
            for T in (3, 17, 64):
                key = "live_w%d_%s_T%d" % (wi, np.dtype(dt).name, T)
                D = 3 * len(ws)
                m = rng.random((T, D)).astype(dt)
                v = (rng.random((T, D)) + 0.01).astype(dt)
                go = rng.standard_normal((T, 3)).astype(np.float32)
                out[key + "_means"], out[key + "_vars"], out[key + "_go"] = m, v, go
                out[key + "_y"] = G.mlpg(m, v, ws)
                out[key + "_grad"] = G.mlpg_grad(m, v, ws, go)
        out["live_w%d_R_T21" % wi] = G.unit_variance_mlpg_matrix(ws, 21)
    # baseline.gmm.MLPGBase parameter split of a random full-covariance joint GMM (M=3, 2 x 4 dims)
    gr = np.random.default_rng(0)
    M, dim = 3, 4
    A = gr.standard_normal((M, 2 * dim, 2 * dim))
    cov = A @ A.transpose(0, 2, 1) + 0.5 * np.eye(2 * dim)
    w = gr.random(M) + 0.1
    gmm = types.SimpleNamespace(means_=gr.standard_normal((M, 2 * dim)), covariances_=cov, weights_=w / w.sum(),
                                covariance_type="full")
    out["split_means"], out["split_covars"], out["split_weights"] = gmm.means_, gmm.covariances_, gmm.weights_
    for swap in (False, True):
        for diff in (False, True):
            ref = RefMLPGBase(gmm, swap=swap, diff=diff)
            key = "split_swap%d_diff%d_" % (swap, diff)
            for name in ("src_means", "tgt_means", "covarXX", "covarXY", "covarYX", "covarYY", "weights"):
                out[key + name] = getattr(ref, name)
            out[key + "num_mixtures"] = np.array(ref.num_mixtures)
            out[key + "prec_chol"] = ref.px.precisions_cholesky_
    np.savez_compressed(os.path.join(HERE, "reference_parity_golden.npz"), **out)


if __name__ == "__main__":
    main()
