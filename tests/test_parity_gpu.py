"""Parity of the CUDA path (through the C-ABI) against golden vectors produced by the real
reference and against the oracle on seeded inputs.  Tolerances: the north_star asks for 1e-4
relative on the final mapping matrix and on the loss trajectory (fp32 arithmetic)."""
import contextlib
import io
import os

import numpy as np
import pytest

from oracle.tangram_oracle import OracleMapper, grid_graph, spatial_weights_from_graph, synthetic_inputs
from tests.helpers import (assert_same_print, traj_err, GOLDEN_CASES, GOLDEN_DIR, load_golden, max_rel, rel_fro,
                           sha256_f32)

pytestmark = pytest.mark.gpu

# Both parity-grade modes run every test in this module: "fp32" (FFMA contractions) and "bf16x3" (tcgen05 tensor
# cores with every fp32 operand split into three bf16 planes, six partial products, fp32 accumulation in TMEM).
_PREC = {"value": "fp32"}


@pytest.fixture(autouse=True, params=["fp32", "bf16x3"])
def parity_precision(request):
    _PREC["value"] = request.param
    yield request.param


def _mapper(**kw):
    from tangram_b200 import Mapper
    kw.setdefault("precision", _PREC["value"])
    return Mapper(device="cuda:0", **kw)


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_golden_one_step(name):
    kw, g = load_golden(name)
    m = _mapper(M0=g["M0"], **kw)
    m.train(1, learning_rate=0.1, print_each=None)
    M1, mom1, mom2, step = m.state()
    assert step == 1
    assert rel_fro(M1, g["M1"]) < 1e-5
    assert abs(float(m.history_matrix[0, 0]) - g["total_loss"][0]) <= 2e-6 * max(1.0, abs(g["total_loss"][0]))


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_golden_trajectory_and_final_mapping(name):
    kw, g = load_golden(name)
    m = _mapper(M0=g["M0"], **kw)
    with contextlib.redirect_stdout(io.StringIO()) as buf:
        out, hist = m.train(int(g["epochs"]), learning_rate=0.1, print_each=10)
    tl = np.array([float(x) for x in hist["total_loss"]])
    assert max_rel(tl, g["total_loss"]) < 1e-4
    assert max_rel(hist["main_loss"], g["main_loss"]) < 1e-4
    for k in ("vg_reg", "kl_reg", "entropy_reg"):
        a, b = np.array(hist[k], dtype=np.float64), g[k]
        assert np.array_equal(np.isnan(a), np.isnan(b))
        if not np.isnan(b).all():
            assert max_rel(a[~np.isnan(b)], b[~np.isnan(b)]) < 1e-3
    assert out.dtype == np.float32 and out.shape == g["output"].shape
    assert rel_fro(out, g["output"]) < 1e-4
    assert isinstance(hist["total_loss"][0], np.ndarray) and hist["total_loss"][0].shape == ()
    assert isinstance(hist["main_loss"][0], float)
    assert len(hist["total_loss"]) == int(g["epochs"]) and hist["val_total_loss"] == []
    # the reference's print line (mapping_optimizer.py:300-307), epoch 0
    assert_same_print(buf.getvalue().splitlines()[0], str(g["printed"]).splitlines()[0])
    assert len(buf.getvalue().splitlines()) == len(str(g["printed"]).splitlines())


@pytest.mark.parametrize("shape", [(1000, 257, 130), (777, 1000, 96), (2048, 512, 256)])
def test_oracle_parity_ragged_shapes(shape):
    """Shapes that are not multiples of any tile size; 10 steps at <= 1e-5, loss at 1e-5."""
    N, V, K = shape
    inp = synthetic_inputs(N, V, K, seed=N + V)
    o = OracleMapper(inp["S"], inp["G"], d=inp["d"], lambda_d=1.0, random_state=42)
    M0 = o.M.numpy().copy()
    oo, oh = o.train(10, print_each=None)
    m = _mapper(S=inp["S"], G=inp["G"], d=inp["d"], lambda_d=1.0, M0=M0)
    out, hist = m.train(10, print_each=None)
    assert max_rel([float(x) for x in hist["total_loss"]], [float(x) for x in oh["total_loss"]]) < 1e-5
    assert rel_fro(out, oo) < 1e-5
    assert np.allclose(out.sum(axis=1), 1.0, atol=1e-5)


def test_oracle_parity_all_terms_medium():
    N, V, K, T = 1500, 400, 200, 8
    inp = synthetic_inputs(N, V, K, seed=2, n_types=T)
    conn, dist = grid_graph(V)
    kw = dict(
        S=inp["S"], G=inp["G"], d=inp["d"], lambda_d=1.0, lambda_g2=0.5, lambda_r=1e-3, lambda_l1=1e-7,
        lambda_l2=1e-7, lambda_neighborhood_g1=0.96, lambda_ct_islands=0.17, lambda_getis_ord=0.71,
        voxel_weights=spatial_weights_from_graph(conn, dist, True, True),
        neighborhood_filter=spatial_weights_from_graph(conn, dist, False, False),
        spatial_weights=spatial_weights_from_graph(conn, dist, False, True),
        ct_encode=inp["ct_encode"])
    o = OracleMapper(random_state=7, **kw)
    M0 = o.M.numpy().copy()
    oo, oh = o.train(15, print_each=None)
    m = _mapper(M0=M0, **kw)
    out, hist = m.train(15, print_each=None)
    assert max_rel([float(x) for x in hist["total_loss"]], [float(x) for x in oh["total_loss"]]) < 1e-4
    assert rel_fro(out, oo) < 1e-4
    # printed terms of the last epoch agree
    last = o.terms_history[-1]
    row = m.history_matrix[-1]
    for col, key in ((7, "gv_neighborhood_sim"), (8, "ct_island_penalty"), (9, "getis_ord_sim")):
        assert abs(row[col] - last[key]) < 1e-4 * max(1.0, abs(last[key]))


def test_clusters_mode_large_voxels():
    """small-N / large-V regime (BASELINE config 4, scaled down)."""
    N, V, K = 48, 5000, 300
    inp = synthetic_inputs(N, V, K, seed=4, clusters=True)
    o = OracleMapper(inp["S"], inp["G"], d=inp["d"], d_source=inp["d_source"], lambda_d=1.0, random_state=3)
    M0 = o.M.numpy().copy()
    oo, oh = o.train(10, print_each=None)
    m = _mapper(S=inp["S"], G=inp["G"], d=inp["d"], d_source=inp["d_source"], lambda_d=1.0, M0=M0)
    out, hist = m.train(10, print_each=None)
    assert max_rel([float(x) for x in hist["total_loss"]], [float(x) for x in oh["total_loss"]]) < 1e-4
    assert rel_fro(out, oo) < 1e-4


def test_reference_draw_is_reproduced():
    """random_state -> the same M0 bits as the reference draw (mapping_optimizer.py:147-157)."""
    inp = synthetic_inputs(64, 40, 16, seed=0)
    m = _mapper(S=inp["S"], G=inp["G"], d=inp["d"], lambda_d=1.0, random_state=42)
    M, _, _, step = m.state()
    np.random.seed(42)
    ref = np.random.normal(0, 1, (64, 40)).astype(np.float32)
    assert step == 0 and np.array_equal(M, ref)


def test_determinism_and_resume():
    """Same inputs -> bit-identical results; 12 steps == 5 steps + checkpoint + 7 steps."""
    inp = synthetic_inputs(900, 300, 150, seed=8)
    kw = dict(S=inp["S"], G=inp["G"], d=inp["d"], lambda_d=1.0, random_state=5)
    a, ha = _mapper(**kw).train(12, print_each=None)
    b, hb = _mapper(**kw).train(12, print_each=None)
    assert np.array_equal(a, b)
    assert np.array_equal(np.array(ha["total_loss"]), np.array(hb["total_loss"]))
    m1 = _mapper(**kw)
    m1.train(5, print_each=None)
    st = m1.state()
    m2 = _mapper(**kw)
    m2.load_state(*st)
    c, _ = m2.train(7, print_each=None, resume=True)       # keep the restored Adam state (default: fresh optimizer per train())
    assert np.array_equal(a, c)


def test_second_train_call_is_a_fresh_optimizer_like_the_reference():
    """mapping_optimizer.py:373: Adam is built inside train().  A second train() on the same mapper restarts the moments and
    the bias correction (oracle pinned to the live reference for this in tests/test_oracle.py); resume=True does not."""
    inp = synthetic_inputs(700, 200, 90, seed=15)
    kw = dict(S=inp["S"], G=inp["G"], d=inp["d"], lambda_d=1.0)
    o = OracleMapper(random_state=6, **kw)
    M0 = o.M.numpy().copy()
    o.train(4, print_each=None)
    oo, oh = o.train(3, print_each=None)
    m = _mapper(M0=M0, **kw)
    m.train(4, print_each=None)
    out, hist = m.train(3, print_each=None)
    assert len(hist["total_loss"]) == 3
    assert rel_fro(out, oo) < 2e-5
    assert max_rel([float(x) for x in hist["total_loss"]], [float(x) for x in oh["total_loss"]]) < 1e-5
    a, _ = _mapper(M0=M0, **kw).train(7, print_each=None)
    m2 = _mapper(M0=M0, **kw)
    m2.train(4, print_each=None)
    b, _ = m2.train(3, print_each=None, resume=True)
    assert np.array_equal(a, b)


def test_live_reference_on_the_same_gpu():
    """The UNMODIFIED reference Mapper (fp32, autograd, torch.optim.Adam; golden from its CPU run,
    tests/golden/make_live_reference_golden.py) against the CUDA path from the reference's own initial draw: loss
    trajectory and final mapping (a fixed sample of 32 rows) within north_star's 1e-4."""
    g = np.load(os.path.join(GOLDEN_DIR, "live_reference_30_epochs.npz"))
    inp = synthetic_inputs(3000, 700, 300, seed=31)
    kw = dict(S=inp["S"], G=inp["G"], d=inp["d"], lambda_d=1.0)
    # the default draw of the drop-in class is the reference's draw, bit for bit
    M0 = _mapper(random_state=42, **kw).state()[0]
    assert sha256_f32(M0) == str(g["M0_sha256"])
    m = _mapper(M0=M0, **kw)
    out, hist = m.train(30, print_each=None)
    assert max_rel([float(x) for x in hist["total_loss"]], g["total_loss"]) < 1e-4
    assert max_rel(hist["main_loss"], g["main_loss"]) < 1e-4
    assert rel_fro(out[g["rows"]], g["out_rows"]) < 1e-4


def test_full_size_properties_config2():
    """BASELINE config 2 size (10k x 1k x 1k): size-independent properties + oracle loss at step 0."""
    N, V, K = 10000, 1000, 1000
    inp = synthetic_inputs(N, V, K, seed=0)
    m = _mapper(S=inp["S"], G=inp["G"], d=inp["d"], lambda_d=1.0, random_state=42)
    out, hist = m.train(30, print_each=None)
    tl = np.array([float(x) for x in hist["total_loss"]])
    assert np.all(np.isfinite(tl)) and tl[-1] < tl[0]                # the optimiser descends
    assert np.all(np.diff(hist["main_loss"]) > -1e-4)                # gene score rises (monotone here)
    assert out.min() >= 0 and np.allclose(out.sum(axis=1), 1.0, atol=2e-5)
    np.random.seed(42)
    M0 = np.random.normal(0, 1, (N, V))
    o = OracleMapper(inp["S"], inp["G"], d=inp["d"], lambda_d=1.0, M0=M0)
    terms, _ = o.loss_and_grad(need_grad=False)
    assert abs(terms["total_loss"] - tl[0]) < 1e-5 * max(1.0, abs(tl[0]))
    # project == softmax(M)^T X
    X = np.random.default_rng(0).random((N, 37)).astype(np.float32)
    assert rel_fro(m.project(X), out.T.astype(np.float64) @ X) < 1e-5


def test_validation_terms_match_oracle():
    inp = synthetic_inputs(400, 120, 60, seed=6)
    kw = dict(S=inp["S"], G=inp["G"], d=inp["d"], lambda_d=1.0)
    o = OracleMapper(random_state=9, **kw)
    M0 = o.M.numpy().copy()
    _, oh = o.train(4, print_each=None, val_each=2)
    m = _mapper(M0=M0, **kw)
    _, hist = m.train(4, print_each=None, val_each=2)
    for k in ("val_total_loss", "val_gene_sim", "val_sp_sparsity_weighted_sim", "val_entropy"):
        assert len(hist[k]) == len(oh[k]) == 2
        assert max_rel(hist[k], oh[k]) < 1e-4


def test_map_cells_to_space_api_end_to_end():
    import pandas as pd
    import tangram_b200 as tg
    N, V, K = 300, 80, 50
    inp = synthetic_inputs(N, V, K, seed=12)
    genes = [f"Gene{i}" for i in range(K)]
    ad_sc = tg.MiniAnnData(X=inp["S"].copy(), obs=pd.DataFrame({"lab": [f"t{i % 3}" for i in range(N)]},
                           index=[f"c{i}" for i in range(N)]), var=pd.DataFrame(index=genes))
    ad_sp = tg.MiniAnnData(X=inp["G"].copy(), obs=pd.DataFrame({"x": np.arange(V)}, index=[f"v{i}" for i in range(V)]),
                           var=pd.DataFrame(index=genes))
    tg.pp_adatas(ad_sc, ad_sp)
    ad_map = tg.map_cells_to_space(ad_sc, ad_sp, device="cuda:0", num_epochs=20, random_state=3, verbose=False,
                                   precision=_PREC["value"])
    assert ad_map.X.shape == (N, V)
    df = ad_map.uns["train_genes_df"]
    assert list(df.columns) == ["train_score", "sparsity_sc", "sparsity_sp", "sparsity_diff"]
    assert df["train_score"].is_monotonic_decreasing and len(df) == K
    assert set(ad_map.uns["training_history"]) >= {"total_loss", "main_loss", "vg_reg", "kl_reg", "entropy_reg"}
    # same answer as the oracle fed the same way
    tr = ad_sc.uns["training_genes"]
    S = np.asarray(ad_sc[:, tr].X, dtype=np.float32)
    G = np.asarray(ad_sp[:, tr].X, dtype=np.float32)
    o = OracleMapper(S, G, d=np.asarray(ad_sp.obs["rna_count_based_density"], dtype=np.float32), lambda_d=1, random_state=3)
    oo, _ = o.train(20, print_each=None)
    assert rel_fro(ad_map.X, oo) < 1e-4
    ad_ge = tg.project_genes(ad_map, ad_sc)                      # default: the mapper was released, host contraction (:368)
    assert not hasattr(ad_map, "_tgb200_mapper")
    assert ad_ge.X.shape == (V, K) and ad_ge.var["is_training"].all()
    assert rel_fro(ad_ge.X, ad_map.X.T.astype(np.float64) @ np.asarray(ad_sc.X)) < 1e-5
    # keep_on_device=True: the same projection through tgb200_project on the GPU, then release()
    ad_map_k = tg.map_cells_to_space(ad_sc, ad_sp, device="cuda:0", num_epochs=20, random_state=3, verbose=False,
                                     precision=_PREC["value"], keep_on_device=True)
    assert np.array_equal(ad_map_k.X, ad_map.X)
    ad_ge_k = tg.project_genes(ad_map_k, ad_sc)
    assert rel_fro(ad_ge_k.X, ad_ge.X) < 1e-5
    ad_map_k._tgb200_mapper.release()
    # clusters mode runs and returns one row per cluster
    ad_map_c = tg.map_cells_to_space(ad_sc, ad_sp, mode="clusters", cluster_label="lab", device="cuda:0",
                                     num_epochs=10, random_state=3, verbose=False)
    assert ad_map_c.X.shape == (3, V)


def _load_c1():
    import os
    import scipy.sparse as sp
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "c1_reference.npz"))
    S = sp.csr_matrix((z["S_data"], z["S_indices"], z["S_indptr"]), shape=tuple(z["S_shape"])).toarray().astype(np.float32)
    return z, S


def test_baseline_config1_real_data_against_reference_run():
    """BASELINE config 1: the reference's own fixtures (26431 cells x 9852 voxels x 249 genes, mode='cells',
    100 epochs, random_state=42).  Golden = the REAL reference Mapper run on the CPU (tests/golden/make_c1_golden.py,
    535 s on 8 cores); the CUDA fp32 path must match its loss trajectory and mapping rows within 1e-4."""
    z, S = _load_c1()
    m = _mapper(S=S, G=z["G"], d=z["d"], lambda_g1=1, lambda_d=1, random_state=int(z["seed"]))
    out, hist = m.train(int(z["epochs"]), print_each=None)
    tl = np.array([float(x) for x in hist["total_loss"]])
    assert traj_err(tl, z["total_loss"]) < 1e-4          # the total loss crosses zero around epoch 12
    assert max_rel(hist["main_loss"], z["main_loss"]) < 1e-4
    assert max_rel(hist["kl_reg"], z["kl_reg"]) < 2e-3
    # 100 epochs is past the horizon where two fp32 runs that only differ in summation order agree to 1e-4 on
    # the mapping itself (SURVEY.md 7.3: reference-vs-reference noise floor 1.5e-4 at 100 epochs; measured here 1.6e-4)
    assert rel_fro(out[z["rows"]], z["out_rows"]) < 5e-4
    assert rel_fro(out.sum(axis=0), z["out_colsum"]) < 3e-5
    assert np.mean(out.argmax(axis=1) == z["out_rowmax_idx"]) > 0.999


def test_baseline_config1_real_data_bf16_tracks_reference():
    z, S = _load_c1()
    from tangram_b200 import Mapper
    if _PREC["value"] != "fp32":
        pytest.skip("bf16 throughput mode: run once")
    m = Mapper(device="cuda:0", S=S, G=z["G"], d=z["d"], lambda_g1=1, lambda_d=1, random_state=int(z["seed"]), precision="bf16")
    out, hist = m.train(int(z["epochs"]), print_each=None)
    tl = np.array([float(x) for x in hist["total_loss"]])
    # bf16 operands on real (wide dynamic range) expression data: up to 7e-3 off during the fast initial descent,
    # 1e-4 once converged -- the throughput mode; bf16x3 is the tensor-core mode that holds 1e-4 throughout
    assert traj_err(tl, z["total_loss"]) < 1.5e-2
    assert traj_err(tl[-20:], z["total_loss"][-20:]) < 5e-4
    assert rel_fro(out.sum(axis=0), z["out_colsum"]) < 5e-3
    assert np.mean(out.argmax(axis=1) == z["out_rowmax_idx"]) > 0.9
