"""Pin the oracle (oracle/tangram_oracle.py) against vectors produced by the real
reference (tests/golden/make_golden.py, tests/golden/make_live_reference_golden.py).  CPU only."""
import contextlib
import io
import os

import numpy as np
import pytest
import torch

from oracle.tangram_oracle import OracleMapper, synthetic_inputs
from tests.helpers import assert_same_print, GOLDEN_CASES, GOLDEN_DIR, load_golden, max_rel, rel_fro, sha256_f32


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_oracle_matches_golden_one_step(name):
    kw, g = load_golden(name)
    o = OracleMapper(M0=g["M0"], **kw)
    terms, dM = o.loss_and_grad()
    o.adam_step(dM, 0.1)
    # loss before the first update
    assert abs(terms["total_loss"] - g["total_loss"][0]) <= 2e-6 * max(1.0, abs(g["total_loss"][0]))
    # first Adam step is +-lr*sign(g) up to eps: compare M after one step
    assert np.max(np.abs(o.M.numpy() - g["M1"])) < 2e-4
    assert rel_fro(o.M.numpy(), g["M1"]) < 1e-5


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_oracle_matches_golden_trajectory(name):
    kw, g = load_golden(name)
    o = OracleMapper(M0=g["M0"], **kw)
    with contextlib.redirect_stdout(io.StringIO()) as buf:
        out, hist = o.train(int(g["epochs"]), learning_rate=0.1, print_each=10)
    tl = np.array([float(x) for x in hist["total_loss"]])
    assert max_rel(tl, g["total_loss"]) < 1e-4                      # north_star tolerance
    assert max_rel(hist["main_loss"], g["main_loss"]) < 1e-4
    for k in ("vg_reg", "kl_reg", "entropy_reg"):
        a, b = np.array(hist[k], dtype=np.float64), g[k]
        assert np.array_equal(np.isnan(a), np.isnan(b))             # NaN conventions
        if not np.isnan(b).all():
            assert max_rel(a[~np.isnan(b)], b[~np.isnan(b)]) < 1e-3
    assert rel_fro(out, g["output"]) < 1e-4                         # final mapping matrix
    assert out.dtype == np.float32 and out.shape == g["output"].shape
    # printed lines: same text (mapping_optimizer.py:300-307)
    assert_same_print(buf.getvalue().splitlines()[0], str(g["printed"]).splitlines()[0])


def test_oracle_float64_gradient_matches_finite_differences():
    inp = synthetic_inputs(20, 12, 8, seed=1, n_types=3)
    from oracle.tangram_oracle import grid_graph, spatial_weights_from_graph
    conn, dist = grid_graph(12)
    o = OracleMapper(
        inp["S"], inp["G"], d=inp["d"], lambda_d=0.8, lambda_g2=0.4, lambda_r=0.01, lambda_l1=1e-3,
        lambda_l2=1e-3, lambda_neighborhood_g1=0.9, lambda_ct_islands=0.3, lambda_getis_ord=0.7,
        voxel_weights=spatial_weights_from_graph(conn, dist, True, True),
        neighborhood_filter=spatial_weights_from_graph(conn, dist, False, False),
        spatial_weights=spatial_weights_from_graph(conn, dist, False, True),
        ct_encode=inp["ct_encode"], random_state=3, dtype=torch.float64)
    _, dM = o.loss_and_grad()
    rng = np.random.default_rng(0)
    for _ in range(12):
        i, j = rng.integers(0, 20), rng.integers(0, 12)
        h = 1e-6
        Mp, Mm = o.M.clone(), o.M.clone()
        Mp[i, j] += h
        Mm[i, j] -= h
        fd = (o.loss_and_grad(Mp, need_grad=False)[0]["total_loss"]
              - o.loss_and_grad(Mm, need_grad=False)[0]["total_loss"]) / (2 * h)
        assert abs(fd - float(dM[i, j])) < 1e-6 + 1e-4 * abs(fd)


def test_oracle_matches_live_reference_autograd():
    """Loss and autograd dL/dM of the reference Mapper's first epoch (random_state=5), from its own initial draw."""
    g = np.load(os.path.join(GOLDEN_DIR, "live_reference_autograd.npz"))
    inp = synthetic_inputs(500, 130, 70, seed=9)
    o = OracleMapper(inp["S"], inp["G"], d=inp["d"], lambda_d=1.0, lambda_g2=0.2, lambda_r=1e-4, random_state=5)
    assert sha256_f32(o.M.numpy()) == str(g["M0_sha256"])        # the reference's draw, bit for bit
    terms, dM = o.loss_and_grad()
    assert abs(terms["total_loss"] - float(g["total_loss"])) < 2e-6
    assert rel_fro(dM.numpy()[g["rows"]], g["grad_rows"]) < 2e-5


def test_unseeded_when_random_state_zero():
    """mapping_optimizer.py:148 -- random_state=0 is falsy -> no seeding (quirk preserved)."""
    inp = synthetic_inputs(8, 6, 5, seed=0)
    np.random.seed(123)
    a = OracleMapper(inp["S"], inp["G"], random_state=0).M.numpy()
    np.random.seed(123)
    b = OracleMapper(inp["S"], inp["G"], random_state=0).M.numpy()
    c = OracleMapper(inp["S"], inp["G"], random_state=0).M.numpy()
    assert np.array_equal(a, b) and not np.array_equal(b, c)


def test_second_train_call_restarts_adam_like_the_reference():
    """mapping_optimizer.py:373: the optimizer is built inside train(), so a second call starts from zero moments.
    Golden: the reference Mapper's second train(3) call after train(4)."""
    g = np.load(os.path.join(GOLDEN_DIR, "live_reference_second_train.npz"))
    inp = synthetic_inputs(60, 25, 12, seed=4)
    kw = dict(S=inp["S"], G=inp["G"], d=inp["d"], lambda_d=1.0, random_state=7)
    o = OracleMapper(**kw)
    o.train(4, print_each=None)
    o_out, o_hist = o.train(3, print_each=None)
    assert rel_fro(o_out, g["output"]) < 1e-5
    assert max_rel([float(x) for x in o_hist["total_loss"]], g["total_loss"]) < 1e-5
