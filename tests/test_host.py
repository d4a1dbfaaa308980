"""Host-side logic of the reference-shaped API (no GPU needed): AnnData stand-in, pp_adatas,
cluster aggregation, sparse spatial weights, argument validation with the reference's messages."""
import numpy as np
import pandas as pd
import pytest
import scipy.sparse as sp

import tangram_b200 as tg
from oracle.tangram_oracle import grid_graph, spatial_weights_from_graph
from tangram_b200 import spatial_weights as sw


def _mock_pair():
    # same shape as the reference's mocks (tests/tangram_test.py:31-47)
    ad_sc = tg.MiniAnnData(X=np.array([[0, 1, 1], [0, 1, 1]], dtype=np.float32),
                           obs=pd.DataFrame(index=["cell_1", "cell_2"]),
                           var=pd.DataFrame(index=["gene_a", "gene_b", "gene_d"]))
    ad_sp = tg.MiniAnnData(X=np.array([[0, 1, 1, 1], [0, 1, 1, 1]], dtype=np.float32),
                           obs=pd.DataFrame(index=["voxel_1", "voxel_2"]),
                           var=pd.DataFrame(index=["gene_c", "gene_b", "gene_a", "gene_d"]))
    return ad_sc, ad_sp


def test_pp_adatas_populates_fields():
    """tests/tangram_test.py:53-61."""
    ad_sc, ad_sp = _mock_pair()
    tg.pp_adatas(ad_sc, ad_sp)
    for ad in (ad_sc, ad_sp):
        assert "training_genes" in ad.uns and "overlap_genes" in ad.uns
    assert sorted(ad_sc.uns["training_genes"]) == ["gene_b", "gene_d"]      # gene_a is all-zero in sc -> filtered
    assert "rna_count_based_density" in ad_sp.obs.keys() and "uniform_density" in ad_sp.obs.keys()
    assert np.isclose(ad_sp.obs["rna_count_based_density"].sum(), 1.0)
    assert np.allclose(ad_sp.obs["uniform_density"], 0.5)


def test_minianndata_indexing():
    ad = tg.MiniAnnData(X=np.arange(12, dtype=np.float32).reshape(3, 4),
                        obs=pd.DataFrame({"lab": list("aba")}, index=["c0", "c1", "c2"]),
                        var=pd.DataFrame(index=["g0", "g1", "g2", "g3"]))
    sub = ad[:, ["g2", "g0"]]
    assert sub.shape == (3, 2) and np.array_equal(sub.X[:, 0], ad.X[:, 2])
    rows = ad[np.asarray(ad.obs["lab"] == "a")]
    assert rows.shape == (2, 4) and list(rows.obs_names) == ["c0", "c2"]
    with pytest.raises(KeyError):
        ad[:, ["nope"]]


def test_cluster_expression_matches_reference_semantics():
    """mapping_utils.py:103-139: sum (scale=True) or mean per label, cluster_density = label frequency."""
    X = np.arange(20, dtype=np.float32).reshape(5, 4)
    ad = tg.MiniAnnData(X=X, obs=pd.DataFrame({"lab": ["x", "y", "x", "x", "y"]}, index=[f"c{i}" for i in range(5)]),
                        var=pd.DataFrame(index=list("abcd")))
    agg = tg.adata_to_cluster_expression(ad, "lab", scale=True)
    labs = list(agg.obs["lab"])
    assert labs[0] == "x"                                                   # value_counts order: most frequent first
    assert np.allclose(agg.X[labs.index("x")], X[[0, 2, 3]].sum(0))
    assert np.allclose(agg.obs["cluster_density"], [0.6, 0.4])
    mean = tg.adata_to_cluster_expression(ad, "lab", scale=False)
    assert np.allclose(mean.X[labs.index("y")], X[[1, 4]].mean(0))
    with pytest.raises(ValueError, match="Provided label must belong"):
        tg.adata_to_cluster_expression(ad, "nope")


def test_sparse_spatial_weights_restate_the_dense_reference_semantics():
    """tangram/spatial_weights.py:5-30 on CSR: row-L1-normalised distances on the connectivity pattern, +I."""
    conn, dist = grid_graph(30)
    ad = tg.MiniAnnData(X=np.ones((30, 2), dtype=np.float32))
    ad.obsp = {"spatial_connectivities": conn, "spatial_distances": dist}
    w = sw.spatial_weights(ad, standardized=True, self_inclusion=True).toarray()
    d = dist.toarray()
    ref = d / np.abs(d).sum(axis=1, keepdims=True) * (conn.toarray() != 0) + np.eye(30)
    assert np.allclose(w, ref, atol=1e-6)
    b = sw.spatial_weights(ad, standardized=False, self_inclusion=False)
    assert sp.issparse(b) and np.array_equal(b.toarray(), conn.toarray())
    assert np.allclose(w, spatial_weights_from_graph(conn, dist, True, True).toarray())
    with pytest.raises(ValueError, match="Missing spatial neighborhood parameters"):
        sw.spatial_weights(tg.MiniAnnData(X=np.ones((3, 2))), True, True)


def _adatas(n=12, v=7, k=5):
    rng = np.random.default_rng(0)
    genes = [f"G{i}" for i in range(k)]
    ad_sc = tg.MiniAnnData(X=rng.random((n, k)).astype(np.float32) + 0.1,
                           obs=pd.DataFrame({"lab": ["a", "b"] * (n // 2)}, index=[f"c{i}" for i in range(n)]),
                           var=pd.DataFrame(index=genes))
    ad_sp = tg.MiniAnnData(X=rng.random((v, k)).astype(np.float32) + 0.1,
                           obs=pd.DataFrame(index=[f"v{i}" for i in range(v)]), var=pd.DataFrame(index=genes))
    return ad_sc, ad_sp


def test_map_cells_to_space_validation_messages():
    """mapping_utils.py:206-254: same exceptions and messages, raised before any device work."""
    ad_sc, ad_sp = _adatas()
    with pytest.raises(ValueError, match="Missing tangram parameters. Run `pp_adatas\\(\\)`."):
        tg.map_cells_to_space(ad_sc, ad_sp)
    tg.pp_adatas(ad_sc, ad_sp)
    with pytest.raises(ValueError, match="lambda_g1 cannot be 0."):
        tg.map_cells_to_space(ad_sc, ad_sp, lambda_g1=0)
    with pytest.raises(ValueError, match="Invalid input for density_prior."):
        tg.map_cells_to_space(ad_sc, ad_sp, density_prior="bogus")
    with pytest.raises(ValueError, match="When lambda_d is set, please define the density_prior."):
        tg.map_cells_to_space(ad_sc, ad_sp, lambda_d=1, density_prior=None)
    with pytest.raises(ValueError, match='Argument "mode" must be'):
        tg.map_cells_to_space(ad_sc, ad_sp, mode="nope")
    with pytest.raises(ValueError, match="A cluster_label must be specified if mode is 'clusters'."):
        tg.map_cells_to_space(ad_sc, ad_sp, mode="clusters")
    with pytest.raises(ValueError, match="target_count, lambda_f_reg and lambda_count must be specified"):
        tg.map_cells_to_space(ad_sc, ad_sp, mode="constrained")
    with pytest.raises(ValueError, match="Given training genes list should be subset of two AnnDatas."):
        tg.map_cells_to_space(ad_sc, ad_sp, cv_train_genes=["zzz"])
    with pytest.raises(NotImplementedError):
        tg.map_cells_to_space(ad_sc, ad_sp, lambda_moran=1.0)


def test_all_zero_gene_is_rejected():
    ad_sc, ad_sp = _adatas()
    tg.pp_adatas(ad_sc, ad_sp)
    ad_sp.X[:, 1] = 0.0
    with pytest.raises(ValueError, match="Genes with all zero values detected"):
        tg.map_cells_to_space(ad_sc, ad_sp)


def test_one_hot_encoding_order_of_first_appearance():
    """tangram/utils.py:105-123."""
    df = tg.one_hot_encoding(pd.Series(["b", "a", "b", "c"]))
    assert list(df.columns) == ["b", "a", "c"]
    assert df.values.tolist() == [[1, 0, 0], [0, 1, 0], [1, 0, 0], [0, 0, 1]]


def test_mapper_refuses_unsupported_terms_and_cpu():
    S = np.ones((4, 3), dtype=np.float32)
    G = np.ones((5, 3), dtype=np.float32)
    with pytest.raises(NotImplementedError):
        tg.Mapper(S, G, lambda_geary=1.0)
    with pytest.raises(NotImplementedError):
        tg.Mapper(S, G, adata_map=object())
    with pytest.raises(ValueError, match="B200 GPUs only"):
        tg.Mapper(S, G, device="cpu")


def test_legacy_normal_rows_is_a_slice_of_the_reference_draw():
    """mapping_optimizer.py:148-150: a rank of a sharded run keeps its rows of the SAME legacy stream, bit for bit."""
    from tangram_b200.mapping_optimizer import legacy_normal_rows
    np.random.seed(11)
    full = np.random.normal(0, 1, (53, 17)).astype(np.float32)
    for r0, r1 in ((0, 53), (0, 20), (20, 41), (41, 53), (7, 8)):
        assert np.array_equal(legacy_normal_rows(11, 53, 17, r0, r1, block_rows=5), full[r0:r1])


class _StrictAnnData(tg.MiniAnnData):
    """Mimics the shape checks of a real anndata.AnnData: X / var of another shape cannot be assigned."""

    def __setattr__(self, name, value):
        if name in ("X", "var") and "obs" in self.__dict__ and "var" in self.__dict__ and not self.__dict__.get("_subsetting"):
            n = value.shape[1] if name == "X" else len(value)
            if n != len(self.__dict__["var"]):
                raise ValueError("Data matrix has wrong shape")
        object.__setattr__(self, name, value)

    def _inplace_subset_var(self, keep):
        object.__setattr__(self, "_subsetting", True)
        try:
            super()._inplace_subset_var(keep)
        finally:
            object.__setattr__(self, "_subsetting", False)


def test_pp_adatas_filters_all_zero_genes_in_place_like_scanpy():
    """mapping_utils.py:47-48 (sc.pp.filter_genes(min_cells=1)): works on an AnnData that refuses reshaping assignments,
    records var['n_cells'], and drops the all-zero gene from X and var together."""
    rng = np.random.default_rng(1)
    genes = ["A", "B", "C", "D"]
    Xs = rng.random((6, 4)).astype(np.float32) + 0.1
    Xs[:, 2] = 0.0
    Xs[0, 1] = 0.0
    ad_sc = _StrictAnnData(X=Xs, obs=pd.DataFrame(index=[f"c{i}" for i in range(6)]), var=pd.DataFrame(index=genes))
    ad_sp = _StrictAnnData(X=rng.random((5, 4)).astype(np.float32) + 0.1, obs=pd.DataFrame(index=[f"v{i}" for i in range(5)]),
                           var=pd.DataFrame(index=genes))
    tg.pp_adatas(ad_sc, ad_sp)
    assert list(ad_sc.var.index) == ["a", "b", "d"] and ad_sc.X.shape == (6, 3)
    assert list(ad_sc.var["n_cells"]) == [6, 5, 6] and list(ad_sp.var["n_cells"]) == [5, 5, 5, 5]
    assert sorted(ad_sc.uns["training_genes"]) == ["a", "b", "d"]


def test_process_group_needs_cells_mode():
    ad_sc, ad_sp = _adatas()
    tg.pp_adatas(ad_sc, ad_sp)
    with pytest.raises(ValueError, match="only mode='cells' can be sharded"):
        tg.map_cells_to_space(ad_sc, ad_sp, mode="clusters", cluster_label="lab", process_group=object())


def test_bench_reference_arm_runs_the_unmodified_reference_on_the_host():
    """`bench.py --impl reference`: the unmodified reference Mapper (oracle/_ref or the reference tree) on the host cores, full
    workload, bounded epochs; the JSON line carries what was actually run."""
    import json
    import os
    import subprocess
    import sys
    from oracle import build_ref
    if not os.path.exists(build_ref.REF_DST) and not os.path.exists(build_ref.REF_SRC):
        pytest.skip("reference file not available (oracle/build_ref.py)")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--workload", "tiny", "--steps", "5",
                          "--warmup", "3"], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stderr[-2000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "map_cells_to_space iterations/sec" and line["unit"] == "iterations/s"
    assert line["cpu_baseline"]["kind"] == "reference" and line["cpu_baseline"]["cores"] >= 1
    assert 2 <= line["steps"] <= 5 and line["steps_requested"] == 5 and line["value"] > 0
    assert abs(line["value"] - 1e3 / line["ms_per_step"]) < 1e-6 * line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["config"]["cells"] == 300 and "unmodified reference" in line["cpu_baseline"]["sample"]


def test_oracle_ref_recipe_is_a_verbatim_copy():
    """oracle/build_ref.py: oracle/_ref/mapping_optimizer.py is the reference file byte for byte (sha256 in SOURCE.txt) and loads
    as a module with the reference's two classes."""
    import hashlib
    import os
    from oracle import build_ref
    if not os.path.exists(build_ref.REF_SRC) and not os.path.exists(build_ref.REF_DST):
        pytest.skip("neither the reference tree nor a copy is present")
    path = build_ref.build()
    assert path == build_ref.REF_DST and os.path.exists(path)
    digest = hashlib.sha256(open(path, "rb").read()).hexdigest()
    assert digest in open(build_ref.STAMP).read()
    if os.path.exists(build_ref.REF_SRC):
        assert open(path, "rb").read() == open(build_ref.REF_SRC, "rb").read()
    mod = build_ref.load()
    assert hasattr(mod, "Mapper") and hasattr(mod, "MapperConstrained")


def test_profiles_traffic_json_matches_the_committed_ncu_capture():
    """bench.py's roofline.traffic comes from profiles/traffic.json, which tools/ncu_traffic.py derives from the committed raw
    `ncu --set full` page: re-derive it and compare (DRAM bytes of the streaming update = its algorithmic 24 B/element)."""
    import csv
    import json
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    traffic = json.load(open(os.path.join(root, "profiles", "traffic.json")))["c3/bf16"]
    rows = list(csv.reader(open(os.path.join(root, traffic["_source"]))))
    hdr, units = rows[0], rows[1]
    ki, ri, wi = hdr.index("Kernel Name"), hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
    scale = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}
    per_launch = [float(r[ri]) * scale[units[ri]] + float(r[wi]) * scale[units[wi]] for r in rows[2:] if "k_adam_rows" in r[ki]]
    assert per_launch and abs(4 * np.mean(per_launch) - traffic["adam_rows"]) < 1e-6 * traffic["adam_rows"]
    assert abs(traffic["adam_rows"] - 24.0 * 100_000 * 10_000) < 0.02 * 24e9          # nothing is re-read


def test_nccl_comm_cache_ignores_non_nccl_groups():
    """gloo groups (the CPU tests) keep the host-driven exchange: nccl_comm_for_group returns None without touching CUDA."""
    import os
    import socket
    import torch.distributed as dist
    from tangram_b200.sharded import nccl_comm_for_group
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=0, world_size=1)
    try:
        assert nccl_comm_for_group(dist.group.WORLD, 0) is None
    finally:
        dist.destroy_process_group()
