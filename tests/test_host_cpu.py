"""CPU-side checks: the C-ABI library loads and exports every symbol the header declares (no compute calls),
the ctypes table matches the header, and the host-side sampler / data prep behave like the reference's."""
import os
import re

import numpy as np
import pytest

from conftest import ROOT


def _header_functions():
    src = open(os.path.join(ROOT, "include", "daisy_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    protos = re.findall(r"DAISY_API\s+[\w\s\*]+?\b(daisy_\w+)\s*\(([^;]*?)\)\s*;", src, flags=re.S)
    return {name: [a.strip() for a in args.split(",")] if args.strip() != "void" else [] for name, args in protos}


def test_library_exports_every_declared_symbol():
    from recommend_lib_b200 import _lib, build
    build.build()
    L = _lib.dlopen()
    decl = _header_functions()
    assert len(decl) >= 20
    for name in decl:
        assert hasattr(L, name), f"{name} declared in include/daisy_b200.h but not exported"


def test_ctypes_table_matches_header():
    from recommend_lib_b200 import _lib
    decl = _header_functions()
    table = dict(_lib.SIGNATURES)
    table["daisy_last_error"] = []
    assert set(table) == set(decl)
    for name, args in decl.items():
        assert len(table[name]) == len(args), f"{name}: header has {len(args)} args, ctypes table {len(table[name])}"


def test_loader_fails_loudly_without_library(monkeypatch, tmp_path):
    from recommend_lib_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(_lib.DaisyError, match="no CPU fallback"):
        _lib.load()


def test_product_does_not_import_the_oracle():
    pkg = os.path.join(ROOT, "recommend_lib_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), f
                assert "mf_oracle" not in text and "bpr_oracle" not in text, f


def test_no_cpu_fallback_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from recommend_lib_b200 import _lib
    from recommend_lib_b200.bpr import BPR, BPRSGD
    m = BPR(10, 10, 8)
    with pytest.raises(_lib.DaisyError):
        m(torch.tensor([1]), torch.tensor([2]), torch.tensor([3]))
    with pytest.raises(_lib.DaisyError):
        BPRSGD(m, 0.1, 0.0).step(torch.tensor([1]), torch.tensor([2]), torch.tensor([3]))


# ---------------------------------------------------------------- sampler (util/data_loader.py:680-700)
def test_sampler_semantics(golden):
    from recommend_lib_b200.sampler import TripleSampler
    s = golden("ml100k_split.npz")
    pairs = s["train_pairs"].astype(np.int64)
    I = int(s["item_num"])
    sm = TripleSampler(pairs, I, num_ng=4, seed=2019)
    t = sm.sample_epoch(0, shuffle=False)
    assert t.shape == (4 * len(pairs), 3) and t.dtype == np.int32 and len(sm) == t.shape[0]
    # features_fill order: positive-major, num_ng consecutive negatives
    assert np.array_equal(t[::4, :2], pairs) and np.array_equal(t[3::4, :2], pairs)
    # rejection: no sampled (u, j) is a training positive
    pos = set(map(tuple, pairs.tolist()))
    assert not any((u, j) in pos for u, _, j in t[:20000].tolist())
    keys = np.unique(pairs[:, 0] * I + pairs[:, 1])
    assert not np.isin(t[:, 0].astype(np.int64) * I + t[:, 2], keys).any()
    assert t[:, 2].min() >= 0 and t[:, 2].max() < I
    # deterministic per (seed, epoch), different across epochs, shuffle is a permutation of the same multiset
    assert np.array_equal(t, sm.sample_epoch(0, shuffle=False))
    assert not np.array_equal(t, sm.sample_epoch(1, shuffle=False))
    sh = sm.sample_epoch(0, shuffle=True)
    key = lambda a: np.sort(a[:, 0].astype(np.int64) * I * I + a[:, 1].astype(np.int64) * I + a[:, 2])
    assert np.array_equal(key(sh), key(t))
    sizes = [b.shape[0] for b in sm.batches(0, 4096)]
    assert len(sizes) == 97 and sizes[-1] == t.shape[0] - 96 * 4096          # SURVEY 8d: 97 steps


def test_negatives_are_uniform_over_non_positives():
    from recommend_lib_b200.sampler import TripleSampler
    pairs = np.array([[0, i] for i in range(0, 50, 2)])          # user 0 likes the even items
    sm = TripleSampler(pairs, 50, num_ng=400, seed=1)
    j = sm.sample_epoch(0)[:, 2]
    assert (j % 2 == 1).all()
    cnt = np.bincount(j, minlength=50)[1::2]
    assert cnt.min() > 0.8 * cnt.mean() and cnt.max() < 1.2 * cnt.mean()


def test_synthetic_generators():
    from recommend_lib_b200.sampler import synthetic_triples, synthetic_ratings
    t = synthetic_triples(200000, 1000, 500, seed=3)
    assert t.dtype == np.int32 and t[:, 0].max() < 1000 and t[:, 1:].max() < 500 and t.min() >= 0
    cnt = np.sort(np.bincount(t[:, 1], minlength=500))[::-1]
    assert cnt[0] > 20 * cnt[100]                                # Zipf(1): rank 1 >> rank 100
    assert np.array_equal(t, synthetic_triples(200000, 1000, 500, seed=3))
    u, i, r = synthetic_ratings(10000, 100, 50, seed=3)
    assert set(np.unique(r)) <= {1.0, 2.0, 3.0, 4.0, 5.0} and u.max() < 100 and i.max() < 50


def test_eval_candidates(golden):
    from recommend_lib_b200 import data
    s = golden("ml100k_split.npz")
    tr, te = s["train_pairs"].astype(np.int64), s["test_pairs"].astype(np.int64)
    allp = np.concatenate([tr, te])
    I = int(s["item_num"])
    eu, ec = data.eval_candidates(allp[:, 0], allp[:, 1], te[:, 0], te[:, 1], I, 999, 2019)
    assert ec.shape == (941, 1000) and len(eu) == 941            # SURVEY D2: users 405 and 655 dropped
    seen = {}
    for u, i in allp.tolist():
        seen.setdefault(u, set()).add(i)
    for u, row in list(zip(eu.tolist(), ec.tolist()))[:50]:
        assert len(set(row)) == 1000 and not (set(row[1:]) & seen[u]) and row[0] in seen[u]


def test_split_loo_ties_and_order():
    from recommend_lib_b200 import data
    users = np.array([0, 0, 0, 1, 1])
    ts = np.array([5, 9, 9, 3, 1])
    tr, te = data.split_loo_by_time(users, np.arange(5), ts)
    assert list(te) == [1, 3] and list(tr) == [0, 2, 4]          # tie at ts=9: first row wins (rank method='first')


def test_rank_metrics_match_the_reference_functions(golden):
    """precision / recall / MAP / NDCG / HR / MRR @k against values computed by the reference's own functions
    (util/metrics.py:99-195; fixture written by tests/golden/make_rank_metrics_golden.py)."""
    from recommend_lib_b200.metrics import rank_metrics
    g = golden("rank_metrics.npz")
    for c in range(3):
        rel, ptr, k = g[f"c{c}_rel"], g[f"c{c}_ur_ptr"], int(g[f"c{c}_k"])
        got = rank_metrics(rel, np.diff(ptr), k)
        want = dict(zip(("precision", "recall", "map", "ndcg", "hr", "mrr"), g[f"c{c}_kpi"]))
        for name in want:
            assert got[name] == pytest.approx(want[name], rel=1e-12, abs=1e-15), (c, name)
    with pytest.raises(ValueError):
        rank_metrics(np.zeros((3, 4)), np.ones(3), top_k=5)              # 'Relevance score length < k'


def test_shard_schedule_deals_every_chunk_to_exactly_one_warp():
    """The owner-interleaved schedule of the row-sharded step kernel (DESIGN section 7): the library's own mapping
    (host instance of the __host__ __device__ function the kernels call) is a bijection onto the chunks, and
    consecutive warps address consecutive owner ranges."""
    import ctypes
    from recommend_lib_b200 import _lib
    L = _lib.load()
    out = ctypes.c_int32()

    def chunk(w, n, g):
        _lib.check(L.daisy_shard_schedule(w, n, g, ctypes.byref(out)))
        return out.value

    for n in (0, 1, 2, 7, 8, 9, 37, 1000, 31250, 31251):
        for g in (0, 1, 2, 3, 4, 8):
            launched = n if g <= 1 else g * ((n + g - 1) // g)
            warps = (launched + 7) // 8 * 8                       # whole blocks of 8 warps are launched
            got = [chunk(w, n, g) for w in range(warps)]
            assert sorted(c for c in got if c >= 0) == list(range(n)), (n, g)
    n, g = 31250, 8                                               # config 5: 1 M triples in chunks of 32, 8 ranks
    per = (n + g - 1) // g
    assert [chunk(w, n, g) // per for w in range(16)] == [0, 1, 2, 3, 4, 5, 6, 7] * 2
    assert [chunk(w, n, 0) for w in range(4)] == [0, 1, 2, 3]
    assert L.daisy_shard_schedule(0, 10, 2, None) != 0            # null output pointer is an error, not a crash


def test_bprfm_bn_module_is_a_drop_in_and_has_no_cpu_path():
    """BPRFMBN (experimental batch-norm path of BPR-FM) keeps the reference class's module structure -- the state_dict
    keys and shapes of BPRFM(num_features, num_factors, True, [0.5, 0.2]) (BPRFMRecommender.py:45-55) -- and refuses to
    compute without a CUDA device."""
    import torch
    from recommend_lib_b200 import _lib
    from recommend_lib_b200.bprfm_bn import BPRFMBN, FMBNAdagrad
    m = BPRFMBN(90, 8, True, [0.5, 0.2], user_num=50)
    sd = m.state_dict()
    assert list(sd.keys()) == ["bias_", "embeddings.weight", "biases.weight", "FM_layers.0.weight", "FM_layers.0.bias",
                               "FM_layers.0.running_mean", "FM_layers.0.running_var", "FM_layers.0.num_batches_tracked"]
    assert tuple(sd["embeddings.weight"].shape) == (90, 8) and tuple(sd["biases.weight"].shape) == (90, 1)
    assert float(sd["biases.weight"].abs().max()) == 0.0 and 0.005 < float(sd["embeddings.weight"].std()) < 0.02
    with pytest.raises(NotImplementedError):
        BPRFMBN(90, 8, False, [0.0, 0.0], user_num=50)
    with pytest.raises(ValueError):
        BPRFMBN(90, 8, True, [0.5, 0.2])                      # user_num is required
    if not torch.cuda.is_available():
        m.eval()
        f = torch.zeros(2, 2, dtype=torch.long)
        with pytest.raises(_lib.DaisyError):
            m(f, None, f, None)
        with pytest.raises(_lib.DaisyError):
            FMBNAdagrad(m).step(f, None, f, None)


def test_item2vec_modules_are_drop_ins_and_have_no_cpu_path():
    """Item2Vec / SGNS (experimental N4 path) keep the reference's module structure (state_dict keys of
    SGNS(Item2Vec(V, D), ...), Item2VecRecommender.py:37-80), its initialisation (padding row zero, U(-0.5/D, 0.5/D)) and
    its negative-sampling table (unigram^0.75); computing without a CUDA device raises."""
    import torch
    from recommend_lib_b200 import _lib
    from recommend_lib_b200.item2vec import Item2Vec, SGNS, SGNSAdam
    counts = np.arange(1, 41, dtype=np.float64)
    sgns = SGNS(Item2Vec(40, 12), vocab_size=40, n_negs=5, weights=counts)
    assert list(sgns.state_dict().keys()) == ["embedding.ivectors.weight", "embedding.ovectors.weight"]
    W = sgns.embedding.ivectors.weight
    assert float(W[0].abs().max()) == 0.0 and float(W.abs().max()) <= 0.5 / 12 and float(W[1:].abs().min()) > 0
    wf = counts ** 0.75
    assert np.allclose(sgns.weights.numpy(), wf / wf.sum(), rtol=1e-6)
    assert tuple(sgns.draw_negatives(3, 2, "cpu").shape) == (3, 10)
    uni = SGNS(Item2Vec(40, 12), vocab_size=40, n_negs=5).draw_negatives(500, 2, "cpu")
    assert int(uni.min()) >= 0 and int(uni.max()) <= 38          # uniform_(0, V - 1).long(): V - 1 is never drawn (:90-91)
    with pytest.raises(RuntimeError):
        sgns(torch.zeros(3, dtype=torch.long), torch.zeros(3, 2, dtype=torch.long))
    if not torch.cuda.is_available():
        with pytest.raises(_lib.DaisyError):
            SGNSAdam(sgns).step(np.arange(3), np.zeros((3, 2), dtype=np.int64))


def test_neumf_module_is_a_drop_in_and_has_no_cpu_path():
    """NeuMF (experimental MLP / NeuMF-end path of NCF) keeps the reference class's module structure: the 12 state_dict
    entries of NCF(U, I, F, 3, 0.0, model) (NCFRecommender.py:45-66) with their shapes; computing without a CUDA device
    raises."""
    import torch
    from recommend_lib_b200 import _lib
    from recommend_lib_b200.ncf_mlp import NeuMF, NeuMFAdam
    U, I, F, L = 40, 30, 8, 3
    for name, P in (("MLP", F), ("NeuMF-end", 2 * F)):
        m = NeuMF(U, I, F, L, 0.0, name)
        sd = {k: tuple(v.shape) for k, v in m.state_dict().items()}
        assert sd == {"embed_user_GMF.weight": (U, F), "embed_item_GMF.weight": (I, F),
                      "embed_user_MLP.weight": (U, 4 * F), "embed_item_MLP.weight": (I, 4 * F),
                      "MLP_layers.1.weight": (4 * F, 8 * F), "MLP_layers.1.bias": (4 * F,),
                      "MLP_layers.4.weight": (2 * F, 4 * F), "MLP_layers.4.bias": (2 * F,),
                      "MLP_layers.7.weight": (F, 2 * F), "MLP_layers.7.bias": (F,),
                      "predict_layer.weight": (1, P), "predict_layer.bias": (1,)}
        assert float(m.predict_layer.bias.abs().max()) == 0.0
    with pytest.raises(NotImplementedError):
        NeuMF(U, I, F, L, 0.5, "NeuMF-end")                      # dropout is not on the accelerated path
    with pytest.raises(NotImplementedError):
        NeuMF(U, I, F, L, 0.0, "GMF")
    if not torch.cuda.is_available():
        z = torch.zeros(2, dtype=torch.long)
        with pytest.raises(_lib.DaisyError):
            m(z, z)
        with pytest.raises(_lib.DaisyError):
            NeuMFAdam(m).step(z, z, torch.zeros(2))


def test_ranking_refuses_cpu_tables():
    """metrics.topk_candidates / topk_full hand the ranking to the model; every rankable model with its tables on the CPU
    raises instead of ranking on the host."""
    from recommend_lib_b200 import _lib, metrics
    from recommend_lib_b200.bpr import BPR
    from recommend_lib_b200.bprfm import BPRFM
    from recommend_lib_b200.ncf import NCF
    from recommend_lib_b200.ncf_mlp import NeuMF
    U, I = 10, 12
    models = [BPR(U, I, 8), NCF(U, I, 8), BPRFM(U + I, 8, user_num=U), BPRFM(U + I, 8, True, user_num=U).eval(),
              NeuMF(U, I, 8)]
    for m in models:
        with pytest.raises(_lib.DaisyError, match="no CPU fallback"):
            metrics.topk_candidates(m, [0, 1], [[1, 2, 3], [4, 5, 6]], 2)
        with pytest.raises(_lib.DaisyError, match="no CPU fallback"):
            metrics.topk_full(m, [0, 1], 2, exclude=[[1], []])


def test_committed_bench_lines_carry_every_contract_key():
    """The JSON lines bench.py printed on a B200 at the end of round 2 (N = 1 at the default and at the driver's flags,
    N = 8 under torchrun) hold every key the bench contract names -- so a change to bench.py that drops one shows up here
    when the lines are regenerated."""
    import json
    root = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "profiles")
    base = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline"}
    for name, n in (("r02s_bench_n1_default.json", 1), ("r02s_bench_n1_driver_flags.json", 1), ("r02r_bench_n8_default.json", 8)):
        d = json.load(open(os.path.join(root, name)))
        assert base <= set(d), (name, base - set(d))
        assert d["metric"] == "bpr_mf_train_triples_per_s" and d["unit"] == "triples/s" and d["n_gpus"] == n
        assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None and d["dtype"] == "f32"
        assert "workload" in d["config"] and "model" not in d["config"]
        assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"])
        assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0 and d["e2e"]["value"] != d["value"]
        assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(d["roofline"])
        assert abs(d["roofline"]["frac"] - d["roofline"]["achieved"] / d["roofline"]["peak"]) < 1e-9
        assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"]) and d["gpu_launches"] > 0
        assert abs(d["value"] - d["config"].get("batch", d["config"].get("global_batch")) / (d["ms_per_step"] * 1e-3)) / d["value"] < 1e-6
    d = json.load(open(os.path.join(root, "r02s_bench_n1_default.json")))
    assert {"value", "unit", "cores", "kind", "sample"} <= set(d["cpu_baseline"]) and d["cpu_baseline"]["kind"] in ("port", "reference")
    assert d["config"]["lazy_decay_materialized_in_timed_region"] is False and d["materialize_ms"] > 0
    n8 = json.load(open(os.path.join(root, "r02r_bench_n8_default.json")))
    chk = n8["config"]["parity_selfcheck"]
    assert chk["ranks"] == 8 and all(v <= chk["tolerance"] for k, v in chk.items() if k.startswith("vs_"))
