"""Algorithms tested locally with ``ClientMockProtocol`` (vantage6's way of testing multi-node
algorithms without a cluster), the wrapper's dispatch / data loading, the message-queue event
mirror, and the repository entry points (bench reference arm, build())."""
import json
import os
import subprocess
import sys
import time

import numpy as np
import pytest

from vantage6_b200.algorithm import IMAGES, resolve_image
from vantage6_b200.algorithm import wrapper
from vantage6_b200.algorithm.builtin import average, glm, weighted_mean
from vantage6_b200.client.mock import ClientMockProtocol
from vantage6_b200.common.serialization import deserialize, serialize

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_weighted_mean_master_over_mock_nodes():
    rng = np.random.default_rng(1)
    data = [rng.normal(size=(n, 1000)) for n in (10, 40, 50)]
    out = weighted_mean.master(ClientMockProtocol(data, weighted_mean), data[0])
    np.testing.assert_allclose(out["mean"], np.concatenate(data).mean(0), rtol=1e-12)
    assert out["count"] == 100 and out["n_nodes"] == 3


def test_glm_control_plane_converges():
    rng = np.random.default_rng(2)
    w_true = rng.normal(size=9) * 0.8
    shards = []
    for n in (400, 600):
        X = rng.normal(size=(n, 8))
        y = (rng.random(n) < 1 / (1 + np.exp(-(X @ w_true[:8] + w_true[8])))).astype(float)
        shards.append({"X": X, "y": y})
    out = glm.master(ClientMockProtocol(shards, glm), shards[0], iterations=200, lr=1.0)
    assert out["losses"][-1] < out["losses"][0]
    assert np.abs(out["coefficients"] - w_true[:8]).max() < 0.4 and out["n"] == 1000


def test_wrapper_dispatch_and_missing_method():
    import pandas as pd

    df = pd.DataFrame({"age": [1.0, 2.0, 3.0]})
    out = wrapper.dispatch(average, {"method": "average_partial", "kwargs": {"column_name": "age"}}, df, lambda: None)
    assert out == {"sum": 6.0, "count": 3}
    with pytest.raises(AttributeError):
        wrapper.dispatch(average, {"method": "nope"}, df, lambda: None)


def test_wrapper_process_contract(tmp_path):
    """INPUT_FILE / OUTPUT_FILE / DATABASE_URI environment contract, as a real child process."""
    db = tmp_path / "vec.npy"
    np.save(db, np.arange(6.0).reshape(2, 3))
    (tmp_path / "in").write_bytes(serialize({"method": "partial_sum"}))
    env = dict(os.environ, INPUT_FILE=str(tmp_path / "in"), OUTPUT_FILE=str(tmp_path / "out"),
               TOKEN_FILE=str(tmp_path / "tok"), DATABASE_URI=str(db), PYTHONPATH=ROOT)
    p = subprocess.run([sys.executable, "-m", "vantage6_b200.algorithm.wrapper",
                        "vantage6_b200.algorithm.builtin.weighted_mean"], env=env, capture_output=True, text=True, timeout=120)
    assert p.returncode == 0, p.stdout + p.stderr
    out = deserialize((tmp_path / "out").read_bytes())
    np.testing.assert_allclose(out["sum"], [3.0, 5.0, 7.0])
    assert out["count"] == 2


def test_data_loaders(tmp_path):
    import pandas as pd
    import torch

    pd.DataFrame({"a": [1, 2]}).to_csv(tmp_path / "d.csv", index=False)
    assert list(wrapper.load_data(str(tmp_path / "d.csv"))["a"]) == [1, 2]
    torch.save({"x": torch.ones(2)}, tmp_path / "d.pt")
    assert wrapper.load_data(str(tmp_path / "d.pt"))["x"].sum() == 2
    assert wrapper.load_data("synthetic://imagenet?n=512") == "synthetic://imagenet?n=512"
    assert wrapper.load_data(None) is None
    with pytest.raises(ValueError):
        wrapper.load_data(str(tmp_path / "d.xyz"))


def test_serialization_roundtrip_numpy_torch_bytes():
    import torch

    obj = {"a": np.arange(4, dtype=np.float32).reshape(2, 2), "t": torch.ones(3, dtype=torch.bfloat16), "b": b"\x00\x01",
           "n": np.int64(3), "f": np.float32(0.5), "s": {1, 2}}
    back = deserialize(serialize(obj))
    np.testing.assert_array_equal(back["a"], obj["a"])
    np.testing.assert_array_equal(back["t"], np.ones(3, dtype=np.float32))
    assert back["b"] == b"\x00\x01" and back["n"] == 3 and back["f"] == 0.5 and sorted(back["s"]) == [1, 2]
    # pickle executes code on load: refused unless the operator opted in (ADVICE r1, medium)
    from vantage6_b200.common.serialization import UnsafePayload

    blob = serialize({"k": [1, 2]}, "pickle")
    with pytest.raises(UnsafePayload):
        deserialize(blob)
    with pytest.raises(UnsafePayload):
        deserialize(blob, "pickle")
    assert deserialize(blob, allow_pickle=True) == {"k": [1, 2]}


def test_image_registry():
    assert resolve_image("v6b200/fedavg").endswith("builtin.fedavg")
    assert resolve_image("harbor2.vantage6.ai/demo/average:latest").endswith("builtin.average")
    assert resolve_image("my/img", {"my/img": "pkg.mod"}) == "pkg.mod"
    with pytest.raises(KeyError):
        resolve_image("module:os")
    assert resolve_image("module:os", allow_modules=True) == "os"
    assert set(IMAGES.values()) >= {"vantage6_b200.algorithm.builtin.glm"}


def test_event_mirror_between_two_servers(v6home):
    """Horizontal scaling: two server apps share events through the message-queue sidecar."""
    from vantage6_b200.dev import free_port
    from vantage6_b200.runtime import from_env
    from vantage6_b200.server.app import ServerApp
    from vantage6_b200.server.mq_broker import attach_app

    port = free_port()
    rt = from_env()
    c = rt.containers.run("mq", command=f"v6-mq-broker serve --port {port}", name="vantage6-mirror-rabbitmq",
                          labels={"vantage6-type": "rabbitmq"})
    try:
        uri = f"amqp://u:p@127.0.0.1:{port}/shared"
        a = ServerApp({"uri": "sqlite://", "api_path": "/api"})
        b = ServerApp({"uri": "sqlite://", "api_path": "/api"})
        attach_app(a, uri)
        attach_app(b, uri)
        got = []
        t0 = time.time()
        while not got and time.time() - t0 < 20:            # pub/sub joins are asynchronous: re-emit until seen
            a.events.emit("new_task", {"task_id": 1}, ["collaboration_1"])
            got = b.events.wait(0, ["collaboration_1"], 0.5)
        assert got and got[0]["name"] == "new_task"
        assert all(e["name"] == "new_task" for e in a.events.wait(0, ["collaboration_1"], 0))   # no echo storm
    finally:
        c.kill()


def test_bench_reference_arm_reports_unavailable():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference"], capture_output=True,
                       text=True, timeout=120)
    assert p.returncode == 0
    d = json.loads(p.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and "unavailable" in d


def test_bench_dump_samples_large_outputs_at_fixed_indices(tmp_path, monkeypatch):
    import torch

    sys.path.insert(0, ROOT)
    import bench

    monkeypatch.setattr(bench, "DUMP_MAX_ELEMS", 1000)
    x = torch.arange(5000, dtype=torch.float64)
    bench.dump_outputs(str(tmp_path / "a"), {"loss": torch.tensor(2.5), "global_model": x})
    bench.dump_outputs(str(tmp_path / "b"), {"global_model": x.clone()})
    loss, a, b = (np.load(tmp_path / p) for p in ("a/loss.npy", "a/global_model.npy", "b/global_model.npy"))
    assert loss.dtype == np.float32 and loss.shape == () and loss == 2.5
    assert a.dtype == np.float32 and a.shape == (1000,) and (a == b).all() and (np.diff(a) > 0).all()


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_round(tmp_path):
    """--steps sets the timed rounds; --dump-outputs writes their last result, and the same arguments give the same inputs
    and so the same dump on every run (what makes two builds comparable output for output).  resnet_mini is the flagship's
    path at 64x64 images -- every convolution on the project's kernels; resnet_tiny's narrow layers fall back to cuDNN,
    whose autotuned algorithm choice may differ between runs."""
    runs = []
    for k in range(2):
        out = tmp_path / f"outputs{k}"
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--model", "resnet_mini", "--steps", "2", "--warmup", "1",
                            "--no-e2e", "--baselines", "", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stderr[-3000:]
        d = json.loads(p.stdout.strip().splitlines()[-1])
        assert d["steps"] == 2 and sorted(f.name for f in out.iterdir()) == ["global_model.npy", "loss.npy"]
        loss, model = np.load(out / "loss.npy"), np.load(out / "global_model.npy")
        assert loss.dtype == np.float32 and float(loss) == d["final_loss"]
        assert model.dtype == np.float32 and model.shape == (min(d["config"]["n_federated_params"], 1 << 23),)
        assert np.isfinite(model).all()
        runs.append((loss, model))
    (l0, m0), (l1, m1) = runs
    np.testing.assert_allclose(l1, l0, rtol=1e-5)
    np.testing.assert_allclose(m1, m0, rtol=1e-5, atol=1e-6 * float(np.abs(m0).max()))


def test_graft_entry_build_is_incremental():
    sys.path.insert(0, ROOT)
    import __graft_entry__ as g

    t0 = time.time()
    g.build()
    assert time.time() - t0 < 120
    from vantage6_b200.ops import native

    C = native()
    for fn in ("fedavg_round", "small_allreduce", "flat_optim", "layernorm_fwd", "rmsnorm_bwd", "rope", "glm_logistic_grad",
               "gemm_bf16", "bcast_gemm_bf16", "flash_attn_fwd", "symm_alloc"):
        assert hasattr(C, fn), fn


def test_peer_channel_single_node_cpu():
    """algorithm/peer.py (the in-box stand-in for vantage6's algorithm VPN): same API on a CPU node."""
    from vantage6_b200.algorithm.peer import PeerChannel

    ch = PeerChannel.open({"addr": "127.0.0.1", "port": 0, "world": 1, "ranks": {"7": 0}}, organization_id=7)
    buf = ch.alloc(100)
    assert buf.local.numel() >= 100 and buf.mc_ptr == 0
    out = ch.allreduce([1.0, 2.0, 3.0], 5.0)
    assert out.tolist() == [1.0, 2.0, 3.0]
    out = ch.allreduce([1.0, 2.0, 3.0], 5.0, normalize=False)
    assert out.tolist() == [5.0, 10.0, 15.0]
    ch.barrier()
    ch.close()


def test_fedavg_confines_researcher_paths(tmp_path, monkeypatch):
    """checkpoint_dir / resume_from / metrics_file arrive in the task input: they may only point into the directories the node
    set aside for algorithms (per-run temporary folder, log directory, V6_ALGORITHM_DATA_DIR)."""
    import pytest

    from vantage6_b200.algorithm.builtin import fedavg

    run_dir, log_dir = tmp_path / "run", tmp_path / "log"
    run_dir.mkdir()
    log_dir.mkdir()
    monkeypatch.setenv("TEMPORARY_FOLDER", str(run_dir))
    monkeypatch.setenv("V6_LOG_DIR", str(log_dir))
    assert fedavg._confined("ckpt", "checkpoint_dir") == str(run_dir / "ckpt")                 # relative: inside the run folder
    assert fedavg._confined(str(log_dir / "m.jsonl"), "metrics_file") == str(log_dir / "m.jsonl")
    with pytest.raises(PermissionError):
        fedavg._confined("/etc/cron.d/x", "metrics_file")
    with pytest.raises(PermissionError):
        fedavg._confined(str(run_dir / ".." / "escape"), "checkpoint_dir")
    with pytest.raises(PermissionError):
        fedavg.train_partial(None, model="resnet_tiny", rounds=1, checkpoint_dir="/root/elsewhere")
    out = fedavg.train_partial(None, model="resnet_tiny", rounds=2, local_steps=1, batch=4, checkpoint_every=1, checkpoint_dir="ckpt",
                               metrics_file=str(log_dir / "m.jsonl"))
    assert len(out["losses"]) == 2 and (run_dir / "ckpt").is_dir() and (log_dir / "m.jsonl").exists()


def _patients(rng, n, shift=0.0):
    import pandas as pd

    return pd.DataFrame({
        "age": rng.normal(60 + shift, 10, n).round(1), "bmi": np.where(rng.random(n) < 0.1, np.nan, rng.normal(26, 4, n)),
        "sex": rng.choice(["f", "m"], n), "stage": rng.choice(["I", "II", "III"], n, p=[0.5, 0.3, 0.2]),
        "time": rng.exponential(24 + shift, n).round(0) + 1, "event": (rng.random(n) < 0.7).astype(int)})


def test_summary_matches_pooled_statistics():
    import pandas as pd

    from vantage6_b200.algorithm.builtin import summary

    rng = np.random.default_rng(3)
    frames = [_patients(rng, 80), _patients(rng, 120, 5.0), _patients(rng, 50, -3.0)]
    pooled = pd.concat(frames)
    out = summary.master(ClientMockProtocol(frames, summary), frames[0], columns=["age", "bmi", "sex", "stage"])
    assert out["n_rows"] == 250 and out["n_nodes"] == 3
    for c in ("age", "bmi"):
        np.testing.assert_allclose(out["columns"][c]["mean"], pooled[c].mean(), rtol=1e-12)
        np.testing.assert_allclose(out["columns"][c]["std"], pooled[c].std(), rtol=1e-10)          # exact pooled variance
        assert out["columns"][c]["min"] == pooled[c].min() and out["columns"][c]["max"] == pooled[c].max()
    assert out["columns"]["bmi"]["missing"] == int(pooled["bmi"].isna().sum()) > 0
    assert out["columns"]["sex"]["counts"] == pooled["sex"].value_counts().to_dict()
    q = summary.master(ClientMockProtocol(frames, summary), frames[0], columns=["age", "bmi"], quantiles=[0.0, 0.25, 0.5, 0.9, 1.0])
    for c in ("age", "bmi"):
        cell = (pooled[c].max() - pooled[c].min()) / 512
        vals = pooled[c].dropna().to_numpy()
        for k, v in q["columns"][c]["quantiles"].items():          # within a cell of a value whose empirical rank is q
            assert (vals <= v + cell).mean() >= float(k) - 1e-12 and (vals < v - cell).mean() <= float(k) + 1e-12, (c, k, v)
        assert q["columns"][c]["quantiles"]["0.0"] <= vals.min() + cell and q["columns"][c]["quantiles"]["1.0"] >= vals.max() - cell
    with pytest.raises(ValueError):
        summary.master(ClientMockProtocol(frames, summary), frames[0], columns=["age"], quantiles=[1.5])
    # privacy guards: a tiny node refuses, rare levels are suppressed
    with pytest.raises(PermissionError):
        summary.RPC_summary_partial(frames[0].head(5))
    rare = frames[0].copy()
    rare.loc[rare.index[:2], "stage"] = "IV"
    part = summary.RPC_summary_partial(rare, columns=["stage"])
    assert part["categorical"]["stage"]["counts"]["IV"] == 0 and part["categorical"]["stage"]["suppressed"]
    with pytest.raises(KeyError):
        summary.RPC_summary_partial(frames[0], columns=["nope"])


def test_crosstab_and_chi_square_match_scipy():
    import pandas as pd
    from scipy.stats import chi2_contingency

    from vantage6_b200.algorithm.builtin import crosstab

    rng = np.random.default_rng(4)
    frames = [_patients(rng, 200), _patients(rng, 300)]
    out = crosstab.master(ClientMockProtocol(frames, crosstab), frames[0], row="sex", column="stage")
    both = pd.concat(frames, ignore_index=True)
    pooled = pd.crosstab(both["sex"], both["stage"])
    assert out["rows"] == list(pooled.index) and out["columns"] == list(pooled.columns)
    assert out["table"] == pooled.to_numpy().tolist() and out["n"] == 500 and not out["suppressed"]
    ref = chi2_contingency(pooled.to_numpy(), correction=False)
    np.testing.assert_allclose(out["chi2"], ref[0], rtol=1e-10)
    assert out["dof"] == ref[2]
    small = crosstab.RPC_crosstab_partial(frames[0].head(12), "sex", "stage")
    assert small["suppressed"] and 0 in {n for cells in small["table"].values() for n in cells.values()}


def test_kaplan_meier_matches_pooled_estimator():
    import pandas as pd

    from vantage6_b200.algorithm.builtin import kaplan_meier

    rng = np.random.default_rng(5)
    frames = [_patients(rng, 150), _patients(rng, 90, 6.0)]
    out = kaplan_meier.master(ClientMockProtocol(frames, kaplan_meier), frames[0], time_column="time", censor_column="event")
    pooled = pd.concat(frames)
    t, e = pooled["time"].to_numpy(), pooled["event"].to_numpy().astype(bool)
    s, ref = 1.0, []
    for ti in sorted(set(t[e])):
        s *= 1.0 - ((t == ti) & e).sum() / (t >= ti).sum()
        ref.append(s)
    np.testing.assert_allclose([c["survival"] for c in out["curve"]], ref, rtol=1e-12)
    assert out["n"] == 240 and out["curve"][0]["at_risk"] <= 240
    assert out["median_survival"] == next(c["time"] for c in out["curve"] if c["survival"] <= 0.5)
    assert all(b["std_err"] >= 0 for b in out["curve"])
    binned = kaplan_meier.master(ClientMockProtocol(frames, kaplan_meier), frames[0], "time", "event", bin_width=6.0)
    assert len(binned["curve"]) < len(out["curve"]) and all(c["time"] % 6.0 == 0 for c in binned["curve"])
    with pytest.raises(PermissionError):
        kaplan_meier.RPC_event_times(frames[0].head(3), "time", "event")


def test_component_inventory_is_current():
    """docs/INVENTORY.md maps every SURVEY.md section-2 item to file:line; the generator fails when a symbol moved."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "inventory.py")], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert out.returncode == 0, out.stderr[-500:]
    import re

    strip = lambda text: re.sub(r"(\.\w+):\d+`", r"\1`", text)          # noqa: E731 -- line numbers drift with every edit; symbols must not
    with open(os.path.join(ROOT, "docs", "INVENTORY.md")) as f:
        assert strip(f.read()) == strip(out.stdout), "docs/INVENTORY.md is stale: python scripts/inventory.py > docs/INVENTORY.md"


def test_serialization_roundtrip_property():
    """Any nesting of JSON scalars, bytes and numpy arrays survives ``serialize`` -> ``deserialize`` (hypothesis)."""
    import math

    from hypothesis import given, settings
    from hypothesis import strategies as st
    from hypothesis.extra import numpy as hnp

    arrays = st.one_of(*[hnp.arrays(dt, hnp.array_shapes(min_dims=0, max_dims=3, max_side=4))
                         for dt in (np.float32, np.float64, np.int32, np.int64, np.uint8, np.bool_)])
    leaves = st.one_of(st.none(), st.booleans(), st.integers(-2**53, 2**53), st.floats(allow_nan=True, allow_infinity=True),
                       st.text(max_size=20), st.binary(max_size=32), arrays)
    trees = st.recursive(leaves, lambda kids: st.one_of(st.lists(kids, max_size=4), st.dictionaries(st.text(max_size=8), kids, max_size=4)),
                         max_leaves=12)

    def same(a, b) -> bool:
        if isinstance(a, np.ndarray):
            return isinstance(b, np.ndarray) and a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a, b, equal_nan=a.dtype.kind == "f")
        if isinstance(a, float):
            return isinstance(b, float) and (a == b or (math.isnan(a) and math.isnan(b)))
        if isinstance(a, dict):
            return isinstance(b, dict) and a.keys() == b.keys() and all(same(a[k], b[k]) for k in a)
        if isinstance(a, list):
            return isinstance(b, list) and len(a) == len(b) and all(same(x, y) for x, y in zip(a, b))
        return type(a) is type(b) and a == b

    @settings(max_examples=150, deadline=None)
    @given(trees)
    def check(tree):
        assert same(tree, deserialize(serialize(tree)))

    check()
    for special in (float("nan"), float("inf"), float("-inf")):           # bare non-finite tokens are still JSON, not "pickle"
        assert same(special, deserialize(serialize(special)))


@pytest.mark.parametrize("family", ["gaussian", "binomial", "poisson"])
def test_glm_irls_matches_pooled_fit(family):
    """Fisher scoring over three mock nodes against scikit-learn fitted on the pooled rows (no penalty)."""
    from sklearn.linear_model import LinearRegression, LogisticRegression, PoissonRegressor

    rng = np.random.default_rng({"gaussian": 1, "binomial": 2, "poisson": 3}[family])
    w_true, b_true = np.array([0.8, -0.5, 0.3, 0.0]), 0.4
    frames = []
    for n in (150, 400, 250):
        X = rng.normal(size=(n, 4))
        eta = X @ w_true + b_true
        y = {"gaussian": eta + rng.normal(scale=0.7, size=n), "binomial": (rng.random(n) < 1 / (1 + np.exp(-eta))).astype(float),
             "poisson": rng.poisson(np.exp(eta)).astype(float)}[family]
        frames.append(np.column_stack([X, y]))
    out = glm.master_irls(ClientMockProtocol(frames, glm), frames[0], family=family)
    pooled = np.concatenate(frames)
    ref = {"gaussian": LinearRegression(), "binomial": LogisticRegression(C=np.inf, tol=1e-10, max_iter=500),
           "poisson": PoissonRegressor(alpha=0.0, tol=1e-10, max_iter=500)}[family].fit(pooled[:, :-1], pooled[:, -1])
    np.testing.assert_allclose(out["coefficients"], np.ravel(ref.coef_), rtol=2e-4, atol=2e-5)
    np.testing.assert_allclose(out["intercept"], float(np.ravel(ref.intercept_)[0]), rtol=2e-4, atol=2e-5)
    assert out["n"] == 800 and out["n_nodes"] == 3 and out["iterations"] <= 12
    assert out["deviance_history"][-1] <= out["deviance_history"][0] + 1e-9
    assert np.all(out["std_errors"] > 0) and np.all(np.abs(out["coefficients"] - w_true) < 5 * out["std_errors"][:-1])
    with pytest.raises(ValueError):
        glm.master_irls(ClientMockProtocol(frames, glm), frames[0], family="gamma")


def test_glm_irls_named_columns_on_frames():
    import pandas as pd

    rng = np.random.default_rng(9)
    frames = []
    for n in (120, 200):
        df = pd.DataFrame({"age": rng.normal(60, 10, n), "dose": rng.normal(2, 1, n), "noise": rng.normal(size=n)})
        df["event"] = (rng.random(n) < 1 / (1 + np.exp(-(0.05 * (df["age"] - 60) + 0.8 * df["dose"] - 1.5)))).astype(float)
        frames.append(df[["event", "age", "dose", "noise"]])            # outcome is NOT the last column
    out = glm.master_irls(ClientMockProtocol(frames, glm), frames[0], family="binomial", columns=["age", "dose"], outcome="event")
    assert len(out["coefficients"]) == 2 and out["coefficients"][1] > 0.3


def test_coxph_matches_pooled_partial_likelihood():
    """Federated Newton iterations against a direct maximisation of the pooled Breslow partial likelihood (scipy)."""
    import pandas as pd
    from scipy.optimize import minimize

    from vantage6_b200.algorithm.builtin import coxph

    rng = np.random.default_rng(11)
    b_true = np.array([0.7, -0.4, 0.0])
    frames = []
    for n in (180, 260, 140):
        X = rng.normal(size=(n, 3))
        t_event = rng.exponential(1.0 / np.exp(X @ b_true))
        t_cens = rng.exponential(2.0, n)
        frames.append(pd.DataFrame({"x1": X[:, 0], "x2": X[:, 1], "x3": X[:, 2], "time": np.round(np.minimum(t_event, t_cens), 2) + 0.01,
                                    "event": (t_event <= t_cens).astype(int)}))
    out = coxph.master(ClientMockProtocol(frames, coxph), frames[0], time_column="time", censor_column="event")
    pooled = pd.concat(frames, ignore_index=True)
    X, t, e = pooled[["x1", "x2", "x3"]].to_numpy(), pooled["time"].to_numpy(), pooled["event"].to_numpy().astype(bool)

    def negll(b):
        r = np.exp(X @ b)
        return -sum((X[(t == u) & e] @ b).sum() - ((t == u) & e).sum() * np.log(r[t >= u].sum()) for u in np.unique(t[e]))

    ref = minimize(negll, np.zeros(3), method="BFGS", options={"gtol": 1e-8})
    np.testing.assert_allclose(out["coefficients"], ref.x, atol=2e-5)
    np.testing.assert_allclose(out["log_likelihood"][-1], -ref.fun, rtol=1e-8)
    assert out["columns"] == ["x1", "x2", "x3"] and out["n"] == 580 and out["n_events"] == int(e.sum()) and out["iterations"] <= 8
    assert all(b > a - 1e-9 for a, b in zip(out["log_likelihood"], out["log_likelihood"][1:]))        # Newton climbs
    assert np.all(np.abs(out["coefficients"] - b_true) < 4 * out["std_errors"])
    np.testing.assert_allclose(out["hazard_ratios"], np.exp(out["coefficients"]))
    with pytest.raises(PermissionError):
        coxph.RPC_event_sums(frames[0].head(4), "time", "event")
    sub = coxph.master(ClientMockProtocol(frames, coxph), frames[0], "time", "event", columns=["x1"], bin_width=0.25)
    assert sub["columns"] == ["x1"] and sub["coefficients"][0] > 0.3


def test_correlation_matches_pooled_complete_cases():
    import pandas as pd

    from vantage6_b200.algorithm.builtin import correlation

    rng = np.random.default_rng(21)
    frames = [_patients(rng, 90), _patients(rng, 140, 4.0), _patients(rng, 60, -2.0)]
    cols = ["age", "bmi", "time"]
    out = correlation.master(ClientMockProtocol(frames, correlation), frames[0], columns=cols)
    pooled = pd.concat(frames, ignore_index=True)[cols].dropna()
    assert out["n"] == len(pooled) < 290                                   # bmi has missing values: complete cases only
    np.testing.assert_allclose(out["mean"], pooled.mean().to_numpy(), rtol=1e-12)
    np.testing.assert_allclose(out["covariance"], pooled.cov().to_numpy(), rtol=1e-9)
    np.testing.assert_allclose(out["correlation"], pooled.corr().to_numpy(), rtol=1e-9)
    assert np.allclose(np.diag(out["correlation"]), 1.0)
    with pytest.raises(PermissionError):
        correlation.RPC_moments(frames[0].head(6), cols)


def test_privacy_floors_belong_to_the_node(monkeypatch):
    """``min_rows`` / ``min_count`` in a task input can tighten the node's floors, never loosen them."""
    from vantage6_b200.algorithm.builtin import crosstab, summary
    from vantage6_b200.algorithm.builtin._common import effective_min_count, effective_min_rows

    rng = np.random.default_rng(5)
    small = _patients(rng, 8)
    with pytest.raises(PermissionError):
        summary.RPC_summary_partial(small, columns=["age"], min_rows=1)          # the researcher asks for less: ignored
    assert effective_min_rows(1) == 10 and effective_min_rows(50) == 50 and effective_min_count(0) == 5
    monkeypatch.setenv("V6B200_MIN_ROWS", "5")                                     # the node's operator lowers the floor
    monkeypatch.setenv("V6B200_MIN_COUNT", "2")
    assert summary.RPC_summary_partial(small, columns=["age"], min_rows=1)["n_rows"] == 8
    with pytest.raises(PermissionError):
        summary.RPC_summary_partial(small, columns=["age"], min_rows=9)           # stricter than the floor: honoured
    frame = _patients(rng, 30)
    lax = crosstab.RPC_crosstab_partial(frame, "sex", "stage", min_count=0)
    strict = crosstab.RPC_crosstab_partial(frame, "sex", "stage", min_count=8)
    cells = lambda part: [n for row in part["table"].values() for n in row.values()]      # noqa: E731
    assert all(n == 0 or n >= 2 for n in cells(lax)) and all(n == 0 or n >= 8 for n in cells(strict))
    monkeypatch.setenv("V6B200_MIN_ROWS", "not-a-number")
    assert effective_min_rows() == 10
