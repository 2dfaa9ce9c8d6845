"""Tier (i) of SURVEY.md section 4 -- CPU multi-process plumbing through the REAL stack:
``vserver import`` + ``vserver start`` + 2x ``vnode start`` as processes, a researcher client, and
algorithms dispatched / collected through the control plane.

* BASELINE config 1: federated weighted mean of a 1k-parameter vector, 2 CPU nodes + 1 server.
* the canonical column-average algorithm on CSV databases.
* FedAvg (tiny ResNet) where the node partials rendezvous over gloo -- the same algorithm code
  that runs over NVLink symmetric memory on the GPU box.
* federated GLM, control-plane flavour and data-plane (K8+K3 reference path) flavour.
* node restart: a task created while a node is down is picked up by the sync at start-up.
"""
import os
import time

import numpy as np
import pytest

from vantage6_b200.dev import DemoNetwork


@pytest.fixture(scope="module")
def network(tmp_path_factory):
    home = tmp_path_factory.mktemp("v6net")
    rng = np.random.default_rng(0)
    mats = [rng.normal(size=(30, 1000)), rng.normal(loc=1.0, size=(70, 1000))]
    import pandas as pd

    dbs = []
    for i, m in enumerate(mats):
        p = home / f"vec{i}.npy"
        np.save(p, m)
        n = 40 + 20 * i
        pd.DataFrame({"age": rng.normal(55 + 10 * i, 8, n).round(1), "sex": rng.choice(["f", "m"], n)}).to_csv(home / f"patients{i}.csv", index=False)
        dbs.append({"default": str(p), "patients": str(home / f"patients{i}.csv")})
    old = os.environ.get("V6B200_HOME")
    # CPU nodes on any machine: the node processes (and the algorithms they start) inherit this environment, and on a GPU
    # box they would otherwise all pick up device 0 -- two NCCL ranks on one GPU
    cpu_only = pytest.MonkeyPatch()
    cpu_only.setenv("CUDA_VISIBLE_DEVICES", "")
    net = DemoNetwork(2, home=str(home), databases=dbs)
    try:
        net.start()
        net.mats = mats
        yield net
    finally:
        net.stop()
        cpu_only.undo()
        if old is None:
            os.environ.pop("V6B200_HOME", None)
        else:
            os.environ["V6B200_HOME"] = old


def run_task(net, image, input_, orgs=None, timeout=240, database="default"):
    c = net.client()
    task = c.task.create(collaboration=net.collaboration_id, organizations=orgs or [net.org_ids[0]], name="t",
                         image=image, input=input_, database=database)
    try:
        return c.wait_for_results(task["id"], timeout=timeout), c, task
    except TimeoutError:
        raise AssertionError(f"task timed out; logs:\n{net.tail_logs()}")


def test_weighted_mean_1k_vector_two_cpu_nodes(network):
    t0 = time.time()
    res, c, task = run_task(network, "v6b200/weighted-mean", {"method": "master", "master": True})
    out = res[0]["result"]
    assert out is not None, res[0]["log"]
    expected = np.concatenate(network.mats).mean(axis=0)          # == sum_i (n_i/n) * mean_i
    assert out["count"] == 100 and out["n_nodes"] == 2
    np.testing.assert_allclose(out["mean"], expected, rtol=1e-12, atol=1e-12)
    assert out["mean"].shape == (1000,)
    # bookkeeping: one master task + one sub-task with a result per organization, same run
    tasks = c.task.list()
    sub = [t for t in tasks if t["parent"] and t["parent"]["id"] == task["id"]]
    assert len(sub) == 1 and len(sub[0]["results"]) == 2 and sub[0]["run_id"] == task["run_id"]
    assert time.time() - t0 < 60


def test_column_average_on_csv(network, tmp_path):
    import pandas as pd

    # this algorithm reads the `default` database: point a one-off task at CSV content via JSON input
    res, _, _ = run_task(network, "v6b200/weighted-mean", {"method": "partial_sum"}, orgs=network.org_ids)
    counts = sorted(r["result"]["count"] for r in res)
    assert counts == [30, 70]
    from vantage6_b200.algorithm.builtin import average
    from vantage6_b200.client.mock import ClientMockProtocol

    dfs = [pd.DataFrame({"age": [10.0, 20.0]}), pd.DataFrame({"age": [30.0, 40.0, 50.0]})]
    out = average.master(ClientMockProtocol(dfs, average), dfs[0], "age")
    assert out == {"average": 30.0, "count": 5}


def test_client_run_is_create_wait_decode(network):
    c = network.client()
    out = c.run("v6b200/weighted-mean", {"method": "master", "master": True})                 # defaults: my collaboration, my organization
    assert out[0]["count"] == 100 and out[0]["n_nodes"] == 2
    parts = c.run("v6b200/weighted-mean", {"method": "partial_sum"}, organizations=network.org_ids)
    assert sorted(p["count"] for p in parts) == [30, 70]
    with pytest.raises(RuntimeError) as e:                                                     # the node's log travels with the error
        c.run("v6b200/weighted-mean", {"method": "no_such_method"})
    assert "RPC_no_such_method" in str(e.value)
    assert c.run("v6b200/weighted-mean", {"method": "no_such_method"}, raise_on_failure=False) == [None]


def test_summary_on_a_labelled_csv_database(network):
    """Second database label per node (``patients``: CSV) + a two-round master through the real control plane."""
    import pandas as pd

    res, _, _ = run_task(network, "v6b200/summary", {"method": "master", "master": True, "kwargs": {"columns": ["age", "sex"]}},
                         database="patients")
    out = res[0]["result"]
    assert out is not None, res[0]["log"]
    pooled = pd.concat([pd.read_csv(network.home / f"patients{i}.csv") for i in range(2)], ignore_index=True)
    assert out["n_rows"] == 100 and out["n_nodes"] == 2, (out, res[0]["log"][-1500:])
    np.testing.assert_allclose(out["columns"]["age"]["mean"], pooled["age"].mean(), rtol=1e-9)
    np.testing.assert_allclose(out["columns"]["age"]["std"], pooled["age"].std(), rtol=1e-9)
    assert out["columns"]["sex"]["counts"] == pooled["sex"].value_counts().to_dict()


def test_fedavg_tiny_resnet_through_control_plane(network):
    res, _, _ = run_task(network, "v6b200/fedavg",
                         {"method": "master", "master": True,
                          "kwargs": {"model": "resnet_tiny", "rounds": 2, "return_weights": True}}, timeout=400)
    out = res[0]["result"]
    assert out is not None, res[0]["log"]
    assert out["world"] == 2 and len(out["global_loss"]) == 2
    assert all(np.isfinite(out["global_loss"]))
    assert out["data_plane"] == "collective"                       # CPU nodes: gloo
    a, b = out["weights_checksum"]
    assert abs(a - b) < 1e-6 * max(1.0, abs(a))                   # both nodes hold the same global model


def test_glm_control_plane_and_fused(network, tmp_path):
    res, _, _ = run_task(network, "v6b200/glm",
                         {"method": "master_fused", "master": True,
                          "kwargs": {"iterations": 30, "lr": 2.0, "rows_per_node": 4000, "features": 256, "synthetic": True}}, timeout=400)
    out = res[0]["result"]
    assert out is not None, res[0]["log"]
    assert out["world"] == 2 and out["losses"][-1] < out["losses"][0]
    assert out["losses"][-1] < 0.9 * out["losses"][0]
    assert out["coef_error_vs_truth"] < 1.0          # 30 plain gradient steps: close to, not at, the optimum


def test_node_restart_picks_up_missed_task(network):
    from click.testing import CliRunner

    from vantage6_b200.cli.node import cli_node_start, cli_node_stop

    r = CliRunner().invoke(cli_node_stop, ["--user", "-n", "demo-node-1"])
    assert "Stopped" in r.output, r.output
    c = network.client()
    task = c.task.create(collaboration=network.collaboration_id, organizations=[network.org_ids[1]], name="late",
                         image="v6b200/weighted-mean", input={"method": "partial_sum"})
    time.sleep(0.5)
    assert not c.task.get(task["id"])["complete"]
    r = CliRunner().invoke(cli_node_start, ["--user", "-n", "demo-node-1"])
    assert r.exit_code == 0, r.output
    res = c.wait_for_results(task["id"], timeout=120)
    assert res[0]["result"]["count"] == 70


def test_kill_request_targets_only_the_named_task():
    """A ``kill_containers`` event for task T ends T's algorithm processes and leaves the others running."""
    from types import SimpleNamespace
    from unittest.mock import MagicMock

    from vantage6_b200.node import Node

    ctx = SimpleNamespace(config={"server_url": "http://127.0.0.1", "port": 1, "api_path": "/api", "api_key": "k"})
    node = Node(ctx)
    procs = {rid: MagicMock(pid=10_000_000 + rid) for rid in (1, 2, 3)}       # pids that do not exist
    node.running.update(procs)
    node._task_of.update({1: 7, 2: 8, 3: 7})
    node.kill_task(7)
    assert procs[1].kill.called and procs[3].kill.called and not procs[2].kill.called
    node.kill_task()
    assert procs[2].kill.called


def test_allowed_images_is_the_nodes_own_veto():
    """``allowed_images`` in the node configuration: regular expressions matched against the full image name."""
    from types import SimpleNamespace

    from vantage6_b200.node import Node

    base = {"server_url": "http://127.0.0.1", "port": 1, "api_path": "/api", "api_key": "k"}
    Node(SimpleNamespace(config=dict(base))).check_image_allowed("anything/at:all")          # no policy: no veto
    node = Node(SimpleNamespace(config=dict(base, allowed_images=[r"v6b200/(average|glm)(:.*)?", r"harbor2\.vantage6\.ai/demo/.*"])))
    node.check_image_allowed("v6b200/average")
    node.check_image_allowed("v6b200/glm:1.2")
    node.check_image_allowed("harbor2.vantage6.ai/demo/average")
    for image in ("v6b200/fedavg", "evil/v6b200/average", "v6b200/average; rm -rf", "harbor2xvantage6.ai/demo/x"):
        with pytest.raises(PermissionError):
            node.check_image_allowed(image)
    Node(SimpleNamespace(config=dict(base, allowed_images="v6b200/.*"))).check_image_allowed("v6b200/fedavg")


def test_encrypted_collaboration_end_to_end(tmp_path):
    """Encrypted collaboration through the real stack: the researcher seals the input per organization, the nodes unseal it,
    the master's sub-task inputs are sealed by the node's proxy for each destination, partial results come back sealed for the
    organization that started the task -- the server only ever stores ciphertext."""
    rng = np.random.default_rng(7)
    mats = [rng.normal(size=(20, 50)), rng.normal(loc=2.0, size=(60, 50))]
    dbs = []
    for i, m in enumerate(mats):
        np.save(tmp_path / f"vec{i}.npy", m)
        dbs.append(str(tmp_path / f"vec{i}.npy"))
    old = os.environ.get("V6B200_HOME")
    net = DemoNetwork(2, home=str(tmp_path / "home"), name="sealed", databases=dbs, encrypted=True)
    try:
        net.start()
        c = net.client()
        assert c.collaboration.get(net.collaboration_id)["encrypted"] is True
        assert all(o["public_key"] for o in c.organization.list() if o["name"] in net.org_names)      # uploaded by the nodes
        task = c.task.create(collaboration=net.collaboration_id, organizations=[net.org_ids[0]], name="t",
                             image="v6b200/weighted-mean", input={"method": "master", "master": True})
        res = c.wait_for_results(task["id"], timeout=120)
        out = res[0]["result"]
        assert out is not None, res[0]["log"]
        np.testing.assert_allclose(out["mean"], np.concatenate(mats).mean(0), rtol=1e-12)
        assert out["count"] == 80 and out["n_nodes"] == 2
        # what the server stores: sealed envelopes, for the input, the sub-task inputs and every result
        import sqlite3

        db = next((tmp_path / "home").rglob("demo.sqlite"))
        rows = sqlite3.connect(db).execute("SELECT input, result FROM result").fetchall()
        assert len(rows) == 3
        import base64

        for inp, result in rows:
            for blob in (inp, result):
                key, iv, body = blob.split("$")                                 # sealed key, iv, ciphertext -- base64 each
                assert len(base64.b64decode(key)) == 256 and len(base64.b64decode(iv)) == 16
                raw = base64.b64decode(body)
                assert raw and not any(marker in raw for marker in (b'"method"', b'"mean"', b'"sum"', b'"count"', b"__ndarray__"))
        # a researcher of the other organization cannot read what was sealed for organization 0
        other = net.client(user=1)
        sealed = other.result.get(res[0]["id"])["result"]
        assert not isinstance(sealed, dict)
    finally:
        net.stop()
        if old is None:
            os.environ.pop("V6B200_HOME", None)
        else:
            os.environ["V6B200_HOME"] = old


def test_finished_result_survives_a_server_outage():
    """The final report is retried with backoff over connection errors and 5xx, not over a definite refusal."""
    from types import SimpleNamespace

    from vantage6_b200.client import ServerError
    from vantage6_b200.node import Node

    node = Node(SimpleNamespace(config={"server_url": "http://127.0.0.1", "port": 1, "api_path": "/api", "api_key": "k"}))
    node.REPORT_BACKOFF_S = (0.01, 0.01, 0.01, 0.01)
    calls = []

    def flaky(endpoint, method="get", json=None, **_):
        calls.append((endpoint, method, json["status"]))
        if len(calls) == 1:
            raise ConnectionRefusedError("server restarting")
        if len(calls) == 2:
            raise ServerError(502, "bad gateway")
        return {}

    node.client.request = flaky
    assert node._report_final(7, {"finished_at": "now", "result": "r", "log": "", "status": "completed"}) is True
    assert calls == [("result/7", "patch", "completed")] * 3
    calls.clear()
    node.client.request = lambda *a, **k: (calls.append(1), (_ for _ in ()).throw(ServerError(400, "Cannot update an already finished result!")))[1]
    assert node._report_final(7, {"status": "completed"}) is False and len(calls) == 1          # refused for good: no retry
    calls.clear()
    node.client.request = lambda *a, **k: (calls.append(1), (_ for _ in ()).throw(ConnectionRefusedError()))[1]
    assert node._report_final(7, {"status": "completed"}) is False and len(calls) == 5          # first try + the whole backoff
    node._stop.set()
    calls.clear()
    assert node._report_final(7, {"status": "completed"}) is False and len(calls) == 1          # a stopping node does not linger


def test_vdev_create_start_use_stop_remove(tmp_path):
    """The developer CLI end to end: separate invocations share the saved network description."""
    from click.testing import CliRunner

    from vantage6_b200.cli.dev import cli_dev
    from vantage6_b200.client import UserClient

    home = str(tmp_path / "devhome")
    old = os.environ.get("V6B200_HOME")
    run = lambda *args: CliRunner().invoke(cli_dev, list(args), catch_exceptions=False)      # noqa: E731
    try:
        r = run("start-demo-network", "-n", "nope", "--home", home)
        assert r.exit_code == 1 and "No demo network" in r.output
        r = run("create-demo-network", "-n", "devnet", "--home", home, "--nodes", "3", "--gpus", "0,1")
        assert r.exit_code == 1 and "--gpus names 2 devices for 3 nodes" in r.output
        for i, n in enumerate((5, 9)):
            np.save(tmp_path / f"v{i}.npy", np.full((n, 4), float(i + 1)))
        r = run("create-demo-network", "-n", "devnet", "--home", home, "--nodes", "2", "--database", str(tmp_path / "v0.npy"),
                "--database", str(tmp_path / "v1.npy"))
        assert r.exit_code == 0 and "Created demo network 'devnet'" in r.output, r.output
        r = run("start-demo-network", "-n", "devnet", "--home", home)
        assert r.exit_code == 0 and "is up" in r.output, r.output
        net = DemoNetwork.load("devnet", home)
        c = UserClient("http://127.0.0.1", net.port, "/api")
        c.authenticate("user-0", net.password)
        c.setup_encryption(None)
        assert sorted(n["status"] for n in c.node.list()) == ["online", "online"]
        collab = c.collaboration.list()[0]
        task = c.task.create(collaboration=collab["id"], organizations=[o["id"] for o in collab["organizations"]], name="t",
                             image="v6b200/weighted-mean", input={"method": "partial_sum"}, database="default")
        res = c.wait_for_results(task["id"], timeout=60)
        assert sorted(r_["result"]["count"] for r_ in res) == [5, 9], [r_["log"] for r_ in res]
        r = run("stop-demo-network", "-n", "devnet", "--home", home)
        assert r.exit_code == 0 and "stopped" in r.output
        with pytest.raises(Exception):
            c.node.list()                                                     # the server is gone
        r = run("remove-demo-network", "-n", "devnet", "--home", home)
        assert r.exit_code == 0
        assert not (tmp_path / "devhome" / "devnet-network.json").exists()
        assert not list((tmp_path / "devhome").rglob("devnet*.yaml"))
    finally:
        CliRunner().invoke(cli_dev, ["stop-demo-network", "-n", "devnet", "--home", home])
        if old is None:
            os.environ.pop("V6B200_HOME", None)
        else:
            os.environ["V6B200_HOME"] = old


def test_tls_network_end_to_end(tmp_path):
    """The whole stack over TLS (``vdev ... --tls`` / ``DemoNetwork(tls=True)``): researcher -> server https, node -> server
    https + wss events, algorithm -> node proxy -> server https, all verified against the server's certificate."""
    for i, n in enumerate((4, 6)):
        np.save(tmp_path / f"v{i}.npy", np.full((n, 3), float(i + 1)))
    old = os.environ.get("V6B200_HOME")
    net = DemoNetwork(2, home=str(tmp_path / "home"), name="tlsnet", databases=[str(tmp_path / "v0.npy"), str(tmp_path / "v1.npy")], tls=True)
    try:
        net.start()
        c = net.client()
        assert c.host.startswith("https://")
        task = c.task.create(collaboration=net.collaboration_id, organizations=[net.org_ids[0]], name="t",
                             image="v6b200/weighted-mean", input={"method": "master", "master": True})
        res = c.wait_for_results(task["id"], timeout=120)
        assert res[0]["result"] is not None, res[0]["log"]
        np.testing.assert_allclose(res[0]["result"]["mean"], np.full(3, (4 * 1.0 + 6 * 2.0) / 10))
        logs = net.tail_logs(200)
        assert "event channel: websocket" in logs and "listening on https://" in logs
        from vantage6_b200.client import UserClient

        with pytest.raises(Exception):                      # no CA file: the self-signed certificate is not trusted
            UserClient("https://127.0.0.1", net.port, "/api").util.get_server_version()
    finally:
        net.stop()
        if old is None:
            os.environ.pop("V6B200_HOME", None)
        else:
            os.environ["V6B200_HOME"] = old
