"""SDK models / ApiClient (reference: sdk/python/v2beta1/test/*.py stubs + mpijob/api_client.py) and the
daemon's REST surface, leader election, healthz, metrics (cmd/mpi-operator/app/server.go)."""
import json
import os
import socket
import time
import urllib.error
import urllib.request

import pytest

import mpijob
from mpi_operator_b200.cmd.options import ServerOption, parse
from mpi_operator_b200.cmd.server import LeaderElector, Operator
from mpi_operator_b200.client import ObjectStore

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def test_models_required_fields_equality_and_serialisation():
    with pytest.raises(ValueError):
        mpijob.V2beta1JobCondition(type="Created")  # status is required
    with pytest.raises(ValueError):
        mpijob.V2beta1MPIJobSpec()  # mpi_replica_specs is required
    with pytest.raises(ValueError):
        mpijob.V2beta1MPIJobList()
    a = mpijob.V2beta1RunPolicy(clean_pod_policy="Running", backoff_limit=3)
    b = mpijob.V2beta1RunPolicy(clean_pod_policy="Running", backoff_limit=3)
    assert a == b and not (a != b) and a != mpijob.V2beta1RunPolicy(clean_pod_policy="All")
    assert a.to_dict()["clean_pod_policy"] == "Running" and "Running" in a.to_str() and repr(a) == a.to_str()
    assert mpijob.V2beta1MPIJobSpec.attribute_map["ssh_auth_mount_path"] == "sshAuthMountPath"
    assert mpijob.V2beta1MPIJobSpec.openapi_types["mpi_replica_specs"] == "dict(str, V2beta1ReplicaSpec)"
    job = mpijob.V2beta1MPIJob(api_version="kubeflow.org/v2beta1", kind="MPIJob", metadata=mpijob.V1ObjectMeta(name="x"),
                               spec=mpijob.V2beta1MPIJobSpec(slots_per_worker=2, mpi_replica_specs={
                                   "Launcher": mpijob.V2beta1ReplicaSpec(replicas=1, template={"spec": {"containers": [{"name": "c"}]}})}))
    body = mpijob.ApiClient().sanitize_for_serialization(job)
    assert body == {"apiVersion": "kubeflow.org/v2beta1", "kind": "MPIJob", "metadata": {"name": "x"},
                    "spec": {"slotsPerWorker": 2, "mpiReplicaSpecs": {"Launcher": {"replicas": 1, "template": {"spec": {"containers": [{"name": "c"}]}}}}}}
    back = mpijob.ApiClient().deserialize(json.dumps(body), "V2beta1MPIJob")
    assert isinstance(back.spec.mpi_replica_specs["Launcher"], mpijob.V2beta1ReplicaSpec) and back.spec.slots_per_worker == 2


def test_configuration_and_exceptions():
    c = mpijob.Configuration(host="http://127.0.0.1:1")
    mpijob.Configuration.set_default(c)
    assert mpijob.Configuration.get_default_copy().host == "http://127.0.0.1:1"
    mpijob.Configuration.set_default(None)
    assert "Python SDK Debug Report" in c.to_debug_report()
    with pytest.raises(mpijob.ApiException) as e:
        mpijob.MPIJobClient("127.0.0.1:1").list()
    assert e.value.status == 0 and "daemon running" in str(e.value)
    assert str(mpijob.ApiValueError("bad", path_to_item=["a", 0, "b"])) == "bad at ['a'][0]['b']"


def test_options_defaults_match_reference_flags():
    o = parse([])
    assert (o.threadiness, o.monitoring_port, o.lock_namespace, o.qps, o.burst, o.controller_rate_limit, o.controller_burst) == (2, 0, "mpi-operator", 5, 10, 10, 100)
    o = parse(["--gang-scheduling", "volcano", "--namespace", "ns", "--cluster-domain", "cluster.local", "--threadiness", "4",
               "--kube-api-qps", "50", "--master", "https://x", "--kubeConfig", "/k", "-alsologtostderr".replace("-a", "--a")])
    assert (o.gang_scheduling_name, o.namespace, o.cluster_domain, o.threadiness, o.qps) == ("volcano", "ns", "cluster.local", 4, 50)


def test_leader_election_is_exclusive_and_records_lease(tmp_path):
    store = ObjectStore()
    a = LeaderElector(store, str(tmp_path), "mpi-operator", "a")
    b = LeaderElector(store, str(tmp_path), "mpi-operator", "b")
    assert a.try_acquire() and not b.try_acquire()
    lease = store.get("leases", "mpi-operator", "mpi-operator")
    assert lease["spec"]["holderIdentity"] == "a" and lease["spec"]["leaseDurationSeconds"] == 15
    assert a.healthy()
    a.release()
    assert b.try_acquire()
    assert store.get("leases", "mpi-operator", "mpi-operator")["spec"]["leaseTransitions"] == 1
    b.release()


def test_rest_api_end_to_end_with_sdk_client(tmp_path):
    port = _free_port()
    op = Operator(ServerOption(fake_gpus=2, leader_elect=False, state_dir=str(tmp_path)))
    op.serve(f"127.0.0.1:{port}")
    op.start()
    try:
        base = f"http://127.0.0.1:{port}"
        assert urllib.request.urlopen(base + "/healthz").read() == b"ok"
        assert "version" in json.load(urllib.request.urlopen(base + "/version"))
        assert json.load(urllib.request.urlopen(base + "/topology"))["free_gpus"] == 2
        cli = mpijob.MPIJobClient(f"127.0.0.1:{port}")
        with pytest.raises(mpijob.ApiException):  # admission: structural validation like a CRD schema
            cli.create({"apiVersion": "kubeflow.org/v2beta1", "kind": "MPIJob", "metadata": {"name": "bad"}, "spec": {}})
        body = {"apiVersion": "kubeflow.org/v2beta1", "kind": "MPIJob", "metadata": {"name": "rest"},
                "spec": {"mpiReplicaSpecs": {"Launcher": {"replicas": 1, "template": {"spec": {"containers": [
                    {"name": "l", "command": ["sh", "-c", "echo hello from launcher"]}]}}}}}}
        out, verb = cli.apply(body)
        assert verb == "created" and cli.apply(body)[1] == "unchanged"
        done = cli.wait_for_condition("rest", "Succeeded", timeout=20)
        assert done["status"]["replicaStatuses"]["Launcher"]["succeeded"] == 1
        assert "hello from launcher" in cli.logs("rest")
        assert [j["metadata"]["name"] for j in cli.list()] == ["rest"]
        assert any(e["reason"] == "MPIJobSucceeded" for e in cli.list_resource("events"))
        text = urllib.request.urlopen(base + "/metrics").read().decode()
        assert "mpi_operator_jobs_successful_total" in text and 'mpi_operator_job_info{launcher="rest-launcher",namespace="default"} 1.0' in text
        cli.delete("rest")
        time.sleep(0.2)
        assert cli.list() == [] and cli.list_resource("jobs") == []  # owner-reference GC
        with pytest.raises(mpijob.exceptions.NotFoundException):
            cli.get("rest")
    finally:
        op.stop()


def test_monitoring_port_serves_metrics_and_healthz_only(tmp_path):
    """The reference serves nothing but /metrics on --monitoring-port (cmd/mpi-operator/main.go:29-40). Here that port
    binds 0.0.0.0, so it must not expose the object API (a POSTed Pod is a command the node agent runs; Secrets hold keys)."""
    port, mon = _free_port(), _free_port()
    op = Operator(ServerOption(fake_gpus=0, leader_elect=False, state_dir=str(tmp_path)))
    op.serve(f"127.0.0.1:{port}")
    op.serve(f"127.0.0.1:{mon}", restricted=True)
    op.start()
    try:
        base = f"http://127.0.0.1:{mon}"
        assert "mpi_operator_jobs_created_total" in urllib.request.urlopen(base + "/metrics").read().decode()
        assert urllib.request.urlopen(base + "/healthz").read() == b"ok"
        for path in ("/api/v1/secrets", "/api/v1/namespaces/default/pods", "/apis/kubeflow.org/v2beta1/mpijobs", "/version", "/topology"):
            with pytest.raises(urllib.error.HTTPError) as e:
                urllib.request.urlopen(base + path)
            assert e.value.code == 404
        pod = {"apiVersion": "v1", "kind": "Pod", "metadata": {"name": "evil"}, "spec": {"containers": [{"name": "c", "command": ["true"]}]}}
        for method in ("POST", "PUT", "PATCH", "DELETE"):
            req = urllib.request.Request(base + "/api/v1/namespaces/default/pods", data=json.dumps(pod).encode(), method=method,
                                         headers={"Content-Type": "application/json"})
            with pytest.raises(urllib.error.HTTPError) as e:
                urllib.request.urlopen(req)
            assert e.value.code == 405
        # the full API is still there on the loopback listener
        assert json.load(urllib.request.urlopen(f"http://127.0.0.1:{port}/api/v1/namespaces/default/pods"))["items"] == []
        # names in URLs are object names, never path components of the state dir
        for path in ("/api/v1/namespaces/default/pods/..%2F..%2Fx/log", "/api/v1/namespaces/../pods/x/log", "/api/v1/namespaces/default/pods/../log",
                     "/api/v1/namespaces/default/pods/UPPER"):
            with pytest.raises(urllib.error.HTTPError) as e:
                urllib.request.urlopen(f"http://127.0.0.1:{port}" + path)
            assert e.value.code == 404, path
        evil = dict(pod, metadata={"name": "../../evil"})
        req = urllib.request.Request(f"http://127.0.0.1:{port}/api/v1/namespaces/default/pods", data=json.dumps(evil).encode(), method="POST",
                                     headers={"Content-Type": "application/json"})
        with pytest.raises(urllib.error.HTTPError) as e:
            urllib.request.urlopen(req)
        assert e.value.code == 422
    finally:
        op.stop()


def test_auth_token_file_protects_the_object_api(tmp_path, monkeypatch):
    """--auth-token-file: the reference leans on the cluster's RBAC (manifests/base/cluster-role.yaml); on a shared box the
    loopback API would otherwise let any local user create pods (= run commands as the daemon's user) and read Secrets."""
    import stat
    port, mon = _free_port(), _free_port()
    tok_file = tmp_path / "token"
    op = Operator(ServerOption(fake_gpus=0, leader_elect=False, state_dir=str(tmp_path / "state"), auth_token_file=str(tok_file)))
    op.serve(f"127.0.0.1:{port}")
    op.serve(f"127.0.0.1:{mon}", restricted=True)
    op.start()
    try:
        token = tok_file.read_text().strip()
        assert len(token) >= 32 and stat.S_IMODE(os.stat(tok_file).st_mode) == 0o600
        base = f"http://127.0.0.1:{port}"
        assert urllib.request.urlopen(base + "/healthz").read() == b"ok"            # liveness stays open
        assert "mpi_operator_jobs_created_total" in urllib.request.urlopen(f"http://127.0.0.1:{mon}/metrics").read().decode()
        pod = {"apiVersion": "v1", "kind": "Pod", "metadata": {"name": "evil"}, "spec": {"containers": [{"name": "c", "command": ["true"]}]}}
        for method, path, body in (("GET", "/api/v1/secrets", None), ("GET", "/apis/kubeflow.org/v2beta1/namespaces/default/mpijobs", None),
                                   ("GET", "/metrics", None), ("POST", "/api/v1/namespaces/default/pods", pod),
                                   ("DELETE", "/api/v1/namespaces/default/pods/evil", None)):
            for hdr in ({}, {"Authorization": "Bearer wrong"}, {"Authorization": token}):
                req = urllib.request.Request(base + path, data=json.dumps(body).encode() if body else None, method=method,
                                             headers={"Content-Type": "application/json", **hdr})
                with pytest.raises(urllib.error.HTTPError) as e:
                    urllib.request.urlopen(req)
                assert e.value.code == 401 and json.load(e.value)["reason"] == "Unauthorized"
        assert op.store.list("pods", "default") == []
        monkeypatch.delenv("MPIJOB_TOKEN", raising=False)
        monkeypatch.delenv("MPIJOB_TOKEN_FILE", raising=False)
        from mpi_operator_b200.sdk.exceptions import UnauthorizedException
        with pytest.raises(UnauthorizedException):
            mpijob.MPIJobClient(f"127.0.0.1:{port}").list()
        monkeypatch.setenv("MPIJOB_TOKEN_FILE", str(tok_file))                       # what mpijobctl and the SDK read
        cli = mpijob.MPIJobClient(f"127.0.0.1:{port}")
        assert cli.list() == []
        events = list(cli.watch("mpijobs", "default", timeout=0.3))
        assert events == []
        monkeypatch.delenv("MPIJOB_TOKEN_FILE")
        monkeypatch.setenv("MPIJOB_TOKEN", token)
        assert mpijob.MPIJobClient(f"127.0.0.1:{port}").list() == []
        # a second daemon on the same file adopts the token instead of replacing it
        from mpi_operator_b200.cmd.server import _load_or_create_token
        assert _load_or_create_token(str(tok_file)) == token
    finally:
        op.stop()


def test_models_match_the_reference_sdk_when_installed():
    """Parity with the upstream, unmodified Python SDK (sdk/python/v2beta1): same openapi_types and attribute_map for all
    9 MPIJob models. tests/golden/sdk_v2beta1_models.json holds {name: [openapi_types, attribute_map]} as read from
    that package's `mpijob.models`."""
    with open(os.path.join(GOLDEN, "sdk_v2beta1_models.json")) as f:
        theirs = json.load(f)
    assert sorted(theirs) == sorted(n for n in mpijob.models.MODEL_CLASSES if n.startswith("V2beta1"))
    for name, (types, amap) in theirs.items():
        ours = mpijob.models.MODEL_CLASSES[name]
        assert ours.attribute_map == amap, name
        # the reference generator spells apimachinery types IoK8sApimachineryPkgApisMetaV1X; we use the
        # kubernetes-client names V1X (and export the long names as aliases)
        norm = {k: v.replace("IoK8sApimachineryPkgApisMetaV1", "V1") for k, v in types.items()}
        assert ours.openapi_types == norm, name
    assert mpijob.models.MODEL_CLASSES["IoK8sApimachineryPkgApisMetaV1ObjectMeta"] is mpijob.V1ObjectMeta


def test_generic_models_match_the_reference_sdk_when_installed():
    """The 100 generic apimachinery models (sdk/meta_models.py, one schema table) against the generated files of the
    upstream, unmodified Python SDK: same class names, module names, attribute maps and required fields.
    tests/golden/sdk_generic_models.json holds {class: [attribute_map, required fields, module]} for every generated
    model file of that package except the V2beta1 ones; a field is required when its setter rejects None."""
    from mpi_operator_b200.sdk.meta_models import snake
    with open(os.path.join(GOLDEN, "sdk_generic_models.json")) as f:
        theirs = json.load(f)
    assert len(theirs) == 100
    for name, (amap, required, module) in theirs.items():
        ours = mpijob.models.MODEL_CLASSES.get(name)
        assert ours is not None, name
        assert snake(name) == module, name
        assert set(amap.items()) <= set(ours.attribute_map.items()), name      # (the pod-template side may carry more fields)
        assert sorted(ours.required) == required, name


def test_sdk_example_flow_through_the_kubernetes_shim(tmp_path, monkeypatch):
    """The flow of the upstream SDK's example (sdk/python/v2beta1/tensorflow-mnist.py): an MPIJob assembled from
    kubernetes.client models and the stale `mpijob.V1ReplicaSpec` name, `config.load_kube_config()` and
    `CustomObjectsApi().create_namespaced_custom_object`, served by the single-box daemon through the in-tree `kubernetes`
    compatibility package."""
    from kubernetes import client, config, watch
    from kubernetes.client import V1Container, V1ObjectMeta, V1PodSpec, V1PodTemplateSpec, V1ResourceRequirements
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    op = Operator(ServerOption(fake_gpus=2, leader_elect=False, state_dir=str(tmp_path)))
    op.serve(f"127.0.0.1:{port}")
    op.start()
    try:
        def replica(n, name, limits):
            # command is a plain string, as in the example; the pods get the list form
            c = V1Container(name=name, image="docker.io/kubeflow/mpi-horovod-mnist", command="mpirun",
                            args=["-np", "2", "python", "/examples/tensorflow_mnist.py"],
                            resources=V1ResourceRequirements(limits=limits))
            return mpijob.V1ReplicaSpec(replicas=n, template=V1PodTemplateSpec(spec=V1PodSpec(containers=[c])))
        job = mpijob.V2beta1MPIJob(kind="MPIJob", api_version="kubeflow.org/v2beta1", metadata=V1ObjectMeta(name="tensorflow-mnist"),
                                   spec=mpijob.V2beta1MPIJobSpec(slots_per_worker=1, mpi_replica_specs={
                                       "Launcher": replica(1, "mpi-launcher", {"cpu": "1", "memory": "2Gi"}),
                                       "Worker": replica(2, "mpi-worker", {"cpu": "2", "memory": "4Gi"})}))
        monkeypatch.setenv("MPIJOB_SERVER", f"127.0.0.1:{port}")
        config.load_kube_config()
        client.CustomObjectsApi().create_namespaced_custom_object(group="kubeflow.org", version="v2beta1", namespace="default",
                                                                  plural="mpijobs", body=job)
        api = client.CustomObjectsApi()
        job = api.get_namespaced_custom_object("kubeflow.org", "v2beta1", "default", "mpijobs", "tensorflow-mnist")
        assert job["spec"]["mpiReplicaSpecs"]["Worker"]["replicas"] == 2 and job["spec"]["slotsPerWorker"] == 1
        c = job["spec"]["mpiReplicaSpecs"]["Launcher"]["template"]["spec"]["containers"][0]
        assert c["resources"] == {"limits": {"cpu": "1", "memory": "2Gi"}} and c["args"][:2] == ["-np", "2"]
        # the example passes command="mpirun" (a string); the launcher pod the controller builds has the list form
        launchers = [p for p in client.CoreV1Api().list_namespaced_pod("default", label_selector="training.kubeflow.org/job-role=launcher").items]
        deadline = time.time() + 10
        while not launchers and time.time() < deadline:
            time.sleep(0.1)
            launchers = client.CoreV1Api().list_namespaced_pod("default", label_selector="training.kubeflow.org/job-role=launcher").items
        assert launchers and launchers[0].spec.containers[0].command == ["mpirun"] and launchers[0].metadata.name.startswith("tensorflow-mnist-launcher")
        assert [j["metadata"]["name"] for j in api.list_namespaced_custom_object("kubeflow.org", "v2beta1", "default", "mpijobs")["items"]] == ["tensorflow-mnist"]
        assert [j["metadata"]["name"] for j in api.list_cluster_custom_object("kubeflow.org", "v2beta1", "mpijobs")["items"]] == ["tensorflow-mnist"]
        ev = next(iter(watch.Watch().stream(api.list_namespaced_custom_object, "kubeflow.org", "v2beta1", "default", "mpijobs", timeout_seconds=5)))
        assert ev["type"] == "ADDED" and ev["object"]["metadata"]["name"] == "tensorflow-mnist"
        api.patch_namespaced_custom_object("kubeflow.org", "v2beta1", "default", "mpijobs", "tensorflow-mnist", {"spec": {"runPolicy": {"suspend": True}}})
        assert api.get_namespaced_custom_object_status("kubeflow.org", "v2beta1", "default", "mpijobs", "tensorflow-mnist")["spec"]["runPolicy"]["suspend"] is True
        with pytest.raises(client.rest.ApiException):
            api.get_namespaced_custom_object("example.com", "v1", "default", "widgets", "x")
        core = client.CoreV1Api()
        assert isinstance(core.list_namespaced_pod("default").items, list)
        api.delete_namespaced_custom_object("kubeflow.org", "v2beta1", "default", "mpijobs", "tensorflow-mnist")
        with pytest.raises(client.rest.ApiException):
            api.get_namespaced_custom_object("kubeflow.org", "v2beta1", "default", "mpijobs", "tensorflow-mnist")
    finally:
        op.stop()


def test_watch_stream_delivers_added_modified_deleted_in_order(tmp_path):
    """`GET ...?watch=true` (client-go informers / `kubectl get -w` in the reference, SURVEY.md §3.1): existing objects first,
    then every change as it happens, filtered by namespace / label selector / metadata.name, until timeoutSeconds."""
    import threading
    from mpi_operator_b200.sdk import MPIJobClient
    from helpers import new_mpijob
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    op = Operator(ServerOption(fake_gpus=2, leader_elect=False, state_dir=str(tmp_path)))
    op.serve(f"127.0.0.1:{port}")
    try:
        cli = MPIJobClient(f"127.0.0.1:{port}")       # controller not started: only what this test writes changes the store
        cli.create(new_mpijob("old", workers=1))
        got, done = [], threading.Event()

        def consume():
            for ev in cli.watch("mpijobs", "default", timeout=3.0):
                got.append((ev["type"], ev["object"]["metadata"]["name"]))
            done.set()
        t = threading.Thread(target=consume)
        t.start()
        deadline = time.time() + 5
        while not got and time.time() < deadline:
            time.sleep(0.02)
        cli.create(new_mpijob("new", workers=1))
        cli.create(new_mpijob("elsewhere", namespace="other", workers=1))          # other namespace: filtered out
        cli.patch("new", {"metadata": {"labels": {"team": "a"}}})
        cli.delete("old")
        assert done.wait(10)
        t.join()
        assert got == [("ADDED", "old"), ("ADDED", "new"), ("MODIFIED", "new"), ("DELETED", "old")], got
        by_name = [(e["type"], e["object"]["metadata"]["name"]) for e in cli.watch("mpijobs", None, timeout=0.5, name="elsewhere")]
        assert by_name == [("ADDED", "elsewhere")]
        by_label = [e["object"]["metadata"]["name"] for e in cli.watch("mpijobs", "default", timeout=0.5, label_selector="team=a")]
        assert by_label == ["new"]
    finally:
        op.stop()


def test_go_style_single_dash_flags_and_klog_flags_are_accepted():
    """The reference's Deployment passes `-alsologtostderr` (Go flag syntax); klog's other flags are registered too."""
    o = parse(["-alsologtostderr", "-v=4", "-threadiness", "3", "-lock-namespace=kubeflow", "-logtostderr=true", "-stderrthreshold=INFO",
               "--monitoring-port", "9090", "-v", "2"])
    assert o.threadiness == 3 and o.lock_namespace == "kubeflow" and o.monitoring_port == 9090


def test_api_discovery_documents(tmp_path):
    """`/api`, `/apis`, `/api/v1`, `/apis/kubeflow.org/v2beta1`, `/openapi/v2`: what kubectl / client libraries read first."""
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    op = Operator(ServerOption(fake_gpus=0, leader_elect=False, state_dir=str(tmp_path)))
    op.serve(f"127.0.0.1:{port}")
    try:
        def get(path):
            return json.loads(urllib.request.urlopen(f"http://127.0.0.1:{port}{path}", timeout=5).read())
        assert get("/api")["versions"] == ["v1"]
        groups = {g["name"]: g["preferredVersion"]["groupVersion"] for g in get("/apis")["groups"]}
        assert groups["kubeflow.org"] == "kubeflow.org/v2beta1" and groups["batch"] == "batch/v1" and "scheduling.volcano.sh" in groups
        core = {r["name"]: r for r in get("/api/v1")["resources"]}
        assert core["pods"]["kind"] == "Pod" and core["pods"]["namespaced"] and "pods/log" in core and "watch" in core["events"]["verbs"]
        mj = {r["name"]: r for r in get("/apis/kubeflow.org/v2beta1")["resources"]}
        assert mj["mpijobs"]["kind"] == "MPIJob" and "mpijob" in mj["mpijobs"]["shortNames"] and "mpijobs/status" in mj
        assert "v2beta1.MPIJob" in get("/openapi/v2")["definitions"]
    finally:
        op.stop()


def test_malformed_requests_get_a_status_never_a_dropped_connection(tmp_path):
    """What kube-apiserver does before the reference's controller ever sees an object: bodies that are not JSON objects are
    400, objects whose fields have the wrong TYPE (CRD structural schema, api/schema.py) or an impossible quantity are 422 with
    the field path, and no request ends without a response. Found by fuzzing the REST surface."""
    port = _free_port()
    op = Operator(ServerOption(fake_gpus=2, leader_elect=False, state_dir=str(tmp_path)))
    op.serve(f"127.0.0.1:{port}")
    op.start()
    coll = f"http://127.0.0.1:{port}/apis/kubeflow.org/v2beta1/namespaces/default/mpijobs"
    pods = f"http://127.0.0.1:{port}/api/v1/namespaces/default/pods"

    def call(method, url, raw):
        req = urllib.request.Request(url, data=raw, method=method, headers={"Content-Type": "application/json"})
        try:
            with urllib.request.urlopen(req, timeout=10) as r:
                return r.status, json.load(r)
        except urllib.error.HTTPError as e:
            return e.code, json.load(e)

    def job(**spec):
        base = {"slotsPerWorker": 1, "mpiReplicaSpecs": {"Launcher": {"replicas": 1, "template": {"spec": {"containers": [{"name": "l", "command": ["true"]}]}}}}}
        base.update(spec)
        return json.dumps({"apiVersion": "kubeflow.org/v2beta1", "kind": "MPIJob", "metadata": {"name": "m"}, "spec": base}).encode()
    try:
        for raw in (b"{", b"[]", b'"text"', b"\xff\xfe", b"7"):
            for method, url in (("POST", coll), ("PUT", coll + "/m"), ("PATCH", coll + "/m"), ("POST", pods), ("PATCH", f"http://127.0.0.1:{port}/topology")):
                code, st = call(method, url, raw)
                assert code == 400 and st["kind"] == "Status" and st["reason"] == "BadRequest", (raw, method, code, st)
        for body, needle in (
                (job(slotsPerWorker="two"), "spec.slotsPerWorker in body must be of type integer"),
                (job(runPolicy={"backoffLimit": {}}), "spec.runPolicy.backoffLimit in body must be of type integer"),
                (job(runPolicy=[]), "spec.runPolicy in body must be of type object"),
                (job(mpiImplementation="LAM"), 'supported values: "OpenMPI", "Intel", "MPICH"'),
                (job(mpiReplicaSpecs={"Launcher": {"replicas": 1.5, "template": {}}}), "spec.mpiReplicaSpecs.Launcher.replicas in body must be of type integer"),
                (job(mpiReplicaSpecs={"Launcher": {"replicas": 1, "template": {"spec": {"containers": {"name": "l"}}}}}), "template.spec.containers in body must be of type array"),
                (job(mpiReplicaSpecs={"Launcher": {"replicas": 1, "template": {"spec": {"containers": [{"name": "l", "resources": {"limits": {"nvidia.com/gpu": "lots"}}}]}}}}),
                 "resources.limits.nvidia.com/gpu: Invalid value: \"lots\": quantities must match"),
                (job(mpiReplicaSpecs={"Launcher": {"replicas": 1, "template": {"spec": {"containers": [{"name": "l", "resources": {"limits": {"nvidia.com/gpu": "0.5"}}}]}}}}), "must be an integer"),
                (json.dumps({"kind": "MPIJob", "metadata": 5, "spec": {}}).encode(), ""),
                (json.dumps({"kind": "MPIJob", "metadata": {"name": "m", "labels": {"a": 1}}, "spec": {"mpiReplicaSpecs": {}}}).encode(), "metadata.labels.a in body must be of type string")):
            code, st = call("POST", coll, body)
            assert code in (400, 422) and st["kind"] == "Status" and needle in st["message"], (body, code, st)
        assert op.store.list("mpijobs") == []
        code, st = call("POST", pods, json.dumps({"metadata": {"name": "p"}, "spec": {"containers": [{"name": "c", "resources": {"limits": {"nvidia.com/gpu": "x"}}}]}}).encode())
        assert code == 422 and "quantities must match" in st["message"]
        code, st = call("POST", pods, json.dumps({"metadata": {"name": "p"}}).encode())
        assert code == 422 and "spec: Required value" in st["message"]
        # a well-formed object still goes through, a PATCH that breaks a type does not
        code, st = call("POST", coll, job(runPolicy={"suspend": True}))
        assert code == 201
        code, st = call("PATCH", coll + "/m", json.dumps({"spec": {"slotsPerWorker": "many"}}).encode())
        assert code == 422 and "spec.slotsPerWorker" in st["message"]
        with socket.create_connection(("127.0.0.1", port), timeout=10) as sk:      # announced size over the limit: refused before reading it
            sk.sendall(b"POST /apis/kubeflow.org/v2beta1/namespaces/default/mpijobs HTTP/1.1\r\nHost: x\r\nContent-Type: application/json\r\n"
                       b"Content-Length: 17825792\r\n\r\n{")
            assert sk.recv(4096).startswith(b"HTTP/1.1 413")
    finally:
        op.stop()
