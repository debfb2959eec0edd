"""Object store / clientset / fake / informers / listers / apply configurations / workqueue
(reference machinery: pkg/client/**, client-go workqueue)."""
import os
import threading
import time

import pytest

from mpi_operator_b200.api import yaml_io
from mpi_operator_b200.client import (ApiError, Clientset, FakeClientset, ObjectStore, SharedInformerFactory, is_already_exists,
                                      is_conflict, is_not_found)
from mpi_operator_b200.client import applyconfiguration as ac
from mpi_operator_b200.controller.workqueue import (BucketRateLimiter, ItemExponentialFailureRateLimiter, MaxOfRateLimiter,
                                                    RateLimitingQueue)

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _pod(name, ns="default", labels=None, owner=None):
    md = {"name": name, "namespace": ns, "labels": labels or {}}
    if owner:
        md["ownerReferences"] = [{"apiVersion": "v1", "kind": "Pod", "name": owner["metadata"]["name"], "uid": owner["metadata"]["uid"], "controller": True}]
    return {"apiVersion": "v1", "kind": "Pod", "metadata": md, "spec": {"containers": [{}]}}


def test_store_crud_resource_version_conflict_and_status_subresource():
    s = ObjectStore()
    a = s.create("pods", _pod("a"))
    assert a["metadata"]["uid"] and a["metadata"]["resourceVersion"] == "1"
    with pytest.raises(ApiError) as e:
        s.create("pods", _pod("a"))
    assert is_already_exists(e.value)
    stale = dict(a)
    a["spec"]["nodeName"] = "n"
    b = s.update("pods", a)
    assert b["metadata"]["resourceVersion"] != a["metadata"]["resourceVersion"] and b["metadata"]["generation"] == 2
    with pytest.raises(ApiError) as e:
        s.update("pods", stale)
    assert is_conflict(e.value)
    b["status"] = {"phase": "Running"}
    b["spec"]["nodeName"] = "IGNORED-by-status-update"
    c = s.update_status("pods", b)
    assert c["status"]["phase"] == "Running" and c["spec"]["nodeName"] == "n"
    c["status"] = {"phase": "Failed"}
    d = s.update("pods", c)  # update() must not touch status of a status-subresource kind
    assert d["status"]["phase"] == "Running"
    assert s.update("pods", d)["metadata"]["resourceVersion"] == d["metadata"]["resourceVersion"]  # no-op: no new version
    with pytest.raises(ApiError) as e:
        s.get("pods", "default", "zzz")
    assert is_not_found(e.value)
    assert [p["metadata"]["name"] for p in s.list("pods", "default")] == ["a"]
    assert s.patch("pods", "default", "a", {"metadata": {"labels": {"x": "y"}}})["metadata"]["labels"] == {"x": "y"}


def test_store_owner_reference_garbage_collection_and_watch():
    s = ObjectStore()
    events = []
    s.watch("pods", lambda t, o, old: events.append((t, o["metadata"]["name"])))
    owner = s.create("pods", _pod("owner"))
    s.create("pods", _pod("child", owner=owner))
    s.create("pods", _pod("grandchild", owner=s.get("pods", "default", "child")))
    s.delete("pods", "default", "owner")
    assert s.list("pods") == []
    assert [e for e in events if e[0] == "DELETED"] == [("DELETED", "owner"), ("DELETED", "child"), ("DELETED", "grandchild")]


def test_store_persistence_roundtrip(tmp_path):
    path = str(tmp_path / "store.json")
    s = ObjectStore(path)
    s.create("configmaps", {"apiVersion": "v1", "kind": "ConfigMap", "metadata": {"name": "cm", "namespace": "ns"}, "data": {"k": "v"}})
    s2 = ObjectStore(path)  # daemon restart re-adopts state (SURVEY.md §5.4)
    assert s2.get("configmaps", "ns", "cm")["data"] == {"k": "v"}
    assert int(s2.create("pods", _pod("p"))["metadata"]["resourceVersion"]) > 1


def test_store_journal_replay_compaction_and_torn_tail(tmp_path):
    """Persistence is a snapshot + an append-only journal: every mutation (including owner-reference garbage collection)
    is one appended record, a restart replays the journal over the snapshot, a torn last record of a crashed writer is
    ignored, and the journal is folded into a new snapshot every kCompactEvery records."""
    import json
    import os
    path = str(tmp_path / "store.json")
    s = ObjectStore(path)
    owner = s.create("configmaps", {"apiVersion": "v1", "kind": "ConfigMap", "metadata": {"name": "owner", "namespace": "ns"}})
    ref = [{"apiVersion": "v1", "kind": "ConfigMap", "name": "owner", "uid": owner["metadata"]["uid"], "controller": True}]
    child = _pod("child")
    child["metadata"]["namespace"] = "ns"
    child["metadata"]["ownerReferences"] = ref
    s.create("pods", child)
    keep = s.create("pods", _pod("keep"))
    keep["spec"]["nodeName"] = "n1"
    s.update("pods", keep)
    s.delete("configmaps", "ns", "owner")              # cascades to the child pod
    assert os.path.exists(path + ".wal") and not os.path.exists(path)   # only journal records so far
    records = [json.loads(ln) for ln in open(path + ".wal")]
    assert [(r["r"], r["k"], "o" in r) for r in records][-2:] == [("configmaps", "ns/owner", False), ("pods", "ns/child", False)]
    with open(path + ".wal", "a") as f:
        f.write('{"rv": 999, "r": "pods", "k": "default/half')   # crash in the middle of an append
    s2 = ObjectStore(path)
    assert [p["metadata"]["name"] for p in s2.list("pods")] == ["keep"] and s2.list("configmaps") == []
    assert s2.get("pods", "default", "keep")["spec"]["nodeName"] == "n1"
    assert os.path.exists(path) and not os.path.exists(path + ".wal")    # replay ends with a fresh snapshot
    assert int(s2.create("pods", _pod("next"))["metadata"]["resourceVersion"]) > int(keep["metadata"]["resourceVersion"])
    # compaction
    s2.kCompactEvery = 20
    for i in range(30):
        s2.create("configmaps", {"apiVersion": "v1", "kind": "ConfigMap", "metadata": {"name": f"c{i}", "namespace": "ns"}})
    snap = json.load(open(path))
    assert len(snap["objects"]["configmaps"]) >= 19
    s3 = ObjectStore(path)
    assert len(s3.list("configmaps")) == 30 and len(s3.list("pods")) == 2


def test_clientset_typed_roundtrip_label_selector_and_delete_collection():
    cs = Clientset(ObjectStore())
    job = yaml_io.load_file(os.path.join(REPO, "examples", "pi", "pi.yaml"))[0]
    c = cs.kubeflow_v2beta1().mpijobs("team-a")
    created = c.create(job)
    assert created.namespace == "team-a" and created.uid
    assert c.get("pi").spec.replica("Worker").replicas == 2
    assert [j.name for j in c.list().items] == ["pi"]
    patched = c.patch("pi", {"spec": {"mpiReplicaSpecs": {"Worker": {"replicas": 5}}}})
    assert patched.spec.replica("Worker").replicas == 5 and patched.spec.replica("Launcher") is not None
    assert c.delete_collection() == 1 and c.list().items == []


def test_fake_clientset_records_actions_and_reactors_inject_faults():
    f = FakeClientset(_pod("seed"))
    kube = f.kube()
    kube.pods("default").create(_pod("x"))
    kube.pods("default").delete("x")
    assert [(a.verb, a.resource, a.name) for a in f.actions] == [("create", "pods", "x"), ("delete", "pods", "x")]

    def boom(action):
        if action.matches("create", "services"):
            raise ApiError("Forbidden", "no", 403)
    f.prepend_reactor(boom)
    with pytest.raises(ApiError):
        kube.services("default").create({"metadata": {"name": "s"}})


def test_informer_namespace_scoping_lister_and_handlers():
    s = ObjectStore()
    s.create("pods", _pod("pre", "a"))
    f = SharedInformerFactory(s, namespace="a")
    inf = f.informer_for("pods")
    seen = []
    inf.add_event_handler(add=lambda o: seen.append(("add", o["metadata"]["name"])),
                          update=lambda old, new: seen.append(("update", new["metadata"]["name"])),
                          delete=lambda o: seen.append(("delete", o["metadata"]["name"])))
    f.start()
    assert f.wait_for_cache_sync()
    s.create("pods", _pod("other-ns", "b"))
    p = s.create("pods", _pod("live", "a", labels={"k": "v"}))
    p["metadata"]["labels"]["k"] = "w"
    s.update("pods", p)
    s.delete("pods", "a", "live")
    assert seen == [("add", "pre"), ("add", "live"), ("update", "live"), ("delete", "live")]
    lister = f.lister_for("pods")
    assert [o["metadata"]["name"] for o in lister.namespaced("a").list()] == ["pre"]
    with pytest.raises(ApiError):
        lister.namespaced("a").get("live")


def test_apply_configuration_builders_and_server_side_apply():
    cfg = (ac.MPIJob("j", "ns").with_labels({"a": "b"})
           .with_spec(ac.MPIJobSpec().with_slots_per_worker(4).with_mpi_implementation("Intel")
                      .with_run_policy(ac.RunPolicy().with_clean_pod_policy("All").with_backoff_limit(2)
                                       .with_scheduling_policy(ac.SchedulingPolicy().with_min_available(3).with_queue("q")))
                      .with_mpi_replica_specs({"Launcher": ac.ReplicaSpec().with_replicas(1).with_template({"spec": {"containers": [{}]}})})))
    body = cfg.build()
    assert body["spec"]["slotsPerWorker"] == 4 and body["spec"]["runPolicy"]["schedulingPolicy"] == {"minAvailable": 3, "queue": "q"}
    assert body["metadata"] == {"name": "j", "namespace": "ns", "labels": {"a": "b"}}
    cs = Clientset(ObjectStore())
    c = cs.kubeflow_v2beta1().mpijobs("ns")
    assert c.apply(cfg).spec.mpi_implementation == "Intel"
    again = c.apply(ac.MPIJob("j", "ns").with_spec(ac.MPIJobSpec().with_slots_per_worker(8)))
    assert again.spec.slots_per_worker == 8 and again.spec.mpi_implementation == "Intel"  # merge, not replace
    st = c.apply_status(ac.MPIJob("j", "ns").with_status(ac.JobStatus().with_conditions(
        ac.JobCondition().with_type("Created").with_status("True"))))
    assert st.status.conditions[0].type == "Created" and st.spec.slots_per_worker == 8


def test_rate_limiters():
    rl = ItemExponentialFailureRateLimiter(0.005, 1000)
    assert [round(rl.when("k"), 3) for _ in range(5)] == [0.005, 0.01, 0.02, 0.04, 0.08]
    assert rl.num_requeues("k") == 5
    rl.forget("k")
    assert rl.when("k") == 0.005
    for _ in range(40):
        d = rl.when("slow")
    assert d == 1000  # capped at 1000 s like the reference
    t = [0.0]
    b = BucketRateLimiter(10, 3, now=lambda: t[0])
    assert [b.when("x") for _ in range(3)] == [0, 0, 0] and b.when("x") == pytest.approx(0.1)
    assert MaxOfRateLimiter(ItemExponentialFailureRateLimiter(1, 10), BucketRateLimiter(1000, 1000)).when("i") == 1


def test_workqueue_dedup_processing_exclusion_and_delay():
    q = RateLimitingQueue()
    q.add("a"); q.add("a"); q.add("b")
    assert len(q) == 2
    item, _ = q.get(1)
    assert item == "a"
    q.add("a")  # re-added while being processed: deferred until done()
    assert len(q) == 1
    assert q.get(1)[0] == "b"
    q.done("a")
    assert q.get(1)[0] == "a"
    q.done("a"); q.done("b")
    t0 = time.time()
    q.add_after("late", 0.15)
    assert q.get(0.05)[0] is None
    assert q.get(1)[0] == "late" and time.time() - t0 >= 0.14
    q.shut_down()
    assert q.get(0.1) == (None, True)


def test_workqueue_single_worker_per_key_under_threads():
    q = RateLimitingQueue()
    active, overlap, done = set(), [], []
    lock = threading.Lock()

    def worker():
        while True:
            item, shut = q.get(0.5)
            if shut or item is None:
                return
            with lock:
                if item in active:
                    overlap.append(item)
                active.add(item)
            time.sleep(0.002)
            with lock:
                active.discard(item)
                done.append(item)
            q.done(item)
    ts = [threading.Thread(target=worker) for _ in range(4)]
    [t.start() for t in ts]
    for i in range(200):
        q.add(f"k{i % 5}")
    time.sleep(0.8)
    q.shut_down()
    [t.join() for t in ts]
    assert overlap == [] and set(done) == {f"k{i}" for i in range(5)}


def test_event_ttl_prunes_old_events():
    from mpi_operator_b200.controller.events import EventRecorder
    s = ObjectStore()
    rec = EventRecorder(s, ttl_seconds=60)
    job = {"apiVersion": "kubeflow.org/v2beta1", "kind": "MPIJob", "metadata": {"name": "j", "namespace": "default", "uid": "u"}}
    rec.event(job, "Normal", "MPIJobCreated", "created")
    rec.event(job, "Normal", "MPIJobRunning", "running")
    assert len(s.list("events")) == 2
    assert rec.prune() == 0
    import time
    assert rec.prune(now=time.time() + 3600) == 2 and s.list("events") == []
    rec.event(job, "Normal", "MPIJobRunning", "running")      # the correlator's stale entry falls back to a fresh event
    assert len(s.list("events")) == 1


def test_indexer_label_index_tracks_updates_and_deletes():
    from mpi_operator_b200.client.informers import Indexer
    ix = Indexer()

    def pod(name, ns="default", **labels):
        return {"metadata": {"name": name, "namespace": ns, "labels": dict(labels)}}
    ix.add(pod("a", job="j1", role="worker"))
    ix.add(pod("b", job="j1", role="launcher"))
    ix.add(pod("c", job="j2", role="worker"))
    ix.add(pod("d", ns="other", job="j1", role="worker"))
    names = lambda objs: [o["metadata"]["name"] for o in objs]  # noqa: E731
    assert names(ix.list("default", {"job": "j1"})) == ["a", "b"]
    assert names(ix.list("", {"job": "j1", "role": "worker"})) == ["a", "d"]          # sorted by namespace/name key
    assert ix.list("default", {"job": "nope"}) == [] and ix.list("default", {"missing": "x"}) == []
    assert names(ix.list("default")) == ["a", "b", "c"]
    ix.update(pod("a", job="j2", role="worker"))                                        # relabelled: leaves j1, joins j2
    assert names(ix.list("default", {"job": "j1"})) == ["b"] and names(ix.list("default", {"job": "j2"})) == ["a", "c"]
    ix.delete(pod("c"))
    assert names(ix.list("default", {"job": "j2"})) == ["a"]
    ix.delete(pod("a"))
    assert ix.list("default", {"job": "j2"}) == [] and ("job", "j2") not in ix._by_label
    got = ix.list("default", {"job": "j1"})[0]
    got["metadata"]["labels"]["job"] = "mutated"                                        # callers get copies
    assert names(ix.list("default", {"job": "j1"})) == ["b"]


def test_object_names_follow_the_apiserver_rule_and_cannot_escape_directories():
    """metadata.name / namespace: DNS-1123 subdomain (apimachinery IsDNS1123Subdomain). Pod names become directory names under the
    node agent's state dir, so '/', '..' and friends must never get into the store."""
    from mpi_operator_b200.api import meta as M
    s = ObjectStore()
    for bad in ("../../etc", "a/b", "..", "Upper", "under_score", "-lead", "trail-", "a..b", "", "x" * 254):
        assert M.name_problem(bad) is not None, bad
        with pytest.raises(ApiError) as e:
            s.create("pods", {"metadata": {"name": bad, "namespace": "default"}, "spec": {}})
        assert e.value.code == 422
    with pytest.raises(ApiError):
        s.create("pods", {"metadata": {"name": "ok", "namespace": "../up"}, "spec": {}})
    for good in ("a", "1-llama", "foo-worker-0", "job.17ab3", "a.b.c", "x" * 253):
        assert M.name_problem(good) is None, good
        s.create("pods", {"metadata": {"name": good, "namespace": "default"}, "spec": {}})
