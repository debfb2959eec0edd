"""API defaulting + validation, ported as *specs* from the reference tables
(pkg/apis/kubeflow/v2beta1/default_test.go:24-164,
pkg/apis/kubeflow/validation/validation_test.go:29-415)."""
import os

import pytest

from mpi_operator_b200.api import constants as C
from mpi_operator_b200.api import yaml_io
from mpi_operator_b200.api.defaults import set_defaults_mpijob
from mpi_operator_b200.api.types import MPIJob, MPIJobSpec, ReplicaSpec, RunPolicy, SchedulingPolicy
from mpi_operator_b200.api.validation import (ERR_INVALID, ERR_NOT_SUPPORTED, ERR_REQUIRED, validate_mpijob)

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ONE_CONTAINER = {"spec": {"containers": [{}]}}


def _spec(**kw):
    base = dict(slots_per_worker=2, run_policy=RunPolicy(clean_pod_policy="Running"), ssh_auth_mount_path="/home/mpiuser/.ssh",
                mpi_implementation="Intel",
                mpi_replica_specs={"Launcher": ReplicaSpec(replicas=1, restart_policy="Never", template=ONE_CONTAINER)})
    base.update(kw)
    return MPIJobSpec(**base)


# ------------------------------------------------------------------ defaults --
def test_defaults_base():
    j = set_defaults_mpijob(MPIJob())
    assert j.spec.slots_per_worker == 1
    assert j.spec.run_policy.clean_pod_policy == "None"
    assert j.spec.ssh_auth_mount_path == "/root/.ssh"
    assert j.spec.mpi_implementation == "OpenMPI"
    assert j.spec.launcher_creation_policy == "AtStartup"


def test_defaults_base_overridden():
    j = MPIJob(spec=MPIJobSpec(slots_per_worker=10, ssh_auth_mount_path="/home/mpiuser/.ssh", mpi_implementation="Intel",
                               launcher_creation_policy="WaitForWorkersReady",
                               run_policy=RunPolicy(clean_pod_policy="Running", ttl_seconds_after_finished=2,
                                                    active_deadline_seconds=3, backoff_limit=4)))
    want = j.deepcopy()
    assert set_defaults_mpijob(j) == want


def test_defaults_launcher_and_worker():
    j = MPIJob(spec=MPIJobSpec(mpi_replica_specs={"Launcher": ReplicaSpec(), "Worker": ReplicaSpec()}))
    set_defaults_mpijob(j)
    assert (j.spec.replica("Launcher").replicas, j.spec.replica("Launcher").restart_policy) == (1, "OnFailure")
    assert (j.spec.replica("Worker").replicas, j.spec.replica("Worker").restart_policy) == (0, "Never")


def test_defaults_replica_overrides_kept():
    j = MPIJob(spec=MPIJobSpec(mpi_replica_specs={"Launcher": ReplicaSpec(restart_policy="Never"),
                                                  "Worker": ReplicaSpec(replicas=3, restart_policy="OnFailure")}))
    set_defaults_mpijob(j)
    assert j.spec.replica("Launcher").restart_policy == "Never"
    assert (j.spec.replica("Worker").replicas, j.spec.replica("Worker").restart_policy) == (3, "OnFailure")


def test_defaults_idempotent_and_roundtrip():
    j = yaml_io.load_file(os.path.join(REPO, "examples", "pi", "pi.yaml"))[0]
    a = set_defaults_mpijob(j.deepcopy())
    assert set_defaults_mpijob(a.deepcopy()) == a
    assert MPIJob.from_dict(a.to_dict()) == a


# ---------------------------------------------------------------- validation --
def _errs(job):
    return [(e.type, e.field) for e in validate_mpijob(job)]


@pytest.mark.parametrize("impl", ["Intel", "MPICH", "OpenMPI"])
def test_valid(impl):
    assert _errs(MPIJob(metadata={"name": "foo"}, spec=_spec(mpi_implementation=impl))) == []
    specs = {"Launcher": ReplicaSpec(replicas=1, restart_policy="OnFailure", template=ONE_CONTAINER),
             "Worker": ReplicaSpec(replicas=3, restart_policy="Never", template=ONE_CONTAINER)}
    assert _errs(MPIJob(metadata={"name": "foo"}, spec=_spec(mpi_implementation=impl, mpi_replica_specs=specs))) == []


def test_empty_job():
    assert _errs(MPIJob()) == [
        (ERR_INVALID, "metadata.name"), (ERR_REQUIRED, "spec.mpiReplicaSpecs"), (ERR_REQUIRED, "spec.slotsPerWorker"),
        (ERR_REQUIRED, "spec.runPolicy.cleanPodPolicy"), (ERR_REQUIRED, "spec.sshAuthMountPath"),
        (ERR_NOT_SUPPORTED, "spec.mpiImplementation")]


def test_invalid_fields():
    specs = {"Launcher": ReplicaSpec(replicas=1, restart_policy="Never", template=ONE_CONTAINER),
             "Worker": ReplicaSpec(replicas=1000, restart_policy="Never", template=ONE_CONTAINER)}
    j = MPIJob(metadata={"name": "this-name-is-waaaaaaaay-too-long-for-a-worker-hostname"},
               spec=_spec(mpi_implementation="Unknown", mpi_replica_specs=specs,
                          run_policy=RunPolicy(clean_pod_policy="unknown", ttl_seconds_after_finished=-1,
                                               active_deadline_seconds=-1, backoff_limit=-1, managed_by="other.sigs.k8s.io/other")))
    assert _errs(j) == [
        (ERR_INVALID, "metadata.name"), (ERR_NOT_SUPPORTED, "spec.runPolicy.cleanPodPolicy"),
        (ERR_INVALID, "spec.runPolicy.ttlSecondsAfterFinished"), (ERR_INVALID, "spec.runPolicy.activeDeadlineSeconds"),
        (ERR_INVALID, "spec.runPolicy.backoffLimit"), (ERR_NOT_SUPPORTED, "spec.runPolicy.managedBy"),
        (ERR_NOT_SUPPORTED, "spec.mpiImplementation")]
    assert all(e.origin == "minimum" for e in validate_mpijob(j) if "Seconds" in e.field or "backoff" in e.field)


def test_empty_replica_specs():
    j = MPIJob(metadata={"name": "foo"}, spec=_spec(mpi_replica_specs={}, mpi_implementation="OpenMPI"))
    assert _errs(j) == [(ERR_REQUIRED, "spec.mpiReplicaSpecs[Launcher]")]


def test_missing_replica_spec_fields():
    j = MPIJob(metadata={"name": "foo"}, spec=_spec(mpi_replica_specs={"Launcher": ReplicaSpec(), "Worker": ReplicaSpec()}))
    assert _errs(j) == [
        (ERR_REQUIRED, "spec.mpiReplicaSpecs[Launcher].replicas"), (ERR_NOT_SUPPORTED, "spec.mpiReplicaSpecs[Launcher].restartPolicy"),
        (ERR_REQUIRED, "spec.mpiReplicaSpecs[Launcher].template.spec.containers"),
        (ERR_REQUIRED, "spec.mpiReplicaSpecs[Worker].replicas"), (ERR_NOT_SUPPORTED, "spec.mpiReplicaSpecs[Worker].restartPolicy"),
        (ERR_REQUIRED, "spec.mpiReplicaSpecs[Worker].template.spec.containers")]


def test_invalid_replica_fields():
    specs = {"Launcher": ReplicaSpec(replicas=2, restart_policy="Always", template=ONE_CONTAINER),
             "Worker": ReplicaSpec(replicas=0, restart_policy="Invalid", template=ONE_CONTAINER)}
    assert _errs(MPIJob(metadata={"name": "foo"}, spec=_spec(mpi_replica_specs=specs))) == [
        (ERR_NOT_SUPPORTED, "spec.mpiReplicaSpecs[Launcher].restartPolicy"), (ERR_INVALID, "spec.mpiReplicaSpecs[Launcher].replicas"),
        (ERR_NOT_SUPPORTED, "spec.mpiReplicaSpecs[Worker].restartPolicy"), (ERR_INVALID, "spec.mpiReplicaSpecs[Worker].replicas")]


def test_invalid_name():
    assert _errs(MPIJob(metadata={"name": "1-foo"}, spec=_spec())) == [(ERR_INVALID, "metadata.name")]
    msg = validate_mpijob(MPIJob(metadata={"name": "1-foo"}, spec=_spec())).to_aggregate()
    assert 'invalid DNS label "1-foo-worker-0"' in msg and "DNS-1035" in msg


def test_aggregate_format():
    agg = validate_mpijob(MPIJob(metadata={"name": "foo"}, spec=_spec(mpi_implementation="X", slots_per_worker=None))).to_aggregate()
    assert agg.startswith("[spec.slotsPerWorker: Required value: must have number of slots per worker, ")
    assert 'spec.mpiImplementation: Unsupported value: "X": supported values: "Intel", "MPICH", "OpenMPI"]' in agg


def test_reference_examples_load_and_validate():
    """The upstream project's v2beta1 example manifests, stored unmodified under tests/golden/reference_examples."""
    for f in ["pi/pi.yaml", "pi/pi-intel.yaml", "pi/pi-mpich.yaml", "horovod/tensorflow-mnist.yaml",
              "tensorflow-benchmarks/tensorflow-benchmarks.yaml"]:
        jobs = yaml_io.load_file(os.path.join(REPO, "tests", "golden", "reference_examples", f))
        assert len(jobs) == 1 and not validate_mpijob(set_defaults_mpijob(jobs[0]))


def test_scheduling_policy_roundtrip():
    sp = SchedulingPolicy(min_available=3, queue="q", min_resources={"nvidia.com/gpu": "4"}, priority_class="high", schedule_timeout_seconds=30)
    d = sp.to_dict()
    assert d == {"minAvailable": 3, "queue": "q", "minResources": {"nvidia.com/gpu": "4"}, "priorityClass": "high", "scheduleTimeoutSeconds": 30}
    assert SchedulingPolicy.from_dict(d) == sp


def test_structural_schema_reports_types_enums_and_quantities_with_field_paths():
    """api/schema.py: the CRD's openAPIV3Schema applied the way kube-apiserver applies it (types, enums, int-or-string), plus the
    core/v1 shapes inside the pod templates the CRD leaves open. Every example manifest in the tree is clean."""
    import glob
    import os

    import yaml

    from mpi_operator_b200.api.schema import core_structural_errors, structural_errors
    repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    seen = 0
    for f in glob.glob(os.path.join(repo, "examples", "*", "*.yaml")):
        for doc in yaml.safe_load_all(open(f)):
            if doc and doc.get("kind") == "MPIJob":
                assert structural_errors(doc) == [], f
                seen += 1
    assert seen >= 6
    tmpl = {"spec": {"containers": [{"name": "c", "command": ["true"], "resources": {"limits": {"nvidia.com/gpu": 1, "cpu": "500m", "memory": "2Gi"}}}]}}
    ok = {"apiVersion": "kubeflow.org/v2beta1", "kind": "MPIJob", "metadata": {"name": "j", "labels": {"a": "b"}},
          "spec": {"slotsPerWorker": 2, "runPolicy": {"backoffLimit": 3, "suspend": False, "ttlSecondsAfterFinished": None,
                                                      "schedulingPolicy": {"minAvailable": 2, "minResources": {"nvidia.com/gpu": 8, "cpu": "4"}}},
                   "mpiImplementation": "Intel", "mpiReplicaSpecs": {"Launcher": {"replicas": 1, "template": tmpl}}}}
    assert structural_errors(ok) == []

    def broken(path, value):
        import copy
        o = copy.deepcopy(ok)
        cur = o
        for k in path[:-1]:
            cur = cur[k]
        cur[path[-1]] = value
        return structural_errors(o)
    assert broken(["spec", "slotsPerWorker"], "2") == ['spec.slotsPerWorker: Invalid value: "string": spec.slotsPerWorker in body must be of type integer: "string"']
    assert broken(["spec", "slotsPerWorker"], True)[0].startswith('spec.slotsPerWorker: Invalid value: "boolean"')
    assert "must be of type int32" in broken(["spec", "slotsPerWorker"], 1 << 40)[0]
    assert broken(["spec", "runPolicy", "suspend"], "yes")[0].startswith("spec.runPolicy.suspend: Invalid value")
    assert "supported values" in broken(["spec", "launcherCreationPolicy"], "Whenever")[0]
    assert broken(["spec", "runPolicy", "schedulingPolicy", "minResources", "nvidia.com/gpu"], [8])[0].endswith('must be of type integer or string: "array"')
    assert "must be an integer" in broken(["spec", "runPolicy", "schedulingPolicy", "minResources", "nvidia.com/gpu"], "1.5")[0]
    assert broken(["spec", "mpiReplicaSpecs", "Launcher", "template"], "pod")[0].startswith("spec.mpiReplicaSpecs.Launcher.template: Invalid value")
    assert "template.spec.containers[0].args[1]" in broken(["spec", "mpiReplicaSpecs", "Launcher", "template", "spec", "containers", 0, "args"], ["-np", 2])[0]
    assert "env[0].value in body must be of type string" in broken(["spec", "mpiReplicaSpecs", "Launcher", "template", "spec", "containers", 0, "env"], [{"name": "A", "value": 1}])[0]
    assert "quantities must match" in broken(["spec", "mpiReplicaSpecs", "Launcher", "template", "spec", "containers", 0, "resources"], {"limits": {"memory": "2 gigs"}})[0]
    assert broken(["metadata"], "name")[0].startswith('metadata: Invalid value: "string"')
    assert structural_errors([]) and structural_errors({"spec": None, "metadata": None}) == []       # nulls are absent fields
    # core objects: types always, required fields only when the REST admission asks
    assert core_structural_errors("pods", {"metadata": {"name": "p"}, "spec": {}}) == []
    assert core_structural_errors("pods", {"metadata": {"name": "p"}, "spec": {}}, required=True) == ["spec.containers: Required value"]
    assert core_structural_errors("pods", {"metadata": {"name": "p"}, "spec": 3})[0].startswith("spec: Invalid value")
    assert core_structural_errors("jobs", {"metadata": {"name": "j"}, "spec": {"backoffLimit": "6", "template": tmpl}})[0].startswith("spec.backoffLimit")
    assert core_structural_errors("configmaps", {"metadata": {"name": "c"}, "data": {"hostfile": 5}})[0].startswith("data.hostfile")
    assert core_structural_errors("volcano-podgroups", {"metadata": {"name": "g"}, "spec": {"minMember": "3"}})[0].startswith("spec.minMember")
    assert core_structural_errors("services", {"metadata": {"name": "s"}, "spec": {"clusterIP": "None"}}) == []
