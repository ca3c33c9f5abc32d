"""Provider C-ABI on a real B200 node: what the Go hypervisor would see through purego."""
import ctypes as C
import json
import os
import subprocess
import sys

import pytest

import conftest
import oracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def prov():
    from tensor_fusion_b200 import provider as P
    lib = P.load()
    logs = []
    cb = P.LogCallback(lambda lvl, msg: logs.append((lvl, msg)))
    assert lib.AccelRegisterLogCallback(cb) == P.SUCCESS       # before AccelInit, like accelerator_unix.go:102-117
    assert lib.AccelInit() == P.SUCCESS
    yield P, lib, logs
    lib.AccelShutdown()
    lib.AccelRegisterLogCallback(P.LogCallback())
    del cb


def test_devices_as_the_hypervisor_sees_them(prov):
    P, lib, logs = prov
    rc, devs = P.all_devices(lib)
    assert rc == P.SUCCESS and len(devs) >= 1
    d = devs[0]
    assert d["uuid"].startswith("GPU-") and d["vendor"] == "NVIDIA"       # quota_controller.go:199-202
    assert "B200" in d["model"] and d["sms"] == 148 and d["tflops"] == 2250.0
    assert 170 << 30 < d["memory"] < 200 << 30
    assert d["props"]["computeCapability"] == "10.0"                       # coresPerSM lookup, legacy.go:690-713
    assert d["props"]["totalComputeUnits"] == "148"                        # worker/controller.go:545-549
    assert d["node"].startswith("/dev/nvidia") and d["index"] == 0
    assert d["caps"]["supportsSoftIsolation"] and d["caps"]["supportsRemoting"] and d["caps"]["maxWorkersPerDevice"] == 16
    assert all(l != b"FATAL" for l, _ in logs)


def test_topology_all_peers_tier0(prov):
    P, lib, _ = prov
    topo = P.ExtendedDeviceTopology()
    assert lib.AccelGetAllDevicesTopology(C.byref(topo)) == P.SUCCESS
    n = topo.deviceCount
    assert n >= 1
    for i in range(n):
        t = topo.devices[i]
        assert t.peerCount == n - 1
        for j in range(t.peerCount):
            assert t.peers[j].topoLevel == 0           # TOPO_LEVEL_INTERNAL over NVSwitch


def test_metrics_and_processes(prov):
    import numpy as np
    P, lib, _ = prov
    from tensor_fusion_b200.worker import Worker
    _, devs = P.all_devices(lib)
    with Worker() as w:                                 # a CUDA context with ~0.6 GiB so this pid shows up
        p = w.dev_alloc(512 << 20)
        w.move_batch([(p, 0, 512 << 20, 7)])
        uu = (C.c_char_p * 1)(devs[0]["uuid"].lower().encode())      # Go passes native case but be lenient
        dm = (P.DeviceMetrics * 1)()
        assert lib.AccelGetDeviceMetrics(uu, 1, dm) == P.SUCCESS
        m = dm[0]
        assert 10 < m.powerUsageWatts < 1200 and 10 < m.temperatureCelsius < 100
        assert m.utilizationPercent <= 100 and m.memoryUsedBytes > 512 << 20
        keys = [m.extraMetrics[i].key.decode() for i in range(m.extraMetricsCount)]
        assert "clockSMMHz" in keys
        pi = (P.ProcessInformation * 1024)()
        n = C.c_size_t()
        assert lib.AccelGetProcessInformation(pi, 1024, C.byref(n)) == P.SUCCESS
        mine = [pi[i] for i in range(n.value) if pi[i].processId.decode() == str(os.getpid())]
        assert mine and mine[0].memoryUsedBytes > 512 << 20 and mine[0].totalSMs == 148
        assert mine[0].deviceUUID.decode() == devs[0]["uuid"]
        w.dev_free(p)
    # unknown device: zeroed row, still SUCCESS (reference falls back the same way)
    uu = (C.c_char_p * 1)(b"GPU-does-not-exist")
    assert lib.AccelGetDeviceMetrics(uu, 1, dm) == P.SUCCESS and dm[0].powerUsageWatts == 0


def test_partition_and_hard_limits(prov):
    P, lib, _ = prov
    _, devs = P.all_devices(lib)
    uuid = devs[0]["uuid"].encode()
    pr = P.PartitionResult()
    assert lib.AccelAssignPartition(b"1g.10gb", uuid, C.byref(pr)) == P.SUCCESS
    env = [bytes(pr.envVars[i]).split(b"\0")[0].decode() for i in range(4)]
    assert env[0] == "NVIDIA_VISIBLE_DEVICES=" + devs[0]["uuid"]
    assert env[1] == "TF_CUDA_SM_PERCENT_LIMIT=15" and env[2] == "TF_CUDA_MEMORY_LIMIT=10240"
    part = pr.deviceUUID
    assert part.startswith(uuid[:40]) and pr.type == 0
    assert lib.AccelRemovePartition(b"1g.10gb", part) == P.SUCCESS
    assert lib.AccelAssignPartition(b"bogus", uuid, C.byref(pr)) == P.INVALID_PARAM
    assert lib.AccelAssignPartition(b"7g.900gb", uuid, C.byref(pr)) == P.RESOURCE_EXHAUSTED
    assert lib.AccelAssignPartition(b"1g.10gb", b"GPU-nope", C.byref(pr)) == P.NOT_FOUND
    assert lib.AccelSetMemHardLimit(uuid, 4 << 30) == P.SUCCESS
    assert lib.AccelSetComputeUnitHardLimit(uuid, 50) == P.SUCCESS
    assert lib.AccelSetMemHardLimit(b"GPU-nope", 1) == P.NOT_FOUND
    ctx = P.SnapshotContext()
    ctx.deviceUUID = uuid
    assert lib.AccelSnapshot(C.byref(ctx)) == P.SUCCESS        # device level, no vGPU worker on it: nothing to freeze
    me = (C.c_int32 * 1)(os.getpid())
    ctx = P.SnapshotContext(processIds=C.cast(me, C.POINTER(C.c_int32)), processCount=1, deviceUUID=None)
    assert lib.AccelSnapshot(C.byref(ctx)) == P.NOT_SUPPORTED  # a live process that is not one of this stack's workers


# The calls of the reference's provider ABI suite (provider/test/test_accelerator.c), made through ctypes in a
# process of its own; prints [section, assertion, passed] in the order and with the names the suite prints them.
ABI_SUITE = r'''
import ctypes as C, json
from tensor_fusion_b200 import provider as P
lib = P.load()
out, sec = [], [None]
def section(name): sec[0] = name
def check(cond, msg): out.append([sec[0], msg, bool(cond)])
INV = P.INVALID_PARAM
dev, n = b"stub-device-0", C.c_size_t()
section("AccelInit")
check(lib.AccelInit() == P.SUCCESS, "AccelInit returns success")
check(lib.AccelShutdown() == P.SUCCESS, "AccelShutdown returns success")
section("AccelGetDeviceCount")
check(lib.AccelGetDeviceCount(C.byref(n)) == P.SUCCESS, "AccelGetDeviceCount returns success")
check(n.value > 0, "Device count > 0")
check(lib.AccelGetDeviceCount(None) == INV, "NULL parameter returns error")
section("AccelGetAllDevices")
devs = (P.ExtendedDeviceInfo * 256)()
check(lib.AccelGetAllDevices(devs, 256, C.byref(n)) == P.SUCCESS, "AccelGetAllDevices returns success")
check(n.value > 0, "Device count > 0")
if n.value > 0:
    b = devs[0].basic
    check(len(b.uuid) > 0, "Device UUID is not empty")
    check(len(b.vendor) > 0, "Vendor is not empty")
    check(len(b.model) > 0, "Model is not empty")
    check(b.totalMemoryBytes > 0, "Total memory > 0")
    check(b.totalComputeUnits > 0, "Total compute units > 0")
    check(b.maxTflops > 0, "Max TFLOPS > 0")
    check(devs[0].virtualizationCapabilities.maxPartitions > 0, "Max partitions > 0")
check(lib.AccelGetAllDevices(None, 256, C.byref(n)) == INV, "NULL devices returns error")
check(lib.AccelGetAllDevices(devs, 0, C.byref(n)) == INV, "Zero maxCount returns error")
section("AccelGetAllDevicesTopology")
topo = P.ExtendedDeviceTopology()
check(lib.AccelGetAllDevicesTopology(C.byref(topo)) == P.SUCCESS, "AccelGetAllDevicesTopology returns success")
check(topo.deviceCount > 0, "Device count > 0")
if topo.deviceCount > 0:
    check(len(topo.devices[0].deviceUUID) > 0, "First device has UUID")
check(lib.AccelGetAllDevicesTopology(None) == INV, "NULL topology returns error")
section("AccelAssignPartition")
pr = P.PartitionResult()
check(lib.AccelAssignPartition(b"1g.10gb", dev, C.byref(pr)) == P.SUCCESS, "AccelAssignPartition returns success")
check(len(pr.deviceUUID) > 0, "Device UUID is set")
check(pr.type in (0, 1), "Partition type is valid")
check(lib.AccelAssignPartition(None, dev, C.byref(pr)) == INV, "NULL templateId returns error")
check(lib.AccelAssignPartition(b"1g.10gb", None, C.byref(pr)) == INV, "NULL deviceUUID returns error")
check(lib.AccelAssignPartition(b"1g.10gb", dev, None) == INV, "NULL partitionResult returns error")
section("AccelRemovePartition")
check(lib.AccelRemovePartition(b"1g.10gb", dev) == P.SUCCESS, "AccelRemovePartition returns success")
check(lib.AccelRemovePartition(None, dev) == INV, "NULL templateId returns error")
check(lib.AccelRemovePartition(b"1g.10gb", None) == INV, "NULL deviceUUID returns error")
section("AccelSetMemHardLimit")
check(lib.AccelSetMemHardLimit(dev, 4 << 30) == P.SUCCESS, "AccelSetMemHardLimit returns success")
check(lib.AccelSetMemHardLimit(None, 4 << 30) == INV, "NULL deviceUUID returns error")
check(lib.AccelSetMemHardLimit(dev, 0) == INV, "Zero memory limit returns error")
section("AccelSetComputeUnitHardLimit")
check(lib.AccelSetComputeUnitHardLimit(dev, 50) == P.SUCCESS, "AccelSetComputeUnitHardLimit returns success")
check(lib.AccelSetComputeUnitHardLimit(dev, 150) == INV, "Invalid limit > 100 returns error")
check(lib.AccelSetComputeUnitHardLimit(None, 50) == INV, "NULL deviceUUID returns error")
check(lib.AccelSetComputeUnitHardLimit(dev, 0) == INV, "Zero limit returns error")
section("AccelGetProcessInformation")
pi = (P.ProcessInformation * 256)()
check(lib.AccelGetProcessInformation(pi, 256, C.byref(n)) == P.SUCCESS, "AccelGetProcessInformation returns success")
if n.value > 0:
    check(0 <= pi[0].computeUtilizationPercent <= 100, "Compute utilization percent in valid range")
    check(pi[0].activeSMs <= pi[0].totalSMs, "Active SMs <= Total SMs")
    check(0 <= pi[0].memoryUtilizationPercent <= 100, "Memory utilization percent in valid range")
check(lib.AccelGetProcessInformation(None, 256, C.byref(n)) == INV, "NULL processInfos returns error")
check(lib.AccelGetProcessInformation(pi, 0, C.byref(n)) == INV, "Zero maxCount returns error")
section("AccelGetDeviceMetrics")
uu, dm = (C.c_char_p * 1)(dev), (P.DeviceMetrics * 1)()
check(lib.AccelGetDeviceMetrics(uu, 1, dm) == P.SUCCESS, "AccelGetDeviceMetrics returns success")
check(len(dm[0].deviceUUID) > 0, "Device UUID is not empty")
check(dm[0].powerUsageWatts >= 0, "Power usage >= 0")
check(dm[0].temperatureCelsius >= 0, "Temperature >= 0")
check(lib.AccelGetDeviceMetrics(None, 1, dm) == INV, "NULL deviceUUIDs returns error")
check(lib.AccelGetDeviceMetrics(uu, 0, dm) == INV, "Zero deviceCount returns error")
section("AccelGetVendorMountLibs")
mp = (P.MountPath * 64)()
check(lib.AccelGetVendorMountLibs(mp, 64, C.byref(n)) == P.SUCCESS, "AccelGetVendorMountLibs returns success")
check(lib.AccelGetVendorMountLibs(None, 64, C.byref(n)) == INV, "NULL mounts returns error")
check(lib.AccelGetVendorMountLibs(mp, 0, C.byref(n)) == INV, "Zero maxCount returns error")
section("AccelRegisterLogCallback")
check(lib.AccelRegisterLogCallback(P.LogCallback()) == P.SUCCESS, "AccelRegisterLogCallback with NULL returns success")
print(json.dumps(out))
'''


def test_reference_abi_suite_passes_against_our_library():
    """The reference's own 49-assertion known-answer test (provider/test/test_accelerator.c) against
    libaccelerator_b200.so: every assertion the suite made of the reference's example provider
    (tests/golden/reference_runs.json) holds for this library too."""
    # the suite addresses a device called "stub-device-0": alias it to GPU 0
    env = dict(os.environ, TF_PROVIDER_DEVICE_ALIASES="stub-device-0=0")
    r = subprocess.run([sys.executable, "-c", "import sys; sys.path.insert(0, %r)\n" % conftest.ROOT + ABI_SUITE],
                       env=env, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr[-3000:]
    ours = [tuple(x) for x in json.loads(r.stdout.strip().splitlines()[-1])]
    assert [x for x in ours if not x[2]] == []
    ref = oracle.abi_suite_results(oracle.reference_run("abi_suite")["stdout"])
    assert len(ref) >= 49 and all(ok for _, _, ok in ref)
    assert [x for x in ref if x not in ours] == []
    assert len(ours) >= 49          # 49 + 3 more when a GPU process is visible
    # the suite itself, compiled from the reference tree against this library, where oracle/Makefile could build it
    exe = os.path.join(oracle.REF_BUILD, "test_accelerator_b200")
    if os.path.exists(exe):
        r = subprocess.run([exe], env=env, capture_output=True, text=True, timeout=120)
        assert "Failed:       0" in r.stdout and r.returncode == 0, r.stdout[-3000:]
        assert [x for x in oracle.abi_suite_results(r.stdout.splitlines()) if x not in ours] == []


def test_reference_provider_baseline_still_passes():
    """Sanity: the unmodified reference provider + its suite, built from its own sources, passes every
    assertion; where oracle/Makefile could build it, it still prints the assertions recorded in tests/golden."""
    rec = oracle.reference_run("abi_suite")
    assert rec["returncode"] == 0 and "Failed:       0" in rec["stdout"]
    exe = os.path.join(oracle.REF_BUILD, "test_accelerator_ref")
    if os.path.exists(exe):
        r = subprocess.run([exe], capture_output=True, text=True, timeout=120, cwd=os.path.dirname(exe))
        assert r.returncode == 0 and "Failed:       0" in r.stdout
        live = oracle.abi_suite_results(r.stdout.splitlines())
        assert [x for x in oracle.abi_suite_results(rec["stdout"]) if x not in live] == []


def test_worker_counters_reach_extra_metrics(prov, tmp_path):
    """SURVEY 8f row 1: what the worker staged / throttled shows up in AccelGetDeviceMetrics.extraMetrics
    (and from there in the hypervisor's tf_gpu_usage line) with no Go change."""
    P, lib, _ = prov
    from tensor_fusion_b200 import trace
    from tensor_fusion_b200.worker import Worker
    _, devs = P.all_devices(lib)
    uuid = devs[0]["uuid"].encode()
    base = str(tmp_path / "shm")
    assert lib.LimiterInit(base.encode()) == P.SUCCESS
    cfg = (P.LimiterDeviceConfig * 1)()
    cfg[0].deviceIdx, cfg[0].deviceUUID, cfg[0].upLimit, cfg[0].memLimit = 0, uuid, 100, 1 << 40
    assert lib.LimiterCreateWorker(b"ns", b"metrics-pod", cfg, 1) == P.SUCCESS
    raw = trace.gen_c1(ncalls=300, error_permille=0)

    def extras():
        uu = (C.c_char_p * 1)(uuid)
        dm = (P.DeviceMetrics * 1)()
        assert lib.AccelGetDeviceMetrics(uu, 1, dm) == P.SUCCESS
        return {dm[0].extraMetrics[i].key.decode(): dm[0].extraMetrics[i].value for i in range(dm[0].extraMetricsCount)}

    before = extras()
    assert before["tfwWorkers"] == 0
    with Worker(shm_path=os.path.join(base, "ns", "metrics-pod", "shm")) as w:
        w.run(raw)
        st = w.stats()
        got = extras()
        assert got["tfwWorkers"] == 1
        assert got["tfwStagedPayloadBytesTotal"] == st["payload_bytes"] > 0
        assert got["tfwMoverLaunchesTotal"] == st["mover_launches"] and got["tfwClientLaunchesTotal"] == st["client_launches"]
        assert got["tfwVramBytes"] == st["vram_bytes"] and "computeThrottledCnt" in got
    assert os.path.exists(os.path.join(base, "ns", "metrics-pod", "tfw_stats"))
    lib.LimiterShutdown()


def test_compiled_hypervisor_harness_runs_the_purego_sequence():
    """tools/hypervisor_harness.c: dlopen(RTLD_NOW|RTLD_GLOBAL), the 14 mandatory symbols, log callback,
    AccelInit, discovery, the 2 Hz metric loops, shutdown -- against our library and the reference stub."""
    exe = os.path.join(conftest.ROOT, "tensor-fusion_b200", "lib", "hypervisor_harness")
    ours = os.path.join(conftest.ROOT, "tensor-fusion_b200", "lib", "libaccelerator_b200.so")
    r = subprocess.run([exe, ours, "2"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "vendor=NVIDIA" in r.stdout and "B200" in r.stdout and "sms=148" in r.stdout and "fatal=0" in r.stdout
    # the same harness against the reference's example provider, as recorded (and live where oracle/Makefile built it):
    # the hypervisor's sequence gets the same kinds of answers from both libraries
    runs = [oracle.reference_run("hypervisor_harness")]
    ref = os.path.join(oracle.REF_BUILD, "libaccelerator_example.so")
    if os.path.exists(ref):
        live = subprocess.run([exe, ref, "1"], capture_output=True, text=True, timeout=120, cwd=os.path.dirname(ref))
        runs.append({"returncode": live.returncode, "stdout": live.stdout.splitlines()})
    def kinds(lines):   # "devices=4 first=...", "tick 0: ...", "ok logs=10 fatal=0" -> devices, tick, ok
        return list(dict.fromkeys(ln.split()[0].split("=")[0] for ln in lines if ln.strip()))

    for run in runs:
        out = "\n".join(run["stdout"])
        assert run["returncode"] == 0 and "vendor=STUB" in out and "devices=4" in out      # hypervisor_suite_test.go:213-218
        assert kinds(run["stdout"]) == kinds(r.stdout.splitlines()) == ["devices", "tick", "ok"]
