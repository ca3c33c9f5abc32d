"""Pins the CPU oracle to every golden vector / known-answer test the reference
holds for this path (SURVEY.md 8c).  Each test cites the Go test it transliterates.
The reference is not needed at run time: its values are restated here and in tests/golden/.
"""
import ctypes as C
import os

import numpy as np
import pytest

import oracle
from oracle import lib as O


def _image(cfgs=(), now=1_700_000_000, pid=None):
    img = np.zeros(O.tfo_shm_file_bytes(), dtype=np.uint8)
    arr = (oracle.DevCfg * max(1, len(cfgs)))()
    for i, (idx, uuid, up, mem, cores) in enumerate(cfgs):
        arr[i].device_idx, arr[i].uuid, arr[i].up_limit, arr[i].mem_limit, arr[i].total_cuda_cores = idx, uuid, up, mem, cores
    assert O.tfo_shm_init_image(C.c_void_p(img.ctypes.data), arr, len(cfgs), now, pid or os.getpid()) == 0
    return img, C.c_void_p(img.ctypes.data)


TEST_CFG = [(0, b"test-device-uuid", 80, 1 << 30, 1024)]  # createTestConfigs, soft_limiter_shm_test.go:27-39


# ---- layout: soft_limiter_shm_test.go:217-232, :177, :197-215 ------------------------------
def test_rust_layout_offsets():
    assert O.tfo_shm_offset(b"v2") == 8
    assert O.tfo_shm_offset(b"heartbeat") == 0x890
    assert O.tfo_shm_offset(b"pids") == 0x898
    assert O.tfo_shm_file_bytes() == 35504          # SURVEY App. B
    assert O.tfo_shm_legacy_bytes() == 35496        # unsafe.Sizeof(SharedDeviceStateV2{})
    assert O.tfo_shm_offset(b"entry") == 136


def test_image_fields_land_on_pinned_offsets():
    img, f = _image(TEST_CFG, now=1234567)
    assert int(img[:4].view(np.uint32)[0]) == 1                     # discriminant V2
    assert bytes(img[8:8 + 16]) == b"test-device-uuid"
    assert int(img[8 + 64: 8 + 68].view(np.uint32)[0]) == 80        # up_limit
    assert int(img[8 + 72: 8 + 80].view(np.uint64)[0]) == 1 << 30   # mem_limit
    assert int(img[8 + 80: 8 + 84].view(np.uint32)[0]) == 1024      # total_cuda_cores
    assert float(img[8 + 96: 8 + 104].view(np.float64)[0]) == 10.0  # refill rate
    assert float(img[8 + 104: 8 + 112].view(np.float64)[0]) == 100.0
    assert float(img[8 + 112: 8 + 120].view(np.float64)[0]) == 100.0
    assert float(img[8 + 120: 8 + 128].view(np.float64)[0]) == 1234567.0
    assert int(img[8 + 128: 8 + 132].view(np.uint32)[0]) == 1       # is_active
    assert int(img[0x888:0x88C].view(np.uint32)[0]) == 1            # device_count
    assert int(img[0x890:0x898].view(np.uint64)[0]) == 1234567      # heartbeat


# ---- TestERLTokenBucketPreservesTokensWhenInsufficient :139-151 ----------------------------
def test_fetch_sub_preserves_tokens_when_insufficient():
    img, f = _image(TEST_CFG)
    O.tfo_shm_set(f, 0, 2, 1.5)
    assert O.tfo_shm_fetch_sub(f, 0, 2.0) == 1.5
    assert O.tfo_shm_get(f, 0, 2) == 1.5
    O.tfo_shm_set(f, 0, 2, 5.0)
    assert O.tfo_shm_fetch_sub(f, 0, 2.0) == 5.0
    assert O.tfo_shm_get(f, 0, 2) == 3.0


# ---- TestERLTokenOperations :590-622 ---------------------------------------------------------
def test_erl_defaults_and_accessors():
    img, f = _image(TEST_CFG)
    assert O.tfo_shm_get(f, 0, 0) == 10.0 and O.tfo_shm_get(f, 0, 1) == 100.0 and O.tfo_shm_get(f, 0, 2) == 100.0
    O.tfo_shm_set(f, 0, 0, 50.0); O.tfo_shm_set(f, 0, 1, 200.0); O.tfo_shm_set(f, 0, 2, 150.0)
    assert (O.tfo_shm_get(f, 0, 0), O.tfo_shm_get(f, 0, 1), O.tfo_shm_get(f, 0, 2)) == (50.0, 200.0, 150.0)
    O.tfo_shm_set(f, 0, 2, 175.0); O.tfo_shm_set(f, 0, 3, 12345.0)
    assert (O.tfo_shm_get(f, 0, 2), O.tfo_shm_get(f, 0, 3)) == (175.0, 12345.0)


# ---- TestFetchAddERLTokens :624-638 ---------------------------------------------------------------
def test_fetch_add_caps_at_capacity():
    img, f = _image(TEST_CFG)
    O.tfo_shm_set(f, 0, 1, 100.0); O.tfo_shm_set(f, 0, 2, 50.0)
    assert O.tfo_shm_fetch_add(f, 0, 30.0) == 50.0 and O.tfo_shm_get(f, 0, 2) == 80.0
    assert O.tfo_shm_fetch_add(f, 0, 50.0) == 80.0 and O.tfo_shm_get(f, 0, 2) == 100.0


# ---- heartbeat :63-102 ----------------------------------------------------------------------------
def test_heartbeat_health():
    now = 1_700_000_000
    img, f = _image((), now=now)
    assert O.tfo_shm_is_healthy(f, 30, now) == 1
    img[0x890:0x898].view(np.uint64)[0] = now - 60
    assert O.tfo_shm_is_healthy(f, 30, now) == 0
    img[0x890:0x898].view(np.uint64)[0] = 0
    assert O.tfo_shm_is_healthy(f, 30, now) == 0
    img[0x890:0x898].view(np.uint64)[0] = now + 5      # from the future: unhealthy (:466-468)
    assert O.tfo_shm_is_healthy(f, 30, now) == 0


# ---- PID set :362-411 ----------------------------------------------------------------------------
def _pids(f):
    out = (C.c_uint64 * 4096)()
    n = O.tfo_shm_pid_values(f, out, 4096)
    return list(out[:n])


def test_pid_set_dedup_remove_capacity():
    img, f = _image(())
    for _ in range(3):
        O.tfo_shm_pid_insert(f, 1234)
    assert _pids(f) == [1234]
    img, f = _image(())
    for p in (111, 222, 333):
        O.tfo_shm_pid_insert(f, p)
    O.tfo_shm_pid_remove(f, 222)
    assert sorted(_pids(f)) == [111, 333]
    img, f = _image(())
    for p in range(2048):
        O.tfo_shm_pid_insert(f, p)
    assert len(_pids(f)) == 2048
    O.tfo_shm_pid_insert(f, 0)
    assert len(_pids(f)) == 2048
    assert O.tfo_shm_pid_insert(f, 99999) == 0           # full


def test_pid_bitmap_is_msb_first():
    img, f = _image(())
    O.tfo_shm_pid_insert(f, 42)       # slot 0 -> word 0, mask 1<<63   (soft_limiter_shm.go:759)
    O.tfo_shm_pid_insert(f, 43)       # slot 1 -> mask 1<<62
    bm = img[0x898 + 16392: 0x898 + 16400].view(np.uint64)[0]
    assert int(bm) == (1 << 63) | (1 << 62)
    assert int(img[0x898 + 8: 0x898 + 16].view(np.uint64)[0]) == 42
    assert int(img[0x898 + 32776: 0x898 + 32784].view(np.uint64)[0]) == 2   # len


# ---- set pod memory :574-588 --------------------------------------------------------------------
def test_set_pod_memory_used():
    img, f = _image(TEST_CFG)
    assert O.tfo_shm_set_pod_memory_used(f, 0, 1 << 30) == 1
    assert O.tfo_shm_pod_memory_used(f, 0) == 1 << 30
    assert O.tfo_shm_set_pod_memory_used(f, 999, 1024) == 0


# ---- paths :239-270, :524-565 -----------------------------------------------------------------------
def test_path_components_and_parsing(tmp_path):
    assert O.tfo_valid_component(b"../escape") == 0
    assert O.tfo_valid_component(b"pod/name") == 0
    assert O.tfo_valid_component(b"namespace") == 1
    ns, name = C.create_string_buffer(256), C.create_string_buffer(256)
    assert O.tfo_from_shm_path(b"/base/namespace/podname/shm", ns, name, 256) == 0
    assert (ns.value, name.value) == (b"namespace", b"podname")
    assert O.tfo_from_shm_path(b"/base/shm", ns, name, 256) != 0
    assert O.tfo_from_shm_path(b"/namespace/shm", ns, name, 256) != 0
    h = C.c_void_p()
    cfg = (oracle.DevCfg * 1)()
    assert O.tfo_shm_create(str(tmp_path).encode(), b"../escape", b"pod", cfg, 0, C.byref(h)) == 1
    assert O.tfo_shm_open(str(tmp_path).encode(), b"namespace", b"pod/name", C.byref(h)) == 1


# ---- create / open / legacy :153-215, :234-237 ---------------------------------------------------------
def test_create_open_share_memory_and_reject_legacy(tmp_path):
    base = str(tmp_path).encode()
    cfg = (oracle.DevCfg * 1)()
    cfg[0].device_idx, cfg[0].uuid, cfg[0].up_limit, cfg[0].mem_limit, cfg[0].total_cuda_cores = 0, b"test-device-uuid", 80, 1 << 30, 1024
    h1, h2 = C.c_void_p(), C.c_void_p()
    assert O.tfo_shm_create(base, b"handle_create_open", b"test", cfg, 1, C.byref(h1)) == 0
    path = tmp_path / "handle_create_open" / "test" / "shm"
    assert path.stat().st_size == 35504
    assert O.tfo_shm_open(base, b"handle_create_open", b"test", C.byref(h2)) == 0
    O.tfo_shm_set_pod_memory_used(O.tfo_shm_data(h1), 0, 42)
    assert O.tfo_shm_pod_memory_used(O.tfo_shm_data(h2), 0) == 42
    O.tfo_shm_close(h1); O.tfo_shm_close(h2)
    # legacy layout: a file of sizeof(SharedDeviceStateV2) must be rejected
    d = tmp_path / "legacy_layout" / "test"
    d.mkdir(parents=True)
    (d / "shm").write_bytes(b"\0" * 35496)
    assert O.tfo_shm_open(base, b"legacy_layout", b"test", C.byref(h2)) == 100
    (d / "shm").write_bytes(b"\0" * 16)                                # corrupt 16-byte file (legacy_test.go:86-392)
    assert O.tfo_shm_open(base, b"legacy_layout", b"test", C.byref(h2)) == 101
    assert O.tfo_shm_open(base, b"non-existent", b"memory", C.byref(h2)) == 2


# ---- ERL controller: quota_controller_test.go:11-73 -------------------------------------------------
def _cfg():
    c = oracle.ErlCfg()
    O.tfo_erl_default_cfg(C.byref(c))
    return c


def test_compute_desired_rate_directions():
    c = _cfg()
    s = oracle.ErlState(current_rate=100, initialized=1)
    assert O.tfo_erl_compute_desired_rate(100, 0.7, 0.35, 0.5, C.byref(s), C.byref(c)) > 100
    s = oracle.ErlState(current_rate=1000, initialized=1)
    assert O.tfo_erl_compute_desired_rate(1000, 0.5, 0.9, 0.5, C.byref(s), C.byref(c)) < 1000


def test_compute_desired_rate_hand_derived_values():
    """Values derived by hand from quota_controller.go:321-347 (exact float64 arithmetic)."""
    c = _cfg()
    # under target: e=.35, I=.175, D=.7, ff=100*.7/.35=200, k=clamp(1+.315+.06125+.07)=1.44625 -> 289.25 -> slew +35% = 135
    s = oracle.ErlState(current_rate=100, initialized=1)
    got = O.tfo_erl_compute_desired_rate(100, 0.7, 0.35, 0.5, C.byref(s), C.byref(c))
    assert got == 100 * (1.0 + 0.35)
    assert s.integral_err == 0.35 * 0.5 and s.last_error == 0.7 - 0.35
    # over target: e=-.4 -> ff=1000*.5/.9, k clamps to 0.5 -> 277.7 -> slew -25% = 750
    s = oracle.ErlState(current_rate=1000, initialized=1)
    assert O.tfo_erl_compute_desired_rate(1000, 0.5, 0.9, 0.5, C.byref(s), C.byref(c)) == 1000 * (1.0 - 0.25)
    # idle: ramp +35% capped at rateMax
    s = oracle.ErlState(current_rate=190000, initialized=1)
    assert O.tfo_erl_compute_desired_rate(190000, 0.5, 0.005, 0.5, C.byref(s), C.byref(c)) == 200000.0
    # deadband: rate unchanged, integral decays
    s = oracle.ErlState(current_rate=500, integral_err=1.0, initialized=1)
    assert O.tfo_erl_compute_desired_rate(500, 0.5, 0.51, 0.5, C.byref(s), C.byref(c)) == 500
    assert s.integral_err == 0.85


def test_rebalance_smoothly_drains_excess_tokens():
    """TestRebalanceTokenBucketSmoothlyDrainsExcessTokens: tokens 200, cap 100, ts 10 -> (35,100)."""
    img, f = _image([(0, b"u", 50, 1 << 30, 1024)])
    O.tfo_shm_set(f, 0, 2, 200.0); O.tfo_shm_set(f, 0, 1, 100.0); O.tfo_shm_set(f, 0, 3, 10.0)
    got = O.tfo_erl_rebalance(f, 0, 10.5, 50.0, 100.0, 0.5, 0.8)
    assert 35 < got < 100
    # hand derivation: FetchAdd caps 200+25 at capacity 100 -> not > capacity; util .8 > .53 and 100 > 35
    # -> drain max(25, 80)*0.5 = 40 -> 60
    assert got == 60.0 and O.tfo_shm_get(f, 0, 2) == 60.0 and O.tfo_shm_get(f, 0, 3) == 10.5


def test_load_erl_config_from_env_json():
    c = oracle.ErlCfg()
    js = b'''{"elasticRateLimitParameters":{"maxRefillRate":"1234","minRefillRate":"12","filterAlpha":"0.4",
             "kp":"1.2","ki":"0.5","kd":"0.2","burstWindow":"0.8","capacityMin":"321","capacityMax":"4321",
             "integralDecayFactor":"0.9"}}'''
    O.tfo_erl_cfg_from_json(js, C.byref(c))
    assert (c.rate_max, c.rate_min, c.util_alpha, c.kp, c.ki, c.kd, c.burst_window, c.capacity_min, c.capacity_max,
            c.integral_decay) == (1234, 12, 0.4, 1.2, 0.5, 0.2, 0.8, 321, 4321, 0.9)
    O.tfo_erl_cfg_from_json(b'{"elasticRateLimitParameters":{"filterAlpha":"7","minRefillRate":"-3","kp":"abc"}}', C.byref(c))
    assert c.util_alpha == 0.95 and c.rate_min == 10.0 and c.kp == 0.9     # clamp / fallbacks (:133-141,:169-177)


def test_compute_up_limit():
    """computeUpLimit worker/controller.go:307-325 == computeLimitPercent handlers/legacy.go:643-661."""
    assert O.tfo_compute_up_limit(25, 0, 2250) == 25
    assert O.tfo_compute_up_limit(0, 562.5, 2250) == 25
    assert O.tfo_compute_up_limit(0, 563, 2250) == 26      # ceil
    assert O.tfo_compute_up_limit(0, 1, 2250) == 1
    assert O.tfo_compute_up_limit(0, 9999, 2250) == 100
    assert O.tfo_compute_up_limit(0, 0, 2250) == 100
    assert O.tfo_compute_up_limit(0, 100, 0) == 100


def test_go_min_max_nan_and_signed_zero():
    nan = float("nan")
    assert np.isnan(O.tfo_go_max(nan, 1.0)) and np.isnan(O.tfo_go_min(1.0, nan))
    assert np.float64(O.tfo_go_max(-0.0, 0.0)).view(np.uint64) == 0
    assert np.float64(O.tfo_go_min(0.0, -0.0)).view(np.uint64) == 1 << 63
    assert O.tfo_go_max(float("inf"), nan) == float("inf")       # Go: Max(x,+Inf)=+Inf even with NaN


# ---- replay oracle self-consistency (parity unpinned at the reference; see DESIGN.md) --------------
def test_splitmix_and_xoshiro_known_answers():
    # splitmix64(seed=0) first outputs: reference implementation by S. Vigna (public domain)
    assert O.tfo_splitmix64_nth(0, 0) == 0xE220A8397B1DCDAF
    assert O.tfo_splitmix64_nth(0, 1) == 0x6E789E6AA1B965F4
    assert O.tfo_splitmix64_nth(0, 2) == 0x06C45D188009454F
    a = oracle.payload(0x7F5EED, 3, 4099)
    b = oracle.payload(0x7F5EED, 3, 4104)
    assert np.array_equal(a, b[:4099])                              # truncation, not re-seeding
    assert not np.array_equal(oracle.payload(0x7F5EED, 4, 64), a[:64])


def test_digest_properties():
    rng = np.random.default_rng(0)
    x = rng.integers(0, 256, 1000, dtype=np.uint8)
    y = x.copy(); y[[10, 18]] = y[[18, 10]]
    assert oracle.digest(x) != oracle.digest(y)                     # order sensitive
    assert oracle.digest(x[:999]) != oracle.digest(x)
    assert oracle.digest(np.zeros(8, np.uint8)) != oracle.digest(np.zeros(16, np.uint8))


def test_vectors_from_golden_file():
    """tests/golden/reference_vectors.json: the reference's constants, each with its file:line."""
    import json
    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "reference_vectors.json")))
    L = g["layout"]
    assert (O.tfo_shm_offset(b"v2"), O.tfo_shm_offset(b"heartbeat"), O.tfo_shm_offset(b"pids")) == (L["v2_payload_offset"], L["last_heartbeat_offset"], L["pids_offset"])
    assert (O.tfo_shm_file_bytes(), O.tfo_shm_legacy_bytes(), O.tfo_shm_offset(b"entry")) == (L["file_bytes"], L["legacy_bytes"], L["entry_bytes"])
    img, f = _image(TEST_CFG)
    d = g["erl_defaults"]
    assert (O.tfo_shm_get(f, 0, 0), O.tfo_shm_get(f, 0, 1), O.tfo_shm_get(f, 0, 2)) == (d["rate"], d["capacity"], d["tokens"])
    for c in g["fetch_sub"]["cases"]:
        O.tfo_shm_set(f, 0, 2, c["tokens"])
        assert O.tfo_shm_fetch_sub(f, 0, c["cost"]) == c["returns"] and O.tfo_shm_get(f, 0, 2) == c["after"]
    O.tfo_shm_set(f, 0, 1, g["fetch_add"]["capacity"]); O.tfo_shm_set(f, 0, 2, g["fetch_add"]["start"])
    for c in g["fetch_add"]["cases"]:
        assert O.tfo_shm_fetch_add(f, 0, c["amount"]) == c["returns"] and O.tfo_shm_get(f, 0, 2) == c["after"]
    cfg = oracle.ErlCfg()
    O.tfo_erl_cfg_from_json(json.dumps(g["erl_config_json"]["env"]).encode(), C.byref(cfg))
    for k, v in g["erl_config_json"]["expect"].items():
        assert getattr(cfg, k) == v, k
    dflt = _cfg()
    for c in g["desired_rate_direction"]["cases"]:
        s = oracle.ErlState(current_rate=c["rate"], initialized=1)
        got = O.tfo_erl_compute_desired_rate(c["rate"], c["target"], c["util"], 0.5, C.byref(s), C.byref(dflt))
        assert (got > c["rate"]) if c["expect"] == "increase" else (got < c["rate"])
    r = g["rebalance"]
    O.tfo_shm_set(f, 0, 2, r["tokens"]); O.tfo_shm_set(f, 0, 1, r["capacity"]); O.tfo_shm_set(f, 0, 3, r["last"])
    got = O.tfo_erl_rebalance(f, 0, r["now"], r["rate"], r["capacity"], r["target"], r["util"])
    assert r["open_interval"][0] < got < r["open_interval"][1]
    for bad in g["paths"]["invalid_components"]:
        assert O.tfo_valid_component(bad.encode()) == 0
    ns, name = C.create_string_buffer(256), C.create_string_buffer(256)
    for c in g["paths"]["from_shm_path"]:
        rc = O.tfo_from_shm_path(c["path"].encode(), ns, name, 256)
        if c.get("error"):
            assert rc != 0
        else:
            assert rc == 0 and (ns.value.decode(), name.value.decode()) == (c["ns"], c["name"])


def test_reference_c_provider_and_mock_driver_known_answers():
    """The reference's C half as it ran when compiled from its own sources (tests/golden/reference_runs.json):
    49/49 ABI assertions, and the mock driver's 100-launches-per-second window."""
    import json
    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "reference_vectors.json")))
    r = oracle.reference_run("abi_suite")
    out = "\n".join(r["stdout"])
    passed = int(out.split("Passed:")[1].split()[0])
    assert r["returncode"] == 0 and "Failed:       0" in out and passed >= g["provider_stub"]["assertions"]   # +3 when a mock process is registered
    assert len(oracle.abi_suite_results(r["stdout"])) == passed
    r = oracle.reference_run("mock_rate_limit")
    out = "\n".join(r["stdout"])
    assert r["returncode"] == 0, out[-500:]
    assert f"Successful launches: {g['mock_rate_limit']['accepted']}" in out
    assert f"Blocked launches: {g['mock_rate_limit']['launches'] - g['mock_rate_limit']['accepted']}" in out
