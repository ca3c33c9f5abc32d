"""ctypes binding of oracle/libtfo_oracle.so -- the CPU checker (test infrastructure only)."""
import ctypes as C
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "oracle", "libtfo_oracle.so")
if not os.path.exists(LIB):
    raise ImportError(f"{LIB} missing: run `make -C oracle` (or __graft_entry__.build())")
lib = C.CDLL(LIB)

_P = C.c_void_p


class DevCfg(C.Structure):
    _fields_ = [("device_idx", C.c_uint32), ("uuid", C.c_char * 128), ("up_limit", C.c_uint32),
                ("mem_limit", C.c_uint64), ("total_cuda_cores", C.c_uint32)]


class ErlCfg(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("burst_window", "rate_min", "rate_max", "capacity_min", "capacity_max",
                                           "util_alpha", "kp", "ki", "kd", "integral_decay")]


class ErlState(C.Structure):
    _fields_ = [("current_rate", C.c_double), ("smoothed_util", C.c_double), ("integral_err", C.c_double),
                ("last_error", C.c_double), ("initialized", C.c_int)]


def _sig(name, res, args):
    f = getattr(lib, name)
    f.restype, f.argtypes = res, args
    return f


_sig("tfo_replay", C.c_int, [_P, C.c_size_t, C.c_uint64, C.c_uint32, C.POINTER(_P)])
_sig("tfo_responses", C.c_size_t, [_P, C.POINTER(_P)])
_sig("tfo_buffer", C.c_int, [_P, C.c_uint32, C.POINTER(_P), C.POINTER(C.c_uint64)])
_sig("tfo_stat", C.c_uint64, [_P, C.c_int])
_sig("tfo_free", None, [_P])
_sig("tfo_set_threads", None, [C.c_int])
_sig("tfo_set_buffer_cache", None, [C.c_int])
_sig("tfo_digest", C.c_uint64, [_P, C.c_uint64])
_sig("tfo_payload", None, [C.c_uint64, C.c_uint32, _P, C.c_uint64])
_sig("tfo_splitmix64_nth", C.c_uint64, [C.c_uint64, C.c_uint32])
_sig("tfo_shm_file_bytes", C.c_size_t, [])
_sig("tfo_shm_legacy_bytes", C.c_size_t, [])
_sig("tfo_shm_offset", C.c_size_t, [C.c_char_p])
_sig("tfo_shm_init_image", C.c_int, [_P, C.POINTER(DevCfg), C.c_size_t, C.c_uint64, C.c_uint64])
_sig("tfo_shm_create", C.c_int, [C.c_char_p, C.c_char_p, C.c_char_p, C.POINTER(DevCfg), C.c_size_t, C.POINTER(_P)])
_sig("tfo_shm_open", C.c_int, [C.c_char_p, C.c_char_p, C.c_char_p, C.POINTER(_P)])
_sig("tfo_shm_data", _P, [_P])
_sig("tfo_shm_close", None, [_P])
_sig("tfo_shm_get", C.c_double, [_P, C.c_uint32, C.c_int])
_sig("tfo_shm_set", None, [_P, C.c_uint32, C.c_int, C.c_double])
_sig("tfo_shm_fetch_sub", C.c_double, [_P, C.c_uint32, C.c_double])
_sig("tfo_shm_fetch_add", C.c_double, [_P, C.c_uint32, C.c_double])
_sig("tfo_shm_has_device", C.c_int, [_P, C.c_uint32])
_sig("tfo_shm_set_pod_memory_used", C.c_int, [_P, C.c_uint32, C.c_uint64])
_sig("tfo_shm_pod_memory_used", C.c_uint64, [_P, C.c_uint32])
_sig("tfo_shm_is_healthy", C.c_int, [_P, C.c_uint64, C.c_uint64])
_sig("tfo_shm_pid_insert", C.c_int, [_P, C.c_uint64])
_sig("tfo_shm_pid_remove", C.c_int, [_P, C.c_uint64])
_sig("tfo_shm_pid_values", C.c_size_t, [_P, C.POINTER(C.c_uint64), C.c_size_t])
_sig("tfo_valid_component", C.c_int, [C.c_char_p])
_sig("tfo_from_shm_path", C.c_int, [C.c_char_p, C.c_char_p, C.c_char_p, C.c_size_t])
_sig("tfo_erl_default_cfg", None, [C.POINTER(ErlCfg)])
_sig("tfo_erl_cfg_from_json", C.c_int, [C.c_char_p, C.POINTER(ErlCfg)])
_sig("tfo_erl_new_state", None, [C.POINTER(ErlState)])
_sig("tfo_erl_compute_desired_rate", C.c_double, [C.c_double, C.c_double, C.c_double, C.c_double, C.POINTER(ErlState), C.POINTER(ErlCfg)])
_sig("tfo_erl_rebalance", C.c_double, [_P, C.c_uint32, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double])
_sig("tfo_erl_tick", C.c_double, [_P, C.c_uint32, C.POINTER(ErlState), C.POINTER(ErlCfg), C.c_uint32, C.c_double, C.c_double])
_sig("tfo_compute_up_limit", C.c_uint32, [C.c_int64, C.c_double, C.c_double])


class Replay:
    """Sequential CPU replay of a TFCS stream."""

    def __init__(self, stream, vram_limit=0, flags=0):
        arr = np.frombuffer(stream, dtype=np.uint8) if isinstance(stream, (bytes, bytearray)) else stream
        self._keep = arr
        s = _P()
        self.rc = lib.tfo_replay(_P(arr.ctypes.data), arr.nbytes, vram_limit, flags, C.byref(s))
        self.s = s

    def responses(self):
        p = _P()
        n = lib.tfo_responses(self.s, C.byref(p))
        return C.string_at(p, n) if n else b""

    def buffer(self, handle):
        p, n = _P(), C.c_uint64()
        if lib.tfo_buffer(self.s, handle, C.byref(p), C.byref(n)) != 0:
            return None
        return np.ctypeslib.as_array((C.c_uint8 * n.value).from_address(p.value)) if n.value else np.empty(0, np.uint8)

    def live_handles(self, upto=4096):
        return [h for h in range(upto) if lib.tfo_buffer(self.s, h, None, None) == 0]

    def stat(self, which): return lib.tfo_stat(self.s, which)

    def close(self):
        if self.s:
            lib.tfo_free(self.s)
            self.s = None

    def __del__(self):
        self.close()


def digest(arr):
    arr = np.ascontiguousarray(arr)
    return lib.tfo_digest(_P(arr.ctypes.data), arr.nbytes)


def payload(seed, call_id, n):
    out = np.empty(n, dtype=np.uint8)
    lib.tfo_payload(seed, call_id, _P(out.ctypes.data), n)
    return out
_sig("tfo_go_max", C.c_double, [C.c_double, C.c_double])
_sig("tfo_go_min", C.c_double, [C.c_double, C.c_double])
_sig("tfo_erl_slew", C.c_double, [C.c_double, C.c_double, C.c_double, C.c_double])
_sig("tfo_pattern", None, [C.c_uint64, _P, C.c_uint64])


def pattern(seed, nbytes):
    out = np.empty(nbytes, dtype=np.uint8)
    lib.tfo_pattern(seed, _P(out.ctypes.data), nbytes)
    return out


# ---- what the reference's own C programs printed (tests/golden/reference_runs.json, oracle/record_golden.py) ----
REF_BUILD = os.path.join(ROOT, "oracle", "_ref")


def reference_run(name):
    """{"returncode", "stdout": [lines]} of one recorded run of the reference's programs."""
    import json
    with open(os.path.join(ROOT, "tests", "golden", "reference_runs.json")) as f:
        return json.load(f)[name]


def abi_suite_results(lines):
    """The assertions of the reference's provider ABI suite output: [(section, message, passed)]."""
    out, section = [], None
    for ln in lines:
        s = ln.strip()
        if s.startswith("=== Testing ") and s.endswith(" ==="):
            section = s[len("=== Testing "):-len(" ===")]
        elif section and s[:2] in ("✓ ", "✗ "):
            out.append((section, s[2:], s[0] == "✓"))
    return out
