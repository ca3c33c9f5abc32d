"""Records what the reference's own C programs print into tests/golden/reference_runs.json.

The tests compare this project with those records, so they do not need the reference tree (or the
binaries `make -C oracle` builds from it into oracle/_ref) when they run.  Rerun after rebuilding
oracle/_ref from a newer reference:

    make -C oracle && python oracle/record_golden.py
"""
import json
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.path.join(HERE, "_ref")
OUT = os.path.join(ROOT, "tests", "golden", "reference_runs.json")

# name -> (command, what it is).  Each runs in oracle/_ref, from a fresh mock driver state (a file in the cwd).
RUNS = {
    "abi_suite": (["./test_accelerator_ref"],
                  "provider/test/test_accelerator.c against the reference's example provider (provider/example/accelerator.c)"),
    "mock_rate_limit": (["./test_rate_limit"], "provider/example/device_mock/test_rate_limit.c"),
    "hypervisor_harness": ([os.path.join(ROOT, "tensor-fusion_b200", "lib", "hypervisor_harness"), os.path.join(REF, "libaccelerator_example.so"), "1"],
                           "tools/hypervisor_harness.c driving the reference's example provider for one metrics tick"),
}


def main():
    rec = {"_about": "stdout of the reference's own C programs, built from its sources by oracle/Makefile and run by "
                     "oracle/record_golden.py. Timings and the mock driver's random metrics vary from run to run; the tests "
                     "read only the lines that do not."}
    for name, (cmd, what) in RUNS.items():
        state = os.path.join(REF, "tmp.example_accelerator.bin")   # the mock driver's processes of earlier runs
        if os.path.exists(state):
            os.unlink(state)
        r = subprocess.run(cmd, cwd=REF, capture_output=True, text=True, timeout=120)
        rec[name] = {"what": what, "returncode": r.returncode, "stdout": r.stdout.splitlines()}
    with open(OUT, "w") as f:
        json.dump(rec, f, indent=1, ensure_ascii=False)
        f.write("\n")
    print("wrote", OUT)


if __name__ == "__main__":
    main()
