#!/usr/bin/env python
"""What the UNMODIFIED reference (oracle/_ref = DuckDB + duckpgq, built by oracle/build_ref.sh) returns for the
statement-level tests, so that they compare the duckpgq_b200 binaries with it without the reference at hand:

    python tests/golden/make_golden_duckdb.py

Writes tests/golden/duckdb_reference.json.gz:
    cases          tests/test_duckdb_shim.py CASES: stdout and stderr of oracle/_ref/duckdb -csv
    operator_time  tests/test_duckdb_shim.py OPERATOR_SQL: the last output row, the Projection and statement times
                   from DuckDB's profiler, and the host they were measured on
    sqllogic       "All tests passed (N assertions in M test cases)" of oracle/_ref/unittest over tests/golden/sqllogic
"""
import gzip
import json
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import test_duckdb_shim as shim  # noqa: E402
import test_sqllogic_override as sqllogic  # noqa: E402

DUCKDB = os.path.join(ROOT, "oracle", "_ref", "duckdb")
UNITTEST = os.path.join(ROOT, "oracle", "_ref", "unittest")


def host() -> str:
    model = "unknown CPU"
    with open("/proc/cpuinfo") as f:
        for line in f:
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    return f"{model}, {os.cpu_count()} hardware threads"


def main():
    cases = {}
    for name, sql in sorted(shim.CASES.items()):
        out, err = shim.run(DUCKDB, sql)
        cases[name] = {"stdout": out, "stderr": err}
    with tempfile.TemporaryDirectory() as tmp:
        row, times = shim.measure_operator_time(DUCKDB, os.path.join(tmp, "profile.json"))
    rc, out = sqllogic.run_suite(UNITTEST)
    m = sqllogic.SUMMARY.search(out)
    assert rc == 0 and m, out[-3000:]
    golden = {"cases": cases,
              "operator_time": dict(times, row=row, measured_on=host()),
              "sqllogic": {"assertions": int(m.group(1)), "test_cases": int(m.group(2))}}
    path = os.path.join(HERE, "duckdb_reference.json.gz")
    with open(path, "wb") as raw, gzip.GzipFile(fileobj=raw, mode="wb", mtime=0) as f:
        f.write(json.dumps(golden, indent=1, sort_keys=True).encode())
    print(path, golden["operator_time"], golden["sqllogic"])


if __name__ == "__main__":
    main()
