#!/usr/bin/env python3
"""Folds reference runs recorded by the test-suite into tests/golden/reference_runs.json.

Record where oracle/_ref holds the reference binaries (`make -C oracle ref`), with the reference's source tree in
CFB_REFERENCE_SRC for the Perl scripts; the GPU tests record on a GPU machine:

  CFB_RECORD_REFERENCE=/tmp/runs.jsonl CFB_REFERENCE_SRC=<reference tree> python -m pytest tests
  python tests/golden/merge_reference_runs.py /tmp/runs.jsonl

A test that skips while recording (the two-GPU tests on a one-GPU machine) makes no calls: record its runs where it
runs, or make the same calls from a script, since the reference's binaries need no GPU.  A key recorded twice must
have the same result (the reference is deterministic on these calls)."""
import json
import os
import sys

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_runs.json")


def main(paths):
    runs = {}
    if os.path.exists(OUT):
        with open(OUT) as f:
            runs = json.load(f)
    for p in paths:
        with open(p) as f:
            for line in f:
                for k, v in json.loads(line).items():
                    if k in runs and runs[k] != v:
                        raise SystemExit("%s: key %s recorded with two different results" % (p, k))
                    runs[k] = v
    with open(OUT, "w") as f:
        f.write("{\n" + ",\n".join("%s: %s" % (json.dumps(k), json.dumps(runs[k], sort_keys=True)) for k in sorted(runs)) + "\n}\n")
    print("%d recorded runs in %s" % (len(runs), OUT))


if __name__ == "__main__":
    main(sys.argv[1:])
