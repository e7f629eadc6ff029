#!/usr/bin/env python
"""Regenerates tests/golden/sam_md5.json: md5 of the UNMODIFIED reference's SAM (oracle/_ref/bwa mem, @PG removed)
on the seeded datasets of tests/test_oracle_pin.py:CASES.  Run from the repo root on a box that has oracle/_ref."""
import json, os, subprocess, sys
sys.path.insert(0, os.path.join(os.path.dirname(__file__), ".."))
import conftest
from test_oracle_pin import CASES
d = conftest.DataSets()
out = {}
for name, ref, kw, extra in CASES:
    fa, fqs = d.reads(ref, **kw)
    r = subprocess.run([os.path.join(conftest.ROOT, "oracle", "_ref", "bwa"), "mem", "-v", "1", "-K", "100000000", "-t", "4"] + extra + [fa] + fqs,
                       stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, check=True)
    out[name] = conftest.md5(conftest.strip_pg(r.stdout))
json.dump(out, open(os.path.join(os.path.dirname(__file__), "sam_md5.json"), "w"), indent=1, sort_keys=True)
print(out)
