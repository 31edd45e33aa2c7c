#!/usr/bin/env python
"""Extracts the input vector of the reference's own KAT TestSocketLine (aggregator/sock_line_test.go:11-349:
the tsList literal and the queried timestamp) into tests/golden/sockline_kat.json, so that the KAT can be
replayed in full (all timestamps) without a checkout of the reference. Run with the path of a getanteon/alaz
checkout at 828b997f:  python tests/golden/make_sockline_fixture.py <alaz checkout>
"""
import json
import os
import re
import sys

REF = os.path.join(sys.argv[1], "aggregator", "sock_line_test.go")
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "sockline_kat.json")

src = open(REF).read()
body = src[src.index("func TestSocketLine"):src.index("func TestXxx")]
lit = body[body.index("tsList := []uint64{"):]
lit = lit[:lit.index("}")]
ts = [int(x) for x in re.findall(r"^\s*(\d{8,})\s*,", lit, flags=re.M)]
q = int(re.search(r"sockLine\.GetValue\((\d+)\)", body).group(1))
json.dump({"source": "aggregator/sock_line_test.go:11-349 (getanteon/alaz @ 828b997f)", "ts_list": ts, "query": q,
           "expect": "GetValue(query) returns a socket (err == nil, si != nil)"}, open(OUT, "w"))
print(len(ts), "timestamps, query", q)
