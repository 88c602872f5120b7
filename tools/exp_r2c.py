#!/usr/bin/env python3
"""Runs ON THE GPU BOX: random-gather ceilings around the directory footprints, whole-line-per-thread vs lane-pair
loads.  One JSON line per measurement."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import rowbowt_b200 as rb  # noqa: E402

lib = rb.lib()
for mb in (64, 128, 160, 192, 224, 256, 384):
    for line in (64, -64, 32, 128):
        g = lib.rbg_gather_roofline(0, mb << 20, line, 256)
        print(json.dumps({"kind": "gather", "footprint_MB": mb, "line_bytes": abs(line), "lane_pairs": line < 0, "gbs": round(g, 1),
                          "glines_per_s": round(g / abs(line), 2)}), flush=True)
