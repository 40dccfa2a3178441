#!/usr/bin/env python
"""Prints the per-layer clock64 trace of trunk_fused's pair 0 (diagnostic; CATTUS_B200_TRACE_TRUNK=1) for a chess net at
each precision:  python tools/trace_fused.py chess10x128 4096 [bf16 fp8]"""
import os, sys
from pathlib import Path
os.environ["CATTUS_B200_TRACE_TRUNK"] = "1"
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from cattus_b200 import CudaNetwork
from cattus_b200.export import export_blob
from oracle import games, net
name, n = sys.argv[1], int(sys.argv[2])
cfg = net.CONFIGS[name]
words, bitmaps = games.synth_chess_positions(n, 1)
for precision in sys.argv[3:] or ["bf16", "fp8"]:
    with CudaNetwork(export_blob(net.make_state_dict(cfg, 0), cfg.game), cfg.game, batch_size=n, n_streams=1, precision=precision) as nw:
        nw.resident_upload(words, bitmaps)
        print(precision, "ms", nw.time_stage(1, n, 3), file=sys.stderr, flush=True)
