"""Live-stream simulation (BASELINE config 5): C channels each carrying a read whose prefix
grows by 1 s of samples per poll (AccumulatingCache semantics, riser/client.py:29-31,44); the
batched SequencerControl classifies every poll's batch.  Reports p50 / p99 of the time from
"batch in hand" to "decisions on host" (the ReadUntil decision budget is ~1 s).  The measurement itself is
riser_b200.sim.measure_latency (bench.py's `latency` key calls the same function).

usage: python tools/live_sim.py [channels] [polls] [kit] [n_models] [scale,offset]

scale,offset: the client hands over calibrated float32 signal, (adc + offset) * scale, instead of int16.
"""
import json
import sys

sys.path.insert(0, ".")
from riser_b200 import sim     # noqa: E402

C = int(sys.argv[1]) if len(sys.argv) > 1 else 512
polls = int(sys.argv[2]) if len(sys.argv) > 2 else 12
kit = sys.argv[3] if len(sys.argv) > 3 else "RNA002"
n_models = int(sys.argv[4]) if len(sys.argv) > 4 else 1
calibration = tuple(float(v) for v in sys.argv[5].split(",")) if len(sys.argv) > 5 else None
print(json.dumps(sim.measure_latency(C, polls, kit, ["mRNA", "mtRNA", "globin"][:n_models], calibration=calibration)))
