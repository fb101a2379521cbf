"""Per-chunk timeline of the pipelined host entry (device planner), B=4096 algo 5."""
import sys, time, json
import numpy as np, torch
sys.path.insert(0, ".")
from scl_deepfake_audio_detection_b200 import workload
from scl_deepfake_audio_detection_b200.engine import Engine
eng = Engine(0)
args = workload.default_args()
B, L = 4096, 64600
chunk = int(sys.argv[1]) if len(sys.argv) > 1 else 0
x = torch.empty((B, L), dtype=torch.float32).pin_memory()
x.normal_(0, 0.1)
y = torch.empty((B, L), dtype=torch.float32).pin_memory()
lengths = np.full(B, L, np.int32)
seeds = np.array([workload.seed_for(u) for u in range(B)], np.uint32)
eng.set_host_chunk(chunk)
for i in range(3):
    t0 = time.perf_counter(); eng.process_host_seeded(5, x.numpy(), lengths, seeds, 16000, args, out=y.numpy()); print("ms", 1e3 * (time.perf_counter() - t0))
eng.trace_host(True)
t0 = time.perf_counter(); eng.process_host_seeded(5, x.numpy(), lengths, seeds, 16000, args, out=y.numpy()); print("traced ms", 1e3 * (time.perf_counter() - t0))
for row in eng.host_timeline():
    print({k: round(v, 2) for k, v in row.items()})
