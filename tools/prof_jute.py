import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from registrar_b200 import _native, synth
ctx = _native.Context(0); ctx.set_option("chunk_records", 0)
b = synth.generate("config3", n=2_000_000)
res = ctx.register_batch(b, copy=False)
for _ in range(3):
    f = ctx.jute_frames(1, 1, device=True)
print(f.kernel_ms)
