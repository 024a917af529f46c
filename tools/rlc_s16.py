import os, sys, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
from aeonflux_b200 import Issuer, PresentationBatch, compact_to_batchable
blob = open(os.path.join(ROOT, "bench_data", "issuer16.bin"), "rb").read()
pres = np.fromfile(os.path.join(ROOT, "bench_data", "s16_256.bin"), np.uint8).reshape(-1, 143, 32)
sp, ip, sk = blob[:1316], blob[1316:1380], blob[1380:]
B = int(sys.argv[1]) if len(sys.argv) > 1 else 32768
k16 = bytes([1, 1, 0, 0, 0, 0, 2, 2] + [3] * 8)
iss = Issuer(sp, ip, sk, device=0, max_batch=B)
items = np.tile(pres, ((B + 255) // 256, 1, 1))[:B]
comp = PresentationBatch.from_items(k16, items)
v, dbg = iss.verify_batch(comp, debug=True)
assert not v.any()
bb_host = torch.from_numpy(compact_to_batchable(k16, comp.fields, dbg["commitments"])).pin_memory()
bb = PresentationBatch(k16, bb_host.numpy())
comp_host = torch.from_numpy(comp.fields).pin_memory()
compp = PresentationBatch(k16, comp_host.numpy())
for name, fn in (("compact", lambda: iss.verify_batch(compp)), ("batchable_exact", lambda: iss.verify_batchable(bb)), ("batchable_rlc", lambda: iss.verify_batchable_rlc(bb, bytes(range(32)))[0])):
    fn()
    t0 = time.perf_counter()
    for _ in range(2):
        v = fn()
    dt = (time.perf_counter() - t0) / 2
    assert not v.any()
    print(name, round(B / dt), "per s", round(dt * 1e3, 1), "ms")
