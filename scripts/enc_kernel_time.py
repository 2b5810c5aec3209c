"""Per-kernel times of the bf16 vision encoder forward+backward (1024 frames of 3x200x200, the bench's encoder batch),
from torch.profiler CUDA activity over `iters` timed passes after warm-up; prints one JSON object, kernel name -> mean
microseconds per pass and launches per pass:  python scripts/enc_kernel_time.py [iters] [out.json]"""
import json
import os
import sys
import tempfile
from collections import defaultdict

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tacorl_b200 import configs, ops  # noqa: E402
from tacorl_b200.utils import synthetic  # noqa: E402
from tacorl_b200.utils.config import instantiate  # noqa: E402

iters = int(sys.argv[1]) if len(sys.argv) > 1 else 20
ops.set_precision("bf16")
enc = instantiate(configs.lmp_vision_encoder()).cuda()
synthetic.init_like_reference(enc, 0)
x = synthetic.play_batch(64, 16, 200, 200, seed=1)["states"]["rgb_static"].view(1024, 3, 200, 200).cuda()


def fb():
    for p in enc.parameters():
        p.grad = None
    e = enc(x)
    e.backward(torch.ones_like(e))


for _ in range(5):
    fb()
torch.cuda.synchronize()
with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
    for _ in range(iters):
        fb()
    torch.cuda.synchronize()
trace = os.path.join(tempfile.mkdtemp(), "trace.json")
prof.export_chrome_trace(trace)
tot, cnt = defaultdict(float), defaultdict(int)
for ev in json.load(open(trace))["traceEvents"]:
    if ev.get("cat") != "kernel":
        continue
    name = ev["name"].split("(")[0].replace("void ", "").replace("tacorl::", "")
    tot[name] += float(ev["dur"])
    cnt[name] += 1
res = {k: {"us_per_pass": round(tot[k] / iters, 2), "launches_per_pass": cnt[k] / iters}
       for k in sorted(tot, key=lambda k: -tot[k])}
res["_gpu"] = torch.cuda.get_device_name()
print(json.dumps(res, indent=1))
if len(sys.argv) > 2:
    with open(sys.argv[2], "w") as f:
        json.dump(res, f, indent=1)
