"""One eager training step of a bench workload from the tree ROOT, on the GPU: kernel launches (gn_launch_count), and the
ordered sequence of library calls with the stream each was issued on (streams numbered by first use) and every
side-stream pick.  usage: python profiles/step_calls.py ROOT WORKLOAD OUT.json"""
import argparse
import hashlib
import json
import os
import sys

root, wl, out = sys.argv[1], sys.argv[2], sys.argv[3]
root = os.path.abspath(root)
sys.path.insert(0, root)
os.chdir(root)

import torch  # noqa: E402

import bench  # noqa: E402
import gripnet_b200 as gb  # noqa: E402
from gripnet_b200 import _lib, streams  # noqa: E402

assert os.path.dirname(gb.__file__) == os.path.join(root, "gripnet_b200"), gb.__file__
dev = torch.device("cuda", 0)
torch.cuda.set_device(0)
args = argparse.Namespace(workload=wl, warmup=3, eager=True, steps=1)
w = bench.build_workload(args, wl, 1, 0, dev, None)
step, _ = bench.capture_step(w, None, args, 1, 0)      # eager: three warm-up steps
torch.cuda.synchronize()

log, ids = [], {}
orig_check, orig_next = _lib.check, streams._next_side


def check(status, what=""):
    s = streams.effective_stream().cuda_stream
    log.append((what, ids.setdefault(s, len(ids))))
    return orig_check(status, what)


def next_side(device, avoid=None, background=False):
    s = orig_next(device, avoid=avoid, background=background)
    log.append(("branch", bool(background), ids.setdefault(s.cuda_stream, len(ids))))
    return s


_lib.check, streams._next_side = check, next_side
step.replay()
torch.cuda.synchronize()
_lib.check, streams._next_side = orig_check, orig_next
rec = {"workload": wl, "launches": step.launches_per_replay, "calls": sum(1 for e in log if e[0] != "branch"),
       "branches": sum(1 for e in log if e[0] == "branch"), "streams": len(ids),
       "sha1": hashlib.sha1(repr(log).encode()).hexdigest()}
print(json.dumps(rec), flush=True)
with open(out, "w") as f:
    json.dump({"summary": rec, "log": log}, f)
