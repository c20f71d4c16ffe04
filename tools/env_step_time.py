"""Times mho_env_step (csrc/env_step.cu) on the recorded items of tests/golden/env_cases.npz.

The 63 recorded items (baseline, local and GNN on networks of 20-200 nodes) are replicated to the size of one
AdHoc_test file (30 items: 10 instances x 3 methods) and of 100 files (3000 items); the outputs are checked against
the recording, then timed with CUDA events over many replays after warm-up: the whole call (upload of the item
arrays, kernel, download of the outputs) and the kernel alone (inputs resident on the device).  Whole recorded cases are replicated, so the two batches hold 36 and 3003 items.  Prints one
JSON line with the device name and power limit read in the same run.

    python tools/env_step_time.py [--reps 200]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)


def power_limit():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=20).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    a = ap.parse_args()
    import torch
    from multihop_offload_b200 import env_step as ES
    from test_env_step import golden_cases
    cases = list(golden_cases(os.path.join(ROOT, "tests", "golden")))
    res = {"device": torch.cuda.get_device_name(0), "power_limit": power_limit(), "reps": a.reps}
    for label, target in (("one_file", 30), ("100_files", 3000)):
        batches, n = [], 0
        while n < target:   # whole recorded cases, in order, until there are at least `target` items
            for net, items, _ in cases:
                if n >= target:
                    break
                batches.append((net, items))
                n += items["n_items"]
        net, items = ES.merge(batches)
        want_items = int(items["n_items"])
        got = ES.launch(net, items, want=())
        jo = 0
        for (_, it), rec in zip(batches, [c[2] for c in cases] * (len(batches) // len(cases) + 1)):
            nj = int(it["job_off"][-1])
            assert np.array_equal(got["delay_emp"][jo:jo + nj], rec["delay_emp"], equal_nan=True), label
            jo += nj
        dev = ES.upload_net(net, "cuda:0")
        for _ in range(a.warmup):
            ES.launch(net, items, want=(), dev_net=dev)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.reps):
            ES.launch(net, items, want=(), dev_net=dev)
        e1.record()
        torch.cuda.synchronize()
        end_to_end = e0.elapsed_time(e1) / a.reps
        call, _, _ = ES.bind(net, items, want=(), dev_net=dev)   # kernel only: inputs resident, outputs stay on the device
        for _ in range(a.warmup):
            call()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(a.reps):
            call()
        e1.record()
        torch.cuda.synchronize()
        res[label] = {"items": want_items, "jobs": int(items["job_off"][-1]), "ms_per_call_with_copies": end_to_end,
                      "ms_per_kernel_launch": e0.elapsed_time(e1) / a.reps}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
