#!/usr/bin/env python
"""Cost of the per-frame SSE, three arms alternated round by round in one process:
  (a) forward_frames_device                      -- the reconstruction only
  (b) forward_frames_device_sse                  -- k_enh_sse: the SSEs in the fused kernel's output stage
  (c) (a) + per frame two qv_sse_device passes   -- the separate-pass alternative (3 more bytes read per pixel)
on 64 x 1920x1080 QP32 (bench.py's workload), 8 x 832x480 and 1 x 416x240.  Per-step times from CUDA events on the launching
stream; per arm the median and min / max over all timed steps, and the median of every round.  (b) and (c) must report the
same SSEs and all three the same reconstruction.  The card's name and power limit are read in the same run.

  python tools/frame_sse_ab.py [--rounds 5] [--steps 30] [--out FILE]"""
import argparse
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = [(64, 1080, 1920), (8, 480, 832), (1, 240, 416)]


def main():
    import torch
    from qcnn_gpu_b200 import api
    from qcnn_gpu_b200.host import formats, synth
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True).stdout.strip()
    say("card: " + " | ".join(card.splitlines()))
    say("rounds %d x steps %d per arm and workload, arms alternated within every round" % (args.rounds, args.steps))
    image = formats.write_model_vect_c(synth.make_model(0xC0FFEE + 32, 32))
    st = torch.cuda.Stream()
    for F, H, W in WORKLOADS:
        a, o = synth.make_frames(0xC0FFEE + 3, min(8, F), H, W)
        reps = (F + len(a) - 1) // len(a)
        d_in = torch.from_numpy(np.tile(a, (reps, 1, 1))[:F]).cuda()
        d_ori = torch.from_numpy(np.tile(o, (reps, 1, 1))[:F]).cuda()
        outs = {k: torch.empty_like(d_in) for k in "abc"}
        sse = {k: torch.zeros((F, 2), dtype=torch.int64, device="cuda") for k in "bc"}
        net = api.QVRCNN(0, min(F, 8), 1, H, W)
        net.load_static_para_mem(image)
        assert net.get_impl() == api.IMPL_FUSED
        fpx = H * W
        s = st.cuda_stream

        def arm(k):
            if k == "a":
                net.forward_frames_device(d_in.data_ptr(), outs["a"].data_ptr(), F, s)
            elif k == "b":
                net.forward_frames_device_sse(d_in.data_ptr(), d_ori.data_ptr(), outs["b"].data_ptr(), F, sse["b"].data_ptr(), s)
            else:
                net.forward_frames_device(d_in.data_ptr(), outs["c"].data_ptr(), F, s)
                base = sse["c"].data_ptr()
                for f in range(F):
                    api.sse_device(d_in.data_ptr() + f * fpx, d_ori.data_ptr() + f * fpx, fpx, base + 16 * f, s)
                    api.sse_device(outs["c"].data_ptr() + f * fpx, d_ori.data_ptr() + f * fpx, fpx, base + 16 * f + 8, s)

        def timed(k, n):
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(n + 1)]
            ev[0].record(st)
            for i in range(n):
                arm(k)
                ev[i + 1].record(st)
            net.synchronize(s)
            return [ev[i].elapsed_time(ev[i + 1]) for i in range(n)]

        for k in "abc":                              # warm-up: module load, every shape of the timed window
            timed(k, 3)
        for t in sse.values():
            t.zero_()
        torch.cuda.synchronize()
        ms = {k: [] for k in "abc"}
        per_round = {k: [] for k in "abc"}
        for r in range(args.rounds):
            for k in "abc":
                x = timed(k, args.steps)
                ms[k] += x
                per_round[k].append(float(np.median(x)))
        # correctness of what was timed: same reconstruction, same SSEs (summed over every call of b and of c)
        same_out = bool(torch.equal(outs["a"], outs["b"]) and torch.equal(outs["a"], outs["c"]))
        same_sse = bool(torch.equal(sse["b"], sse["c"]))
        want = ((d_in.long() - d_ori.long()) ** 2).view(F, -1).sum(1)
        calls = args.rounds * args.steps                # the warm-up calls were zeroed out
        ok_sse = bool(torch.equal(sse["b"][:, 0], want * calls))
        say("\n%d x %dx%d  (same reconstruction in all arms: %s; SSE b == c: %s; b == numpy x calls: %s)" % (F, W, H, same_out, same_sse, ok_sse))
        med_a = float(np.median(ms["a"]))
        for k, label in (("a", "forward_frames_device"), ("b", "forward_frames_device_sse"), ("c", "forward + 2 qv_sse_device per frame")):
            x = ms[k]
            say("  (%s) %-38s median %8.3f ms  min %8.3f  max %8.3f  (%+.2f %% vs a)  round medians: %s" % (
                k, label, float(np.median(x)), min(x), max(x), 100.0 * (float(np.median(x)) / med_a - 1.0),
                " ".join("%.3f" % v for v in per_round[k])))
        net.close()
        del d_in, d_ori, outs, sse
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as fp:
            fp.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
