#!/usr/bin/env python
"""Frames of several resolutions in one launch (qv_forward_frame_list_device) against one launch per resolution, arms
alternated round by round on one stream in one process:
  (a) one tick of a mixed-resolution service: 4 x 416x240 + 4 x 832x480 + 2 x 1280x720 + 2 x 1920x1080 + 1 x 2560x1600
      (list)   one qv_forward_frame_list_device over the 13 frames, on one handle
      (per)    one qv_forward_frames_device per resolution, on handles created for those resolutions
  (b) a uniform batch through the list path: 64 x 1920x1080 (bench.py's workload)
      (list)   qv_forward_frame_list_device over the 64 frames
      (per)    qv_forward_frames_device on the same frames
Per-call times from CUDA events on the launching stream; per arm the median and min / max over all timed calls, and the
median of every round.  Both arms of a workload must give the same bytes.  (a) works on 24 MB (in + out), which stays in
the 126 MB L2 from call to call; (b) on 265 MB, which does not.  The card's name and power limit are read in the same run.

  python tools/frame_list_ab.py [--rounds 5] [--steps 30] [--out FILE]"""
import argparse
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

TICK = [(4, 240, 416), (4, 480, 832), (2, 720, 1280), (2, 1080, 1920), (1, 1600, 2560)]
UNIFORM = [(64, 1080, 1920)]


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

    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True).stdout.strip()
    say("card: " + " | ".join(card.splitlines()))
    say("rounds %d x steps %d per arm and workload, arms alternated within every round" % (args.rounds, args.steps))
    image = formats.write_model_vect_c(synth.make_model(0xC0FFEE + 32, 32))
    st = torch.cuda.Stream()
    s = st.cuda_stream
    for name, groups in (("(a) mixed tick", TICK), ("(b) uniform 64 x 1080p", UNIFORM)):
        blocks, outs_per, outs_list, nets = [], [], [], []
        for g, (F, H, W) in enumerate(groups):
            a, _ = synth.make_frames(0xC0FFEE + 5 + g, min(F, 8), H, W)
            reps = (F + len(a) - 1) // len(a)
            blocks.append(torch.from_numpy(np.tile(a, (reps, 1, 1))[:F]).cuda())
            outs_per.append(torch.empty_like(blocks[-1]))
            outs_list.append(torch.empty_like(blocks[-1]))
            net = api.QVRCNN(0, min(F, 8), 1, H, W)
            net.load_static_para_mem(image)
            assert net.get_impl() == api.IMPL_FUSED
            nets.append(net)
        list_net = api.QVRCNN(0, 1, 1, 16, 16)
        list_net.load_static_para_mem(image)
        desc = [(blk[i], out[i]) for blk, out in zip(blocks, outs_list) for i in range(blk.shape[0])]
        px = sum(F * H * W for F, H, W in groups)

        def arm(k):
            if k == "list":
                list_net.forward_frame_list_device(desc, None, s)
            else:
                for net, blk, out in zip(nets, blocks, outs_per):
                    net.forward_frames_device(blk.data_ptr(), out.data_ptr(), blk.shape[0], s)

        def timed(k, n):
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(n + 1)]
            ev[0].record(st)
            for i in range(n):
                arm(k)
                ev[i + 1].record(st)
            list_net.synchronize(s)
            return [ev[i].elapsed_time(ev[i + 1]) for i in range(n)]

        arms = ("list", "per")
        for k in arms:                               # warm-up: module load, every shape of the timed window
            timed(k, 3)
        ms = {k: [] for k in arms}
        per_round = {k: [] for k in arms}
        for r in range(args.rounds):
            for k in arms:
                x = timed(k, args.steps)
                ms[k] += x
                per_round[k].append(float(np.median(x)))
        same = all(torch.equal(a, b) for a, b in zip(outs_per, outs_list))
        launches = list_net.launch_count()
        say("\n%s: %s  (%.2f Mpixel per call; same bytes in both arms: %s; list launches so far: %d)" % (
            name, " + ".join("%d x %dx%d" % (F, W, H) for F, H, W in groups), px / 1e6, same, launches))
        med_per = float(np.median(ms["per"]))
        for k, label in (("list", "qv_forward_frame_list_device"), ("per", "qv_forward_frames_device per geometry")):
            x = ms[k]
            med = float(np.median(x))
            say("  %-4s %-40s median %8.3f ms  min %8.3f  max %8.3f  %8.1f Mpixel/s  (%+.2f %% vs per)  round medians: %s" % (
                k, label, med, min(x), max(x), px / 1e3 / med, 100.0 * (med / med_per - 1.0), " ".join("%.3f" % v for v in per_round[k])))
        for n in nets + [list_net]:
            n.close()
        del blocks, outs_per, outs_list, desc
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as fp:
            fp.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
