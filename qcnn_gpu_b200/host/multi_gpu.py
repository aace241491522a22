"""Multi-GPU driver for the QVRCNN pass: one process per GPU (torchrun).  Compute goes through the C ABI.

  * frames mode: contiguous frame blocks per rank (qv_forward_frames_device), no communication during compute;
  * strips mode: one very large frame in horizontal strips (qv_strip_*): every rank keeps its rows in a block of its own
    HBM, the neighbours map that block through CUDA IPC and the fused kernel reads its 6 halo rows straight from the
    neighbour's memory over NVLink -- no NCCL call between frames.  torch.distributed carries the 192-byte descriptors
    once at setup and the int64 SSE all-reduce of the PSNR report at the end.

  torchrun --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 -m qcnn_gpu_b200.host.multi_gpu \\
      --mode frames --qp 27 --frames 240 --height 2160 --width 3840        # BASELINE config 4
  torchrun ... -m qcnn_gpu_b200.host.multi_gpu --mode strips --qp 22 --height 4320 --width 7680   # config 5

--check additionally computes the whole job on rank 0 alone and asserts the N-GPU result is bit-identical; in strips mode
every step of the check uploads a DIFFERENT frame (alternating the two input slots), so a halo row read too early or too
late shows up as a mismatch.

--per-frame adds the per-frame PSNR before and after the net (vrcnn_data::psnr_pf, inference/yuv_data.cpp:98-112): every rank
fills its part of a zeroed [frames, 2] int64 tensor of exact SSEs -- its frame range (forward_frames_device_sse) or its rows of
the frame (strip_forward_sse) -- and one all-reduce adds them up, so the result is the one-GPU result bit for bit.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


class StripRank:
    """This rank's strip of an h x w frame: handle, strip block, neighbours attached (descriptors exchanged once)."""

    def __init__(self, api, shard, local: int, image: bytes, h: int, w: int, rank: int, world: int, dist):
        self.y0, n = shard.split(h, rank, world)
        self.y1 = self.y0 + n
        if world > 1 and h // world < shard.HALO:
            raise ValueError("strips of %d rows are shorter than the %d-row halo: use fewer ranks" % (h // world, shard.HALO))
        self.net = api.QVRCNN(local, 1, 1, n, w)
        self.net.load_static_para_mem(image)
        self.net.strip_setup(h, self.y0, self.y1)
        descs = [self.net.strip_export()]
        if world > 1:
            descs = [None] * world
            dist.all_gather_object(descs, self.net.strip_export())
            if rank > 0:
                self.net.strip_attach(api.STRIP_ABOVE, descs[rank - 1])
            if rank < world - 1:
                self.net.strip_attach(api.STRIP_BELOW, descs[rank + 1])
            dist.barrier()                      # every rank has mapped its neighbours before anyone runs


def main():
    import torch
    import torch.distributed as dist
    from qcnn_gpu_b200 import api
    from qcnn_gpu_b200.host import formats, shard, synth

    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", choices=["frames", "strips"], default="frames")
    ap.add_argument("--qp", type=int, default=27)
    ap.add_argument("--frames", type=int, default=16)
    ap.add_argument("--height", type=int, default=2160)
    ap.add_argument("--width", type=int, default=3840)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--check", action="store_true")
    ap.add_argument("--per-frame", action="store_true", help="per-frame PSNR before / after the net in the JSON line")
    ap.add_argument("--uniq", type=int, default=4, help="distinct synthetic frames per rank (repeated)")
    args = ap.parse_args()
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    from qcnn_gpu_b200.host import numa
    numa.bind_to_gpu(local)
    cdev = "cuda"
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    h, w = args.height, args.width
    model = synth.make_model(0xC0FFEE + args.qp, args.qp)
    image = formats.write_model_vect_c(model)
    # an explicit non-default stream: everything of this rank's data path is ordered on it
    stream = torch.cuda.Stream()
    sp = stream.cuda_stream

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def rank_frames(r):
        """frames mode: the anchor and original frames of rank r (`uniq` distinct synthetic frames, repeated)"""
        f0, nf = shard.split(args.frames, r, world)
        uniq = max(1, min(args.uniq, nf))
        a, o = synth.make_frames(0xC0FFEE + 4, uniq, h, w, first_frame=f0 % 1024)
        reps = (nf + uniq - 1) // uniq
        return np.tile(a, (reps, 1, 1))[:nf], np.tile(o, (reps, 1, 1))[:nf]

    check_outs = []
    if args.mode == "frames":
        f0, nf = shard.split(args.frames, rank, world)
        a, o = rank_frames(rank)
        d_in = torch.from_numpy(a).cuda()
        d_ori = torch.from_numpy(o).cuda()
        d_out = torch.empty_like(d_in)
        net = api.QVRCNN(local, max(1, min(nf, 8)), 1, h, w)
        net.load_static_para_mem(image)
        run = lambda k: net.forward_frames_device(d_in.data_ptr(), d_out.data_ptr(), nf, sp)
        npx_local = nf * h * w
        halo = "none (frames are independent)"
    else:
        sr = StripRank(api, shard, local, image, h, w, rank, world, dist)
        net, y0, y1 = sr.net, sr.y0, sr.y1
        a, o = synth.make_frames(0xC0FFEE + 5, 1, h, w, rows=(y0, y1))     # only this rank's rows ever exist on this rank
        d_ori = torch.from_numpy(o[0]).cuda()
        d_out = torch.empty_like(d_ori)
        net.strip_load(0, a[0], sp)
        if args.check:
            step_frames = [synth.make_frames(0xC0FFEE + 5, 1, h, w, first_frame=1 + k, rows=(y0, y1))[0][0] for k in range(args.steps)]

            def run(k):                          # a different frame every step, alternating input slots
                if k < 0:
                    return net.strip_forward(0, d_out.data_ptr(), sp)
                net.strip_load(k & 1, step_frames[k], sp)
                net.strip_forward(k & 1, d_out.data_ptr(), sp)
                with torch.cuda.stream(stream):
                    check_outs.append(d_out.clone())
        else:
            run = lambda k: net.strip_forward(0, d_out.data_ptr(), sp)
        npx_local = (y1 - y0) * w
        halo = "peer-mapped HBM over NVLink (CUDA IPC), read by the fused kernel; no collective between frames"

    torch.cuda.synchronize()
    for _ in range(2):
        run(-1)
    net.synchronize(sp)
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for k in range(args.steps):
        run(k)
    e1.record(stream)
    net.synchronize(sp)
    sync_all()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=cdev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    if args.mode == "strips" and args.check:
        net.strip_load(0, a[0], sp)              # the report below is about the frame d_ori belongs to
        net.strip_forward(0, d_out.data_ptr(), sp)
        net.synchronize(sp)
    acc = torch.zeros(1, dtype=torch.int64, device="cuda")
    api.sse_device(d_out.data_ptr(), d_ori.data_ptr(), npx_local, acc.data_ptr(), api.CUDA_STREAM_LEGACY)
    torch.cuda.synchronize()
    psnr, sse, n = shard.psnr_from_global_sse(int(acc.item()), npx_local, dist if world > 1 else None, device=cdev)
    result = {"mode": args.mode, "qp": args.qp, "n_gpus": world, "height": h, "width": w,
              "frames": args.frames if args.mode == "frames" else 1,
              "Mpixel_per_s": n * args.steps / (float(ms.item()) * 1e-3) / 1e6, "ms_per_step": float(ms.item()) / args.steps,
              "after_quantized_net_PSNR": psnr, "sse": sse, "halo": halo}
    if args.per_frame:
        n_frames = args.frames if args.mode == "frames" else 1
        pf = torch.zeros((n_frames, 2), dtype=torch.int64, device="cuda")
        if args.mode == "frames":
            net.forward_frames_device_sse(d_in.data_ptr(), d_ori.data_ptr(), d_out.data_ptr(), nf, pf[f0:].data_ptr(), sp)
        else:                                    # slot 0 holds this rank's rows of the frame d_ori belongs to
            net.strip_forward_sse(0, d_ori.data_ptr(), d_out.data_ptr(), pf.data_ptr(), sp)
        net.synchronize(sp)
        if world > 1:
            dist.all_reduce(pf, op=dist.ReduceOp.SUM)
        pf_host = pf.cpu().numpy()
        before = [api.psnr_from_sse(int(v), h * w) for v in pf_host[:, 0]]
        after = [api.psnr_from_sse(int(v), h * w) for v in pf_host[:, 1]]
        result.update({"psnr_per_frame_before": before, "psnr_per_frame_after": after,
                       "psnr_per_frame_mean_before": float(np.mean(before)), "psnr_per_frame_mean_after": float(np.mean(after))})
    if args.check:
        # gather every rank's output on rank 0 and compare with rank 0 computing everything alone
        mine = d_out.cpu().numpy() if args.mode == "frames" else np.stack([t.cpu().numpy() for t in check_outs])
        outs = [mine]
        if world > 1:
            outs = [None] * world
            dist.all_gather_object(outs, mine)
        if rank == 0:
            if args.mode == "frames":
                got = np.concatenate(outs)
                full = np.concatenate([rank_frames(r)[0] for r in range(world)])
                solo = api.QVRCNN(local, 4, 1, h, w)
            else:
                got = np.concatenate(outs, axis=1)                      # [steps, h, w]
                full = np.concatenate([synth.make_frames(0xC0FFEE + 5, 1, h, w, first_frame=1 + k)[0] for k in range(args.steps)])
                solo = api.QVRCNN(local, 1, 1, h, w)
            solo.load_static_para_mem(image)
            want = solo.forward_frames_host(full)
            result["bit_identical_to_1gpu"] = bool(np.array_equal(got.reshape(want.shape), want))
            result["distinct_frames_checked"] = int(want.shape[0])
            if args.per_frame:
                # the all-reduced per-frame SSEs against rank 0's own computation of the frames of the report
                if args.mode == "frames":
                    anc, ori = full, np.concatenate([rank_frames(r)[1] for r in range(world)])
                    rec = want
                else:
                    anc, ori = synth.make_frames(0xC0FFEE + 5, 1, h, w)
                    rec = solo.forward_frames_host(anc)
                sse = lambda x: ((x.astype(np.int64) - ori.astype(np.int64)) ** 2).reshape(len(ori), -1).sum(axis=1)
                result["per_frame_sse_identical_to_1gpu"] = bool(np.array_equal(pf_host, np.stack([sse(anc), sse(rec)], axis=1)))
    if rank == 0:
        print(json.dumps(result))
    if world > 1:
        dist.barrier()
    if args.mode == "strips":
        net.strip_release()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
