#!/usr/bin/env python
"""bench.py -- luma Mpixel/s of the QVRCNN int8 pass (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--kernel auto|fused|layered] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic luma: BASELINE config 3,
QP=32, 64 frames of 1920x1080 per GPU (weak scaling: every rank processes its own 64 frames,
frame-sharded, no data-path collective; the only collective is the int64 SSE all-reduce of the
PSNR report, outside the timed region).  `value` = whole-job Mpixel/s with the frames already
resident in HBM; `e2e` = the same metric through the host-buffer entry point
qv_forward_frames_host (pinned host memory -> H2D -> net -> D2H every step), with the box's measured
concurrent copy ceiling beside it.  Further blocks of the same JSON line: `sustained` (320 back-to-back
steps under the power cap, own clock sample), `config4` (BASELINE config 4: 240 x 4K frames sharded over the
ranks) and `config5` (config 5: one 8K frame in N strips, halo rows read from the neighbour GPUs' memory),
each with a bit-identity check against one GPU.

--impl reference times the reference path's CPU restatement (oracle/, the only CPU implementation
of this path that exists: the reference itself is cuDNN-only) on the box's host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

OPS_PER_PIXEL = 109024          # 2 * 54512 MAC, BASELINE.md section 2
HBM_BYTES_PER_PIXEL = 2          # 1 B luma in + 1 B recon out
QP, FRAMES, H, W = 32, 64, 1080, 1920
WORKLOAD = "config3: QVRCNN QP=32, 64x1920x1080 synthetic luma frames per GPU"


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_burst=d["bf16_tflops"], bf16_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_burst=1590.0, bf16_sustained=1400.0, source="fallback (B200_PROFILING.md)")


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the fused kernel on this workload, from the committed
    `ncu --set full` capture (profiles/ncu_fused_traffic.json, written by tools/ncu_summary.py); None if absent."""
    p = os.path.join(ROOT, "profiles", "ncu_fused_traffic.json")
    try:
        d = json.load(open(p))
        if d.get("workload") != WORKLOAD:
            return None
        return {"dram_bytes_per_launch": d["dram_bytes_read"] + d["dram_bytes_write"], "algorithmic_bytes_per_launch": FRAMES * H * W * HBM_BYTES_PER_PIXEL,
                "unit": "B", "source": d.get("source")}
    except Exception:
        return None


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (one streaming nvidia-smi
    process at 50 ms period; only lines that arrive between start() and stop() are kept)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag, self.proc = index, [], threading.Event(), None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag.is_set():
                    break
                parts = [s.strip() for s in line.split(",")]
                if len(parts) >= 7:
                    self.samples.append(parts)
        except Exception:
            pass

    def stop(self):
        self.stop_flag.set()
        if self.proc is not None:
            try:
                self.proc.terminate()
            except Exception:
                pass
        self.join(timeout=2)

    def summary(self):
        def num(v):
            try:
                return float(v)
            except ValueError:
                return None
        sm = [num(s[0]) for s in self.samples if num(s[0]) is not None]
        mx = [num(s[1]) for s in self.samples if num(s[1]) is not None]
        pw = [num(s[2]) for s in self.samples if num(s[2]) is not None]
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons), "samples": len(self.samples)}


def build_inputs(rank: int):
    from qcnn_gpu_b200.host import formats, synth
    model = synth.make_model(0xC0FFEE + QP, QP)
    uniq = 8                                    # 8 distinct frames per rank, repeated to 64
    anchor, ori = synth.make_frames(0xC0FFEE + 3, uniq, H, W, first_frame=rank * uniq)
    reps = FRAMES // uniq
    return model, formats.write_model_vect_c(model), np.tile(anchor, (reps, 1, 1)), np.tile(ori, (reps, 1, 1))


def copy_ceiling(torch, dist, world, nbytes, reps=6):
    """What the host side of this box can move: every rank copies `nbytes` host->device and `nbytes` device->host between
    pinned memory and HBM CONCURRENTLY (two streams, one cudaMemcpyAsync per copy), all ranks at once -- the traffic pattern of
    the e2e step without any compute.  Returns aggregate GB/s each way (bytes of all ranks / slowest rank's time)."""
    h_a = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    h_b = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    d_a = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    d_b = torch.zeros(nbytes, dtype=torch.uint8, device="cuda")
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()

    def once():
        with torch.cuda.stream(s1):
            d_a.copy_(h_a, non_blocking=True)
        with torch.cuda.stream(s2):
            h_b.copy_(d_b, non_blocking=True)
    once()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        once()
    torch.cuda.synchronize()
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    gbs = world * nbytes * reps / float(dt.item()) / 1e9
    return {"h2d_plus_d2h_concurrent_gbs_each_way": gbs, "per_gpu_gbs_each_way": gbs / world, "bytes_per_copy": nbytes, "reps": reps,
            "how": "pinned <-> HBM, one cudaMemcpyAsync per copy, H2D and D2H on two streams, all ranks at once, no compute"}


def run_config4(torch, dist, api, rank, world, local, steps=5, warmup=2):
    """BASELINE config 4: QVRCNN QP=27, 240 frames of 3840x2160, frame-sharded (240/N per GPU, no collective), device
    resident.  Bit-identity with one GPU: every rank's distinct frames and their outputs are gathered on rank 0, which runs
    them alone; the tiled copies are compared on the rank that made them."""
    from qcnn_gpu_b200.host import formats, shard, synth
    qp, total, h, w, uniq = 27, 240, 2160, 3840, 2
    f0, nf = shard.split(total, rank, world)
    model = synth.make_model(0xC0FFEE + qp, qp)
    image = formats.write_model_vect_c(model)
    a, _ = synth.make_frames(0xC0FFEE + 4, uniq, h, w, first_frame=rank * uniq)
    d_u = torch.from_numpy(a).cuda()
    d_in = d_u.repeat((nf + uniq - 1) // uniq, 1, 1)[:nf].contiguous()
    d_out = torch.empty_like(d_in)
    net = api.QVRCNN(local, 8, 1, h, w)
    net.load_static_para_mem(image)
    st = torch.cuda.Stream()
    torch.cuda.synchronize()
    run = lambda: net.forward_frames_device(d_in.data_ptr(), d_out.data_ptr(), nf, st.cuda_stream)
    for _ in range(warmup):
        run()
    net.synchronize(st.cuda_stream)
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for _ in range(steps):
        run()
    e1.record(st)
    net.synchronize(st.cuda_stream)
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    # every copy of a distinct frame gave the same output (checked where it was computed) ...
    ok_local = all(bool(torch.equal(d_out[j], d_out[j % uniq])) for j in range(uniq, nf))
    flag = torch.tensor([1 if ok_local else 0], dtype=torch.int64, device="cuda")
    g_in = [torch.empty_like(d_u) for _ in range(world)]
    g_out = [torch.empty_like(d_u) for _ in range(world)]
    mine_out = d_out[:uniq].contiguous()
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        dist.all_gather(g_in, d_u)
        dist.all_gather(g_out, mine_out)
    else:
        g_in, g_out = [d_u], [mine_out]
    block = None
    if rank == 0:
        # ... and the distinct frames of every rank, run by rank 0 alone, give what the ranks got
        solo_in = torch.cat(g_in)
        solo_out = torch.empty_like(solo_in)
        net.forward_frames_device(solo_in.data_ptr(), solo_out.data_ptr(), solo_in.shape[0], st.cuda_stream)
        net.synchronize(st.cuda_stream)
        same = bool(torch.equal(solo_out, torch.cat(g_out))) and bool(flag.item() == 1)
        t = float(ms.item()) / steps
        block = {"workload": "config4: QVRCNN QP=27, 240x3840x2160 frames, frame-sharded (%d per GPU)" % nf, "n_gpus": world,
                 "Mpixel_per_s": total * h * w / (t * 1e-3) / 1e6, "ms_per_step": t, "steps": steps, "scaling": "strong",
                 "bit_identical_to_1gpu": same, "bytes_exchanged_per_step": 0, "collectives_in_timed_region": 0,
                 "distinct_frames_per_gpu": uniq}
    del net, d_in, d_out
    torch.cuda.empty_cache()
    return block


def run_config5(torch, dist, api, rank, world, local, steps=20, warmup=3):
    """BASELINE config 5: QVRCNN QP=22, ONE 7680x4320 frame cut into N horizontal strips, one per GPU.  Each GPU keeps only
    its own rows; the fused kernel reads the 6 halo rows either side out of the neighbour GPUs' HBM (peer-mapped through CUDA
    IPC, NVLink), ordered by sequence words the kernels write and poll themselves: no NCCL call and no host
    synchronisation between frames (qv_strip_forward).  The check uploads a DIFFERENT frame for each of two further
    steps, alternating the two input slots, and rank 0 recomputes those frames alone."""
    from qcnn_gpu_b200.host import formats, multi_gpu, shard, synth
    qp, h, w = 22, 4320, 7680
    model = synth.make_model(0xC0FFEE + qp, qp)
    image = formats.write_model_vect_c(model)
    sr = multi_gpu.StripRank(api, shard, local, image, h, w, rank, world, dist)
    net, y0, y1 = sr.net, sr.y0, sr.y1
    st = torch.cuda.Stream()
    sp = st.cuda_stream
    a, _ = synth.make_frames(0xC0FFEE + 5, 1, h, w, rows=(y0, y1))
    d_out = torch.empty((y1 - y0, w), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    net.strip_load(0, a[0], sp)
    l0 = net.launch_count()
    for _ in range(warmup):
        net.strip_forward(0, d_out.data_ptr(), sp)
    net.synchronize(sp)
    per_step_launches = (net.launch_count() - l0) / max(1, warmup)
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for _ in range(steps):
        net.strip_forward(0, d_out.data_ptr(), sp)
    e1.record(st)
    net.synchronize(sp)
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    # check: further, different frames, alternating the input slots
    n_chk = 2
    outs, fks = [], []
    for k in range(n_chk):
        fk = synth.make_frames(0xC0FFEE + 5, 1, h, w, first_frame=1 + k, rows=(y0, y1))[0][0]
        fks.append(fk)
        net.strip_load((k + 1) & 1, fk, sp)
        net.strip_forward((k + 1) & 1, d_out.data_ptr(), sp)
        with torch.cuda.stream(st):
            outs.append(d_out.clone())
    net.synchronize(sp)
    mine = torch.stack(outs)                                         # [n_chk, rows, w]
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        rows = [shard.split(h, r, world)[1] for r in range(world)]
        parts = [torch.empty((n_chk, rows[r], w), dtype=torch.uint8, device="cuda") for r in range(world)]
        # rows per rank may differ by one: gather through rank 0 with point-to-point copies (outside the timed region)
        if rank == 0:
            parts[0] = mine
            for r in range(1, world):
                dist.recv(parts[r], src=r)
        else:
            dist.send(mine, dst=0)
    else:
        parts = [mine]
    block = None
    if rank == 0:
        got = torch.cat(parts, dim=1)
        full = np.stack(fks) if world == 1 else np.concatenate([synth.make_frames(0xC0FFEE + 5, 1, h, w, first_frame=1 + k)[0] for k in range(n_chk)])
        solo = api.QVRCNN(local, 1, 1, h, w)
        solo.load_static_para_mem(image)
        d_full = torch.from_numpy(full).cuda()
        d_want = torch.empty_like(d_full)
        solo.forward_frames_device(d_full.data_ptr(), d_want.data_ptr(), n_chk, sp)
        solo.synchronize(sp)
        t = float(ms.item()) / steps
        halo_bytes = (2 * world - 2) * shard.HALO * w
        block = {"workload": "config5: QVRCNN QP=22, one 7680x4320 frame in %d horizontal strip(s)" % world, "n_gpus": world,
                 "Mpixel_per_s": h * w / (t * 1e-3) / 1e6, "ms_per_frame": t, "steps": steps, "scaling": "strong",
                 "bit_identical_to_1gpu": bool(torch.equal(got, d_want)), "distinct_frames_checked": n_chk,
                 "halo": "6 rows each way read by the fused kernel from the neighbour GPU's HBM (peer-mapped, CUDA IPC, NVLink)" if world > 1 else "none (one strip)",
                 "bytes_exchanged_per_step": halo_bytes, "nccl_calls_between_frames": 0, "kernel_launches_per_step_per_gpu": per_step_launches}
        del solo
    if world > 1:
        dist.barrier()
    net.strip_release()
    del net
    torch.cuda.empty_cache()
    return block


DUMP_SEED, DUMP_FRAMES, DUMP_PIXELS = 20261020, 4, 1 << 22


def dump_outputs(out_dir: str, d_out) -> None:
    """What the timed step hands its caller, the reconstructed luma d_out (uint8 [FRAMES, H, W], 133 MB), as float32 .npy
    files of 50 MB: recon_frames.npy = DUMP_FRAMES whole frames, recon_pixels.npy = DUMP_PIXELS pixels over the whole batch.
    Which frames and pixels depends on DUMP_SEED alone, so two builds of the project can be compared file for file."""
    import torch
    rng = np.random.default_rng(DUMP_SEED)
    frames = np.sort(rng.choice(FRAMES, DUMP_FRAMES, replace=False))
    pixels = np.sort(rng.integers(0, FRAMES * H * W, DUMP_PIXELS))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "recon_frames.npy"), d_out[torch.from_numpy(frames).cuda()].cpu().numpy().astype(np.float32))
    np.save(os.path.join(out_dir, "recon_pixels.npy"), d_out.view(-1)[torch.from_numpy(pixels).cuda()].cpu().numpy().astype(np.float32))


REF_BIN = os.path.join(ROOT, "oracle", "_ref", "qcnn_ref_witness")


def _gpu_present() -> bool:
    try:
        return subprocess.run(["nvidia-smi", "-L"], capture_output=True, timeout=20).returncode == 0
    except Exception:
        return False


def run_reference(args, rank: int, world: int):
    """Reference arm.  The reference has NO CPU implementation of this path: its forward_blu is six
    cudnnConvolutionForward calls plus glue kernels (inference/cnn.cu:145-160).  When the witness binary
    (the reference's own unmodified sources compiled against cuDNN by oracle/ref_witness/Makefile) and a GPU
    are present, this arm runs THAT, with the reference's own driver sequence and timer scope (one frame at a
    time on device 0: H2D, forward_blu, sync, D2H -- inference/kernel.cu:89-101), kind = "reference".
    The CPU restatement (oracle port, all host threads) is timed beside it as `cpu_baseline`; it is also
    the fallback `value` when the binary or the GPU is missing (kind = "port").  Each step is a bounded
    sample of the workload: `sample_frames` 1920x1080 frames of the same synthetic batch."""
    if rank != 0:
        return
    import tempfile
    from oracle import oracle
    from qcnn_gpu_b200.host import formats, synth
    model = synth.make_model(0xC0FFEE + QP, QP)
    image = formats.write_model_vect_c(model)
    # The reference itself (witness binary) runs the WHOLE batch of our arm every step -- the same 64 frames, one forward_blu per
    # frame as its driver does; the CPU port beside it is timed on a bounded sample of that batch.
    use_witness = args.reference_kind != "cpu" and os.path.exists(REF_BIN) and _gpu_present()
    sample_frames = FRAMES if use_witness else 4
    _, _, anchor, _ = build_inputs(0)
    anchor = anchor[:sample_frames]
    om = oracle.OracleModel(image)
    # CPU port: one frame per step
    om.forward_blu(anchor[:1, :270])
    cpu_steps = args.steps
    t0 = time.perf_counter()
    for i in range(cpu_steps):
        cpu_out = om.forward_blu(anchor[i % sample_frames:i % sample_frames + 1])
    cpu_dt = time.perf_counter() - t0
    cpu_mpx = cpu_steps * H * W / cpu_dt / 1e6
    cores = oracle.num_threads()
    cpu_block = {"value": cpu_mpx, "unit": "Mpixel/s", "cores": cores, "kind": "port",
                 "sample": "%d x one 1920x1080 frame, OpenMP C oracle (oracle/qvrcnn_oracle.c)" % cpu_steps}
    kind, value, ms_per_step, note, matches = "port", cpu_mpx, cpu_dt / cpu_steps * 1e3, "CPU oracle port (no GPU or no witness binary)", None
    if use_witness:
        with tempfile.TemporaryDirectory() as td:
            mf, fi, fo = os.path.join(td, "m.data"), os.path.join(td, "in.luma"), os.path.join(td, "out.luma")
            open(mf, "wb").write(image)
            anchor.tofile(fi)
            reps = args.warmup + args.steps
            p = subprocess.run([REF_BIN, mf, str(H), str(W), str(sample_frames), fi, fo, str(reps)], capture_output=True, text=True,
                               timeout=300 + 30 * reps)     # a step of the reference takes ~3 s on a B200
            times = [int(l.split(":")[1]) for l in p.stdout.splitlines() if l.startswith("time_us:")]
            if p.returncode == 0 and len(times) == reps:
                timed = times[args.warmup:]
                tot = sum(timed) * 1e-6
                value = len(timed) * sample_frames * H * W / tot / 1e6
                ms_per_step = tot / len(timed) * 1e3
                kind = "reference"
                note = "unmodified reference sources (inference/*.cu) + cuDNN on GPU 0, one frame per forward_blu, " \
                       "timer scope of inference/kernel.cu:89-101 (H2D + forward_blu + sync + D2H)"
                rec = np.fromfile(fo, np.uint8).reshape(sample_frames, H, W)
                matches = bool(np.array_equal(rec[:1], om.forward_blu(anchor[:1])))
            else:
                note = "witness binary failed (rc=%d): %s" % (p.returncode, (p.stderr or p.stdout)[-200:].replace("\n", " "))
    line = {"impl": "reference", "metric": "luma Mpixel/s (QVRCNN int8, 1080p)", "value": value, "unit": "Mpixel/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int8", "data": "synthetic",
            "config": {"workload": WORKLOAD, "sample": ("the whole batch: %d frames of 1920x1080 per step" if sample_frames == FRAMES else "%d frames of 1920x1080 from the batch per step") % sample_frames,
                       "reference_kind": kind, "note": note},
            "cpu_baseline": cpu_block,
            "e2e": {"value": value, "unit": "Mpixel/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if matches is not None:
        line["reference_output_matches_oracle"] = matches
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--kernel", default="auto", choices=["auto", "fused", "layered"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sustained", action="store_true")
    ap.add_argument("--sustained-steps", type=int, default=320, help="back-to-back steps of the `sustained` block (>= 2 s)")
    ap.add_argument("--no-extra-configs", action="store_true", help="skip the config4 / config5 blocks")
    ap.add_argument("--reference-kind", default="auto", choices=["auto", "cpu"],
                    help="--impl reference: auto = the real reference (cuDNN) when it can run, cpu = the CPU port only")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write a fixed, seeded sample of what the last one computed (rank 0) to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from qcnn_gpu_b200 import api

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    from qcnn_gpu_b200.host import numa
    # host threads + pinned staging on the GPU's NUMA node: matters for e2e when N ranks share the host; at N = 1 the
    # process keeps all cores (the cpu_baseline leg uses them)
    numa_info = numa.bind_to_gpu(local) if world > 1 else {"bound": False}
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    model, image, anchor, ori = build_inputs(rank)
    net = api.QVRCNN(local, FRAMES, 1, H, W)
    net.load_static_para_mem(image)
    net.set_impl({"auto": api.IMPL_AUTO, "fused": api.IMPL_FUSED, "layered": api.IMPL_LAYERED}[args.kernel])
    impl_name = {api.IMPL_FUSED: "fused-tcgen05", api.IMPL_LAYERED: "layered-dp4a"}[net.get_impl()]

    h_in = torch.from_numpy(anchor).pin_memory()
    h_out = torch.empty_like(h_in).pin_memory()
    d_in = h_in.cuda()
    d_ori = torch.from_numpy(ori).cuda()
    d_out = torch.empty_like(d_in)
    stream = torch.cuda.Stream()                 # an explicit stream: launches and the timing events share it
    torch.cuda.synchronize()
    npx = FRAMES * H * W

    def step_device():
        net.forward_frames_device(d_in.data_ptr(), d_out.data_ptr(), FRAMES, stream.cuda_stream)

    sampler = ClockSampler(local)
    sampler.start()
    t_s = time.perf_counter()
    while not sampler.samples and time.perf_counter() - t_s < 8.0:      # nvidia-smi takes a second or two to come up:
        time.sleep(0.05)                                                 # the timed region must not be over before it does
    for _ in range(max(args.warmup, 3)):
        step_device()
    barrier()
    sampler.samples.clear()
    l0 = net.launch_count()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    evs[0].record(stream)
    for i in range(args.steps):
        step_device()
        evs[i + 1].record(stream)
    net.synchronize(stream.cuda_stream)          # also surfaces a failure a CTA reported
    barrier()
    launches = net.launch_count() - l0
    sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, d_out)
    total_ms = evs[0].elapsed_time(evs[-1])
    step_ms = [evs[i].elapsed_time(evs[i + 1]) for i in range(args.steps)]

    # The steady state: the default region above is ~0.2 s, over before the board's power reading catches up; SUSTAINED_STEPS
    # back-to-back steps (>= 2 s) with their own clock sample show the operating point under the 1000 W cap.
    sustained = None
    if not args.no_sustained:
        s2 = ClockSampler(local)
        s2.start()
        t_s = time.perf_counter()
        while not s2.samples and time.perf_counter() - t_s < 8.0:
            time.sleep(0.05)
        barrier()
        n_sus = max(args.sustained_steps, 1)
        es = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        es[0].record(stream)
        for i in range(n_sus):
            if i == n_sus // 2:
                s2.samples.clear()               # clocks of the second half only
                es[1].record(stream)
            step_device()
        es[2].record(stream)
        net.synchronize(stream.cuda_stream)
        barrier()
        s2.stop()
        sus = torch.tensor([es[0].elapsed_time(es[2]), es[1].elapsed_time(es[2])], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(sus, op=dist.ReduceOp.MAX)
        sustained = {"steps": n_sus, "seconds": float(sus[0].item()) * 1e-3, "ms_per_step": float(sus[0].item()) / n_sus,
                     "ms_per_step_second_half": float(sus[1].item()) / (n_sus - n_sus // 2), "clocks_second_half": s2.summary()}

    # PSNR report + exact SSE (outside the timed region); the one collective of the job
    acc = torch.zeros(2, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    api.sse_device(d_in.data_ptr(), d_ori.data_ptr(), npx, acc[0:1].data_ptr(), stream.cuda_stream)
    api.sse_device(d_out.data_ptr(), d_ori.data_ptr(), npx, acc[1:2].data_ptr(), stream.cuda_stream)
    stream.synchronize()
    tmax = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(acc, op=dist.ReduceOp.SUM)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    torch.cuda.synchronize()
    total_ms = float(tmax.item())
    psnr_before = api.psnr_from_sse(int(acc[0].item()), npx * world)
    psnr_after = api.psnr_from_sse(int(acc[1].item()), npx * world)

    # end to end through the host-buffer entry point (pinned host memory in and out, every step)
    for _ in range(2):
        net.forward_frames_host_ptr(h_in.data_ptr(), h_out.data_ptr(), FRAMES)
    barrier()
    t0 = time.perf_counter()
    e2e_steps = max(3, min(args.steps, 10))
    for _ in range(e2e_steps):
        net.forward_frames_host_ptr(h_in.data_ptr(), h_out.data_ptr(), FRAMES)
    barrier()
    e2e_s = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_mpx = world * npx * e2e_steps / float(e2e_s.item()) / 1e6
    same = bool(torch.equal(h_out.cuda(), d_out))
    ceiling = copy_ceiling(torch, dist, world, npx)
    cfg4 = cfg5 = None
    if not args.no_extra_configs and net.get_impl() == api.IMPL_FUSED:
        cfg4 = run_config4(torch, dist, api, rank, world, local)
        cfg5 = run_config5(torch, dist, api, rank, world, local)

    # The reference driver's own call pattern (inference/kernel.cu:91-97: per frame load_data, forward_blu, D2H of x_rec),
    # one 1920x1080 frame per call through the drop-in surface -- what a user who only relinks the driver gets.
    per_frame = None
    if rank == 0:
        net1 = api.QVRCNN(local, 1, 1, H, W)
        net1.load_static_para_mem(image)
        frames1 = [np.ascontiguousarray(anchor[i:i + 1]) for i in range(8)]
        for f in frames1[:3]:
            net1.load_data(f); net1.forward_blu(); net1.get_recon()
        reps = 24
        t0 = time.perf_counter()
        for i in range(reps):
            net1.load_data(frames1[i % 8]); net1.forward_blu(); rec1 = net1.get_recon()
        dt_pageable = (time.perf_counter() - t0) / reps
        # the vrcnn_data shim hands the driver page-locked frame buffers (qv_host_alloc): same calls, plain DMA
        import ctypes
        L = api.lib()
        fpx1 = H * W
        pin_in, pin_out = L.qv_host_alloc(8 * fpx1), L.qv_host_alloc(fpx1)
        for i in range(8):
            ctypes.memmove(pin_in + i * fpx1, frames1[i].ctypes.data, fpx1)
        t0 = time.perf_counter()
        for i in range(reps):
            L.qv_load_data(net1._h, pin_in + (i % 8) * fpx1); L.qv_forward_blu(net1._h); L.qv_get_recon(net1._h, pin_out)
        dt = (time.perf_counter() - t0) / reps
        last = np.ctypeslib.as_array(ctypes.cast(pin_out, ctypes.POINTER(ctypes.c_uint8)), shape=(H, W)).copy()
        ok1 = bool(np.array_equal(last, rec1[0]))
        L.qv_host_free(pin_in); L.qv_host_free(pin_out)
        per_frame = {"ms_per_frame": dt * 1e3, "Mpixel_per_s": H * W / dt / 1e6, "ms_per_frame_pageable": dt_pageable * 1e3,
                     "same_frame_both_ways": ok1,
                     "calls": "qv_load_data + qv_forward_blu + qv_get_recon, one 1920x1080 frame per call, the shim's page-locked buffers"}
        del net1

    if rank == 0:
        peaks = measured_peaks()
        value = world * npx * args.steps / (total_ms * 1e-3) / 1e6
        per_gpu_px_s = npx * args.steps / (total_ms * 1e-3)
        tops = per_gpu_px_s * OPS_PER_PIXEL / 1e12
        # int8 dense peak = 2 x the bf16 figure.  The kernel runs alone at the full SM clock (1965 MHz, ~310 W, no power
        # throttling), so the BURST cuBLAS measurement is the denominator; the fraction of the sustained (power-capped,
        # ~1.36 GHz) figure and of the nominal 4.5 POP/s are reported beside it.
        int8_peak = 2.0 * peaks["bf16_burst"]
        line = {
            "metric": "luma Mpixel/s (QVRCNN int8, 1080p)", "value": value, "unit": "Mpixel/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int8", "data": "synthetic",
            "config": {"workload": WORKLOAD, "kernel": impl_name, "frames_per_gpu": FRAMES, "parallelism": "frame-sharded dp%d" % world,
                       "l2": "inputs+outputs (265 MB/step) larger than L2 (126 MB)"},
            "gpu_launches": int(launches),
            "e2e": {"value": e2e_mpx, "unit": "Mpixel/s", "h2d_bytes_per_step": npx, "d2h_bytes_per_step": npx,
                    "api": "qv_forward_frames_host (pinned host in/out)", "bit_identical_to_device_path": same,
                    # what could bind the end-to-end rate: the kernels (device-resident rate) or the host side (the box's
                    # measured concurrent pinned-copy rate, 1 byte per pixel each way)
                    "copy_ceiling": ceiling, "copy_gbs_each_way": e2e_mpx * 1e6 / 1e9,
                    "frac_of_copy_ceiling": e2e_mpx * 1e6 / 1e9 / ceiling["h2d_plus_d2h_concurrent_gbs_each_way"],
                    "frac_of_device_rate": e2e_mpx / value,
                    "bound": "copies (host memory / PCIe)" if ceiling["h2d_plus_d2h_concurrent_gbs_each_way"] * 1e3 < value else "kernel",
                    "frac_of_binding_limit": e2e_mpx / min(value, ceiling["h2d_plus_d2h_concurrent_gbs_each_way"] * 1e3),
                    "numa": numa_info, "reference_call_pattern": per_frame},
            "roofline": {"bound": "tensor", "achieved": tops, "peak": int8_peak, "unit": "TOP/s (int8)", "frac": tops / int8_peak,
                         "traffic": ncu_traffic(), "peak_source": "2 x bf16_tflops (burst), " + peaks["source"],
                         "frac_of_2x_bf16_sustained": tops / (2.0 * peaks["bf16_sustained"]), "frac_of_nominal_4500": tops / 4500.0,
                         "hbm": {"achieved_gbs": per_gpu_px_s * HBM_BYTES_PER_PIXEL / 1e9, "peak_gbs": peaks["hbm_gbs"],
                                 "frac": per_gpu_px_s * HBM_BYTES_PER_PIXEL / 1e9 / peaks["hbm_gbs"]},
                         "kernel_ms_per_launch": total_ms / max(1, launches)},
            "clocks": sampler.summary(),
            "psnr": {"before_net": psnr_before, "after_quantized_net": psnr_after},
            "step_ms": [round(x, 3) for x in step_ms],
        }
        if sustained:
            t_s = npx / (sustained["ms_per_step_second_half"] * 1e-3) * OPS_PER_PIXEL / 1e12
            sustained.update({"Mpixel_per_s": world * npx / (sustained["ms_per_step"] * 1e-3) / 1e6,
                              "tops_per_gpu_second_half": t_s, "frac_of_2x_bf16_sustained": t_s / (2.0 * peaks["bf16_sustained"]),
                              "frac_of_2x_bf16_burst": t_s / int8_peak, "frac_of_nominal_4500": t_s / 4500.0})
            line["sustained"] = sustained
        if cfg4:
            line["config4"] = cfg4
        if cfg5:
            line["config5"] = cfg5
        if world == 1 and not args.no_cpu_baseline:
            from oracle import oracle
            from qcnn_gpu_b200.host import formats
            om = oracle.OracleModel(formats.write_model_vect_c(model))
            om.forward_blu(anchor[:1, :135])
            t0 = time.perf_counter()
            nb = 4
            ref = om.forward_blu(anchor[:nb])
            dt = time.perf_counter() - t0
            line["cpu_baseline"] = {"value": nb * H * W / dt / 1e6, "unit": "Mpixel/s", "cores": oracle.num_threads(), "kind": "port",
                                    "sample": "%d of the 64 frames (1920x1080), OpenMP C oracle" % nb,
                                    "gpu_matches_oracle_on_sample": bool(np.array_equal(ref, d_out[:nb].cpu().numpy()))}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
