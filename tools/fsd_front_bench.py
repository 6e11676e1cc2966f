"""The FSD segmentation front at configs/fsd size - dynamic voxelisation, DynamicScatterVFE(5 -> [64, 64]), SimpleSparseUNet
(flagship.FSD_UNET, 34 sparse convolutions), Voxel2PointScatterNeck - on 150k-point sweeps (synth_frame(seed, 150000, extra_dims=2), four
distinct sweeps cycled), per precision: the registered module chain (host syncs between the stages) against graph replay of
sst_b200.fsd_engine.FSDSegEngine, one engine and 8 engines on 8 streams.  CUDA events over >= 20 frames after warm-up; the card's name
and power limit are read in the same run.  Prints one JSON document.

    python tools/fsd_front_bench.py [--frames 40] [--out profiles/r03_fsd_front.json]"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sst_b200 import flagship as fl  # noqa: E402
from sst_b200.fsd_engine import FSDSegEngine, module_front  # noqa: E402
from sst_b200.spconv_modules import set_spconv_precision  # noqa: E402

P, SWEEPS, STREAMS = 150000, 4, 8


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clk = ([s.strip() for s in q.stdout.strip().split(",")] + ["?", "?", "?"])[:3] if q.returncode == 0 else ("?", "?", "?")
    return dict(name=torch.cuda.get_device_name(0), nvidia_smi_name=name, power_limit=power, max_sm_clock=clk)


def events(fn, frames):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    fn(frames)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=40)
    ap.add_argument("--precisions", default="bf16,fp32_tc,fp32")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert args.frames >= 20
    dev = torch.device("cuda:0")
    sweeps = [fl.synth_frame(100 + i, P, extra_dims=2).to(dev) for i in range(SWEEPS)]
    offs = torch.tensor([0, P], dtype=torch.int32, device=dev)
    vfe, unet, neck = fl.build_fsd_front(seed=0)
    vfe, unet = vfe.to(dev), unet.to(dev)
    rec = dict(workload="FSD segmentation front, configs/fsd: voxel (0.25, 0.25, 0.2), range [-80,-80,-2,80,80,4], DynamicScatterVFE(5->[64,64]), "
                        "SimpleSparseUNet flagship.FSD_UNET, Voxel2PointScatterNeck; 150k-point sweeps (synth_frame extra_dims=2, 4 cycled), batch 1",
               frames=args.frames, card=card(), results={})
    for prec in args.precisions.split(","):
        vfe.precision = "bf16" if prec == "bf16" else "fp32"
        set_spconv_precision(unet, prec)

        def modules(n):
            with torch.no_grad():
                for i in range(n):
                    module_front(vfe, unet, neck, [sweeps[i % SWEEPS]], fl.FSD_SEG_VOXEL_SIZE, fl.FSD_PC_RANGE)

        engines = [FSDSegEngine(fl.FSD_SEG_VOXEL_SIZE, fl.FSD_PC_RANGE, vfe, unet, neck, max_points=P, batch_size=1, precision=prec, device=dev)
                   for _ in range(STREAMS)]
        for e in engines:
            e.load_frames_device(sweeps[0], offs)

        def one(n):
            e = engines[0]
            for i in range(n):
                e.load_frames_device(sweeps[i % SWEEPS], offs)
                e.run()
            torch.cuda.current_stream().wait_stream(e.stream)

        def many(n):
            for i in range(n):
                for j, e in enumerate(engines):
                    e.load_frames_device(sweeps[(i + j) % SWEEPS], offs)
                    e.run()
            for e in engines:
                torch.cuda.current_stream().wait_stream(e.stream)

        # same result: the engine against the module chain on one sweep (bit-identical expected)
        ref = None
        with torch.no_grad():
            ref = module_front(vfe, unet, neck, [sweeps[1]], fl.FSD_SEG_VOXEL_SIZE, fl.FSD_PC_RANGE)
        engines[0].load_frames_device(sweeps[1], offs)
        got = engines[0].run()
        torch.cuda.synchronize()
        K, M = int(got["num_pts"].item()), int(got["num_voxels"].item())
        identical = (K == ref[0].shape[0] and M == ref[2].shape[0] and torch.equal(got["pts_feats"][:K], ref[0])
                     and torch.equal(got["voxel_feats"][:M], ref[2]) and torch.equal(got["pts_mask"][:P], ref[1]))
        for fn in (modules, one, many):   # warm-up
            fn(3)
        # alternate the three arms twice; report the faster pass of each (shared host: other people's work)
        t = {"modules": [], "engine_1": [], "engine_8": []}
        for _ in range(2):
            t["modules"].append(events(modules, args.frames) / args.frames)
            t["engine_1"].append(events(one, args.frames) / args.frames)
            t["engine_8"].append(events(many, args.frames) / (args.frames * STREAMS))
        e = engines[0]
        rec["results"][prec] = dict(
            voxels=M, kept_points=K, identical_to_modules=bool(identical),
            modules_ms_per_frame=min(t["modules"]), engine_ms_per_frame=min(t["engine_1"]),
            engine_8_streams_ms_per_frame=min(t["engine_8"]), passes_ms=t,
            speedup_1=min(t["modules"]) / min(t["engine_1"]), speedup_8=min(t["modules"]) / min(t["engine_8"]),
            launches_per_frame=e.launches_per_frame, other_nodes_per_frame=e.other_nodes_per_frame,
            buffer_bytes_per_engine=e.buffer_bytes)
        print(f"[{prec}] modules {min(t['modules']):.3f} ms  engine {min(t['engine_1']):.3f} ms  8 engines {min(t['engine_8']):.3f} ms/frame  "
              f"identical={identical}  launches {e.launches_per_frame}", file=sys.stderr)
        del engines
        torch.cuda.empty_cache()
    js = json.dumps(rec, indent=1)
    print(js)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(js + "\n")


if __name__ == "__main__":
    main()
