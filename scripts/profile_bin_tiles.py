"""GPU timing of the tile binning (csrc/splat_bin_tiles.cu) at the bench shape: build the 300k-Gaussian / 1024x667 bench
scene, project it, then time gb_bin_tiles_pack through the C ABI under each ordering (GOLIATH_B200_BINSORT=tile|rank),
L2 flushed before every call as the bench does:
  - the whole call replayed from a CUDA graph, CUDA events around each replay (no host launch gaps);
  - per kernel, device times from torch.profiler (CUDA activity records) over eager calls.
Usage: python scripts/profile_bin_tiles.py [reps] [out.json]"""
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench
from goliath_b200 import _lib, synthetic
from goliath_b200.gsplat import project_gaussians

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 20
out_path = sys.argv[2] if len(sys.argv) > 2 else None
dev = torch.device("cuda:0")
H, W, BW = bench.H, bench.W, bench.BW
u = bench.unpack(bench.packed_scene(300_000).to(dev))
c = synthetic.ring_camera(0, img_h=H, img_w=W)
xys, depths, radii, conics, comp, nth, cov3d = project_gaussians(
    u["primpos"].contiguous(), u["primscale"].contiguous(), 1.0, u["primqvec"].contiguous(), c["viewmat"].to(dev),
    c["fx"], c["fy"], c["cx"], c["cy"], H, W, BW, 0.1)
G = xys.shape[0]
T = ((W + BW - 1) // BW) * ((H + BW - 1) // BW)
cap = 8 * G
L = _lib.lib()
col3, op1 = u["diff_color"].contiguous(), u["opacity"].contiguous()
ws = torch.empty(L.gb_bin_tiles_workspace_bytes(G, T, cap), dtype=torch.uint8, device=dev)
bins = torch.empty(T, 2, dtype=torch.int32, device=dev)
order = torch.empty(T, dtype=torch.int32, device=dev)
gids = torch.empty(cap, dtype=torch.int32, device=dev)
rec = torch.empty(cap, 12, device=dev)
n_out = torch.zeros(1, dtype=torch.int32, device=dev)
ovf = torch.zeros(1, dtype=torch.int32, device=dev)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)


def call():
    _lib.check(L.gb_bin_tiles_pack(G, xys.data_ptr(), depths.data_ptr(), radii.data_ptr(), conics.data_ptr(),
                                   col3.data_ptr(), op1.data_ptr(), comp.data_ptr(), H, W, BW, cap, bins.data_ptr(),
                                   order.data_ptr(), 0, gids.data_ptr(), rec.data_ptr(), n_out.data_ptr(), ovf.data_ptr(),
                                   ws.data_ptr(), _lib.stream_ptr(dev)), "bin_tiles_pack")


def graph_time():
    for _ in range(3):
        flush.fill_(1)
        call()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        call()
    torch.cuda.current_stream().wait_stream(side)
    with torch.cuda.graph(g):
        call()
    ts = []
    for _ in range(reps):
        flush.fill_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        g.replay()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b) * 1e3)
    return ts


def kernel_times():
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            flush.fill_(1)
            call()
        torch.cuda.synchronize()
    per = {}
    for e in prof.key_averages():
        dt = getattr(e, "self_device_time_total", None)
        if dt is None:
            dt = getattr(e, "self_cuda_time_total", 0)
        if dt <= 0 or "elementwise" in e.key:  # host-side rows, and the L2 flush fill
            continue
        name = e.key.replace("(anonymous namespace)::", "").split("(")[0]
        per[name] = per.get(name, 0.0) + dt / reps
    return dict(sorted(per.items(), key=lambda kv: -kv[1]))


props = torch.cuda.get_device_properties(dev)
result = {"gpu": props.name, "G": G, "T": T, "reps": reps, "modes": {}}
try:
    import subprocess

    result["power_limit"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                                           capture_output=True, text=True).stdout.strip()
except Exception:
    pass
before = L.gb_get_bin_sort_mode()
ref = None
for name, mode in (("rank", 1), ("tile", 0), ("rank", 1), ("tile", 0)):
    L.gb_set_bin_sort_mode(mode)
    ts = graph_time()
    ks = kernel_times()
    torch.cuda.synchronize()
    outs = (bins.clone(), gids[:int(n_out)].clone(), rec[:int(n_out)].clone())
    if ref is None:
        ref = outs
    same = all(torch.equal(a.view(torch.int32), b.view(torch.int32)) for a, b in zip(outs, ref))
    m = result["modes"].setdefault(name, {"graph_us": [], "kernels_us": [], "same_outputs_as_rank": []})
    m["graph_us"].append(sorted(ts)[len(ts) // 2])
    m["kernels_us"].append(ks)
    m["same_outputs_as_rank"].append(same)
    print("%s: whole call from a CUDA graph, median %.1f us (min %.1f); outputs identical to rank: %s"
          % (name, sorted(ts)[len(ts) // 2], min(ts), same))
    for k, v in ks.items():
        print("    %8.1f us  %s" % (v, k))
L.gb_set_bin_sort_mode(before)
if out_path:
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(result, f, indent=1)
