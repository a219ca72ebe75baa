"""Per-pass GPU time of the voxel sampler on the 1 M-point cloud of the bench (CUDA events).  Grids of up to
kVoxelSmemMax voxels (csrc/samplers.cu) take the shared-memory pre-aggregation path, larger ones the global one."""
import importlib, os, sys, time
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sampling = importlib.import_module("eigen-pinns_b200.sampling")
dev = torch.device("cuda", 0)
cloud = torch.from_numpy(np.random.default_rng(1234).standard_normal((1_000_000, 3))).to(dev)
lo, hi = sampling.bounds(cloud)
extent = hi - lo
for target in (256, 1024, 16384):
    base = (np.prod(extent) / (target * 2)) ** (1 / 3)
    for scale in (0.7, 1.0, 1.5):
        vs = base * scale
        dims = np.ceil(extent / vs).astype(int) + 1
        sampling.voxel_select(cloud, lo, vs, dims, max_out=target)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        cnt, _ = sampling.voxel_select(cloud, lo, vs, dims, max_out=target)
        e1.record()
        torch.cuda.synchronize()
        print("target %5d scale %.2f n_vox %7d count %6d: gpu %.3f ms wall %.3f ms" % (
            target, scale, int(np.prod(dims)), cnt, e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3))
t0 = time.perf_counter()
sampling.voxel_levels(cloud, [256, 512, 1024])
print("hierarchy [256, 512, 1024]: %.2f ms wall" % ((time.perf_counter() - t0) * 1e3))
