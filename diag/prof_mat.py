import sys, types
sys.path.insert(0, ".")
import torch
import bench, pertrenderer_b200 as pb
dev = torch.device("cuda", 0)
fr, _ = bench.rasterised_fragments(types.SimpleNamespace(views=8, image_size=256, faces_per_pixel=50), dev)
atlas = torch.rand((10240, 4, 4, 3), device=dev, requires_grad=True)
g = torch.randn(fr.pix_to_face.shape + (3,), device=dev)
def step():
    t = pb.AtlasTexels(atlas).materialize(fr.pix_to_face, fr.bary_coords)
    t.backward(g)
step(); torch.cuda.synchronize()
from torch.profiler import profile, ProfilerActivity
with profile(activities=[ProfilerActivity.CUDA]) as p:
    step(); torch.cuda.synchronize()
print(p.key_averages().table(sort_by="cuda_time_total", row_limit=8), flush=True)
