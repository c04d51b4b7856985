"""Device time of the fused graph build (k_build_tile) at 512^3 for several terms: separates instruction cost (exp vs the
cheap linear / division terms) from the memory side (the bytes moved are the same).  The regional cases run the lazy
build by default (cold blocks write 5 of the 79 B/voxel); the "eager" case forces the full build for comparison, and
lazy lines report the algorithmic bytes of build plus on-demand materialisation from the materialised-block count."""
import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy, torch
from medpy_b200 import synthetic
from medpy_b200.graphcut.device import graph_from_device_arrays
size = int(sys.argv[1]) if len(sys.argv) > 1 else 512
vol = synthetic.two_blob_volume((size,) * 3, seed=0)
d_img = torch.from_numpy(vol["image"]).cuda(); d_prob = torch.from_numpy(vol["prob"]).cuda()
d_fg = torch.from_numpy(vol["fg"].view(numpy.uint8)).cuda(); d_bg = torch.from_numpy(vol["bg"].view(numpy.uint8)).cuda()
n = size ** 3
CASES = [("exp+regional", dict(boundary="difference_exponential", prob=d_prob, alpha=0.1)),
         ("exp+regional, eager", dict(boundary="difference_exponential", prob=d_prob, alpha=0.1, _env={"MEDPY_GC_LAZY": "0"})),
         ("exp+regional, prob NOT loaded (dbg)", dict(boundary="difference_exponential", prob=d_prob, alpha=0.1, _env={"MEDPY_GC_BUILD_DBG": "1"})),
         ("exp+regional, plain image staging", dict(boundary="difference_exponential", prob=d_prob, alpha=0.1, _env={"MEDPY_GC_BUILD_TMA": "0"})),
         ("exp+regional, no markers", dict(boundary="difference_exponential", prob=d_prob, alpha=0.1, _nomark=True)),
         ("exp", dict(boundary="difference_exponential")),
         ("exp, no markers", dict(boundary="difference_exponential", _nomark=True))]
for name, kw in CASES + [("exp+regional (again)", dict(boundary="difference_exponential", prob=d_prob, alpha=0.1)),
                 ("exp", dict(boundary="difference_exponential")),
                 ("division+regional", dict(boundary="difference_division", prob=d_prob, alpha=0.1)),
                 ("linear", dict(boundary="difference_linear")),
                 ("max_exp+regional", dict(boundary="maximum_exponential", prob=d_prob, alpha=0.1))]:
    g = None
    best = 1e9
    env = kw.pop("_env", {})
    nomark = kw.pop("_nomark", False)
    for k in ("MEDPY_GC_BUILD_DBG", "MEDPY_GC_BUILD_TMA", "MEDPY_GC_LAZY"):
        os.environ.pop(k, None)
    os.environ.update(env)
    zeros = torch.zeros_like(d_fg)
    for rep in range(4):
        g = graph_from_device_arrays(zeros if nomark else d_fg, zeros if nomark else d_bg, image=d_img, sigma=vol["sigma"], graph=g, **kw)
        g._nat().synchronize()
        g._commit() if hasattr(g, "_commit") else None
        torch.cuda.synchronize()
        try:
            g.maxflow()
        except Exception as exc:
            pass
        best = min(best, g.stats()["ms_boundary"])
    out = {"term": name, "ms_build": round(best, 3), "GBps_alg79": round(n * 79 / best / 1e6, 1)}
    st = g.stats()
    if st["build_blocks"]:          # 8 x 8 x 32 voxels per block: 79 B/voxel where materialised, 10 R + 5 W elsewhere
        m, b = st["blocks_materialised"], st["build_blocks"]
        out.update(build_blocks=b, blocks_materialised=m, lazy_alg_GB=round((m * 79 + (b - m) * 15) * 2048 / 1e9, 2))
    print(json.dumps(out), flush=True)
