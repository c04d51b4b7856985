"""MetaImage IO of the import shim (CPU part) and our own CLIs against the oracle on the GPU."""
import os
import subprocess
import sys

import numpy
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COMPAT = os.path.join(ROOT, "medpy_b200", "compat")


def _write_case(tmp_path, shape=(12, 10, 9), ext=".mha"):
    sys.path.insert(0, COMPAT)
    try:
        from medpy.io import save, Header
    finally:
        sys.path.remove(COMPAT)
    from medpy_b200 import synthetic
    vol = synthetic.two_blob_volume(shape, seed=2, with_prob=False)
    # MedPy's convention: arrays are x,y,z -> transpose our z,y,x volume
    img_xyz = numpy.ascontiguousarray(vol["image"]).T
    markers = (vol["fg"].astype(numpy.uint8) + 2 * vol["bg"].astype(numpy.uint8)).T
    hdr = Header(spacing=(1.0, 1.0, 2.0), offset=(0.0, 0.0, 0.0))
    ip, mp = str(tmp_path / ("img" + ext)), str(tmp_path / ("markers" + ext))
    save(img_xyz, ip, hdr, True)
    save(markers, mp, hdr, True)
    return vol, ip, mp


def test_metaimage_roundtrip_and_xyz_order(tmp_path):
    sys.path.insert(0, COMPAT)
    try:
        import importlib
        import medpy.io as mio
        importlib.reload(mio)
        a = numpy.arange(2 * 3 * 4, dtype=numpy.float32).reshape(2, 3, 4)  # x, y, z
        p = str(tmp_path / "a.mha")
        mio.save(a, p, mio.Header(spacing=(1, 2, 3), offset=(0, 0, 0)), True)
        b, hdr = mio.load(p)
        assert b.shape == (2, 3, 4) and numpy.array_equal(a, b)
        assert not b.flags.c_contiguous and b.flags.f_contiguous      # transposed view, like the reference's load()
        assert mio.header.get_voxel_spacing(hdr) == (1.0, 2.0, 3.0)
        with pytest.warns(DeprecationWarning):
            assert mio.header.get_pixel_spacing(hdr) == (1.0, 2.0, 3.0)
    finally:
        sys.path.remove(COMPAT)
        for k in [k for k in sys.modules if k == "medpy" or k.startswith("medpy.")]:
            del sys.modules[k]


@pytest.mark.gpu
@pytest.mark.parametrize("ext", [".mha", ".nii.gz"])
def test_own_cli_matches_oracle(tmp_path, ext):
    from oracle import energy_terms as et, solvers
    vol, ip, mp = _write_case(tmp_path, shape=(20, 16, 18), ext=ext)
    out = str(tmp_path / ("out" + ext))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "medpy_b200", "cli", "graphcut_voxel.py"), "15.0", ip, mp, out,
                        "--boundary", "diff_exp", "-s", "-f"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    sys.path.insert(0, COMPAT)
    try:
        from medpy.io import load
        mask_xyz, _ = load(out)
    finally:
        sys.path.remove(COMPAT)
    # spacing (1,1,2) is in x,y,z order = the CLI's array order; our volume is z,y,x -> reversed
    prob = et.build_problem(vol["fg"], vol["bg"], boundary=("difference_exponential", vol["image"], 15.0, (2.0, 1.0, 1.0)))
    oflow, omask, _ = solvers.solve_port(prob)
    assert numpy.array_equal(mask_xyz.T.astype(numpy.uint8), omask)


def _write_label_case(tmp_path, shape=(12, 10, 9)):
    sys.path.insert(0, COMPAT)
    try:
        from medpy.io import save, Header
    finally:
        sys.path.remove(COMPAT)
    from medpy_b200 import synthetic
    vol = synthetic.two_blob_volume(shape, seed=5, with_prob=False)
    grids = numpy.meshgrid(*[numpy.arange(s) for s in shape], indexing="ij")
    regions = sum((g // 3) * m for g, m in zip(grids, (100, 10, 1))) + 7          # arbitrary ids: the CLI relabels
    grad = numpy.sqrt(sum(d ** 2 for d in numpy.gradient(vol["image"].astype(numpy.float64)))).astype(numpy.float32)
    markers = (vol["fg"].astype(numpy.uint8) + 2 * vol["bg"].astype(numpy.uint8))
    hdr = Header(spacing=(1.0, 1.0, 1.0), offset=(0.0, 0.0, 0.0))
    paths = {}
    for name, arr in (("grad", grad), ("regions", regions.astype(numpy.int32)), ("markers", markers)):
        paths[name] = str(tmp_path / (name + ".mha"))
        save(numpy.ascontiguousarray(arr).T, paths[name], hdr, True)
    return vol, regions, grad, paths


@pytest.mark.gpu
def test_own_label_cli_matches_oracle(tmp_path):
    from oracle import energy_label_terms as elt, solvers
    vol, regions, grad, paths = _write_label_case(tmp_path, shape=(18, 15, 12))
    out = str(tmp_path / "out.mha")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "medpy_b200", "cli", "graphcut_label.py"), paths["grad"],
                        paths["regions"], paths["markers"], out, "-f"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    sys.path.insert(0, COMPAT)
    try:
        from medpy.io import load
        from medpy.filter import relabel
        mask_xyz, _ = load(out)
        lab_xyz = relabel(numpy.ascontiguousarray(regions.astype(numpy.int32)).T)     # what the CLI cut: x,y,z order
    finally:
        sys.path.remove(COMPAT)
    g_xyz, fg_xyz, bg_xyz = grad.T, vol["fg"].T, vol["bg"].T
    i, j, w, wr = elt.stawiaski_calls(lab_xyz, g_xyz)
    fgr, bgr = elt.marker_regions(lab_xyz, fg_xyz), elt.marker_regions(lab_xyz, bg_xyz)
    tw = [(fgr, numpy.full(fgr.size, 65535.0), numpy.zeros(fgr.size)), (bgr, numpy.zeros(bgr.size), numpy.full(bgr.size, 65535.0))]
    _, rmask, _ = solvers.solve_sparse(int(lab_xyz.max()), i, j, w, wr, tw)
    assert numpy.array_equal(numpy.asarray(mask_xyz).astype(numpy.uint8), rmask[lab_xyz - 1])

