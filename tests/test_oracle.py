"""CPU tests: the oracle (oracle/energy_terms.py + oracle/bk_lattice.c) against the golden vectors
produced by the unmodified reference, and against the outputs of the real reference solver and graph builder
recorded on seeded random inputs (tests/golden/reference_runs_v1.npz)."""
import os
import sys

import numpy
import pytest

from conftest import golden
from oracle import energy_terms as et
from oracle import solvers

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import make_golden_reference_runs as reference_runs  # noqa: E402

NAMES = golden().names()


def _problem(c):
    boundary = None
    if c["boundary"]:
        boundary = (c["boundary"], c["image"], c["sigma"], tuple(c["spacing"]) if c["spacing"] else False)
    regional = (c["prob"], c["alpha"]) if c["prob"] is not None else None
    return et.build_problem(c["fg"], c["bg"], regional=regional, boundary=boundary)


@pytest.mark.parametrize("name", NAMES)
def test_terms_bit_exact_vs_reference(name):
    """n-link weights and net t-links equal the reference's get_edge / get_trcap bit for bit."""
    c = golden().case(name)
    with numpy.errstate(all="ignore"):
        prob = _problem(c)
    nd = len(prob["shape"])
    for d in range(nd):
        got = prob["wf"][d] if prob["wf"] is not None else numpy.zeros(prob["tr"].size)
        assert numpy.array_equal(got, c["w"][d], equal_nan=True), "axis %d weights differ" % d
    assert numpy.array_equal(prob["tr"], c["tr"])


@pytest.mark.parametrize("name", NAMES)
def test_port_flow_and_mask_vs_reference(name):
    """BK restatement: flow bit-identical, mask identical to the reference run."""
    c = golden().case(name)
    with numpy.errstate(all="ignore"):
        prob = _problem(c)
    flow, mask, _ = solvers.solve_port(prob)
    assert numpy.array_equal(mask, c["mask"].reshape(mask.shape))
    if numpy.isnan(c["flow"]):
        assert numpy.isnan(flow)
    else:
        assert flow == c["flow"], (flow.hex(), c["flow"].hex())
        if not numpy.isnan(prob["wf"][0]).any() if prob["wf"] is not None else True:
            e = et.cut_energy(prob["shape"], prob["wf"], prob["wb"], prob["tr"], prob["flow_const"], mask)
            assert abs(e - flow) <= 1e-12 * max(1.0, abs(flow))


def test_reference_known_answers():
    """The reference's own KATs survive the trip: cut.py maxflow == 3, fixtures' masks."""
    c = golden().case("ref_fixture_cut3d")
    assert c["flow"] == 3.0
    expect = numpy.asarray([[[1, 1, 1, 0, 0]] * 3] * 2, dtype=numpy.uint8)
    assert numpy.array_equal(c["mask"], expect)
    flow, mask, _ = solvers.solve_port(_problem(c))
    assert flow == 3.0 and numpy.array_equal(mask, expect)


def test_port_equals_real_reference_on_random_lattices():
    """120 random integer lattices (1-D..4-D): the restatement's flow and mask equal the reference BK's."""
    z = reference_runs.load()
    off = 0
    for k, prob in enumerate(reference_runs.random_lattices()):
        f1, m1, _ = solvers.solve_port(prob)
        m2 = z["lattice/mask"][off:off + m1.size].reshape(m1.shape)
        off += m1.size
        assert f1 == z["lattice/flow"][k] and numpy.array_equal(m1, m2), k
    assert off == z["lattice/mask"].size


def test_port_equals_real_reference_float_32cubed():
    """The bench workload's generator at 32^3 (float64 capacities): flow and mask equal the reference BK's."""
    z = reference_runs.load()
    f1, m1, _ = solvers.solve_port(reference_runs.blob32_problem())
    assert f1 == z["blob32/flow"] and numpy.array_equal(m1, z["blob32/mask"])
    assert 0 < m1.sum() < m1.size


def test_voxel_oracle_fuzzed_against_the_live_reference():
    """120 random lattices (1-D..4-D, the eight boundary terms, five image dtypes, random sigma / spacing / regional term /
    overlapping markers) through the reference's own graph_from_voxels: weights, t-links, flow and mask equal the
    restatement's bit for bit; weight <= 0 ValueErrors occur in the same cases
    (tests/golden/fuzz_voxels_against_reference.py, replayed against the reference's recorded outputs)."""
    import fuzz_voxels_against_reference as fuzz
    z = reference_runs.load()
    cases, seed = reference_runs.VOX_FUZZ
    fuzz.check(cases, seed, {k[4:]: z[k] for k in z.files if k.startswith("vox/")})
