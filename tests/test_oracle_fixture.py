"""The oracle is pinned by the reference's only known-answer material: the bag fixture
traversability_estimation/maps/elevation_map.bag (SURVEY.md Appendix B), decoded into tests/golden/."""
import zlib

import numpy as np


def _geo(ob, m):
    return ob.Geometry(m["rows"], m["cols"], m["resolution"], m["length_x"], m["length_y"], *m["position"])


def test_golden_manifest_matches_arrays(fixture_map):
    m, d = fixture_map
    for k, crc in m["crc32"].items():
        raw = np.ascontiguousarray(d[k].T).tobytes()
        assert f"{zlib.crc32(raw):08x}" == crc, k
    assert d["elevation"].shape == (100, 133)
    # spot values, SURVEY.md B.2
    assert d["traversability_slope"][0, 0] == np.float32(0.9074399471282959)
    assert d["traversability_step"][50, 66] == np.float32(0.3709149956703186)
    assert d["traversability"][37, 101] == np.float32(0.9801885485649109)


def test_chain_bit_exact_on_fixture(oracle, fixture_map):
    m, d = fixture_map
    g = _geo(oracle, m)
    o = oracle.chain(g, oracle.ChainParams.yaml_defaults(0), d["elevation"])
    for k, ref in (("slope", "traversability_slope"), ("step", "traversability_step"),
                   ("roughness", "traversability_roughness"), ("traversability", "traversability")):
        assert np.array_equal(o[k].view(np.uint32), d[ref].view(np.uint32)), k


def test_raw_moment_normals_differ_only_on_planar_edge_windows(oracle, fixture_map):
    m, d = fixture_map
    g = _geo(oracle, m)
    o = oracle.chain(g, oracle.ChainParams.yaml_defaults(1), d["elevation"])
    bad = np.argwhere(o["slope"].view(np.uint32) != d["traversability_slope"].view(np.uint32))
    assert sorted(map(tuple, bad.tolist())) == [(99, 117), (99, 118)]
    assert np.array_equal(o["step"].view(np.uint32), d["traversability_step"].view(np.uint32))


def test_single_filters_compose_to_chain(oracle, fixture_map):
    m, d = fixture_map
    g = _geo(oracle, m)
    p = oracle.ChainParams.yaml_defaults(0)
    nx, ny, nz = oracle.normals(g, p, d["elevation"])
    s = oracle.slope(g, p.slope_critical, nz)
    t = oracle.step(g, p, d["elevation"])
    r = oracle.roughness(g, p, d["elevation"], nx, ny, nz)
    f = oracle.fuse(p.fuse_weight, s, t, r)
    assert np.array_equal(f.view(np.uint32), d["traversability"].view(np.uint32))
    assert np.all(nz >= 0)
    nrm = nx.astype(np.float64) ** 2 + ny.astype(np.float64) ** 2 + nz.astype(np.float64) ** 2
    assert np.allclose(nrm, 1.0, atol=1e-6)


def test_golden_vectors_can_be_regenerated_from_the_reference_bag(fixture_map, tmp_path):
    """tests/golden/ equals a fresh decode of the reference's bag, which is stored beside it xz-compressed
    (elevation_map.bag.xz; its sha256 is the manifest's)."""
    import hashlib
    import lzma
    import os
    from bag import read_gridmap_bag
    m, d = fixture_map
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "elevation_map.bag.xz"), "rb") as f:
        raw = lzma.decompress(f.read())
    assert hashlib.sha256(raw).hexdigest() == m["sha256"]
    bag = tmp_path / "elevation_map.bag"
    bag.write_bytes(raw)
    msg = read_gridmap_bag(str(bag))
    assert (msg.rows, msg.cols, msg.resolution) == (m["rows"], m["cols"], m["resolution"])
    assert msg.outer_start_index == 0 and msg.inner_start_index == 0
    for k, v in d.items():
        assert np.array_equal(msg.data[k].view(np.uint32), v.view(np.uint32)), k
