"""Extract the reference's golden vector into tests/golden/.

Source: the reference's traversability_estimation/maps/elevation_map.bag — its only
known-answer material (SURVEY.md Appendix B), kept xz-compressed as
tests/golden/elevation_map.bag.xz; a path to an uncompressed bag may be given instead.
The decoded layers are committed as a small .npz next to this script's output manifest
(crc32 per layer, so a reader can re-derive them from the bag and compare).

    python tools/make_golden.py [path/to/elevation_map.bag]
"""
import json
import lzma
import os
import sys
import tempfile
import zlib

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bag import read_gridmap_bag  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests", "golden")
KEEP = ["elevation", "traversability_slope", "traversability_step", "traversability_roughness",
        "traversability", "traversability_footprint", "slope_footprint", "step_footprint"]


def main():
    if len(sys.argv) > 1:
        m = read_gridmap_bag(sys.argv[1])
    else:
        with open(os.path.join(OUT, "elevation_map.bag.xz"), "rb") as f, tempfile.TemporaryDirectory() as tmp:
            bag = os.path.join(tmp, "elevation_map.bag")
            with open(bag, "wb") as g:
                g.write(lzma.decompress(f.read()))
            m = read_gridmap_bag(bag)
    os.makedirs(OUT, exist_ok=True)
    arrays = {k: m.data[k] for k in KEEP}
    np.savez_compressed(os.path.join(OUT, "fixture_gridmap.npz"), **arrays)
    manifest = {
        "source": "traversability_estimation/maps/elevation_map.bag",
        "sha256": "02cba247d0526fb9aaa84b19dffd87e31abb3e8b3bdaa11e0a50f14c18e38448",
        "frame_id": m.frame_id, "stamp": list(m.stamp),
        "resolution": m.resolution, "length_x": m.length_x, "length_y": m.length_y,
        "position": [m.pose[0], m.pose[1]],
        "rows": m.rows, "cols": m.cols,
        "outer_start_index": m.outer_start_index, "inner_start_index": m.inner_start_index,
        "layout": "column-major float32: value(i,j) = data[j*rows + i]",
        "crc32": {k: f"{zlib.crc32(np.ascontiguousarray(v.T).tobytes()):08x}" for k, v in arrays.items()},
    }
    with open(os.path.join(OUT, "fixture_gridmap.json"), "w") as f:
        json.dump(manifest, f, indent=1)
    print(json.dumps(manifest, indent=1))


if __name__ == "__main__":
    main()
