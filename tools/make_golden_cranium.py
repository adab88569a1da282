"""Generate tests/golden/cranium_crop.npz and tests/golden/cranium_sample.npz from the
sample project samples/Cranium.inv3 of the InVesalius 3 sources:

    python tools/make_golden_cranium.py <path to Cranium.inv3>

The .inv3 format is a tar of main.plist + matrix.dat + mask_N.dat/.plist
(invesalius/project.py:378-470, invesalius/data/mask.py:315-366). We keep a crop of the
int16 matrix plus the two shipped, reference-produced threshold masks (bit-packed), and
whole-volume voxel counts. The whole matrix (14 MB) is too large to store; the sample file
keeps it on a lattice plus every voxel that sits on a bound of either threshold range.
"""
import io
import plistlib
import sys
import tarfile
from pathlib import Path

import numpy as np

GOLDEN = Path(__file__).resolve().parents[1] / "tests" / "golden"
DST = GOLDEN / "cranium_crop.npz"
DST_SAMPLE = GOLDEN / "cranium_sample.npz"
CROP = (slice(30, 78), slice(64, 192), slice(64, 192))  # z, y, x
LATTICE = (2, 4, 4)  # z, y, x strides of the whole-volume sample; CROP's starts lie on it


def load_inv3(path):
    with tarfile.open(path, "r:*") as tf:
        files = {Path(m.name).name: tf.extractfile(m).read() for m in tf.getmembers() if m.isfile()}
    main = plistlib.loads(files["main.plist"])
    shape = tuple(main["matrix"]["shape"])
    matrix = np.frombuffer(files[main["matrix"]["filename"]], dtype=main["matrix"]["dtype"]).reshape(shape)
    masks = []
    for key in sorted(main["masks"], key=int):
        mp = plistlib.loads(files[main["masks"][key]])
        mshape = tuple(mp["mask_shape"])
        m = np.frombuffer(files[mp["mask_file"]], dtype=np.uint8).reshape(mshape)
        masks.append((tuple(mp["threshold_range"]), m))
    return main, matrix, masks


def write_sample(matrix, masks):
    """The matrix on the LATTICE, and the flat indices and values of every voxel equal to a
    bound of a threshold range or one past it (where an off-by-one would show)."""
    lattice = np.ascontiguousarray(matrix[tuple(slice(None, None, s) for s in LATTICE)])
    edge = np.zeros(matrix.shape, bool)
    for (lo, hi), _ in masks:
        for v in (lo - 1, lo, hi, hi + 1):
            edge |= matrix == v
    idx = np.flatnonzero(edge)
    np.savez_compressed(DST_SAMPLE, lattice=lattice, lattice_step=np.array(LATTICE), bound_index=idx.astype(np.int64),
                        bound_value=matrix.reshape(-1)[idx])
    print(DST_SAMPLE, DST_SAMPLE.stat().st_size, lattice.shape, idx.size)


def main(src):
    meta, matrix, masks = load_inv3(src)
    out = {"matrix_crop": np.ascontiguousarray(matrix[CROP]), "crop": np.array([[s.start, s.stop] for s in CROP]),
           "full_shape": np.array(matrix.shape), "spacing": np.array(meta["spacing"], dtype=np.float64)}
    for i, (thr, m) in enumerate(masks):
        body = m[1:, 1:, 1:]
        assert set(np.unique(body)) <= {0, 255}
        out[f"thr_{i}"] = np.array(thr, dtype=np.int64)
        out[f"mask_{i}_crop_bits"] = np.packbits(body[CROP] == 255)
        out[f"mask_{i}_count_full"] = np.array(int((body == 255).sum()))
        # per-slice counts pin the whole volume without shipping it
        out[f"mask_{i}_slice_counts"] = (body == 255).sum(axis=(1, 2)).astype(np.int64)
    out["matrix_slice_sums"] = matrix.astype(np.int64).sum(axis=(1, 2))
    # the two WHOLE reference masks, bit-packed (the marching-cubes envelope check contours them), and
    # what the reference recorded for the surfaces it built from them (surface_N.plist: volume in mm^3
    # of the smoothed / decimated mesh shipped in the project — an envelope, not a golden mesh)
    with tarfile.open(src, "r:*") as tf:
        files = {Path(m.name).name: tf.extractfile(m).read() for m in tf.getmembers() if m.isfile()}
    for i, (thr, m) in enumerate(masks):
        out[f"mask_{i}_bits_full"] = np.packbits(m[1:, 1:, 1:] == 255)
        out[f"surface_{i}_volume_mm3"] = np.array(float(plistlib.loads(files[f"surface_{i}.plist"])["volume"]))
    np.savez_compressed(DST, **out)
    print(DST, DST.stat().st_size, {k: v.shape for k, v in out.items()})
    write_sample(matrix, masks)


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    sys.exit(main(Path(sys.argv[1])))
