"""Generate the mesh fixtures under tests/golden/ from the reference's own test data.

Run once, with the test/ directory of a checkout of the reference (kopacja/rho2sdf.jl) as the argument:

    python tests/golden/make_fixtures.py <rho2sdf.jl checkout>/test

The tests read the committed .npz files only.
Layout follows the reference's `MeshInformations` (src/MeshGrid/MeshInformations.jl:3-12):
X is 3 x nnp (Julia column-major == numpy (nnp,3) C-order), IEN is nen x nel and is stored here
1-BASED exactly as `rho2sdf` receives it (i.e. after the unconditional `+1` of MeshInformations.jl:8
and, for the cantilever files, after the `-1` data correction of test/runtests.jl:193).
"""
import os
import sys

import numpy as np
import scipy.io as sio

OUT = os.path.dirname(os.path.abspath(__file__))


def sphere(ref):
    # sphere.mat is MAT v7.3 (HDF5); no h5py here.  Its three datasets are contiguous and
    # uncompressed (SURVEY.md section 4): X float64 1331x3 @4608, IEN int64 1000x8 @36552, rho @104648.
    raw = open(os.path.join(ref, "sphere.mat"), "rb").read()
    X = np.frombuffer(raw, dtype="<f8", count=1331 * 3, offset=4608).reshape(1331, 3).copy()
    IEN = np.frombuffer(raw, dtype="<i8", count=1000 * 8, offset=36552).reshape(1000, 8).copy()
    rho = np.frombuffer(raw, dtype="<f8", count=1000, offset=104648).copy()
    assert IEN.min() == 0 and IEN.max() == 1330
    IEN = IEN + 1  # MeshInformations.jl:8
    return X, IEN, rho


def mat5(ref, name, correction):
    d = sio.loadmat(os.path.join(ref, name + ".mat"))
    m = d["msh"][0, 0]
    X = np.ascontiguousarray(m["X"].T.astype(np.float64))          # (nnp,3)
    IEN = np.ascontiguousarray(m["IEN"].T.astype(np.int64)) + 1     # MeshInformations.jl:8
    IEN = IEN + correction                                           # runtests.jl:193 for 1-based files
    rho = d["rho"].astype(np.float64).ravel()
    assert IEN.min() == 1 and IEN.max() == X.shape[0]
    return X, IEN, rho


if __name__ == "__main__":
    ref = sys.argv[1]
    for name, (X, IEN, rho) in {
        "sphere": sphere(ref),
        "cantilever_beam_vfrac_03": mat5(ref, "cantilever_beam_vfrac_03", -1),
        "chapadlo": mat5(ref, "chapadlo", 0),
    }.items():
        np.savez_compressed(os.path.join(OUT, name + ".npz"), X=X, IEN=IEN, rho=rho)
        print(name, X.shape, IEN.shape, rho.shape, rho.mean())
