"""Generates the committed fixtures in tests/golden/ from the read-only reference tree.

Run HERE (the container that has /root/reference); the GPU box only sees the generated files.

  sphere_tables.npz    the datasets HydroChrono reads from demos/sphere/hydroData/sphere.h5
                       (src/h5fileinfo.cpp:27-91), raw/unscaled, via tests/h5lite.py
  sphere_goldens.npz   the reference's golden heave trajectories for the sphere
                       (tests/regression/reference_data/sphere/**), stored as int32 micro-metres
                       (the files print 6 decimals) + the step count; plus time / heave of
                       tests/regression/run_hydrochrono/iea_sphere/decay/expected/results.still.h5.
  yaml_reference_dumps.json.gz
                       what the reference's hydro.yaml parser (oracle/_ref/ref_yaml_dump, built by oracle/Makefile from
                       the reference tree) prints for the synthetic, block-form and fuzzed corpus of
                       tests/test_yaml_vs_reference.py.  The committed file was recorded from this repository's parser at
                       the commit where the live comparison had found it identical to the reference's on every synthetic
                       and fuzzed file, with the reference's rejection of the block-form sweeps (the known deviation).
"""
import gzip
import json
import os
import sys
import tempfile
from pathlib import Path

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from h5lite import load_bemio  # noqa: E402

REF = "/root/reference"


def tables():
    d = load_bemio(os.path.join(REF, "demos/sphere/hydroData/sphere.h5"), 1)
    b = d["bodies"][0]
    np.savez_compressed(os.path.join(HERE, "sphere_tables.npz"), rho=d["rho"], g=d["g"], water_depth=d["water_depth"],
                        w=d["w"], **{k: np.asarray(v) for k, v in b.items()})


def _traj(path, skip):
    rows = []
    with open(path) as f:
        for i, line in enumerate(f):
            if i < skip:
                continue
            p = line.split()
            if len(p) == 2:
                rows.append((float(p[0]), float(p[1])))
    a = np.array(rows)
    return a


def goldens():
    rd = os.path.join(REF, "tests/regression/reference_data/sphere")
    out = {}
    a = _traj(os.path.join(rd, "decay/hc_ref_sphere_decay.txt"), 1)
    out["decay_um"] = np.round(a[:, 1] * 1e6).astype(np.int32)
    out["decay_t0_dt"] = np.array([a[0, 0], a[1, 0] - a[0, 0]])
    for i in range(1, 11):
        a = _traj(os.path.join(rd, "reg_waves/hc_ref_sphere_reg_waves_%d.txt" % i), 5)
        out["reg%d_um" % i] = np.round(a[:, 1] * 1e6).astype(np.int32)
    a = _traj(os.path.join(rd, "irreg_waves/hc_ref_sphere_irreg_waves.txt"), 2)
    out["irreg_um"] = np.round(a[:, 1] * 1e6).astype(np.int32)
    # CLI regression golden (HHT integrator, g = 9.8, dt = 0.01): heave of body1 + time, float64
    from h5lite import H5Lite
    h = H5Lite(os.path.join(REF, "tests/regression/run_hydrochrono/iea_sphere/decay/expected/results.still.h5"))
    out["iea_decay_t"] = h.read("results/time/time")
    out["iea_decay_z"] = h.read("results/model/bodies/body1/position")[:, 2].copy()
    np.savez_compressed(os.path.join(HERE, "sphere_goldens.npz"), **out)
    for k, v in out.items():
        print(k, v.shape)


def yaml_dumps(binary=None):
    import test_yaml_vs_reference as tyr
    binary = binary or tyr.REF_BIN
    with tempfile.TemporaryDirectory() as d:
        d = Path(d)
        out = {"synthetic": {n: tyr.dump_in(binary, [f], d)[0] for n, f in tyr.synthetic_corpus(d).items()},
               "block": {n: list(tyr.dump_in(binary, [f], d)) for n, f in tyr.block_corpus(d).items()},
               "fuzz": tyr.dump_in(binary, tyr.fuzz_corpus(d), d)[0]}
    with gzip.GzipFile(os.path.join(HERE, "yaml_reference_dumps.json.gz"), "wb", mtime=0) as f:
        f.write(json.dumps(out, indent=0, sort_keys=True).encode())


if __name__ == "__main__":
    tables()
    goldens()
    yaml_dumps()
