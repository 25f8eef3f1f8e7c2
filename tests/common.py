"""Shared helpers for the test-suite (TEST INFRASTRUCTURE)."""
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")

# model constants of the reference's sphere cases
# (tests/regression/sphere/demo_sphere_decay.cpp:55-60,86-87; reg_waves/sphere_reg_waves_test.cpp:23-30,58)
SPHERE_MASS = 261.8e3
SPHERE_DT = 0.015
TASK10_AMPS = [0.177, 0.314, 0.380, 0.491, 0.706, 0.961, 1.256, 1.589, 1.962, 2.374]
TASK10_OMEGAS = [2.094395102, 1.570796327, 1.427996661, 1.256637061, 1.047197551,
                 0.897597901, 0.785398163, 0.698131701, 0.628318531, 0.571198664]
TASK10_DAMPING = [398736.034, 118149.758, 90080.857, 161048.558, 322292.419,
                  479668.979, 633979.761, 784083.286, 932117.647, 1077123.445]


def sphere_raw():
    """Raw (unscaled) sphere.h5 datasets as the dict layout of tests/h5lite.load_bemio."""
    z = np.load(os.path.join(GOLDEN, "sphere_tables.npz"))
    body = {k: z[k] for k in ("cg", "cb", "lin_matrix", "inf_added_mass", "rirf_K", "rirf_t", "exc_mag",
                              "exc_phase", "exc_irf_f", "exc_irf_t")}
    body["disp_vol"] = float(z["disp_vol"])
    return {"rho": float(z["rho"]), "g": float(z["g"]), "water_depth": float(z["water_depth"]), "w": z["w"],
            "bodies": [body]}


def asymmetric_tables(raw, seed=11):
    """Copy of raw tables whose matrices are not symmetric, so a row / column swap anywhere in a D x D path shows.
    rirf_K: an independent factor 1 + 0.4 U(-1, 1) per (row, column), so the coupling blocks between bodies are
    unrelated.  lin_matrix: every entry non-zero, off-diagonal terms small next to the diagonal (the stepping tests stay
    stable).  inf_added_mass: 15 % of each entry's diagonal scale added per (row, column), the mass matrix stays well
    conditioned.  Everything else is shared with raw."""
    rng = np.random.Generator(np.random.MT19937(seed))
    N = len(raw["bodies"])
    D = 6 * N
    fK = 1.0 + 0.4 * rng.uniform(-1.0, 1.0, size=(D, D))
    A = np.concatenate([b["inf_added_mass"] for b in raw["bodies"]])
    d = np.sqrt(np.abs(np.diag(A)))
    A = A + 0.15 * np.outer(d, d) * rng.uniform(-1.0, 1.0, size=(D, D))
    out = dict(raw, bodies=[])
    for b, body in enumerate(raw["bodies"]):
        Kh = np.asarray(body["lin_matrix"], dtype=np.float64)
        scale = max(np.abs(np.diag(Kh)).max(), 1.0)
        diag = np.where(np.diag(Kh) != 0.0, np.diag(Kh), 0.05 * scale * rng.uniform(0.5, 1.0, size=6))
        off = 0.02 * np.sqrt(np.outer(np.abs(diag), np.abs(diag))) * rng.uniform(0.2, 1.0, size=(6, 6)) \
            * rng.choice([-1.0, 1.0], size=(6, 6))
        Kh = np.where(np.eye(6, dtype=bool), np.diag(diag), Kh + off)
        nb = dict(body)
        nb["rirf_K"] = np.asarray(body["rirf_K"]) * fK[6 * b:6 * b + 6, :, None]
        nb["lin_matrix"] = Kh
        nb["inf_added_mass"] = A[6 * b:6 * b + 6].copy()
        out["bodies"].append(nb)
    return out


def transposed_tables(raw):
    """raw with every matrix transposed: K per lag, each body's lin_matrix, the D x D infinite-frequency added mass."""
    K = np.concatenate([b["rirf_K"] for b in raw["bodies"]]).transpose(1, 0, 2)
    A = np.concatenate([b["inf_added_mass"] for b in raw["bodies"]]).T
    out = dict(raw, bodies=[])
    for b, body in enumerate(raw["bodies"]):
        nb = dict(body)
        nb["rirf_K"] = np.ascontiguousarray(K[6 * b:6 * b + 6])
        nb["lin_matrix"] = np.ascontiguousarray(np.asarray(body["lin_matrix"]).T)
        nb["inf_added_mass"] = np.ascontiguousarray(A[6 * b:6 * b + 6])
        out["bodies"].append(nb)
    return out


def sphere_goldens():
    return np.load(os.path.join(GOLDEN, "sphere_goldens.npz"))


def traj_norms(sim, ref):
    """The reference's regression metric (tests/regression/utilities/compare_template.py:365-369):
    n1 = ||d||_2 / n, n2 = ||d||_inf; pass iff n1 <= 1e-4 and n2 <= 0.02."""
    d = np.asarray(sim) - np.asarray(ref)
    return np.linalg.norm(d) / d.size, np.abs(d).max()


def force_tol(ref_series, rel=1e-9, floor_frac=1e-3):
    """Per-component tolerance for force parity: rel * max(|F_ref|, floor_frac * max_t |F_ref component|).
    1e-9 relative is the north-star bar; the floor handles components crossing zero (SURVEY.md section 7)."""
    ref_series = np.asarray(ref_series)
    comp_max = np.abs(ref_series).reshape(-1, ref_series.shape[-1]).max(axis=0)
    return rel * np.maximum(np.abs(ref_series), floor_frac * comp_max)


def rms_relative_error(ref, pred):
    """Gate of the reference's CLI regression harness (tests/regression/run_hydrochrono/compare_results.py:103-107)."""
    ref, pred = np.asarray(ref), np.asarray(pred)
    ref_rms = float(np.sqrt(np.mean(np.square(ref))))
    if ref_rms == 0.0:
        return float(np.sqrt(np.mean(np.square(pred))))
    return float(np.sqrt(np.mean(np.square(pred - ref))) / ref_rms)
