"""Oracle: the generators' dataset shell -- x0 sampling, noisy/clean rows, CSV (fp64, pandas) -- and
the consumer's loader.

Test infrastructure -- see ``oracle/__init__.py``.  Restates generation_type2.py:162-220,309-322
and generation_type1.py:139-158,260-339 (x0 ranges, clean/noisy DataFrames, CSV schema
``t,X,Y,[phi],vx,vy,omega,d,delta,trajectory_id``; last row's d,delta = NaN -> empty field), and
KalmanNet/data_loader.py:5-109 (CSV pair -> shuffled float32 tensors).
The sensor noise values come from ``oracle/philox.py`` (the B200 path's Philox stream) or, for
pinning the shell itself against the reference, from NumPy PCG64 exactly as the reference does.
"""
import numpy as np
import pandas as pd

from . import philox

CLEAN_COLS = ["t", "X", "Y", "phi", "vx", "vy", "omega", "d", "delta", "trajectory_id"]
NOISY_COLS = ["t", "X", "Y", "vx", "vy", "omega", "d", "delta", "trajectory_id"]

# generation_type1.py:260-265 / generation_type2.py:171-174
X0_RANGES_TYPE1 = ((-2.0, 2.0), (-2.0, 2.0), (-np.pi, np.pi), (0.4, 1.5), (-0.05, 0.05), (-1.0, 1.0))
X0_RANGES_TYPE2 = ((-2.0, 2.0), (-2.0, 2.0), (-np.pi, np.pi), (0.2, 0.6), (-0.05, 0.05), (-1.0, 1.0))


def sample_x0_type2(num_traj, seed=42):
    """x0[i] = six successive rng.uniform draws of default_rng(seed).  generation_type2.py:164,171-174
    (that generator is used for nothing else, so the draws of trajectory i are 6i..6i+5)."""
    rng = np.random.default_rng(seed)
    out = np.zeros((num_traj, 6))
    for i in range(num_traj):
        for j, (lo, hi) in enumerate(X0_RANGES_TYPE2):
            out[i, j] = rng.uniform(lo, hi)
    return out


def sample_x0_type1_first(seed=42):
    """x0 of trajectory 0 of generation_type1.py (legacy global RNG seeded at :17; later
    trajectories interleave with the open-loop control synthesis draws :280-285)."""
    rs = np.random.RandomState(seed)
    return np.array([rs.uniform(lo, hi) for lo, hi in X0_RANGES_TYPE1])


def pcg64_noise(traj_id, n_rows, seed_base=philox.NOISE_SEED_BASE, std=philox.NOISE_STD):
    """The reference's own noise draw (generation_type2.py:190-199): column-wise normals."""
    rng = np.random.default_rng(seed_base + traj_id)
    return np.column_stack([rng.normal(0, s, n_rows) for s in std])


def trajectory_frames(X_truth, U, traj_id, Ts, noise):
    """-> (clean DataFrame, noisy DataFrame) for one trajectory.
    generation_type2.py:202-216 / generation_type1.py:139-158,308-310."""
    n = X_truth.shape[0]
    X_meas = X_truth + noise
    t = np.arange(n) * Ts
    d = np.append(U[:, 0], np.nan)
    delta = np.append(U[:, 1], np.nan)
    frames = []
    for S in (X_truth, X_meas):
        frames.append(pd.DataFrame({
            "t": t, "X": S[:, 0], "Y": S[:, 1], "phi": S[:, 2], "vx": S[:, 3], "vy": S[:, 4],
            "omega": S[:, 5], "d": d, "delta": delta, "trajectory_id": traj_id}))
    return frames[0][CLEAN_COLS], frames[1][NOISY_COLS]


def write_csv(clean_frames, noisy_frames, clean_path, noisy_path):
    """pd.concat(..., ignore_index=True).to_csv(index=False).  generation_type2.py:218,319-322."""
    pd.concat(clean_frames, ignore_index=True).to_csv(clean_path, index=False)
    pd.concat(noisy_frames, ignore_index=True).to_csv(noisy_path, index=False)


def load_vehicle_dataset(noisy_path, clean_path, T_steps):
    """KalmanNet/data_loader.py:5-109 (load_vehicle_dataset) on a clean / noisy CSV pair -> (y[n,5,T], u[n,2,T], x[n,6,T],
    n_train): both files read with pandas' default parser (:22-23); n = number of distinct trajectory_id (:29); trajectory i =
    the group with id i (:44-47, so ids must be 0..n-1), its first T_steps rows (:51-53); y = noisy X,Y,vx,vy,omega,
    u = the noisy file's d,delta, x = clean X,Y,phi,vx,vy,omega (:14-18), float32, laid out [n, channel, T].  Trajectories
    come in the loader's shuffled order (default_rng(42), :60-62), i.e. its train, validation and test tensors concatenated;
    the first n_train = int(0.7 n) of them are the training split.  The loader's None returns on missing data
    (:24-26, :54-56) are not restated."""
    noisy, clean = pd.read_csv(noisy_path), pd.read_csv(clean_path)
    n = clean["trajectory_id"].nunique()
    gn, gc = noisy.groupby("trajectory_id"), clean.groupby("trajectory_id")
    y, u, x = [], [], []
    for i in range(n):
        a, b = gn.get_group(i).iloc[:T_steps], gc.get_group(i).iloc[:T_steps]
        y.append(a[["X", "Y", "vx", "vy", "omega"]].to_numpy().T)
        u.append(a[["d", "delta"]].to_numpy().T)
        x.append(b[["X", "Y", "phi", "vx", "vy", "omega"]].to_numpy().T)
    perm = np.arange(n)
    np.random.default_rng(42).shuffle(perm)
    return tuple(np.stack(v).astype(np.float32)[perm] for v in (y, u, x)) + (int(0.7 * n),)
