"""Byte-for-byte comparison of two `bench.py --dump-outputs DIR` directories (the same config, steps and warmup run with
two library builds, e.g. the second through NMPC_B200_LIB): python tools/compare_dumps.py DIR_A DIR_B
Prints one line per array and exits non-zero unless both directories hold the same files with identical bytes."""
import sys
from pathlib import Path
import numpy as np

a_dir, b_dir = Path(sys.argv[1]), Path(sys.argv[2])
names = sorted({p.name for p in a_dir.glob("*.npy")} | {p.name for p in b_dir.glob("*.npy")})
ok = bool(names)
for name in names:
    pa, pb = a_dir / name, b_dir / name
    if not (pa.exists() and pb.exists()):
        print(f"{name}: only in {a_dir if pa.exists() else b_dir}"); ok = False; continue
    if pa.read_bytes() == pb.read_bytes():
        print(f"{name}: identical ({pa.stat().st_size} bytes)"); continue
    ok = False
    a, b = np.load(pa), np.load(pb)
    if a.shape != b.shape:
        print(f"{name}: DIFFERENT shapes {a.shape} vs {b.shape}"); continue
    rows = np.unique(np.nonzero(a.view(np.uint64) != b.view(np.uint64))[0]) if a.dtype == np.float64 else []
    diff = np.abs(a - b)
    print(f"{name}: DIFFERENT in {len(rows)} of {len(a)} rows, max |a - b| {np.nanmax(diff) if diff.size else 0.0:.3e}")
print("identical" if ok else "DIFFERENT")
sys.exit(0 if ok else 1)
