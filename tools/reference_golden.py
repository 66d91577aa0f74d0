#!/usr/bin/env python3
"""Freeze the data tables and literals of rs_pbrt that the restatements depend on into tests/golden/reference_tables.npz.

    python tools/reference_golden.py <rs_pbrt checkout> [out.npz]

tests/test_reference_tables.py holds data/sobol_tables.bin, the oracle's prime tables and the constants of the oracle and
the kernels against this file, so the suite runs without the rs_pbrt sources.  What is stored:
  sobol_sha256        SHA-256 of the blob tools/extract_sobol_tables.py makes from src/core/sobolmatrices.rs (all three tables)
  sobol32_index/value a fixed, seeded sample of 2048 entries of SOBOL_MATRICES_32 (locates a mismatch the digest only reports)
  vdc, vdc_inv        VD_C_SOBOL_MATRICES(_INV) as the blob stores them (u64, rows zero padded to 52)
  primes, prime_sums  PRIMES / PRIME_SUMS of src/core/lowdiscrepancy.rs
  shadow_epsilon, inv_2_pi, pcg32 (default state, stream, multiplier), k_max_resolution, rng_threshold_op
                      literals of src/core/pbrt.rs, src/core/rng.rs, src/samplers/halton.rs
Re-run only against a new rs_pbrt revision.
"""
import hashlib
import re
import subprocess
import sys
import tempfile
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
N_SAMPLE = 2048


def literal(text, pattern):
    m = re.search(pattern, text)
    if m is None:
        raise SystemExit("not found: %s" % pattern)
    return m.group(1).replace("_", "")


def rust_array(text, name):
    i = text.index("pub const %s:" % name)
    j = text.index("[", text.index("=", i))
    k = text.index("];", j)
    return [int(t.replace("_", "")) for t in re.findall(r"[\d_]+", text[j + 1:k]) if t.strip("_")]


def main():
    if len(sys.argv) < 2:
        raise SystemExit(__doc__)
    ref = Path(sys.argv[1]) / "src"
    out = Path(sys.argv[2]) if len(sys.argv) > 2 else ROOT / "tests" / "golden" / "reference_tables.npz"
    with tempfile.TemporaryDirectory() as tmp:
        blob_path = Path(tmp) / "sobol.bin"
        subprocess.run([sys.executable, str(ROOT / "tools" / "extract_sobol_tables.py"), str(ref / "core" / "sobolmatrices.rs"), str(blob_path)],
                       check=True, capture_output=True)
        blob = blob_path.read_bytes()
    hdr = np.frombuffer(blob, "<u4", 8)
    n_dims, size, n_vdc, n_vdc_inv = (int(x) for x in hdr[1:5])
    sobol32 = np.frombuffer(blob, "<u4", n_dims * size, 32)
    off = 32 + 4 * n_dims * size
    vdc = np.frombuffer(blob, "<u8", n_vdc * 52, off).reshape(n_vdc, 52)
    vdc_inv = np.frombuffer(blob, "<u8", n_vdc_inv * 52, off + 8 * n_vdc * 52).reshape(n_vdc_inv, 52)
    idx = np.sort(np.random.default_rng(20240).choice(sobol32.size, N_SAMPLE, replace=False)).astype(np.int64)

    low = (ref / "core" / "lowdiscrepancy.rs").read_text()
    primes, sums = rust_array(low, "PRIMES"), rust_array(low, "PRIME_SUMS")
    assert len(primes) == len(sums) == 1000
    pbrt = (ref / "core" / "pbrt.rs").read_text()
    rng = (ref / "core" / "rng.rs").read_text()
    halton = (ref / "samplers" / "halton.rs").read_text()
    op = literal(rng, r"let threshold = \(!b \+ 1\) (\S) b;")
    np.savez_compressed(
        out, sobol_sha256=np.str_(hashlib.sha256(blob).hexdigest()), sobol32_index=idx, sobol32_value=sobol32[idx], vdc=vdc, vdc_inv=vdc_inv,
        primes=np.array(primes, np.uint32), prime_sums=np.array(sums, np.uint32),
        shadow_epsilon=np.float32(literal(pbrt, r"pub const SHADOW_EPSILON: Float = ([\d._]+);")),
        inv_2_pi=np.float32(literal(pbrt, r"pub const INV_2_PI: Float = ([\d._]+);")),
        pcg32=np.array([int(literal(rng, r"pub const PCG32_%s: u64 = (0x[0-9a-f_]+);" % n), 16) for n in ("DEFAULT_STATE", "DEFAULT_STREAM", "MULT")], np.uint64),
        k_max_resolution=np.int32(literal(halton, r"pub const K_MAX_RESOLUTION: i32 = ([\d_]+)_i32;")),
        rng_threshold_op=np.str_(op))
    print("wrote", out)


if __name__ == "__main__":
    main()
