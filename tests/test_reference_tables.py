"""The only pieces of the reference that CAN be held against it mechanically: its data tables and a few literals, frozen from
rs_pbrt's sources into tests/golden/reference_tables.npz (tools/reference_golden.py)."""
import hashlib
import re
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
GOLD = np.load(Path(__file__).resolve().parent / "golden" / "reference_tables.npz")


def test_sobol_blob_is_the_reference_tables():
    """data/sobol_tables.bin (embedded in the library, loaded by the oracle) == SOBOL_MATRICES_32 / VD_C_SOBOL_MATRICES(_INV) of
    src/core/sobolmatrices.rs as tools/extract_sobol_tables.py lays them out."""
    blob = (ROOT / "data" / "sobol_tables.bin").read_bytes()
    hdr = np.frombuffer(blob, "<u4", 8)
    assert hdr.tolist() == [0x4C424F53, 1024, 52, 25, 26, 0, 0, 0]
    sobol32 = np.frombuffer(blob, "<u4", 1024 * 52, 32)
    np.testing.assert_array_equal(sobol32[GOLD["sobol32_index"]], GOLD["sobol32_value"])
    off = 32 + 4 * sobol32.size
    np.testing.assert_array_equal(np.frombuffer(blob, "<u8", 25 * 52, off).reshape(25, 52), GOLD["vdc"])
    np.testing.assert_array_equal(np.frombuffer(blob, "<u8", 26 * 52, off + 8 * 25 * 52).reshape(26, 52), GOLD["vdc_inv"])
    assert hashlib.sha256(blob).hexdigest() == str(GOLD["sobol_sha256"])


def test_prime_tables_are_the_reference_tables(oracle):
    """PRIMES / PRIME_SUMS (src/core/lowdiscrepancy.rs:18-147) are generated, not transcribed, on our side."""
    L = oracle.load()
    assert [L.orc_prime(i) for i in range(1000)] == GOLD["primes"].tolist()
    assert [L.orc_prime_sum(i) for i in range(1000)] == GOLD["prime_sums"].tolist()


def test_constants_match_the_reference_source():
    """The literals the restatements depend on (pbrt.rs SHADOW_EPSILON / INV_2_PI, rng.rs PCG32 constants and its bounded-draw
    threshold, halton.rs K_MAX_RESOLUTION) are the ones the oracle and the kernels define."""
    o_math = (ROOT / "oracle" / "o_math.hpp").read_text()
    o_sampler = (ROOT / "oracle" / "o_sampler.hpp").read_text()
    csrc = ROOT / "rs_pbrt_b200" / "csrc"
    pb_math = (csrc / "pb_math.cuh").read_text()
    gpu = (csrc / "pbrt_gpu.cu").read_text()

    def f32(text, pattern):
        return np.float32(re.search(pattern + r"\s*=?\s*([\d.]+)f", text).group(1))

    assert f32(o_math, r"Float SHADOW_EPSILON") == GOLD["shadow_epsilon"] == f32(pb_math, r"#define PB_SHADOW_EPSILON")
    assert f32(o_math, r"Float INV_2_PI") == GOLD["inv_2_pi"] == f32(pb_math, r"#define PB_INV_2_PI")
    for v in GOLD["pcg32"].tolist():
        lit = "0x%016xULL" % v
        assert lit in o_sampler and lit in gpu, lit
    threshold = "(~b + 1u) %s b" % GOLD["rng_threshold_op"]
    assert threshold in o_sampler and threshold in gpu
    k = int(GOLD["k_max_resolution"])
    assert "K_MAX_RESOLUTION = %d;" % k in o_sampler
    assert "(px / %d) * %d" % (k, k) in (csrc / "pb_sobol.cuh").read_text()
