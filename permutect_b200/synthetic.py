"""Synthetic variants shaped like the reference's datasets (SURVEY.md §8d), generated in bulk with numpy.

Record layout follows datum.py:51-89: int16[16 + 2L], float16[6 + I], uint8[reads][row_bytes] (12 in the reference's
datasets: 7 bytes of 56 packed binary features, then one quantised float per byte).
"""
import numpy as np

HAP_LEN = 21
N_INFO = 71


def wgs_counts(n: int, rng) -> tuple:
    """Ingest caps applied as the reference would (plain_text_data.py:172-174): ref = min(10, Poisson(15));
    alt: 65% min(15, 1 + Geometric0(0.55)), 35% min(15, max(1, Binomial(30, 0.5)))."""
    ref = np.minimum(10, rng.poisson(15, n))
    geo = np.minimum(15, rng.geometric(0.55, n))             # numpy's geometric starts at 1 == 1 + Geometric0
    het = np.minimum(15, np.maximum(1, rng.binomial(30, 0.5, n)))
    alt = np.where(rng.random(n) < 0.65, geo, het)
    return ref.astype(np.int64), alt.astype(np.int64)


def panel_counts(n: int, rng) -> tuple:
    """High-depth panel stress (caps bypassed): ref ~ clip(N(1900,150), 0, 30000); alt 70% 1+Geometric(0.2),
    30% Binomial(2000, U(0.01, 0.5))."""
    ref = np.clip(rng.normal(1900, 150, n), 0, 30000).astype(np.int64)
    geo = rng.geometric(0.2, n)
    binom = np.maximum(1, rng.binomial(2000, rng.uniform(0.01, 0.5, n)))
    alt = np.where(rng.random(n) < 0.7, geo, binom).astype(np.int64)
    return ref, alt


def make_arrays(ref: np.ndarray, alt: np.ndarray, rng, n_info: int = N_INFO, hap_len: int = HAP_LEN, row_bytes: int = 12):
    n = len(ref)
    ia = np.zeros((n, 16 + 2 * hap_len), np.int16)
    fa = np.zeros((n, 6 + n_info), np.float16)
    ia[:, 0], ia[:, 1] = ref, alt
    u = rng.random(n)
    ia[:, 2] = np.where(u < 0.1, 2, np.where(u < 0.55, 0, 1))           # ~10% unlabeled, rest 50/50
    ia[:, 3] = np.where(rng.random(n) < 0.8, 0, rng.integers(1, 5, n))   # 80% SNV
    ref_hap = rng.integers(0, 4, (n, hap_len))
    alt_hap = ref_hap.copy()
    centre = hap_len // 2
    alt_hap[:, centre] = (ref_hap[:, centre] + rng.integers(1, 4, n)) % 4
    indel = ia[:, 3] > 0
    alt_hap[indel, centre] = 4
    ia[:, 16:16 + hap_len], ia[:, 16 + hap_len:] = ref_hap, alt_hap
    fa[:, 2:6] = np.nan
    info = np.clip(rng.standard_normal((n, n_info)), -4, 4)
    info[:, 1::2] = (rng.random((n, (n_info) // 2)) < 0.3)
    fa[:, 6:] = info.astype(np.float16)
    total = int(ref.sum() + alt.sum())
    reads = np.empty((total, row_bytes), np.uint8)
    reads[:, :7] = rng.integers(0, 256, (total, 7), dtype=np.uint8)
    reads[:, 6] &= 0xF0                                                 # 4 pad bits of the last packed byte are zero
    reads[:, 7:] = np.clip(np.rint(32 * rng.standard_normal((total, row_bytes - 7)) + 128), 0, 255).astype(np.uint8)
    return ia, fa, reads


def make_wgs_arrays(n: int, seed: int = 0):
    rng = np.random.default_rng(seed)
    ref, alt = wgs_counts(n, rng)
    return make_arrays(ref, alt, rng)


def make_panel_arrays(n: int, seed: int = 0):
    rng = np.random.default_rng(seed)
    ref, alt = panel_counts(n, rng)
    return make_arrays(ref, alt, rng)
