"""GPU parity tests for the exact integer GRM of packed dosage matrices (tcgen05 kind::i8,
csrc/grm_i8.cu) against the NumPy oracle."""
import numpy as np
import pytest

from oracle import gwas_oracle as go, synth

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("n,p,kind", [
    (128, 128, synth.KIND_DIPLOID),      # one tile, one ring slot
    (128, 1000, synth.KIND_TETRAPLOID),  # one tile, ragged marker tail
    (300, 4097, synth.KIND_DIPLOID),     # 6 tiles, ragged rows and markers
    (129, 40000, synth.KIND_TETRAPLOID), # two accumulation slices (32768 + 7232 markers)
    (1000, 70000, synth.KIND_DIPLOID),   # 20 tiles x 3 slices = 60 work items (test_gpu_waves.py: past the first wave)
])
def test_int8_grm_matches_oracle(gbm, n, p, kind):
    A = synth.block(31, n, 0, p, kind)
    dm = gbm.DeviceMatrix.upload(A)
    pk = dm.pack()
    assert pk is not None
    Ks, _ = pk.grm(0, 2, 0)
    Ku, _ = pk.grm(0, 2, 1)
    Kp, _ = pk.grm(1, 4, 0)
    Kf, _ = dm.grm(0, 2, 0)  # Float64 DMMA path on the same data
    dm.free()
    pk.free()
    for got, want in ((Ks, go.grm_simple(A)), (Ku, go.grm_simple(A, center=False)), (Kp, go.grm_ploidy_aware(A, 4))):
        assert np.array_equal(got, got.T)
        scale = np.abs(want).max()
        assert np.max(np.abs(got - want)) < 1e-11 * scale
    assert np.max(np.abs(Ks - Kf)) < 1e-11 * np.abs(Kf).max()
    # the uncentred product of dyadic dosages is exact in both routes
    if kind in (synth.KIND_DIPLOID, synth.KIND_TETRAPLOID):
        exact = (A @ A.T) / p
        assert np.max(np.abs(Ku - exact)) <= 4 * np.finfo(float).eps * np.abs(exact).max()
