"""Every compiled plan of the frequency-domain transforms against float64 references.

The transforms of kernels_fd.cuh are compiled per block length B = 64 .. 1024 and tile width C (complex columns per CTA): the
H-side kernels (fft_h, ifft_numH) take the C of fd_cols_h (8 at B = 1024, else 16, or 8 / 16 / 32 from CMF_FD_COLS when the
tile fits in 160 KB), the W-side kernels (fft_w, ifft_numW) that of fd_cols_w, and fft_x / ifft_resid always run C = 16.
Benchmark shapes reach only a few of these instantiations, so each (B, C, Kq) is forced here on a small shape and checked
through the contractions that use its transforms:
  - the direct loss: fft_w (the TC_FQX operand), fft_h (full blocks) and ifft_resid;
  - numW: fft_x, fft_h (owned columns) and ifft_numW<float>;
  - the Gram partial: fft_h (full blocks) and ifft_numW<double>;
  - numH: fft_w and ifft_numH;
  - denomH: fft_w on the lag table, fft_h at hop B - 2L + 2 and ifft_numH.
K = 7 (Kq = 64) takes the unpaired load / store paths of odd K; K = 72 fills Kq = 128.  N = 72 leaves a partial tile.
"""
import pytest

from tests.test_gpu_engine_plans import _check_contractions, case_data, cmf, fd_plan, refs  # noqa: F401  (fixtures)

gpu = pytest.mark.gpu

N, T, L = 72, 2500, 12
BLOCKS = [64, 128, 256, 512, 1024]
KS = {64: 7, 128: 72}


def cols_h_accepted(B, c):
    """fd_cols_h: CMF_FD_COLS = c is taken when c is 8, 16 or 32 and the B x c tile fits in 160 KB."""
    return c in (8, 16, 32) and B * c * 8 <= 160 * 1024


PLANS = [(B, c, kq) for B in BLOCKS for c in (8, 16, 32) if cols_h_accepted(B, c) for kq in (64, 128)]


def test_plans_cover_every_instantiation():
    # every (B, C) the host can launch an H-side transform with, at both Kq; the W side and fft_x / ifft_resid ride along
    assert {(B, c) for B, c, _ in PLANS} == {(B, c) for B in BLOCKS for c in (8, 16, 32) if (B, c) != (1024, 32)}
    assert {kq for _, _, kq in PLANS} == {64, 128}
    for B in BLOCKS:
        for K in KS.values():
            p = fd_plan(N, T, K, L, B)
            assert p["forced"] and p["B"] == B
    assert fd_plan(N, T, KS[64], L)["Kq"] == 64 and fd_plan(N, T, KS[128], L)["Kq"] == 128


@gpu
@pytest.mark.parametrize("plan", PLANS, ids=lambda p: f"B{p[0]}-C{p[1]}-Kq{p[2]}")
def test_fd_transforms_at_every_plan(cmf, refs, plan, monkeypatch):
    B, c, kq = plan
    monkeypatch.setenv("CMF_FD_B", str(B))
    monkeypatch.setenv("CMF_FD_COLS", str(c))
    dims = (N, T, KS[kq], L)
    p = fd_plan(*dims, B)
    s = cmf.DeviceShard(N, T, 0, T, KS[kq], L, dtype="f32", device=0)
    try:
        s.set_engine(2)
        assert s.get_engine() == 2
        assert s.fd_layout() == (p["B"], p["V"], p["nblkp"])

        def again():
            """numW on a second run"""

        _check_contractions(s, refs(dims), dims, [again])
    finally:
        s.close()
