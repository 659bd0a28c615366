"""bench.py helpers that feed the JSON line (no GPU): the `roofline.traffic` lookup must read the column of the kernel
it is asked for from a committed multi-launch `ncu --set full` summary, and the per-proof operation count behind
`whole_step` must match DESIGN.md section 3.5."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_ncu_traffic_picks_the_kernels_column():
    import bench
    got, name = bench._ncu_traffic(["does_not_exist.csv", "r2f_ncu_full_msm2p20.csv"], "k_bucket_accum")
    assert name == "r2f_ncu_full_msm2p20.csv"
    assert 1.3e9 < got < 1.6e9            # 1.31 GB read + 0.13 GB written per launch at 2^20 points
    scat, _ = bench._ncu_traffic(["r2f_ncu_full_msm2p20.csv"], "k_digit_scatter")
    assert scat is not None and scat < 0.3e9
    fb, name = bench._ncu_traffic(["r2f_ncu_full_fb_msm_warp.csv"], "k_fb_msm_warp_d")
    assert name and 2.2e9 < fb < 2.8e9    # 192 B per gather x 13.7 M gathers
    assert bench._ncu_traffic(["r2f_ncu_full_fb_msm_warp.csv"], "no_such_kernel") == (None, None)


def test_whole_step_operation_counts():
    import bench
    # 52 cards: n = 104, Q = 208, m = 105; 16 table windows, 16 windows in the combined verification MSM
    ref = bench.shuffle_imad_per_proof(104, 208, 105, "reference-fixed", 16, 16)
    fix = bench.shuffle_imad_per_proof(104, 208, 105, "fixed", 16, 16)
    assert ref["mixed_adds"] == 10336 and fix["mixed_adds"] == 39456
    assert ref["imad"] == 8243528 and fix["imad"] == 23952856
    # the roofline bound quoted for the `fixed` mode: 9.31 T IMAD/s / 23.95 M per proof = 389 K proofs/s
    assert 385e3 < 148 * 32 * 1.965e9 / fix["imad"] < 392e3


def test_dump_outputs_helpers(tmp_path):
    """--dump-outputs: the same sample of rows in every run, every byte value exact, float arrays only, 64 MB in all."""
    import numpy as np
    import pytest
    import bench
    rows = bench.dump_rows(4096)
    assert len(rows) == bench.DUMP_ROWS and np.all(np.diff(rows) > 0) and rows[-1] < 4096
    assert np.array_equal(rows, bench.dump_rows(4096))
    assert np.array_equal(bench.dump_rows(100), np.arange(100))
    buf = bytes(range(256)) * 2
    a = bench.bytes_f32(buf, 4)
    assert a.dtype == np.float32 and a.shape == (4, 128)
    assert bytes(a.astype(np.uint8).tobytes()) == buf
    bench.write_dump(str(tmp_path / "out"), {"x": a, "y": np.zeros(3)})
    assert np.array_equal(np.load(tmp_path / "out" / "x.npy"), a)
    assert np.load(tmp_path / "out" / "y.npy").dtype == np.float64
    with pytest.raises(TypeError):
        bench.write_dump(str(tmp_path / "bad"), {"z": np.zeros(3, dtype=np.uint8)})
    with pytest.raises(ValueError):
        bench.write_dump(str(tmp_path / "big"), {"z": np.zeros(bench.DUMP_LIMIT // 8 + 1)})
    assert not (tmp_path / "bad").exists() and not (tmp_path / "big").exists()
