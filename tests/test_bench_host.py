"""Host-side arithmetic of bench.py that must hold on a box this suite never sees (8 ranks sharing one host)."""
import bench

GIB = 1 << 30
SAMPLE = 2 * 3 * 1080 * 1920 * 4  # source + destination bytes of one sample in pinned memory


def test_whole_batch_is_pinned_when_the_host_can_spare_it():
    assert bench.host_ring_samples(256, 16, available_bytes=2000 * GIB, local_ranks=8) == 256
    assert bench.host_ring_samples(256, 16, available_bytes=3 * 256 * SAMPLE, local_ranks=1) == 256


def test_ring_is_whole_chunks_within_a_third_of_the_ranks_share():
    for avail, ranks in ((200 * GIB, 8), (64 * GIB, 8), (20 * GIB, 4), (1 * GIB, 8)):
        n = bench.host_ring_samples(256, 16, available_bytes=avail, local_ranks=ranks)
        assert n % 16 == 0 and 16 <= n < 256
        assert n == 16 or n * SAMPLE * 3 * ranks <= avail


def test_small_batches_are_never_cut():
    assert bench.host_ring_samples(8, 16, available_bytes=GIB, local_ranks=8) == 8


def test_dump_outputs_fits_the_budget_and_samples_the_same_elements(tmp_path, monkeypatch):
    import numpy as np
    import torch

    monkeypatch.setattr(bench, "DUMP_BYTES", 4000)
    big = torch.arange(10_000, dtype=torch.float32).reshape(10, 1000)
    small = torch.arange(9, dtype=torch.float64).reshape(3, 3)
    half = torch.ones(4, dtype=torch.float16)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"big": big, "small": small, "half": half})
    a = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in ("big", "small", "half")}
    assert a["small"].dtype == np.float64 and np.array_equal(a["small"], small.numpy())  # fits: written whole
    assert a["half"].dtype == np.float32 and a["half"].shape == (4,)
    assert a["big"].dtype == np.float32 and a["big"].ndim == 1 and 0 < a["big"].size < big.numel()
    assert np.all(np.diff(a["big"]) > 0)  # the elements of sorted, distinct flat indices
    assert sum(x.nbytes for x in a.values()) <= 4000
    assert np.array_equal(a["big"], np.load(tmp_path / "b" / "big.npy"))
