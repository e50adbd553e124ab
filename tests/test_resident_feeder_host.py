"""Host side of the resident feeder: it sizes bags with the host augmentation's own count and shares PackedBagFeeder's
schedule code; it refuses a non-CUDA device.  The device leg is in tests/test_gpu_resident_feeder.py."""
import random

import pytest

import mil_b200
from mil_b200 import feeder


def test_augmentation_count_is_the_host_subset_size():
    rng = random.Random(1)
    for n in (1, 2, 3, 9, 10, 11, 127, 128, 129, 1000, 20_000, 70_000):
        for t in ("Biopsy", "Resection"):
            assert feeder.augmentation_count(n, t) == len(feeder.augmentation_rows(n, t, rng)) == int(n * feeder.AUGMENT_KEEP[t])
    assert feeder.augmentation_count(50, "Other") is None and feeder.augmentation_rows(50, "Other", rng) is None


def test_both_feeders_share_one_schedule():
    for name in ("set_epoch", "order", "batches", "__len__"):
        assert getattr(feeder.ResidentBagFeeder, name) is getattr(feeder.PackedBagFeeder, name)
    assert mil_b200.ResidentBagFeeder is feeder.ResidentBagFeeder


def test_resident_feeder_needs_a_cuda_device():
    import numpy as np
    with pytest.raises(mil_b200.MilB200Error, match="CUDA"):
        feeder.ResidentBagFeeder([np.zeros((3, 16), np.float32)], batch_bags=1, L_feat=16, device="cpu")
