"""CPU: bench.py --dump-outputs writes every array of the scan result exactly, and a fixed sample under its cap."""
import numpy as np

import conftest  # noqa: F401
import bench
import kvgpu
from kvgpu.context import PciResult


def _result(S=50_000):
    rng = np.random.default_rng(11)
    surv = np.zeros(S, dtype=kvgpu.PCI_SURV)
    surv["addr"] = np.arange(S) * 3
    surv["iommu_group"] = rng.integers(0, 1 << 32, S, dtype=np.uint64).astype(np.uint32)
    surv["device"] = rng.integers(0, 1 << 16, S).astype(np.uint16)
    surv["name_slot"] = 0xFFFFFFFF
    return PciResult(3 * S, surv, np.arange(7, dtype=np.uint16), np.arange(8, dtype=np.uint32),
                     rng.permutation(S).astype(np.uint32), np.zeros(7, dtype=np.uint32),
                     np.arange(900, dtype=np.uint32), np.arange(901, dtype=np.uint32),
                     rng.permutation(S).astype(np.uint32), b"\x03\x00ABC")


def _load(d, names):
    return {n: np.load(d / (n + ".npy")) for n in names}


def test_dump_is_exact_under_the_cap(tmp_path):
    res = _result()
    arrays = bench.result_arrays(res)
    assert set(arrays) == {"survivors_addr", "survivors_iommu_group", "survivors_device", "survivors_numa",
                           "survivors_name_slot", "dev_keys", "dev_off", "dev_perm", "dev_name_slot",
                           "grp_keys", "grp_off", "grp_perm", "name_pool"}
    bench.dump_outputs(str(tmp_path), arrays, bench.DUMP_BYTES)
    got = _load(tmp_path, arrays)
    assert all(a.dtype == np.float64 for a in got.values())
    assert np.array_equal(got["survivors_iommu_group"], res.survivors["iommu_group"])
    assert np.array_equal(got["survivors_name_slot"], res.survivors["name_slot"])
    assert np.array_equal(got["grp_perm"], res.grp_perm)
    assert np.array_equal(got["name_pool"], [3, 0, 65, 66, 67])


def test_dump_samples_the_same_elements_past_the_cap(tmp_path):
    arrays = bench.result_arrays(_result())
    budget = 8 * sum(a.size for a in arrays.values()) // 4
    a, b = tmp_path / "a", tmp_path / "b"
    bench.dump_outputs(str(a), arrays, budget)
    bench.dump_outputs(str(b), arrays, budget)
    ga, gb = _load(a, arrays), _load(b, arrays)
    assert sum(x.nbytes for x in ga.values()) <= budget
    assert all(np.array_equal(ga[n], gb[n]) for n in arrays)
    addr = ga["survivors_addr"]                       # a sorted subset of the original elements
    assert 0 < len(addr) < len(arrays["survivors_addr"]) and np.all(np.diff(addr) > 0) and np.all(addr % 3 == 0)
