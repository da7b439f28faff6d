"""The rescan diff of csrc/kvg_rescan.cuh (k_rescan_merge for PCI and mdev survivors, k_rescan_keys), executed on
the CPU from its real kernel source under the warp emulator of tools/emu/ and checked against a restatement of the
rules in include/kvgpu.h: survivors added / removed / moved by identity, and map keys added / removed / changed
where "changed" compares member lists as each map stores them."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

import conftest  # noqa: F401

sys.path.insert(0, os.path.join(conftest.ROOT, "tools", "emu"))
import build as emu_build  # noqa: E402

from kvgpu import _lib as KL  # noqa: E402

RS_TILE = 1024


@pytest.fixture(scope="module")
def emu():
    L = C.CDLL(emu_build.build_rescan())
    P = C.POINTER
    L.emu_rescan.argtypes = [C.c_int, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, P(C.c_void_p),
                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, P(C.c_void_p), C.c_void_p,
                             P(C.c_void_p), C.c_void_p]
    L.emu_rescan.restype = C.c_int
    return L


# ---- survivor lists ----------------------------------------------------------------------------------------------
def ident(s, mdev):
    return bytes(s["uuid"]) if mdev else int(s["addr"])


def fields(s, mdev):
    """(map-0 key, map-1 key, numa)"""
    if mdev:
        return int(s["type_key"]), int(s["parent"]), int(s["numa"])
    return int(s["device"]), int(s["iommu_group"]), int(s["numa"])


def keys_of(surv, mdev):
    k0 = np.unique(np.array([fields(s, mdev)[0] for s in surv], dtype=np.uint32))
    k1 = np.unique(np.array([fields(s, mdev)[1] for s in surv], dtype=np.uint32))
    return k0, k1


def members(surv, mdev, m):
    """each map as it stores its members: {key: [member, ...]} in Walk order"""
    out = {}
    for s in surv:
        f = fields(s, mdev)
        numa_kept = m == 0 or not mdev  # gpuVgpuMap keeps uuids only
        out.setdefault(f[m], []).append((ident(s, mdev), f[2]) if numa_kept else ident(s, mdev))
    return out


def expected(A, B, mdev):
    ia = {ident(s, mdev): s for s in A}
    ib = {ident(s, mdev): k for k, s in enumerate(B)}
    added = [k for k, s in enumerate(B) if ident(s, mdev) not in ia]
    removed = [ident(s, mdev) for s in A if ident(s, mdev) not in ib]
    moved = [k for k, s in enumerate(B) if ident(s, mdev) in ia and fields(ia[ident(s, mdev)], mdev) != fields(s, mdev)]
    keys = []
    for m in (0, 1):
        old, new = members(A, mdev, m), members(B, mdev, m)
        keys.append((sorted(set(new) - set(old)), sorted(set(old) - set(new)),
                     sorted(k for k in set(old) & set(new) if old[k] != new[k])))
    return added, removed, moved, keys


def run(emu, A, B, mdev):
    dt = KL.MDEV_SURV if mdev else KL.PCI_SURV
    U = 2 if mdev else 1
    na, nb = len(A), len(B)
    a = np.zeros(na + 1, dtype=dt)
    a[:na] = A
    b = np.zeros(nb + 1, dtype=dt)
    b[:nb] = B
    ka, kb = keys_of(A, mdev), keys_of(B, mdev)
    key_lists = [np.append(ka[0], 0).astype(np.uint32), np.append(kb[0], 0).astype(np.uint32),
                 np.append(ka[1], 0).astype(np.uint32), np.append(kb[1], 0).astype(np.uint32)]
    nkeys = np.array([len(ka[0]), len(kb[0]), len(ka[1]), len(kb[1])], dtype=np.uint32)
    added = np.full(nb + 1, 0xdeadbeef, dtype=np.uint32)
    moved = np.full(nb + 1, 0xdeadbeef, dtype=np.uint32)
    removed = np.zeros(na + 1, dtype=dt)
    kcap = int(nkeys.max()) + 1
    kout = [np.full(kcap, 0xdeadbeef, dtype=np.uint32) for _ in range(6)]
    b_next = np.zeros(nb + 1, dtype=dt)
    kb_next = [np.zeros(len(kb[0]) + 1, dtype=np.uint32), np.zeros(len(kb[1]) + 1, dtype=np.uint32)]
    ctrl = np.zeros(16, dtype=np.uint32)
    ptrs = lambda arrs: (C.c_void_p * len(arrs))(*[x.ctypes.data for x in arrs])  # noqa: E731
    bad = emu.emu_rescan(1 if mdev else 0, a.ctypes.data, na, b.ctypes.data, nb, ptrs(key_lists),
                         nkeys.ctypes.data, added.ctypes.data, removed.ctypes.data, moved.ctypes.data, ptrs(kout),
                         b_next.ctypes.data, ptrs(kb_next), ctrl.ctypes.data)
    assert U in (1, 2)
    return dict(bad=bad, ctrl=ctrl, added=added, removed=removed, moved=moved, kout=kout, b_next=b_next[:nb],
                kb_next=[kb_next[0][:len(kb[0])], kb_next[1][:len(kb[1])]])


def check(emu, A, B, mdev):
    got = run(emu, A, B, mdev)
    assert got["bad"] == 0
    c = got["ctrl"]
    added, removed, moved, keys = expected(A, B, mdev)
    assert list(c[:3]) == [len(added), len(removed), len(moved)]
    assert got["added"][:c[0]].tolist() == added
    assert [ident(s, mdev) for s in got["removed"][:c[1]]] == removed
    assert got["moved"][:c[2]].tolist() == moved
    for m in (0, 1):
        for q in range(3):
            n = int(c[3 + 3 * m + q])
            assert got["kout"][3 * m + q][:n].tolist() == keys[m][q], (m, q)
    assert got["b_next"].tobytes() == np.asarray(B).tobytes()
    ka = keys_of(B, mdev)
    assert got["kb_next"][0].tolist() == ka[0].tolist() and got["kb_next"][1].tolist() == ka[1].tolist()
    assert emu.emu_rescan_flags_clear() == 1
    return keys


def gen_pci(rng, n, addr_space=None):
    s = np.zeros(n, dtype=KL.PCI_SURV)
    space = addr_space or max(4 * n, 16)
    s["addr"] = np.sort(rng.choice(space, size=n, replace=False)).astype(np.uint32)
    s["iommu_group"] = rng.integers(0, max(2, n // 4), n)
    s["device"] = rng.choice([0x1b38, 0x2330, 0x2901, 0x20b5], n)
    s["numa"] = rng.integers(0, 2, n)
    s["name_slot"] = rng.integers(0, 1000, n)
    return s


def gen_mdev(rng, n):
    s = np.zeros(n, dtype=KL.MDEV_SURV)
    u = rng.integers(0, 256, size=(n, 16), dtype=np.uint8)
    u = u[np.lexsort(u.T[::-1])]
    keep = np.ones(n, dtype=bool)
    keep[1:] = np.any(u[1:] != u[:-1], axis=1)
    u = u[keep]
    s = s[:len(u)]
    s["uuid"] = u
    s["parent"] = rng.integers(0, max(2, len(u) // 8), len(u))
    s["type_key"] = rng.integers(0, 40, len(u))
    s["numa"] = rng.integers(0, 2, len(u))
    s["src"] = np.arange(len(u))
    return s


def churn(rng, A, mdev, frac=0.05):
    """drop some, move some (each field), add some"""
    n = len(A)
    keep = rng.random(n) > frac
    B = A[keep].copy()
    for f in (("type_key", "parent", "numa") if mdev else ("device", "iommu_group", "numa")):
        idx = rng.choice(len(B), size=max(1, int(len(B) * frac / 3)), replace=False) if len(B) else []
        for i in idx:
            B[i][f] = (int(B[i][f]) + 1) % (2 if f == "numa" else 50)
    extra = gen_mdev(rng, max(1, int(n * frac))) if mdev else gen_pci(rng, max(1, int(n * frac)), 1 << 30)
    if not mdev:
        extra["addr"] += 1 << 30  # outside A's address space: new identities
    allv = np.concatenate([B, extra])
    order = np.argsort(np.array([ident(s, mdev) for s in allv], dtype=object), kind="stable") if mdev else \
        np.argsort(allv["addr"], kind="stable")
    allv = allv[order]
    ids = [ident(s, mdev) for s in allv]
    uniq = [k == 0 or ids[k] != ids[k - 1] for k in range(len(ids))]
    return allv[np.array(uniq, dtype=bool)] if len(allv) else allv


@pytest.mark.parametrize("mdev", [False, True])
def test_empty_and_full(emu, mdev):
    rng = np.random.default_rng(1)
    full = gen_mdev(rng, 3000) if mdev else gen_pci(rng, 3000)
    empty = full[:0]
    check(emu, empty, empty, mdev)
    keys = check(emu, empty, full, mdev)
    assert keys[0][0] == sorted(set(int(fields(s, mdev)[0]) for s in full))
    check(emu, full, empty, mdev)
    keys = check(emu, full, full, mdev)
    assert keys == [([], [], []), ([], [], [])]


@pytest.mark.parametrize("na,nb", [(1, 0), (0, 1), (1, 1), (RS_TILE, 0), (RS_TILE - 1, 1), (RS_TILE, RS_TILE),
                                   (RS_TILE + 1, RS_TILE - 1), (2 * RS_TILE - 3, 5), (511, 513), (3 * RS_TILE + 7, 2)])
def test_tile_and_diagonal_boundaries(emu, na, nb):
    rng = np.random.default_rng(na * 7919 + nb)
    for mdev in (False, True):
        pool = gen_mdev(rng, na + nb + 50) if mdev else gen_pci(rng, na + nb + 50)
        pick = rng.permutation(len(pool))
        A = pool[np.sort(pick[:na])]
        B = pool[np.sort(pick[max(0, na - nb // 2):max(0, na - nb // 2) + nb])]
        check(emu, A, B, mdev)


@pytest.mark.parametrize("mdev", [False, True])
def test_ten_thousand_with_every_kind_of_change(emu, mdev):
    rng = np.random.default_rng(10)
    A = gen_mdev(rng, 10_000) if mdev else gen_pci(rng, 10_000)
    B = churn(rng, A, mdev)
    added, removed, moved, keys = expected(A, B, mdev)
    assert added and removed and moved and any(k[2] for k in keys)
    check(emu, A, B, mdev)


def one_move(mdev, field):
    rng = np.random.default_rng(3)
    A = gen_mdev(rng, 200) if mdev else gen_pci(rng, 200)
    A["numa"] = 0
    B = A.copy()
    B[57][field] = int(B[57][field]) + (1 if field == "numa" else 1000)
    return A, B


def test_group_only_move_changes_iommu_map_not_device_map(emu):
    A, B = one_move(False, "iommu_group")
    keys = check(emu, A, B, False)
    assert keys[0] == ([], [], [])
    assert keys[1][0] == [int(B[57]["iommu_group"])] or keys[1][2]  # new group is new or changed
    assert int(A[57]["iommu_group"]) in keys[1][1] + keys[1][2]


def test_device_only_move_changes_device_map_not_iommu_map(emu):
    A, B = one_move(False, "device")
    keys = check(emu, A, B, False)
    assert keys[1] == ([], [], [])
    assert keys[0][0] == [int(B[57]["device"])]


def test_pci_numa_only_move_changes_both_maps(emu):
    A, B = one_move(False, "numa")
    keys = check(emu, A, B, False)
    assert keys[0][2] == [int(A[57]["device"])] and keys[1][2] == [int(A[57]["iommu_group"])]


def test_mdev_numa_only_move_changes_vgpu_map_not_gpu_vgpu_map(emu):
    A, B = one_move(True, "numa")
    keys = check(emu, A, B, True)
    assert keys[0] == ([], [], [int(A[57]["type_key"])])
    assert keys[1] == ([], [], [])


def test_mdev_parent_only_move(emu):
    A, B = one_move(True, "parent")
    keys = check(emu, A, B, True)
    assert keys[0] == ([], [], [])
    assert keys[1][0] == [int(B[57]["parent"])]


@pytest.mark.parametrize("mdev", [False, True])
@pytest.mark.parametrize("where", [1, RS_TILE, RS_TILE + 1, 2500])  # inside a tile and on tile boundaries
def test_non_ascending_input_raises_the_flag(emu, mdev, where):
    rng = np.random.default_rng(where)
    A = gen_mdev(rng, 3000) if mdev else gen_pci(rng, 3000)
    B = A.copy()
    B[where - 1], B[where] = A[where].copy(), A[where - 1].copy()
    assert run(emu, A, B, mdev)["bad"] == 1
    dup = A.copy()
    dup[where] = dup[where - 1]
    assert run(emu, A, dup, mdev)["bad"] == 1
    assert emu.emu_rescan_flags_clear() == 1


@pytest.mark.parametrize("mdev", [False, True])
def test_back_to_back_diffs_on_the_same_buffers(emu, mdev):
    """the second diff runs on the flags and look-back words the first one left: nothing is cleared in between"""
    rng = np.random.default_rng(77)
    A = gen_mdev(rng, 5000) if mdev else gen_pci(rng, 5000)
    B = churn(rng, A, mdev)
    Cc = churn(rng, B, mdev)
    check(emu, A, B, mdev)
    check(emu, B, Cc, mdev)
    check(emu, Cc, A, mdev)
