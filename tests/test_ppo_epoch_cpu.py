"""CPU side of the epoch update phase (kbs_minibatch_permutation / kbs_shuffle_minibatches / ppo.PpoUpdater.epoch): the
ctypes mirror of kbs_ppo_minibatches, the profiler's kernel-id count, and the NumPy restatement of the permutation law that
tests/test_gpu_ppo_epoch.py checks the device against (Philox4x32-10 against the Random123 known-answer vectors)."""

import re
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
M32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(c, key):
    """Philox4x32-10 on arrays: c = 4 uint32-valued arrays (broadcastable), key = (k0, k1).  uint64 arithmetic, masked."""
    c = [np.asarray(x, np.uint64) & M32 for x in c]
    k0, k1 = np.uint64(key[0]) & M32, np.uint64(key[1]) & M32
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c[0], np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & M32, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & M32]
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & M32, (k1 + np.uint64(0xBB67AE85)) & M32
    return c


def permutation(seed: int, pass_: int, env0: int, n: int) -> np.ndarray:
    """The law of kbs_minibatch_permutation (include/kbotstep.h): sort (key(e) << 32) | e, keep the low 32 bits."""
    e = np.arange(n, dtype=np.uint64)
    x = philox4x32_10((pass_ & 0xFFFFFFFF, pass_ >> 32, (env0 + e) & M32, 0xFFFFFFFF), (seed & 0xFFFFFFFF, seed >> 32))
    v = (x[0] << np.uint64(32)) | e
    return (np.sort(v) & M32).astype(np.int32)


def test_philox_restatement_matches_known_answers():
    """Random123's kat_vectors for philox4x32_10."""
    kat = [((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
           ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
           ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
            (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]
    for c, k, want in kat:
        assert tuple(int(w) for w in philox4x32_10(c, k)) == want


def test_permutation_law_is_a_permutation():
    for n in (1, 4, 63, 4096):
        p = permutation(7, 3, 0, n)
        assert sorted(p.tolist()) == list(range(n))
    assert not np.array_equal(permutation(7, 3, 0, 64), permutation(7, 4, 0, 64))
    assert not np.array_equal(permutation(7, 3, 0, 64), permutation(7, 3, 64, 64))
    assert not np.array_equal(permutation(7, 3, 0, 64), permutation(8, 3, 0, 64))


def test_minibatches_struct_and_kernel_ids_match_header(lib_built):
    from kbot_joystick_b200 import _lib as L

    hdr = (ROOT / "include" / "kbotstep.h").read_text()
    body = re.search(r"typedef struct kbs_ppo_minibatches \{(.*?)\} kbs_ppo_minibatches;", hdr, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = []
    for decl in filter(None, (d.strip() for d in body.split(";"))):
        decl = re.sub(r"^(const\s+)?(float|int64_t|uint8_t)\s*\*?\s*", "", decl)
        names += [re.sub(r"[\*\s]", "", nm) for nm in decl.split(",")]
    assert names == [f[0] for f in L.KbsPpoMinibatches._fields_]
    assert L.KbsPpoMinibatches._fields_[-2:] == [("batch_size", L._i64), ("num_batches", L._i64)]
    assert int(re.search(r"#define KBS_NUM_KERNEL_IDS (\d+)", hdr).group(1)) == L.NUM_KERNEL_IDS
    assert int(re.search(r"#define KBS_MAX_PERMUTATION_ENVS (\d+)", hdr).group(1)) == L.MAX_PERMUTATION_ENVS
    lib = L.load()
    assert {"kbs_minibatch_permutation", "kbs_shuffle_minibatches"} <= set(L.EXPORTS)
    names = [lib.kbs_kernel_name(i).decode() for i in range(L.NUM_KERNEL_IDS)]
    assert names[-2:] == ["minibatch_permutation_kernel", "shuffle_minibatches_kernels"] and "?" not in names
