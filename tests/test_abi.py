"""CPU checks of the C-ABI boundary: the library loads without a GPU, exports every function
declared in include/rr_b200.h, the ctypes table matches the header, and host-only entry points
(MT19937 seeding, tokenizer) give reference answers."""
import ctypes as C
import random
import re
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]


def _declared():
    text = (ROOT / "include" / "rr_b200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(rr_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from rr_b200 import _lib
    names = _declared()
    assert len(names) >= 30
    missing = [n for n in names if not hasattr(_lib.lib, n)]
    assert not missing, missing
    assert not _lib.MISSING
    assert sorted(_lib.PROTOTYPES) == names


def test_struct_sizes_match_header():
    from rr_b200 import _lib
    assert C.sizeof(_lib.Event) == 24 and C.sizeof(_lib.Decision) == 16
    assert C.sizeof(_lib.DeploymentDesc) == 24 and C.sizeof(_lib.RouterSettings) == 32
    assert C.sizeof(_lib.DeploymentState) == 48
    assert C.sizeof(_lib.ModelDesc) == 36 and C.sizeof(_lib.Completion) == 48


def test_mt19937_seeding_matches_cpython():
    from rr_b200 import _lib
    for seed in [0, 1, 42, 1234, 2**31 - 1, 2**32 - 1, 2**32, 2**40 + 12345, 2**64 - 1]:
        buf = (C.c_uint32 * 625)()
        assert _lib.lib.rr_mt_seed_state(seed, buf) == 0
        want = random.Random(seed).getstate()[1]
        assert tuple(buf) == tuple(want), seed


def test_tokenizer_counts():
    from rr_b200 import _lib
    n = C.c_int32()
    s = "What is machine learning?".encode()
    assert _lib.lib.rr_count_tokens(s, len(s), C.byref(n)) == 0 and n.value == len(s) + 1
    ids = (C.c_int32 * 64)()
    assert _lib.lib.rr_tokenize(s, len(s), 128256, ids, 64, C.byref(n)) == 0
    assert n.value == len(s) + 1 and ids[0] == 1 and ids[1] == 3 + ord("W")
    assert _lib.lib.rr_tokenize(s, len(s), 128256, ids, 4, C.byref(n)) != 0   # buffer too small


def test_version_and_errors():
    from rr_b200 import _lib
    assert b"sm_100a" in _lib.lib.rr_version()
    assert b"429" in _lib.lib.rr_strerror(1)


@pytest.mark.parametrize("grid,inter,hidden,slice_kb", [(148, 14336, 4096, 28), (148, 8192, 3072, 16), (132, 2816, 1024, 15),
                                                        (148, 1024, 512, 16), (7, 14336, 4096, 28)])
def test_fused_mlp_schedule_is_a_partition_and_deadlock_free(grid, inter, hidden, slice_kb):
    """Host logic of the fused decode MLP kernel (csrc/rr_gemm.cu, mlp_schedule): every gate/up tile and every
    (down tile, K-slice) appears exactly once; in every CTA's list all gate/up items precede all down items (a down
    item waits on gate/up tiles of OTHER CTAs, which therefore can never be queued behind a waiting item); slices
    cover the K range without gaps; the lists are balanced."""
    import ctypes as C
    import numpy as np
    from rr_b200 import _lib as lib
    mx = C.c_int32()
    cap = grid * 128
    buf = np.full((cap, 4), -7, dtype=np.int32)
    rc = lib.lib.rr_debug_mlp_schedule(grid, inter, hidden, slice_kb, buf.ctypes.data_as(C.POINTER(C.c_int32)), cap, C.byref(mx))
    assert rc == 0 and 1 <= mx.value <= 128
    items = buf[: grid * mx.value].reshape(grid, mx.value, 4)
    tiles0, kb0n = 2 * inter // 128, (hidden + 63) // 64
    tiles1, kb1n = (hidden + 127) // 128, inter // 64
    n_slices = (kb1n + slice_kb - 1) // slice_kb
    seen0, seen1, loads = set(), set(), []
    for c in range(grid):
        phase_seen, load, ended = 0, 0, False
        for tp, k0, k1, z in items[c]:
            if tp < 0:
                ended = True
                continue
            assert not ended                                   # no entry after the terminator
            ph, tile = tp >> 16, tp & 0xFFFF
            assert ph >= phase_seen                            # gate/up first, then down
            phase_seen = ph
            if ph == 0:
                assert (k0, k1) == (0, kb0n) and tile < tiles0 and tile not in seen0
                seen0.add(tile)
            else:
                assert tile < tiles1 and 0 <= z < n_slices and (tile, z) not in seen1
                assert k0 == z * slice_kb and k1 == min(kb1n, k0 + slice_kb)
                seen1.add((tile, z))
            load += k1 - k0
        loads.append(load)
    assert len(seen0) == tiles0 and len(seen1) == tiles1 * n_slices
    total = tiles0 * kb0n + tiles1 * kb1n
    assert sum(loads) == total
    if grid >= 64 and total // grid >= 100:                    # the production shapes: within 15 % of the mean
        assert max(loads) <= 1.15 * total / grid + slice_kb
