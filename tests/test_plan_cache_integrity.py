"""On-disk plan cache (plan_cache_dir) against damaged files and concurrent writers (host only).

A cache file is uploaded to the device as it is read, so a file whose payload differs from what
was stored must be a miss, whatever its sizes say: an out-of-range source column would make the
kernels read outside x.  And one process may build the same operator on several threads at once
(dask workers, benchmark ranks sharing a cache directory); their writes must not mix.
"""
import os
import threading

import numpy as np
import pytest

from test_plan import HostPlan

ARRAYS = ("rowptr", "col", "val", "tiles", "segs", "wplan", "iplan")


def _c4(lib):
    from smmregrid_b200 import synth
    w = synth.config_weights("C4", 10)
    n_src, n_dst = w.sizes["src_grid_size"], w.sizes["dst_grid_size"]
    return (lib, w["src_address"], w["dst_address"], w["remap_matrix"], n_src, n_dst), n_src


def _assert_same_plan(got, want, what):
    for name in ARRAYS:
        assert np.array_equal(getattr(got, name), getattr(want, name)), f"{what}: {name}"
    strip = lambda info: {k: v for k, v in info.items() if k != "plan_cache_hit"}      # noqa: E731
    assert strip(got.info) == strip(want.info), what


def _only_file(d):
    files = os.listdir(d)
    assert len(files) == 1 and files[0].endswith(".plan"), files
    return os.path.join(d, files[0])


def _offset_of(data, arr):
    """Byte offset of the array's payload in the file: found by content, not by layout."""
    needle = np.ascontiguousarray(arr).tobytes()
    pos = data.find(needle)
    assert pos >= 0 and data.find(needle, pos + 1) < 0, "payload not found exactly once"
    return pos


ALTERATIONS = ("col-in-range", "col-out-of-range", "val", "wplan")


def _alteration(what, fresh, n_src):
    """(array, flat index, new value): one element of col (a column still in range, one beyond
    n_src), val or wplan (one ulp), changed in place so that every length stays intact."""
    col, i = fresh.col, fresh.col.size // 2
    wp = fresh.wplan.reshape(-1)
    j = int(np.argmax(np.abs(wp)))
    return {"col-in-range": (col, i, np.int32((int(col[i]) + 1) % n_src)),
            "col-out-of-range": (col, i, np.int32(n_src + 4096)),
            "val": (fresh.val, i, np.nextafter(fresh.val[i], np.inf)),
            "wplan": (wp, j, np.nextafter(wp[j], -np.inf))}[what]


@pytest.mark.parametrize("what", ALTERATIONS)
def test_altered_payload_is_a_miss(smm_lib, tmp_path, what):
    """The altered file is a miss, and the rebuilt plan equals a build without the cache; the
    file is rewritten and the next load is a hit again."""
    args, n_src = _c4(smm_lib)
    fresh = HostPlan(*args)
    assert fresh.info["kernel_name"] == "staged" and fresh.wplan.size > 0
    d = str(tmp_path / "plans")
    assert HostPlan(*args, cache_dir=d).info["plan_cache_hit"] == 0
    path = _only_file(d)
    with open(path, "rb") as f:
        good = f.read()
    arr, idx, value = _alteration(what, fresh, n_src)
    assert value != arr.reshape(-1)[idx]
    pos = _offset_of(good, arr) + idx * arr.itemsize
    bad = bytearray(good)
    bad[pos:pos + arr.itemsize] = np.asarray(value, arr.dtype).tobytes()
    with open(path, "wb") as f:
        f.write(bad)
    got = HostPlan(*args, cache_dir=d)
    assert got.info["plan_cache_hit"] == 0, "altered file accepted"
    _assert_same_plan(got, fresh, what)
    with open(path, "rb") as f:
        assert f.read() == good, "the miss did not rewrite the file"
    again = HostPlan(*args, cache_dir=d)
    assert again.info["plan_cache_hit"] == 1
    _assert_same_plan(again, fresh, what)


def test_trailing_bytes_are_a_miss(smm_lib, tmp_path):
    """A valid file with bytes appended is not the file that was stored."""
    args, _ = _c4(smm_lib)
    d = str(tmp_path / "plans")
    HostPlan(*args, cache_dir=d)
    path = _only_file(d)
    with open(path, "ab") as f:
        f.write(b"\0" * 8)
    assert HostPlan(*args, cache_dir=d).info["plan_cache_hit"] == 0
    assert HostPlan(*args, cache_dir=d).info["plan_cache_hit"] == 1


def test_concurrent_writers_of_one_operator(smm_lib, tmp_path):
    """8 threads build the same operator with one cache directory at the same moment (all miss,
    all write), then load it twice each while slower threads may still be writing: every plan
    equals the fresh build, no temporary file is left behind and the file that stays is a hit.
    The file is removed between rounds."""
    args, _ = _c4(smm_lib)
    fresh = HostPlan(*args)
    d = str(tmp_path / "plans")
    n = 8
    for r in range(4):
        barrier = threading.Barrier(n)
        plans, errors = [[] for _ in range(n)], []

        def work(t):
            try:
                barrier.wait()
                for _ in range(3):
                    plans[t].append(HostPlan(*args, cache_dir=d))
            except Exception as e:          # noqa: BLE001
                errors.append(f"thread {t}: {e!r}")

        threads = [threading.Thread(target=work, args=(t,)) for t in range(n)]
        for th in threads:
            th.start()
        for th in threads:
            th.join()
        assert not errors, errors
        for t, ps in enumerate(plans):
            for k, p in enumerate(ps):
                _assert_same_plan(p, fresh, f"round {r} thread {t} call {k}")
        path = _only_file(d)                        # (a leftover temporary file fails here)
        last = HostPlan(*args, cache_dir=d)
        assert last.info["plan_cache_hit"] == 1, f"round {r}: the stored file is not a hit"
        _assert_same_plan(last, fresh, f"round {r} final load")
        os.remove(path)
