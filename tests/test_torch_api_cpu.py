"""The torch-facing functions against the call table of their calling-context tests, without a GPU."""
import inspect

import b200sort

import torch_calls as tc

# order_array and order_with_trust sort host (numpy) arrays; lib and lib_path load the library
NOT_TORCH_SORTS = {"order_array", "order_with_trust", "lib", "lib_path"}


def test_every_sorting_function_is_in_the_call_table():
    """tests/test_torch_capture_gpu.py captures and side-streams every call of tests/torch_calls.CALLS: a sorting
    function added to b200sort.__all__ must be added there too."""
    exported = {name for name in b200sort.__all__ if inspect.isfunction(getattr(b200sort, name))} - NOT_TORCH_SORTS
    assert exported == {c.fn for c in tc.CALLS.values()}
    assert {c.algo for c in tc.CALLS.values() if c.fn == "sort"} == {"", "merge"}


def test_call_table_entries_are_well_formed():
    """Every entry's key type is one its function accepts, its form matches the function's name, and the
    references sort a small data set of every kind."""
    import numpy as np
    import torch
    for name, c in tc.CALLS.items():
        assert (c.form == "rows") == c.fn.startswith("segmented_"), name
        assert (c.out == "pairs") == c.fn.endswith("_by_key") and (c.out == "indices") == c.fn.endswith("_indices")
        width = 16 if "16" in c.fn else 64 if "64" in c.fn else 32
        assert c.width == width == getattr(torch, tc.TORCH_DTYPES[c.kt]).itemsize * 8, name
        for kind in ("random", "all_equal", "masked"):
            shape = (4, 33) if c.form == "rows" else (133,)
            data = tc.dataset(c, shape, kind, 1)
            keys, second = tc.expected(c, shape, data)
            img = tc.KO[c.width].image(keys, c.kt, c.desc).reshape(-1, shape[-1])
            assert (np.diff(img.astype(np.float64), axis=1) >= 0).all(), (name, kind)
            if kind == "masked":
                assert not (img & ~type(img[0, 0])(tc.MASKED[c.width])).any(), (name, kind)
            if c.out == "indices":
                assert second.dtype == np.int64 and (second < shape[-1]).all()
