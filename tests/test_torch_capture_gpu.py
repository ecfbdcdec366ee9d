"""The torch-facing sorts in the two calling contexts their docstrings promise besides an eager call: inside a CUDA
graph capture as the first library call of a process, and on a side stream without synchronising the host.

1. Capture first (one fresh process per case, so the lane-order self-test's verdict starts unknown): the process
   builds its inputs with torch ops only, then captures the call with ``torch.cuda.graph`` in the default global
   capture mode, which is the first call into the library.  The self-test runs inside that capture.  It must neither
   break the capture nor cache a failed verdict.  The graph is replayed on random bit patterns with float specials,
   all keys equal, and images masked to skip passes, and every result is compared with the numpy reference.  The
   process then prints the device's verdict and effective pass kernel, which must equal those of a control process
   that ran ``b200sort_device_check()`` eagerly.  The same holds when the first sort runs eagerly on one thread while
   another thread holds a global-mode capture, and for the first call on a second GPU after an eager one on the first.
2. Side streams (in the pytest process): under ``torch.cuda.stream(s)`` with ``s`` held back by a 0.3 s sleep kernel,
   each call on an input that is overwritten on ``s`` must return while ``s`` is still busy (no host synchronisation)
   and sort what ``s`` wrote (it ran on ``s``).  The inputs start one element into larger tensors.

The calls, data sets and references are tests/torch_calls.py.
"""
import json
import os
import subprocess
import sys

import pytest

import torch_calls as tc

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REPLAYS = [("random", 11), ("all_equal", 12), ("masked", 13), ("random", 14)]


# ---- 1. the first call of a process inside a capture -----------------------------------------------------------------
def _verdict(L) -> dict:
    return {"atomic_order_ok": L.b200sort_radix_atomic_order_ok(),
            "variant": L.b200sort_radix_effective_variant_name().decode()}


def _print_verdict(v: dict):
    print("VERDICT " + json.dumps(v, sort_keys=True), flush=True)


def child_control():
    from b200sort._lib import check, lib
    check(lib().b200sort_device_check())
    _print_verdict(_verdict(lib()))


def child_capture(name: str):
    import torch
    from b200sort import _lib
    c = tc.CALLS[name]
    inputs = [tc.Inputs(c, shape) for shape in c.shapes()]
    for i, inp in enumerate(inputs):
        inp.load(tc.dataset(c, inp.shape, "random", i))
    torch.cuda.synchronize()
    assert _lib._lib is None, "the library was loaded before the capture"
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):                                   # capture_error_mode "global"
        outs = [c.run(*inp.args()) for inp in inputs]
    for kind, seed in REPLAYS:
        data = [tc.dataset(c, inp.shape, kind, seed + i) for i, inp in enumerate(inputs)]
        for inp, d in zip(inputs, data):
            inp.load(d)
        g.replay()
        torch.cuda.synchronize()
        for inp, d, out in zip(inputs, data, outs):
            tc.compare(c, inp.shape, d, out, f"{name} {inp.shape} replay {kind}")
    _print_verdict(_verdict(_lib.lib()))


def child_threads():
    """Thread A holds a global-mode capture of a torch op while this thread makes the process's first sort, eagerly."""
    import threading
    import torch
    import b200sort
    from b200sort import _lib
    c = tc.CALLS["sort_by_key"]
    shape = tc.SIZES_1D[-1]
    inp = tc.Inputs(c, shape)
    data = tc.dataset(c, shape, "random", 21)
    inp.load(data)
    x = torch.arange(4096, dtype=torch.float32, device="cuda")
    y = torch.empty_like(x)
    # Give torch's caching allocator blocks for the sort's outputs and workspace, so that torch itself needs no
    # cudaMalloc while A captures: only the library's own calls are under test.
    cached = [torch.empty(64 << 20, dtype=torch.uint8, device="cuda"), torch.empty(256 << 10, dtype=torch.uint8,
                                                                                   device="cuda")]
    del cached
    torch.cuda.synchronize()
    assert _lib._lib is None
    g, s = torch.cuda.CUDAGraph(), torch.cuda.Stream()
    capturing, release, errors = threading.Event(), threading.Event(), []

    def thread_a():
        try:
            with torch.cuda.stream(s):
                g.capture_begin(capture_error_mode="global")
                try:
                    torch.mul(x, 3, out=y)
                    capturing.set()
                    if not release.wait(timeout=300):
                        raise TimeoutError("the sorting thread did not finish")
                finally:
                    g.capture_end()
        except BaseException as e:                                  # reported by the main thread
            errors.append(e)
            capturing.set()

    a = threading.Thread(target=thread_a)
    a.start()
    try:
        assert capturing.wait(timeout=300)
        out = b200sort.sort_by_key(*inp.args())                     # thread B: the first call into the library
    finally:
        release.set()
        a.join(timeout=300)
    assert not a.is_alive() and not errors, f"thread A's capture: {errors}"
    torch.cuda.synchronize()
    tc.compare(c, shape, data, out, "sort_by_key during another thread's capture")
    y.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(y, x * 3), "thread A's graph"
    _print_verdict(_verdict(_lib.lib()))


def child_two_gpus():
    """An eager sort on cuda:0, then the first sort on cuda:1 inside a capture: the verdict is kept per device."""
    import torch
    from b200sort import _lib
    c = tc.CALLS["sort_by_key"]
    shape = tc.SIZES_1D[-1]
    first = tc.Inputs(c, shape, device="cuda:0")
    data = tc.dataset(c, shape, "random", 31)
    first.load(data)
    tc.compare(c, shape, data, c.run(*first.args()), "eager on cuda:0")
    with torch.cuda.device(1):
        inp = tc.Inputs(c, shape, device="cuda:1")
        inp.load(data)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            out = c.run(*inp.args())
        for kind, seed in REPLAYS:
            d = tc.dataset(c, shape, kind, seed)
            inp.load(d)
            g.replay()
            torch.cuda.synchronize()
            tc.compare(c, shape, d, out, f"cuda:1 replay {kind}")
    verdicts = []
    for dev in (0, 1):
        with torch.cuda.device(dev):
            verdicts.append(_verdict(_lib.lib()))
    assert verdicts[0] == verdicts[1], verdicts
    _print_verdict(verdicts[1])


def child(argv):
    {"control": child_control, "capture": child_capture, "threads": child_threads,
     "two_gpus": child_two_gpus}[argv[0]](*argv[1:])


def _run_child(*argv) -> dict:
    code = ("import sys; sys.path[:0] = ['.', 'tests']\n"
            "import test_torch_capture_gpu as t\n"
            "t.child(sys.argv[1:])\n")
    env = {k: v for k, v in os.environ.items() if k != "B200SORT_RANK_SAFE"}
    r = subprocess.run([sys.executable, "-c", code, *argv], cwd=ROOT, env=env, capture_output=True, text=True,
                       timeout=900)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("VERDICT ")]
    assert r.returncode == 0 and lines, \
        f"child {argv} exited with {r.returncode}:\n{r.stdout[-3000:]}\n{r.stderr[-6000:]}"
    return json.loads(lines[-1][len("VERDICT "):])


@pytest.fixture(scope="module")
def control():
    """The verdict and pass kernel of a process that ran b200sort_device_check() before anything else."""
    return _run_child("control")


@pytest.mark.parametrize("name", list(tc.CALLS))
def test_first_call_of_a_process_inside_a_capture(name, control):
    assert _run_child("capture", name) == control


def test_first_call_while_another_thread_captures(control):
    assert _run_child("threads") == control


def test_first_call_on_a_second_gpu_inside_a_capture(control):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    assert _run_child("two_gpus") == control


# ---- 2. side streams -------------------------------------------------------------------------------------------------
SLEEP_CYCLES = 600_000_000          # about 0.3 s at the B200's 1.9-2 GHz SM clock


@pytest.fixture(scope="module")
def checked_device():
    from b200sort._lib import check, lib
    check(lib().b200sort_device_check())


@pytest.mark.parametrize("name", list(tc.CALLS))
def test_side_stream_without_host_synchronisation(name, checked_device):
    import torch
    c = tc.CALLS[name]
    s = torch.cuda.Stream()
    for i, shape in enumerate(c.shapes()):
        inp = tc.Inputs(c, shape, offset=1)
        first, second = tc.dataset(c, shape, "random", 41 + i), tc.dataset(c, shape, "masked", 51 + i)
        src = tc.staged(inp, second)
        inp.load(first)
        # One eager call first: the CUDA driver loads a kernel's module on its first launch, and that load may wait
        # for the device (lazy loading), which is not the wrapper's doing.
        tc.compare(c, shape, first, c.run(*inp.args()), f"{name} {shape} warm-up")
        torch.cuda.synchronize()
        with torch.cuda.stream(s):
            torch.cuda._sleep(SLEEP_CYCLES)
            inp.load(src=src)                                   # the second data set, written on s after the sleep
            out = c.run(*inp.args())
            busy = not s.query()
        assert busy, f"{name} {shape}: the call returned after s had drained (it synchronised the host)"
        s.synchronize()
        tc.compare(c, shape, second, out, f"{name} {shape} on a side stream")
