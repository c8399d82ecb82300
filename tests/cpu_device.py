"""TEST HARNESS (never imported by the product): runs the product's Python host layer — ministark_b200/prover.py
(`GpuProver`), prover_mgpu.py (`ShardedProver`), channel / air / proof / deep / the examples — WITHOUT a GPU by putting
the CPU oracle's build of the C ABI (oracle/libms_cpu_abi.so, oracle/cpu_abi.c) underneath `ministark_b200._lib` and
giving the prover host ("cpu") torch tensors and no-op streams.  The product itself has no such switch: outside a
process that called install() the library loader only ever opens libministark_b200.so and fails without a CUDA device.

What this buys in the CPU suite: the Fiat–Shamir driver, the program binding, the query phase, the sharding arithmetic
and the collectives of the multi-GPU prover (over gloo, world size 2 and 4) are executed end to end and their proof
bytes compared with oracle/stark_oracle.cpu_prove before any GPU run."""
import ctypes as C
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE = os.path.join(ROOT, "oracle")


def build():
    subprocess.check_call(["make", "-s", "-C", ORACLE, "libms_cpu_abi.so"])
    return os.path.join(ORACLE, "libms_cpu_abi.so")


class _Stream:
    cuda_stream = 0

    def wait_stream(self, other):
        pass

    def wait_event(self, event):
        pass

    def synchronize(self):
        pass


class _Event:
    def __init__(self, *a, **k):
        pass

    def record(self, stream=None):
        pass

    def synchronize(self):
        pass


def install():
    """idempotent; returns the ctypes handle of the CPU ABI"""
    # the process must see no GPU even on a machine that has one: with a device visible, torch.cuda.stream() stops being a
    # no-op and tries to make the harness's _Stream objects current.  Takes effect because CUDA is not initialised yet here.
    os.environ["CUDA_VISIBLE_DEVICES"] = ""
    import torch
    assert not torch.cuda.is_available(), "cpu_device.install() must run before CUDA is initialised in this process"
    from ministark_b200 import _lib, prover
    from ministark_b200 import Context
    if getattr(_lib, "_cpu_device_installed", False):
        return _lib._lib
    lib = C.CDLL(build())
    for name, (res, args) in _lib._SIGS.items():
        if hasattr(lib, name):          # the six device-only entry points are absent (tests/test_cpp_cpu_abi.py lists them)
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
    _lib._lib = lib
    _lib._cpu_device_installed = True

    def init(self, device=0):
        self.device = torch.device("cpu")
        self.stream, self.copy_stream = _Stream(), _Stream()
        self.ctx = Context(0)
        self._airs = {}

    prover.GpuProver.__init__ = init
    prover.GpuProver._shared = {}
    torch.cuda.Event = _Event
    return lib
