"""ctypes driver of integration/_build/libsearch_gpu.so: the reference-side adapter (integration/search_gpu.cpp -- the
six Search* entry points of gps/gps.h:140-145 over libacq_b200.so) inside the receiver harness the tests use
(integration/harness_gpu.cpp).  The library is compiled against integration/ref_api, the declarations of the
reference's types.h, gps/gps.h and its gps/sats.cpp table restated in this repository (integration/Makefile)."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
INTEGRATION = os.path.join(os.path.dirname(HERE), "integration")
LIB = os.path.join(INTEGRATION, "_build", "libsearch_gpu.so")
REF = os.path.join(INTEGRATION, "ref_api")

EVENT_DTYPE = np.dtype([("kind", "<i4"), ("a", "<i4"), ("b", "<i4"), ("c", "<i4"), ("d", "<i4"),
                        ("e", "<i4"), ("x", "<f8"), ("y", "<f8")])
# the reference's prototypes (gps/gps.h:140-145) as the Itanium C++ ABI mangles them
REFERENCE_SYMBOLS = {
    "SearchInit()": "_Z10SearchInitv", "SearchFree()": "_Z10SearchFreev", "SearchTask(void*)": "_Z10SearchTaskPv",
    "SearchTaskRun()": "_Z13SearchTaskRunv", "SearchEnable(int)": "_Z12SearchEnablei",
    "SearchParams(int, char**)": "_Z12SearchParamsiPPc",
}


def build():
    """Build the adapter (make keeps a fresh library); returns the library path."""
    from . import _build
    if _build.needs_build():
        _build.build()
    subprocess.run(["make", "-C", INTEGRATION, "--no-print-directory"], check=True, stdout=subprocess.DEVNULL)
    return LIB


class Adapter:
    def __init__(self):
        if not os.path.exists(LIB):
            build()
        L = C.CDLL(LIB)
        L.adp_init.argtypes = [C.c_int, C.POINTER(C.c_char_p)]
        L.adp_search_task.argtypes = [C.c_void_p] + [C.c_int] * 8
        L.adp_get_events.argtypes = [C.c_void_p, C.c_int]
        L.adp_prn_label.restype = C.c_char_p
        L.adp_prn_label.argtypes = [C.c_int]
        L.adp_task_run.argtypes = [C.c_int] * 5
        self.L = L

    def init(self, *argv):
        a = (C.c_char_p * (len(argv) + 1))(b"kiwid", *[x.encode() for x in argv])
        return self.L.adp_init(len(argv) + 1, a)

    def search_task(self, blocks, passes=1, free_chans=12, acq=(1, 1, 1), debug_prn=0, e1b_only=0):
        blocks = np.ascontiguousarray(blocks, np.uint8)
        n = self.L.adp_search_task(blocks.ctypes.data, blocks.size // 8192, passes, free_chans, *[int(x) for x in acq],
                                   debug_prn, e1b_only)
        ev = np.zeros(n, EVENT_DTYPE)
        if n:
            self.L.adp_get_events(ev.ctypes.data, n)
        return ev

    def task_run(self, good, users, clk_corrections, always_acq=0, locked=0):
        v = self.L.adp_task_run(good, users, clk_corrections, always_acq, locked)
        return v >> 8, v & 0xff   # (TaskSleepID calls, TaskWakeup calls) so far
