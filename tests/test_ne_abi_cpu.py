"""include/ns_ne_abi.h restates struct ne_tensor / ne_compute_params and a few enum values of the reference's graph engine (the
structs bestla_support / bestla_parallel_for receive).  Every offset, size and enum value of ns_ne_abi.h must equal the one the
reference's core/ne.h gives; the reference's numbers (x86-64 LP64) are stored in tests/golden/reference.npz, recorded by compiling
the same program against that header."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from oracle import golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

FIELDS = ["type", "backend", "n_dims", "ne", "nb", "op", "is_param", "op_params", "grad", "src0", "src1", "opt", "n_tasks", "perf_runs",
          "perf_cycles", "perf_time_us", "data", "size", "name", "padding"]
PFIELDS = ["type", "ith", "nth", "wsize", "wdata", "dev_wsize", "dev_wdata", "dev_queue"]
ENUMS = {"NE_TYPE_F32": "NS_NE_TYPE_F32", "NE_TYPE_F16": "NS_NE_TYPE_F16", "NE_TYPE_Q4_0": "NS_NE_TYPE_Q4_0", "NE_TYPE_Q6_K": "NS_NE_TYPE_Q6_K",
         "NE_TYPE_BTLA": "NS_NE_TYPE_BTLA", "NE_BACKEND_CPU": "NS_NE_BACKEND_CPU", "NE_BACKEND_SYCL": "NS_NE_BACKEND_SYCL",
         "NE_TASK_INIT": "NS_NE_TASK_INIT", "NE_TASK_COMPUTE": "NS_NE_TASK_COMPUTE", "NE_TASK_FINALIZE": "NS_NE_TASK_FINALIZE",
         "NE_OP_ADD": "NS_NE_OP_ADD", "NE_OP_MUL": "NS_NE_OP_MUL", "NE_OP_NORM": "NS_NE_OP_NORM", "NE_OP_RMS_NORM": "NS_NE_OP_RMS_NORM",
         "NE_OP_MUL_MAT": "NS_NE_OP_MUL_MAT", "NE_OP_MUL_MAT_BIAS": "NS_NE_OP_MUL_MAT_BIAS", "NE_OP_MUL_MAT_ID": "NS_NE_OP_MUL_MAT_ID",
         "NE_OP_ROPE": "NS_NE_OP_ROPE", "NE_OP_MUL_QKV": "NS_NE_OP_MUL_QKV", "NE_OP_MUL_FFN_SILU": "NS_NE_OP_MUL_FFN_SILU",
         "NE_OP_MUL_FFN_GELU": "NS_NE_OP_MUL_FFN_GELU", "NE_OP_MUL_FFN_GELU_MUL": "NS_NE_OP_MUL_FFN_GELU_MUL",
         "NE_OP_MUL_FFN_ADD_GELU": "NS_NE_OP_MUL_FFN_ADD_GELU", "NE_OP_MUL_ID_FFN_SILU": "NS_NE_OP_MUL_ID_FFN_SILU",
         "NE_OP_MUL_ID_FFN_GELU": "NS_NE_OP_MUL_ID_FFN_GELU", "NE_MAX_DIMS": "NS_NE_MAX_DIMS", "NE_MAX_OPT": "NS_NE_MAX_OPT",
         "NE_MAX_OP_PARAMS": "NS_NE_MAX_OP_PARAMS"}


def _layout(header, tensor, params, enums, incs):
    """offsets of FIELDS / PFIELDS, both sizeofs and the enum values, as one header declares them"""
    vals = [f"offsetof(struct {tensor}, {f})" for f in FIELDS] + [f"offsetof(struct {params}, {f})" for f in PFIELDS]
    vals += [f"sizeof(struct {tensor})", f"sizeof(struct {params})"] + [f"(long)({e})" for e in enums]
    body = "".join(f'printf("%ld\\n", (long)({v}));' for v in vals)
    with tempfile.TemporaryDirectory() as d:
        src, exe = os.path.join(d, "layout.c"), os.path.join(d, "layout")
        open(src, "w").write(f'#include <stdio.h>\n#include <stddef.h>\n#include "{header}"\nint main(void){{{body}return 0;}}\n')
        r = subprocess.run(["gcc", "-std=c11", *[f"-I{i}" for i in incs], src, "-o", exe], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        out = subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()
    return np.array([int(v) for v in out], np.int64)


def test_layout_matches_the_reference_header():
    def reference():
        ref = os.path.join(golden.SOURCE, "neural_speed")
        return _layout("core/ne.h", "ne_tensor", "ne_compute_params", list(ENUMS), [ref, f"{ref}/core"])

    golden.check("ne_abi.layout", _layout("ns_ne_abi.h", "ns_ne_tensor", "ns_ne_compute_params", list(ENUMS.values()), [f"{ROOT}/include"]),
                 reference)


def test_committed_layout_numbers():
    """the numbers the compile above produced here (x86-64 LP64): sizeof(struct ne_tensor) = 512, ne_compute_params = 56"""
    with tempfile.TemporaryDirectory() as d:
        src = os.path.join(d, "sz.c")
        open(src, "w").write('#include <stdio.h>\n#include <stddef.h>\n#include "ns_ne_abi.h"\nint main(void){printf("%zu %zu %zu %zu %zu %d %d\\n",'
                             'sizeof(struct ns_ne_tensor), sizeof(struct ns_ne_compute_params), offsetof(struct ns_ne_tensor, src0),'
                             'offsetof(struct ns_ne_tensor, n_tasks), offsetof(struct ns_ne_tensor, data), (int)NS_NE_TYPE_BTLA, (int)NS_NE_OP_MUL_QKV);return 0;}')
        exe = os.path.join(d, "sz")
        subprocess.run(["gcc", "-std=c11", f"-I{ROOT}/include", src, "-o", exe], check=True)
        out = subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()
    assert out == ["512", "56", "128", "432", "456", "19", "52"], out


def test_library_exports_the_graph_engine_entry_points():
    import neural_speed_b200 as ns
    L = ns.lib()
    for name in ("bestla_support", "bestla_backend_support", "bestla_parallel_for", "bestla_mul", "bestla_add", "bestla_layernormalization"):
        assert hasattr(L, name), name


def test_parallel_for_runs_the_three_phases_on_every_task():
    """bestla_parallel_for (ne_bestla.cpp:42-70): INIT once on task 0, then COMPUTE and FINALIZE on every task index, phases
    separated by barriers; nth == 1 runs inline.  Host logic only -- no GPU involved."""
    import neural_speed_b200 as ns
    L = ns.lib()

    class Params(C.Structure):
        _fields_ = [("type", C.c_int), ("ith", C.c_int), ("nth", C.c_int), ("wsize", C.c_size_t), ("wdata", C.c_void_p),
                    ("dev_wsize", C.c_size_t), ("dev_wdata", C.c_void_p), ("dev_queue", C.c_void_p)]

    assert C.sizeof(Params) == 56
    log = []
    import threading
    lock = threading.Lock()
    CB = C.CFUNCTYPE(None, C.POINTER(Params), C.c_void_p)

    def cb(p, node):
        with lock:
            log.append((p.contents.type, p.contents.ith, p.contents.nth))

    fn = CB(cb)
    L.bestla_parallel_for.argtypes = [CB, C.POINTER(Params), C.c_void_p]
    L.bestla_parallel_for.restype = None
    for nth in (1, 4):
        log.clear()
        p = Params(0, 0, nth, 0, None, 0, None, None)
        L.bestla_parallel_for(fn, C.byref(p), None)
        init = [e for e in log if e[0] == 0]
        comp = sorted(e[1] for e in log if e[0] == 1)
        fin = sorted(e[1] for e in log if e[0] == 2)
        assert init == [(0, 0, nth)]
        assert comp == list(range(nth)) and fin == list(range(nth))
        # phase order: INIT before any COMPUTE, every COMPUTE before any FINALIZE
        kinds = [e[0] for e in log]
        assert kinds == sorted(kinds)
