"""16-bit (fp16 / bf16) inputs without an fp32 copy, the parts that need no GPU: the header declares the typed entry
points and the dtype codes, the built library exports them, the Python layer routes every input to the right entry
point with the right dtype code and hands 16-bit rows over without converting them, and the sharded index's query
upload keeps their dtype.  The kernels and the bit-equality contract are covered by tests/test_gpu_h16_inputs.py."""
import ctypes
import os
import re
import socket
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

REPO = Path(__file__).resolve().parent.parent
HEADER = (REPO / "include" / "knn_b200.h").read_text()
TYPED = ["knn_index_add_typed", "knn_index_add_typed_dev", "knn_index_search_typed", "knn_index_search_typed_dev",
         "knn_index_search_begin_typed_dev", "knn_index_search_filter_typed_dev", "knn_index_search_finish_typed_dev"]


def test_header_declares_dtype_codes_and_typed_entry_points():
    codes = dict(re.findall(r"#define (KNN_DTYPE_\w+) (\d+)", HEADER))
    assert codes == {"KNN_DTYPE_F32": "0", "KNN_DTYPE_F16": "1", "KNN_DTYPE_BF16": "2"}
    for name in TYPED:
        m = re.search(r"\bint %s\(([^)]*)\);" % name, HEADER)
        assert m, "%s is not declared" % name
        args = " ".join(m.group(1).split())
        assert "const void*" in args and "int dtype" in args, (name, args)
    # the fp32 entry points keep their signatures
    for decl in ["int knn_index_add(knn_index* idx, int64_t n, const float* x);",
                 "int knn_index_search(knn_index* idx, int64_t nq, const float* xq, int64_t k, float* D, int64_t* I);"]:
        assert decl in HEADER


def test_python_dtype_codes_match_the_header():
    from knn_b200 import _lib

    codes = dict(re.findall(r"#define (KNN_DTYPE_\w+) (\d+)", HEADER))
    assert (_lib.DTYPE_F32, _lib.DTYPE_F16, _lib.DTYPE_BF16) == tuple(int(codes["KNN_DTYPE_" + s]) for s in ("F32", "F16", "BF16"))
    for name in TYPED:
        assert name in _lib.SIGNATURES


def test_library_exports_typed_entry_points():
    from knn_b200 import _lib

    if not _lib.LIB_PATH.exists():
        pytest.skip("libknn_b200.so is not built")
    lib = ctypes.CDLL(str(_lib.LIB_PATH))
    for name in TYPED + ["knn_index_add", "knn_index_add_dev", "knn_index_search", "knn_index_search_dev",
                         "knn_index_search_begin_dev", "knn_index_search_filter_dev", "knn_index_search_finish_dev"]:
        assert hasattr(lib, name), name


# ---- Python dtype routing against a stub library ---------------------------------------------------------------
class _StubLib:
    """Records the calls IndexFlat makes (and, with `snap`, the first `snap` bytes at the row address of the call,
    read while the rows are still alive); every call succeeds."""

    def __init__(self, snap=0):
        self.calls, self.snap, self.bytes = [], snap, []

    def __getattr__(self, name):
        if not name.startswith("knn_"):
            raise AttributeError(name)

        def call(*args):
            self.calls.append((name, args))
            if self.snap:
                self.bytes.append(ctypes.string_at(args[2], self.snap))
            return 0

        return call


def _stub_index(d=8, snap=0):
    from knn_b200.index import IndexFlat

    idx = IndexFlat.__new__(IndexFlat)  # no library, no device
    idx._lib, idx._h, idx.d, idx.metric_type, idx.device = _StubLib(snap), ctypes.c_void_p(1), d, 0, 0
    return idx


def _host_inputs(n=5, d=8):
    rng = np.random.default_rng(0)
    x = rng.standard_normal((n, d)).astype(np.float32)
    return {
        "np_f16": (x.astype(np.float16), 1),
        "torch_f16": (torch.from_numpy(x).to(torch.float16), 1),
        "torch_bf16": (torch.from_numpy(x).to(torch.bfloat16), 2),
    }


@pytest.mark.parametrize("kind", ["np_f16", "torch_f16", "torch_bf16"])
def test_host_16bit_rows_pass_through_without_a_copy(kind):
    x, code = _host_inputs()[kind]
    ptr = x.ctypes.data if isinstance(x, np.ndarray) else x.data_ptr()
    idx = _stub_index()
    idx.add(x)
    idx.search(x, 3)
    (add_name, add_args), (search_name, search_args) = idx._lib.calls
    assert add_name == "knn_index_add_typed" and add_args[1:] == (5, ptr, code)
    assert search_name == "knn_index_search_typed" and search_args[1:5] == (5, ptr, code, 3)


@pytest.mark.parametrize("kind", ["np_f16", "torch_f16", "torch_bf16"])
def test_non_contiguous_16bit_rows_are_made_contiguous_not_converted(kind):
    x, code = _host_inputs(n=10)[kind]
    view = x[::2]
    idx = _stub_index(snap=5 * 8 * 2)
    idx.add(view)
    name, args = idx._lib.calls[0]
    assert name == "knn_index_add_typed" and args[1] == 5 and args[3] == code
    # the rows handed over are the view's rows, in the view's dtype
    got = idx._lib.bytes[0]
    want = np.ascontiguousarray(view).tobytes() if isinstance(view, np.ndarray) else view.contiguous().view(torch.int16).numpy().tobytes()
    assert got == want


@pytest.mark.parametrize("dtype", [np.float32, np.float64, np.int32])
def test_other_host_dtypes_become_float32(dtype):
    x = np.arange(40).reshape(5, 8).astype(dtype)
    idx = _stub_index(snap=5 * 8 * 4)
    idx.add(x)
    name, args = idx._lib.calls[0]
    assert name == "knn_index_add_typed" and args[3] == 0
    assert np.array_equal(np.frombuffer(idx._lib.bytes[0], np.float32).reshape(5, 8), x.astype(np.float32))
    if dtype is np.float32:
        assert args[2] == x.ctypes.data  # contiguous float32: no copy, as before


def test_search_into_passes_the_dtype():
    idx = _stub_index()
    idx.search_into(1234, 7, 5, 11, 22, dtype=2)
    idx.search_into(1234, 7, 5, 11, 22)
    assert idx._lib.calls == [("knn_index_search_typed", (idx._h, 7, 1234, 2, 5, 11, 22)),
                              ("knn_index_search_typed", (idx._h, 7, 1234, 0, 5, 11, 22))]


def test_normalize_l2_still_refuses_16bit_arrays():
    from knn_b200.index import normalize_L2

    with pytest.raises(TypeError):
        normalize_L2(np.ones((3, 4), np.float16))


def test_cpu_float32_tensor_is_still_refused():
    """Only 16-bit CPU tensors take the host path (numpy has no bf16); other CPU tensors are refused as before."""
    idx = _stub_index()
    with pytest.raises(ValueError, match="cuda"):
        idx.add(torch.ones((2, 8)))


# ---- sharded query upload keeps the dtype (gloo, CPU) ----------------------------------------------------------
class _NoShard:
    device = 0
    ntotal = 0


def _upload_worker(rank, world, port, out):
    sys.path.insert(0, str(REPO))
    sys.path.insert(0, str(REPO / "knn-for-homology_b200"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist

    dist.init_process_group("gloo", rank=rank, world_size=world)
    from knn_b200.distributed import ShardedIndexFlat

    index = ShardedIndexFlat(8, 0, index_factory=_NoShard)
    x = torch.randn(11, 8, generator=torch.Generator().manual_seed(3))  # every rank holds the same queries
    for src, want in [(x.to(torch.float16).numpy(), torch.float16), (x.to(torch.bfloat16), torch.bfloat16),
                      (x.to(torch.float16), torch.float16), (x.numpy(), torch.float32), (x.double().numpy(), torch.float32)]:
        got = index.upload_queries(src)
        ref = torch.from_numpy(src) if isinstance(src, np.ndarray) else src
        assert got.dtype == want, (type(src), got.dtype)
        assert torch.equal(got, ref.to(want)), type(src)
    if rank == 0:
        Path(out).write_text("ok")
    dist.destroy_process_group()


def test_upload_queries_keeps_16bit_dtypes_world2_gloo(tmp_path):
    import torch.multiprocessing as mp

    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    out = tmp_path / "ok"
    mp.spawn(_upload_worker, args=(2, port, str(out)), nprocs=2, join=True)
    assert out.read_text() == "ok"
