"""CPU tests of the drop-in boundary: the C-ABI library loads, exports every symbol that
include/knn_b200.h declares, and fails loudly (no CPU fallback) when there is no device."""
import ctypes
import os
import re
import subprocess
import sys
import textwrap
from pathlib import Path

import numpy as np
import pytest

REPO = Path(__file__).resolve().parent.parent


def _declared_symbols():
    text = (REPO / "include" / "knn_b200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(knn_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    import knn_b200

    lib = knn_b200._lib.load()
    declared = _declared_symbols()
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/knn_b200.h but not exported"
    # the ctypes table binds exactly the declared surface
    assert sorted(knn_b200._lib.SIGNATURES) == declared


def test_no_torch_types_in_abi():
    text = (REPO / "include" / "knn_b200.h").read_text()
    assert "torch" not in text and "at::" not in text and "#include <cuda" not in text


def test_alias_module_exposes_reference_surface():
    """Names the reference drivers touch: cath/search.py:15-24, seqvec_search/main.py:23-45,
    pfam/proteins_search.py:22-40, seqvec_search/create_index.py:41-47."""
    import faiss

    for name in ["METRIC_INNER_PRODUCT", "METRIC_L2", "normalize_L2", "IndexFlat", "IndexFlatIP", "IndexFlatL2",
                 "IndexLSH", "IndexHNSWFlat", "write_index", "read_index"]:
        assert hasattr(faiss, name), name
    assert faiss.METRIC_INNER_PRODUCT == 0 and faiss.METRIC_L2 == 1
    with pytest.raises(NotImplementedError):
        faiss.IndexLSH(1024, 1024)


def test_argument_errors_before_any_device_work():
    import knn_b200

    x = np.zeros((3, 8), np.float64)
    with pytest.raises(TypeError):
        knn_b200.normalize_L2(x)
    with pytest.raises(ValueError):
        knn_b200.normalize_L2(np.zeros((4, 8), np.float32)[:, ::2])
    with pytest.raises(ValueError):
        knn_b200.IndexFlat(8, 7)
    lib = knn_b200._lib.load()
    assert lib.knn_index_create(None, 8, 0, 0, 0) == -1
    assert b"invalid" in lib.knn_last_error()
    assert lib.knn_index_free(None) == 0


def test_fails_loudly_without_a_device():
    """In a child process with every CUDA device hidden, so that a machine with a GPU checks it too."""
    script = textwrap.dedent(f"""
        import sys
        sys.path.insert(0, {str(REPO / "knn-for-homology_b200")!r})
        import numpy as np
        import pytest
        import knn_b200
        with pytest.raises(knn_b200._lib.KnnError, match="no CPU fallback"):
            knn_b200.IndexFlat(16, 0)
        with pytest.raises(knn_b200._lib.KnnError):
            knn_b200.normalize_L2(np.ones((2, 4), np.float32))
        """)
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    subprocess.run([sys.executable, "-c", script], env=env, check=True, timeout=300)


def test_missing_library_is_an_import_error(monkeypatch, tmp_path):
    import knn_b200._lib as L

    monkeypatch.setattr(L, "_lib", None)
    monkeypatch.setattr(L, "LIB_PATH", tmp_path / "nope.so")
    with pytest.raises(ImportError, match="no CPU fallback"):
        L.load()


def test_product_never_imports_the_oracle():
    for p in (REPO / "knn-for-homology_b200").rglob("*"):
        if p.suffix in {".py", ".cu", ".cuh", ".h"}:
            assert "oracle" not in p.read_text().replace("see oracle/flat_oracle.py", "").replace(
                "oracle/flat_oracle.py", ""), p


def test_flat_index_file_byte_layout(tmp_path):
    """write_index / read_index on a host-side stand-in: the bytes of a faiss 1.7.x flat index file, field by
    field (fourcc, d, ntotal, two dummies of 1 << 20, is_trained, metric, vector count, float32 rows).  The
    layout is restated from upstream knowledge (no faiss in this image); this pins it against accidental change."""
    import struct

    import numpy as np

    from knn_b200 import io as kio

    class HostFlat:
        def __init__(self, d, metric):
            self.d, self.metric_type, self.rows = d, metric, np.empty((0, d), np.float32)

        ntotal = property(lambda self: self.rows.shape[0])

        def reconstruct_n(self, i0, n):
            return self.rows[i0:i0 + n]

        def add(self, x):
            self.rows = np.concatenate([self.rows, x])

    for metric, fourcc in [(0, b"IxFI"), (1, b"IxF2")]:
        src = HostFlat(3, metric)
        src.add(np.arange(6, dtype=np.float32).reshape(2, 3) / 4)
        path = tmp_path / f"m{metric}.index"
        kio.write_index(src, str(path))
        raw = path.read_bytes()
        want = (fourcc + struct.pack("<i", 3) + struct.pack("<q", 2) + struct.pack("<qq", 1 << 20, 1 << 20) + b"\x01"
                + struct.pack("<i", metric) + struct.pack("<Q", 6) + (np.arange(6, dtype="<f4") / 4).tobytes())
        assert raw == want and len(raw) == 4 + 4 + 8 + 16 + 1 + 4 + 8 + 24
        back = kio.read_index(str(path), index_factory=HostFlat)
        assert (back.d, back.ntotal, back.metric_type) == (3, 2, metric) and np.array_equal(back.rows, src.rows)
    (tmp_path / "bad").write_bytes(b"IxHN" + b"\0" * 60)
    with pytest.raises(NotImplementedError):
        kio.read_index(str(tmp_path / "bad"), index_factory=HostFlat)
    with pytest.raises(TypeError):
        kio.write_index(object(), str(tmp_path / "x"))
