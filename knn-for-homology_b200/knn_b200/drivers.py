"""The reference's driver functions around the flat search (SURVEY.md section 8 rows a7-a10), with the
same names, arguments, return values and files - but ONE upload of the embeddings: normalisation,
index build and search all run on the device copy, where the reference (and a plain faiss alias)
crosses the host/device boundary for every step (normalize_L2: up and down, add: up, search: up).

  search            cath/search.py:13-26
  search_and_save   cath/search.py:29-53
  faiss_search      seqvec_search/main.py:22-50
  proteins_search   pfam/proteins_search.py:11-57 (flat branch)
  create_index      seqvec_search/create_index.py:16-47 (index build + persist; flat index instead of LSH)

Results are bit-identical to calling the faiss-style API step by step (same kernels, same order).
"""
from __future__ import annotations

import time
from pathlib import Path

import numpy as np

from .index import METRIC_INNER_PRODUCT, METRIC_L2, IndexFlat, _default_device, normalize_L2
from .io import write_index

# What users of the approximate branches get (SURVEY.md section 8 f5): the exact index answers every query the
# approximate ones answer, with better neighbours, and on this hardware faster than a Hamming scan would
# (DESIGN.md section 8) - so the message points there instead of failing silently or returning other results.
APPROXIMATE_INDEX_HINT = ("%s is an approximate index and not part of this engine (its codes depend on faiss's own random "
                          "rotation, so results could never match the reference's); use the exact 'flat' index - on a "
                          "B200 it is faster than the Hamming scan it would replace")


_CHUNK_BYTES = 64 << 20
_pinned = {}


def _pinned_pair(device: int):
    """Two page-locked 64 MB bounce buffers per device: pageable numpy memory <-> device in chunks, the (multi-threaded)
    host copy of chunk i + 1 under the DMA of chunk i.  A plain pageable cudaMemcpy stages through the driver's own
    buffers on one thread; the drivers move gigabytes both ways (the reference's in-place normalisation is written back
    to the caller's arrays), which is most of their wall time once the search takes a fraction of a second."""
    import torch

    if device not in _pinned:
        _pinned[device] = [torch.empty(_CHUNK_BYTES, dtype=torch.uint8, pin_memory=True) for _ in range(2)]
    return _pinned[device]


def _upload(x: np.ndarray, device: int):
    """Host matrix -> a device tensor of the same values: float16 stays float16 (half the PCIe bytes; the device
    up-converts, exactly, where the caller needs float32), any other dtype becomes float32."""
    import torch

    x = np.ascontiguousarray(x, dtype=None if x.dtype == np.float16 else np.float32)
    dev = torch.device("cuda", device)
    if x.nbytes < 2 * _CHUNK_BYTES:
        return torch.from_numpy(x).to(dev)
    src = torch.from_numpy(x)
    out = torch.empty(x.shape, dtype=src.dtype, device=dev)
    src, dst = src.view(-1), out.view(-1)
    n = _CHUNK_BYTES // src.element_size()
    bufs = [b.view(src.dtype) for b in _pinned_pair(device)]
    done = [torch.cuda.Event(), torch.cuda.Event()]
    for c, i in enumerate(range(0, src.numel(), n)):
        w = c & 1
        m = min(n, src.numel() - i)
        if c >= 2:
            done[w].synchronize()
        bufs[w][:m].copy_(src[i:i + m])
        dst[i:i + m].copy_(bufs[w][:m], non_blocking=True)
        done[w].record()
    return out


def _download_into(host: np.ndarray, dev_tensor) -> None:
    """Device tensor -> the caller's (pageable) numpy memory, chunked through the pinned pair."""
    import torch

    t = dev_tensor.contiguous().view(-1)
    if host.nbytes < 2 * _CHUNK_BYTES or not host.flags.c_contiguous:
        torch.from_numpy(host).copy_(dev_tensor)
        return
    dst = torch.from_numpy(host).view(-1)
    n = _CHUNK_BYTES // t.element_size()
    bufs = [b.view(t.dtype) for b in _pinned_pair(dev_tensor.device.index)]
    done = [torch.cuda.Event(), torch.cuda.Event()]
    chunks = list(range(0, t.numel(), n))
    for c, i in enumerate(chunks):  # D2H of chunk c is in flight while chunk c - 1 is copied out on the host
        w = c & 1
        m = min(n, t.numel() - i)
        bufs[w][:m].copy_(t[i:i + m], non_blocking=True)
        done[w].record()
        if c >= 1:
            j = chunks[c - 1]
            mj = min(n, t.numel() - j)
            done[w ^ 1].synchronize()
            dst[j:j + mj].copy_(bufs[w ^ 1][:mj])
    j = chunks[-1]
    mj = min(n, t.numel() - j)
    done[(len(chunks) - 1) & 1].synchronize()
    dst[j:j + mj].copy_(bufs[(len(chunks) - 1) & 1][:mj])


def _to_host(dev_tensor) -> np.ndarray:
    import torch

    out = np.empty(tuple(dev_tensor.shape), dtype={torch.float32: np.float32, torch.int64: np.int64}[dev_tensor.dtype])
    _download_into(out, dev_tensor)
    return out


def search(embeddings: np.ndarray, hits: int = 10, metric: int = METRIC_INNER_PRODUCT, device: int | None = None,
           index: IndexFlat | None = None):
    """All-vs-all search; one more hit is searched internally because the first one is the self hit
    (cath/search.py:16).  The caller's array is not modified (the reference normalises a copy).
    ``index``: an IndexFlat of the same width and metric to reuse (it is reset first): a loop over many matrices
    then pays for the device storage and the ~1 GB of search workspaces once instead of once per matrix."""
    device = _default_device() if device is None else device
    # float16 embeddings cross PCIe as they are and are up-converted on the device (exact): normalisation runs in
    # float32, as the reference's does after its host-side cast (cath/search.py:39-40)
    x = _upload(embeddings, device).float()
    if metric == METRIC_INNER_PRODUCT:
        normalize_L2(x)
    if index is None:
        index = IndexFlat(x.shape[1], metric, device=device)
    else:
        assert (index.d, index.metric_type) == (x.shape[1], metric), "reused index has another width or metric"
        index.reset()
    index.add(x)
    scores, results = index.search(x, hits + 1)
    scores, results = _to_host(scores), _to_host(results)
    # Remove the self hit (blindly column 0, like cath/search.py:26)
    return results[:, 1:], scores[:, 1:]


def search_and_save(cath_data: Path, device: int | None = None) -> None:
    """cath/search.py:29-53: both metrics over every *.npy of the directory; writes
    `<stem>.<metric>-search-time.txt`, `hits_<metric>.npz` and `scores_<metric>.npz`."""
    cath_data = Path(cath_data)
    for name, metric in [("Cosine", METRIC_INNER_PRODUCT), ("Euclidean", METRIC_L2)]:
        print(f"Searching with {name}")
        hits, scores = {}, {}
        indexes = {}  # one index per embedding width, reused across the files (the embedders differ in width)
        for file_path in sorted(cath_data.glob("*.npy")):
            # fp16 embeddings of the half precision model stay fp16 on the host: `search` uploads them as they are and
            # casts to fp32 on the device, with the same values as the reference's host-side cast (cath/search.py:39-40)
            embeddings = np.load(file_path)
            if embeddings.dtype != np.float16:
                embeddings = embeddings.astype(np.float32)
            print(file_path.stem, embeddings.shape)
            start = time.time()
            if embeddings.shape[1] not in indexes:
                indexes[embeddings.shape[1]] = IndexFlat(embeddings.shape[1], metric,
                                                         device=_default_device() if device is None else device)
            hits[file_path.stem], scores[file_path.stem] = search(embeddings, metric=metric, device=device,
                                                                  index=indexes[embeddings.shape[1]])
            end = time.time()
            print(end - start)
            cath_data.joinpath(file_path.with_suffix(f".{name.lower()}-search-time.txt")).write_text(str(end - start))
        np.savez(cath_data.joinpath(f"hits_{name.lower()}.npz"), **hits)
        np.savez(cath_data.joinpath(f"scores_{name.lower()}.npz"), **scores)


def faiss_search(haystack, queries: np.ndarray, hits: int = 13, metric: int = METRIC_INNER_PRODUCT, device: int | None = None):
    """seqvec_search/main.py:22-50.  ``haystack`` is a matrix or a ready index.  Returns
    ``(ids, scores, search_seconds)`` - ids first.  Like the reference, queries (and a matrix
    haystack) are L2-normalised IN PLACE for the inner-product metric."""
    import threading

    import torch

    device = _default_device() if device is None else device
    q = _upload(queries, device).float()  # float32 on the device, as the in-place normalisation needs
    if metric == METRIC_INNER_PRODUCT:
        normalize_L2(q)
        _write_back(queries, q)
    writer = None
    if isinstance(haystack, np.ndarray):
        h = _upload(haystack, device).float()
        if metric == METRIC_INNER_PRODUCT:
            normalize_L2(h)
            if haystack.dtype != np.float32 or not haystack.flags.c_contiguous:
                raise TypeError("normalize_L2 expects a C-contiguous float32 array (it normalises in place)")
            # The reference's in-place normalisation has to reach the caller's array (main.py:34), gigabytes over PCIe
            # that nothing below depends on: they travel on a side stream, driven by a helper thread, while the index
            # is built and searched, and are home before this function returns.
            ready = torch.cuda.Event()
            ready.record(torch.cuda.current_stream(device))
            writer = threading.Thread(target=_write_back_async, args=(haystack, h, device, ready), daemon=True)
            writer.start()
        index = IndexFlat(h.shape[1], metric, device=device)
        index.train(h)
        index.add(h)
    else:
        index = haystack
    torch.cuda.current_stream(device).synchronize()
    start = time.time()
    scores, result = index.search(q, hits)
    if writer is not None:  # the bounce buffers are shared: the results travel after the write-back
        torch.cuda.current_stream(device).synchronize()
        writer.join()
    scores, result = _to_host(scores), _to_host(result)
    search_time = time.time() - start  # like faiss's index.search: until (D, I) are numpy arrays
    if _write_back_error:
        raise _write_back_error.pop()
    return result, scores, search_time


_write_back_error = []


def _write_back_async(host: np.ndarray, dev, device: int, ready) -> None:
    import torch

    try:
        torch.cuda.set_device(device)
        side = torch.cuda.Stream(device=device)
        side.wait_event(ready)
        with torch.cuda.stream(side):
            _download_into(host, dev)
        side.synchronize()
    except Exception as e:  # surfaced by the caller
        _write_back_error.append(e)


def _write_back(host: np.ndarray, dev) -> None:
    """faiss.normalize_L2 mutates the caller's float32 C-contiguous array; anything else it refuses."""
    if host.dtype != np.float32 or not host.flags.c_contiguous:
        raise TypeError("normalize_L2 expects a C-contiguous float32 array (it normalises in place)")
    _download_into(host, dev)  # device -> the caller's memory directly (no intermediate host array)


def proteins_search(full_sequences_data: Path, index_mode: str = "flat", k: int = 1000, device: int | None = None):
    """pfam/proteins_search.py:11-57, flat branch: `full_sequences.npy` -> `full_sequences_flat.index`,
    `full_sequences_flat_scores.npy`, `full_sequences_flat_hits.npy` in the same directory."""
    if index_mode != "flat":
        raise ValueError(APPROXIMATE_INDEX_HINT % {"lsh": "IndexLSH", "hnsw": "IndexHNSWFlat"}.get(index_mode, repr(index_mode)))
    device = _default_device() if device is None else device
    full_sequences_data = Path(full_sequences_data)
    npy = full_sequences_data.joinpath("full_sequences.npy")
    embeddings = np.load(npy)
    if embeddings.dtype != np.float16:  # fp16 is uploaded as it is and cast on the device (same values, half the bytes)
        embeddings = embeddings.astype(np.float32)
    print("full_sequences", embeddings.shape)
    start = time.time()
    x = _upload(embeddings, device).float()
    normalize_L2(x)
    index = IndexFlat(x.shape[1], METRIC_INNER_PRODUCT, device=device)
    index.train(x)
    index.add(x)
    print(f"Index creation took {int(time.time() - start)}s")
    index_file = full_sequences_data.joinpath(f"full_sequences_{index_mode}.index")
    write_index(index, str(index_file))
    start = time.time()
    flat_scores, flat_hits = index.search(x, k)
    flat_scores, flat_hits = _to_host(flat_scores), _to_host(flat_hits)
    print(f"Search took {int(time.time() - start)}s")
    np.save(full_sequences_data.joinpath(f"full_sequences_{index_mode}_scores.npy"), flat_scores)
    np.save(full_sequences_data.joinpath(f"full_sequences_{index_mode}_hits.npy"), flat_hits)
    return flat_scores, flat_hits


def create_index(args=None):
    """seqvec_search/create_index.py:16-47: `<dir>/train.npy` -> an index file that `main.py --knn-index`
    (seqvec_search/main.py:131-132: `faiss.read_index`) loads and hands to `faiss_search`.

    Same command line (`--dir`, `--index`, `--param`).  The reference builds an `IndexLSH(d, param)` here; this engine
    is the exact one, so the file written is a FLAT inner-product index (`IxFI`, faiss's on-disk format): `--param`
    (LSH bits) is accepted and has no meaning for it.  `faiss_search` normalises a matrix haystack in place before
    adding it (main.py:34) but takes a ready index as it is, so the rows are L2-normalised here, on the device, before
    they are added - searching the file gives exactly what searching `train.npy` gives.  `--kind lsh` raises.
    Returns the index (the reference returns None)."""
    import argparse
    import logging

    logger = logging.getLogger(__name__)
    parser = argparse.ArgumentParser()
    parser.add_argument("--dir", type=Path, default=Path(), help="The name of the directory containing the database")
    parser.add_argument("--index", type=Path, required=True, help="The location to write the index to")
    parser.add_argument("--param", type=int, default=1024,
                        help="The tuning parameter of the (LSH) index of the reference; ignored by the exact flat index")
    parser.add_argument("--kind", default="flat", choices=["flat", "lsh"], help="flat: exact index (this engine)")
    parser.add_argument("--device", type=int, default=None)
    args = parser.parse_args(args)
    if args.kind != "flat":
        raise NotImplementedError(APPROXIMATE_INDEX_HINT % "IndexLSH")
    device = _default_device() if args.device is None else args.device
    logger.info(f"Loading database from {args.dir.joinpath('train.npy')}")
    embeddings = np.load(str(args.dir.joinpath("train.npy")))
    logger.info(f"Building exact flat index on {embeddings.shape}")
    x = _upload(embeddings, device).float()
    normalize_L2(x)
    index = IndexFlat(x.shape[1], METRIC_INNER_PRODUCT, device=device)
    index.train(x)
    index.add(x)
    logger.info("Writing out the flat index")
    write_index(index, str(args.index))
    return index
