"""Local tensor sources with the part of HFMultiModelIndex's interface (shard/index.py:60-276)
that the merge path calls: add_model, model_indexes, get_model_keys, get_layer_order,
get_tensor -> promise, preload_tensor.  Network download, claim counting and the HF cache
layout are out of scope (SURVEY.md section 2 rows 5/6); a reference HFMultiModelIndex instance
can be passed to FourierMerge instead of these classes.

  InMemoryIndex        tensors handed over as dicts (tests, benchmarks, synthetic models)
  LocalSafetensorsIndex {storage_dir}/{org}/{model}/model.safetensors.index.json + shards on disk,
                       read lazily, uploaded with pinned staging, nothing kept after use
                       (the reference keeps every tensor it ever read in RAM, index.py:79,265);
                       or a PEFT LoRA adapter directory (shardmerge_b200/lora.py), bound to a base.
"""
from __future__ import annotations

import json
import re
from pathlib import Path
from typing import Dict, List, Optional, Set

import torch

from . import lora


class TensorPromise:
    """Awaitable handle for one tensor (interface of shard/index.py:38-58)."""

    def __init__(self, model_uri: str, tensor_name: str, device: str, loader):
        self.model_uri, self.tensor_name, self.device = model_uri, tensor_name, device
        self._loader = loader

    async def get(self) -> torch.Tensor:
        return self._loader()


def canonical_layer_order(names) -> List[str]:
    """embed_tokens, then model.layers.<n>.<component> by (n, component name as discovered on layer 0),
    then model.norm.weight, lm_head, then everything else sorted (shard/index.py:132-187)."""
    names = list(names)
    embed = sorted(n for n in names if "embed_tokens" in n)
    layer = [n for n in names if "layers." in n]
    norm = sorted(n for n in names if "model.norm.weight" in n)
    head = sorted(n for n in names if "lm_head" in n)
    claimed = set(embed) | set(layer) | set(norm) | set(head)
    other = sorted(n for n in names if n not in claimed)
    numbers = sorted({int(n.split("layers.")[1].split(".")[0]) for n in layer})
    prefix0 = "model.layers.0."
    components = sorted(n[len(prefix0):] for n in layer if n.startswith(prefix0))
    ordered_layers = [f"model.layers.{i}.{c}" for i in numbers for c in components]
    ordered = embed + ordered_layers + norm + head + other
    if set(ordered) != set(names):
        raise ValueError(f"Weight ordering mismatch! Missing: {set(names) - set(ordered)}, Extra: {set(ordered) - set(names)}")
    return ordered


class _IndexBase:
    def __init__(self):
        self.model_indexes: Dict[str, dict] = {}
        self._order: Dict[str, List[str]] = {}
        self._prefetched: dict = {}
        self._copy_streams: dict = {}
        self.copy_events = None          # set to a list to collect (start, end) CUDA events of every upload (bench.py)

    def _register(self, model_uri: str, index: dict):
        self.model_indexes[model_uri] = index
        self._order[model_uri] = canonical_layer_order(index["weight_map"].keys())

    def get_model_keys(self, model_uri: str) -> Set[str]:
        return set(self.model_indexes[model_uri]["weight_map"].keys())

    def get_layer_order(self, model_uri: str) -> List[str]:
        return list(self._order[model_uri])

    async def preload_tensor(self, model_uri: str, tensor_name: str):
        return None

    # ---- one-tensor-ahead upload (SURVEY.md 8f N2) ------------------------------------------------------
    # The reference loads a tensor when _merge_layer asks for it, synchronously (shard/index.py:238-270), so the
    # GPU idles during every host-to-device copy.  prefetch() starts the copy of a tensor the merge loop will ask
    # for next on a dedicated copy stream; the matching get_tensor(...).get() hands the device tensor over after
    # making the caller's stream wait for the copy.
    def _host_tensor(self, model_uri: str, tensor_name: str) -> torch.Tensor:
        raise NotImplementedError

    def prefetch(self, model_uri: str, tensor_name: str, device: str):
        dev = torch.device(device)
        if dev.type != "cuda":
            return
        key = (model_uri, tensor_name, str(dev))
        if key in self._prefetched:
            return
        host = self._host_tensor(model_uri, tensor_name)
        if host.device.type == "cuda":
            return
        if not host.is_pinned():
            host = host.pin_memory()
        stream = self._copy_streams.get(str(dev))
        if stream is None:
            stream = self._copy_streams[str(dev)] = torch.cuda.Stream(device=dev)
        with torch.cuda.stream(stream):
            if self.copy_events is not None:
                e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
                e0.record(stream)
            t = host.to(dev, non_blocking=True)
            if self.copy_events is not None:
                e1.record(stream)
                self.copy_events.append((e0, e1))
            ev = stream.record_event()
        self._prefetched[key] = (t, ev, host)

    def _take_prefetched(self, model_uri: str, tensor_name: str, device: str):
        ent = self._prefetched.pop((model_uri, tensor_name, str(torch.device(device))), None)
        if ent is None:
            return None
        t, ev, _host = ent
        cur = torch.cuda.current_stream(t.device)
        cur.wait_event(ev)
        t.record_stream(cur)
        return t


class InMemoryIndex(_IndexBase):
    """models: {model_uri: {tensor_name: tensor}}; `shard_of(tensor_name) -> file name` lays out the
    output shards (default: one shard per transformer layer, like HF checkpoints roughly do)."""

    def __init__(self, models: Dict[str, Dict[str, torch.Tensor]], shard_of=None):
        super().__init__()
        self.models = models
        self._shard_of = shard_of or _default_shard_of

    async def add_model(self, model_uri: str, revision: str = "main"):
        if model_uri in self.model_indexes:
            return
        tensors = self.models[model_uri]
        self._register(model_uri, {"metadata": {"total_size": sum(t.numel() * t.element_size() for t in tensors.values())},
                                   "weight_map": {n: self._shard_of(n) for n in tensors}})

    def tensor_numels(self, model_uri: str) -> Dict[str, int]:
        return {n: t.numel() for n, t in self.models[model_uri].items()}

    def tensor_shapes(self, model_uri: str) -> Dict[str, tuple]:
        return {n: tuple(t.shape) for n, t in self.models[model_uri].items()}

    def _host_tensor(self, model_uri: str, tensor_name: str) -> torch.Tensor:
        return self.models[model_uri][tensor_name]

    def get_tensor(self, model_uri: str, tensor_name: str, device: str = "cpu") -> TensorPromise:
        t = self.models[model_uri][tensor_name]

        def load():
            if str(t.device) == str(device):
                return t
            pre = self._take_prefetched(model_uri, tensor_name, device)
            return pre if pre is not None else t.to(device, non_blocking=t.is_pinned())

        return TensorPromise(model_uri, tensor_name, device, load)


def _default_shard_of(name: str) -> str:
    m = re.match(r"model\.layers\.(\d+)\.", name)
    return f"model-layer{int(m.group(1)):05d}.safetensors" if m else "model-misc.safetensors"


_ST_TO_TORCH = {"BOOL": torch.bool, "U8": torch.uint8, "I8": torch.int8, "F8_E5M2": torch.float8_e5m2, "F8_E4M3": torch.float8_e4m3fn,
                "I16": torch.int16, "U16": torch.uint16, "F16": torch.float16, "BF16": torch.bfloat16, "I32": torch.int32,
                "U32": torch.uint32, "F32": torch.float32, "F64": torch.float64, "I64": torch.int64, "U64": torch.uint64}


class LocalSafetensorsIndex(_IndexBase):
    """Models stored under storage_dir/<model_uri>/ as model.safetensors.index.json + shard files
    (the layout the reference's DownloadManager leaves behind, shard/index.py:88-95).

    Reader side of SURVEY.md 8f N2.  The reference reads a tensor when `_merge_layer` asks for it (safe_open().get_tensor,
    shard/index.py:261-266), keeps every tensor it ever read (:79, :265) and uploads it with a pageable copy.  Here
    `prefetch()` hands the tensor to a reader thread: a positional read straight from the safetensors file (header parsed
    once per shard) into a POOLED pinned buffer, then the host-to-device copy on a copy stream, issued from that thread --
    file read, upload and the merge kernels of earlier tensors overlap, nothing is pinned per tensor and nothing is kept."""

    def __init__(self, storage_dir, reader_threads: int = 8):
        super().__init__()
        self.storage_dir = Path(storage_dir)
        self._shard_meta: Dict[str, tuple] = {}          # shard path -> (data start, {name: (dtype, shape, begin, end)})
        self._reader_threads = reader_threads
        self._readers = None
        self._pin_free: Dict[int, list] = {}             # pinned buffers by size
        self._pin_busy: list = []                        # (event, buffer): handed back once the upload has finished
        self._adapters: Dict[str, lora.Adapter] = {}     # adapter model uri -> its parsed config and header
        import threading
        self._pin_lock = threading.Lock()

    async def add_model(self, model_uri: str, revision: str = "main"):
        if model_uri in self.model_indexes or model_uri in self._adapters:
            return
        directory = self.storage_dir / model_uri
        path = directory / "model.safetensors.index.json"
        if not path.exists() and lora.is_adapter_dir(directory):
            _, entries = self._meta(directory / lora.WEIGHTS_FILE)
            self._adapters[model_uri] = lora.Adapter(model_uri, lora.read_config(directory),
                                                     {k: (d, s) for k, (d, s, _, _) in entries.items()})
            return
        if not path.exists():
            raise FileNotFoundError(f"{path} not found (shardmerge_b200 does not download models)")
        with open(path) as fh:
            self._register(model_uri, json.load(fh))

    # ---- LoRA adapters ---------------------------------------------------------------------------------------
    # An adapter has no tensors under base names: once bound to a base it reports that base's keys, order and shapes.
    # `prefetch(adapter, name)` uploads only the factors or the full replacement of `name` (the keys of
    # adapter_part(adapter, name)), and `get_tensor(adapter, key)` hands each over by its key in the adapter's file.
    def is_adapter(self, model_uri: str) -> bool:
        return model_uri in self._adapters

    def bind_adapter(self, model_uri: str, base_uri: str):
        """Bind an added adapter to the added full model `base_uri`; raises lora.UnsupportedAdapter."""
        if base_uri in self._adapters:
            raise lora.UnsupportedAdapter(f"adapter {model_uri}: its base {base_uri} is an adapter, not a full model")
        self._adapters[model_uri].bind(base_uri, self.tensor_shapes(base_uri))
        self.model_indexes[model_uri] = self.model_indexes[base_uri]
        self._order[model_uri] = self._order[base_uri]

    def adapter_part(self, model_uri: str, tensor_name: str) -> Optional[lora.Part]:
        """How `model_uri`'s `tensor_name` is formed when `model_uri` is a bound adapter, else None."""
        adapter = self._adapters.get(model_uri)
        return None if adapter is None else adapter.part(tensor_name)

    # ---- safetensors headers ---------------------------------------------------------------------------------
    def _meta(self, shard: Path) -> tuple:
        key = str(shard)
        meta = self._shard_meta.get(key)
        if meta is None:
            import struct
            with open(shard, "rb") as fh:
                (n,) = struct.unpack("<Q", fh.read(8))
                header = json.loads(fh.read(n))
            entries = {k: (_ST_TO_TORCH[v["dtype"]], tuple(v["shape"]), v["data_offsets"][0], v["data_offsets"][1])
                       for k, v in header.items() if k != "__metadata__"}
            meta = self._shard_meta[key] = (8 + n, entries)
        return meta

    def _shard_of(self, model_uri: str, tensor_name: str) -> Path:
        adapter = self._adapters.get(model_uri)
        if adapter is not None:
            if tensor_name not in adapter.tensors:
                raise KeyError(f"Tensor {tensor_name} not found in adapter {model_uri}")
            return self.storage_dir / model_uri / lora.WEIGHTS_FILE
        index = self.model_indexes[model_uri]
        if tensor_name not in index["weight_map"]:
            raise KeyError(f"Tensor {tensor_name} not found in model {model_uri}")
        return self.storage_dir / model_uri / index["weight_map"][tensor_name]

    def tensor_shapes(self, model_uri: str) -> Dict[str, tuple]:
        """shapes from the safetensors headers (no tensor data is read); a bound adapter has its base's."""
        if model_uri in self._adapters:
            return self.tensor_shapes(self._adapters[model_uri].base)
        out: Dict[str, tuple] = {}
        index = self.model_indexes[model_uri]
        for shard in sorted(set(index["weight_map"].values())):
            for key, (_, shape, _, _) in self._meta(self.storage_dir / model_uri / shard)[1].items():
                out[key] = shape
        return out

    def tensor_numels(self, model_uri: str) -> Dict[str, int]:
        """element counts from the safetensors headers (no tensor data is read)."""
        out: Dict[str, int] = {}
        for key, shape in self.tensor_shapes(model_uri).items():
            n = 1
            for d in shape:
                n *= d
            out[key] = n
        return out

    # ---- reads -----------------------------------------------------------------------------------------------
    def _read_into(self, model_uri: str, tensor_name: str, buf: torch.Tensor) -> torch.Tensor:
        """Fill `buf` (uint8, >= the tensor's bytes) from the file -> typed view of it."""
        import os
        shard = self._shard_of(model_uri, tensor_name)
        start, entries = self._meta(shard)
        dtype, shape, b0, b1 = entries[tensor_name]
        n = b1 - b0
        view = memoryview(buf[:n].numpy()) if n else memoryview(b"")
        fd = os.open(str(shard), os.O_RDONLY)
        try:
            done = 0
            while done < n:
                got = os.preadv(fd, [view[done:]], start + b0 + done)
                if got <= 0:
                    raise IOError(f"short read of {tensor_name} from {shard}")
                done += got
        finally:
            os.close(fd)
        return buf[:n].view(dtype).reshape(shape)

    def _host_tensor(self, model_uri: str, tensor_name: str) -> torch.Tensor:
        shard = self._shard_of(model_uri, tensor_name)
        _, entries = self._meta(shard)
        _, _, b0, b1 = entries[tensor_name]
        return self._read_into(model_uri, tensor_name, torch.empty(max(b1 - b0, 1), dtype=torch.uint8))

    def _pinned(self, nbytes: int) -> torch.Tensor:
        with self._pin_lock:
            still = []
            for ev, buf in self._pin_busy:               # uploads that have finished give their buffers back
                if ev.query():
                    self._pin_free.setdefault(buf.numel(), []).append(buf)
                else:
                    still.append((ev, buf))
            self._pin_busy = still
            lst = self._pin_free.get(nbytes)
            if lst:
                return lst.pop()
        return torch.empty(max(nbytes, 1), dtype=torch.uint8).pin_memory()

    def prefetch(self, model_uri: str, tensor_name: str, device: str):
        adapter = self._adapters.get(model_uri)
        for key in adapter.part(tensor_name).keys if adapter is not None else (tensor_name,):
            self._prefetch_key(model_uri, key, device)

    def _prefetch_key(self, model_uri: str, tensor_name: str, device: str):
        dev = torch.device(device)
        if dev.type != "cuda":
            return
        key = (model_uri, tensor_name, str(dev))
        if key in self._prefetched:
            return
        if self._readers is None:
            from concurrent.futures import ThreadPoolExecutor
            self._readers = ThreadPoolExecutor(max_workers=self._reader_threads, thread_name_prefix="shardmerge-reader")
        stream = self._copy_streams.get(str(dev))
        if stream is None:
            stream = self._copy_streams[str(dev)] = torch.cuda.Stream(device=dev)
        shard = self._shard_of(model_uri, tensor_name)
        _, entries = self._meta(shard)
        _, _, b0, b1 = entries[tensor_name]

        def job():
            buf = self._pinned(b1 - b0)
            host = self._read_into(model_uri, tensor_name, buf)
            with torch.cuda.device(dev), torch.cuda.stream(stream):
                t = host.to(dev, non_blocking=True)
                ev = stream.record_event()
            with self._pin_lock:
                self._pin_busy.append((ev, buf))
            return t, ev

        self._prefetched[key] = self._readers.submit(job)

    def _take_prefetched(self, model_uri: str, tensor_name: str, device: str):
        fut = self._prefetched.pop((model_uri, tensor_name, str(torch.device(device))), None)
        if fut is None:
            return None
        t, ev = fut.result()
        cur = torch.cuda.current_stream(t.device)
        cur.wait_event(ev)
        t.record_stream(cur)
        return t

    def get_tensor(self, model_uri: str, tensor_name: str, device: str = "cpu") -> TensorPromise:
        self._shard_of(model_uri, tensor_name)            # KeyError now, like the reference, not inside the promise

        def load():
            if torch.device(device).type == "cuda":
                pre = self._take_prefetched(model_uri, tensor_name, device)
                if pre is not None:
                    return pre
                self._prefetch_key(model_uri, tensor_name, device)          # not announced: the same path, waited for at once
                return self._take_prefetched(model_uri, tensor_name, device)
            return self._host_tensor(model_uri, tensor_name)

        return TensorPromise(model_uri, tensor_name, device, load)
