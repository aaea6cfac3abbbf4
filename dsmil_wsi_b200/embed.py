"""The patch-embedding loop (SURVEY §8 a13; reference compute_feats.py:19-82), B200-side re-design.

Reference loop per bag: DataLoader(batch 128, 4 workers: PIL open + VF.to_tensor) -> `.float().cuda()`
(synchronous, pageable, 77 MB per batch) -> `i_classifier(patches)` -> `.cpu().numpy()` (a sync per batch)
-> Python list -> DataFrame.to_csv('%.4f').

Here:
  * the patch FILES cross PCIe (~2 MB per 128-patch batch instead of 77 MB of fp32) and are decoded on the device
    (jpeg.py / csrc/jpeg_kernels.cuh: Huffman decoding one warp per patch, IDCT, upsampling, colour, /255 -- bit for
    bit PIL's output), on a side stream under the backbone of the previous batch; the worker threads only read files;
  * a batch holding a file the device path does not take (progressive, CMYK, ...) goes through PIL -- the reference's
    own decoder -- and crosses PCIe as **uint8 HWC** from pinned staging buffers (19 MB per batch);
    uint8 -> fp32 CHW / 255 is then `dsmil_patches_u8_to_f32` (bit-identical to VF.to_tensor).
    `DSMIL_B200_JPEG=host` forces that route for every batch, `=gpu` forbids it (raises instead);
  * the backbone is the caller's module (torchvision ResNet via cuDNN -- library code, as in the reference);
    the instance classifier head is `dsmil_instance_scores` (our kernel) through IClassifier;
  * features stay on the device for the whole bag: ONE D2H per bag, or none when `sink` hands the bag
    straight to the aggregator (`milnet.b_classifier`, `MILNet.forward_bags`);
  * the CSV wire format of the reference (`header 0..D-1`, '%.4f', no index) is written by `write_bag_csv`.
The function signature mirrors compute_feats.compute_feats(args, bags_list, i_classifier, save_path, magnification).
"""
from __future__ import annotations

import glob
import os
import sys
import weakref
from concurrent.futures import ThreadPoolExecutor
from typing import Callable, List, Optional, Sequence

import numpy as np
import torch

from . import _lib
from . import functional as Fn


def list_patches(bag_dir: str, magnification: str = "single") -> List[str]:
    """compute_feats.py:64-68: jpg + jpeg of the bag folder ('high': one level deeper)."""
    if magnification in ("single", "low"):
        return glob.glob(os.path.join(bag_dir, "*.jpg")) + glob.glob(os.path.join(bag_dir, "*.jpeg"))
    if magnification == "high":
        return (glob.glob(os.path.join(bag_dir, "*" + os.sep + "*.jpg")) +
                glob.glob(os.path.join(bag_dir, "*" + os.sep + "*.jpeg")))
    raise ValueError(f"magnification {magnification!r} is not a single-level listing; tree mode has its own "
                     "traversal (list_tree_patches / compute_tree_feats)")


def list_tree_patches(bag_dir: str):
    """Two-magnification traversal of compute_feats.py:91,100-103: the low-magnification patches of the bag
    folder (jpg then jpeg) and, per low patch `<x>.jp(e)g`, the high-magnification patches in folder `<x>/`.
    Returns (low_paths, [high_paths of low 0, high_paths of low 1, ...])."""
    low = glob.glob(os.path.join(bag_dir, "*.jpg")) + glob.glob(os.path.join(bag_dir, "*.jpeg"))
    high = []
    for lp in low:
        folder = os.path.dirname(lp) + os.sep + os.path.splitext(os.path.basename(lp))[0]
        high.append(glob.glob(folder + os.sep + "*.jpg") + glob.glob(folder + os.sep + "*.jpeg"))
    return low, high


def _decode_u8(src) -> np.ndarray:
    """PIL decode of a path or of the bytes of a file (the host route of a batch)."""
    import io
    from PIL import Image
    with Image.open(io.BytesIO(src) if isinstance(src, (bytes, bytearray, memoryview)) else src) as im:
        a = np.asarray(im.convert("RGB") if im.mode != "RGB" else im, dtype=np.uint8)
    return np.array(a, copy=True) if not a.flags.writeable else a  # HWC uint8 (writable: torch.from_numpy)


def _read_file(path: str) -> bytes:
    with open(path, "rb") as f:
        return f.read()


def patches_to_float(u8_hwc: torch.Tensor) -> torch.Tensor:
    """uint8 [B,H,W,C] (CUDA) -> float32 [B,C,H,W] = x / 255 (== VF.to_tensor per image), on the device."""
    Fn.require_cuda(u8_hwc, "patches")
    if u8_hwc.dtype != torch.uint8 or u8_hwc.dim() != 4:
        raise TypeError("patches_to_float expects a uint8 [B,H,W,C] tensor")
    u8_hwc = u8_hwc.contiguous()
    B, H, W, Cc = (int(s) for s in u8_hwc.shape)
    with torch.cuda.device(u8_hwc.device):
        out = torch.empty(B, Cc, H, W, dtype=torch.float32, device=u8_hwc.device)
        _lib.check(_lib.load().dsmil_patches_u8_to_f32(u8_hwc.data_ptr(), B, H, W, Cc, out.data_ptr(), Fn._stream()),
                   "dsmil_patches_u8_to_f32")
    return out


def format_bag_csv(feats: np.ndarray) -> str:
    """The reference's wire format as a string (compute_feats.py:80-82: pandas to_csv(index=False,
    float_format='%.4f')), produced by the native formatter in blocks of rows."""
    import ctypes as C
    from . import _hostlib
    lib = _hostlib.load()
    x = np.ascontiguousarray(np.asarray(feats), dtype=np.float32)
    if x.ndim != 2 or x.shape[1] < 1:
        raise ValueError(f"feats must be [N, D], got shape {x.shape}")
    N, D = x.shape
    block = max(1, (8 << 20) // (49 * D))
    header_len = len(",".join(str(i) for i in range(D))) + 1
    parts = []
    for lo in range(0, max(N, 1), block):
        rows = x[lo:lo + block]
        cap = 12 * D + 49 * rows.shape[0] * D + 16
        buf = C.create_string_buffer(cap)
        n = lib.dsmil_csv_format_bag(rows.ctypes.data, rows.shape[0], D, buf, cap)
        if n < 0:
            raise RuntimeError(f"dsmil_csv_format_bag: {_hostlib.ERRORS.get(n, n)}")
        parts.append(buf.raw[(header_len if lo else 0):n].decode("ascii"))
    return "".join(parts)


def write_bag_csv(feats: np.ndarray, save_path: str, bag_dir: str) -> str:
    """`<save_path>/<class>/<bag>.csv` in the reference's wire format (compute_feats.py:80-82), written by the
    native formatter (csrc_host/bagcsv.c): byte-identical to `DataFrame.to_csv(index=False,
    float_format='%.4f')`, ~70x faster (7 s -> 0.1 s for a 10 000 x 512 bag)."""
    import ctypes as C
    from . import _hostlib
    cls, name = bag_dir.split(os.path.sep)[-2], bag_dir.split(os.path.sep)[-1]
    os.makedirs(os.path.join(save_path, cls), exist_ok=True)
    out = os.path.join(save_path, cls, name + ".csv")
    x = np.ascontiguousarray(np.asarray(feats), dtype=np.float32)
    if x.ndim != 2 or x.shape[1] < 1:
        raise ValueError(f"feats must be [N, D], got shape {x.shape}")
    rc = _hostlib.load().dsmil_csv_write_bag(out.encode(), x.ctypes.data, x.shape[0], x.shape[1])
    if rc < 0:
        raise OSError(f"writing {out}: {_hostlib.ERRORS.get(rc, rc)}")
    return out


class _Staging:
    """Two slots, each: pinned file blob + headers (device route) or a pinned uint8 batch (host route) and their
    device twins; batch b+1 is read / parsed / copied / decoded while batch b is embedded."""

    def __init__(self, batch: int, H: int, W: int, device, memory_format=torch.contiguous_format):
        from . import jpeg
        self.batch, self.H, self.W, self.device, self.memory_format = batch, H, W, device, memory_format
        self.host_u8 = [None, None]                      # allocated on first use of the host route
        self.dev_u8 = [None, None]
        self.dev_f32 = [None, None]                      # allocated on first use of the device route
        self.blob = [jpeg._Pinned(), jpeg._Pinned()]
        self.hdr = [jpeg._Pinned(), jpeg._Pinned()]
        self.status_host = [torch.zeros(batch, dtype=torch.int32).pin_memory() for _ in range(2)]
        self.status_names = [None, None]
        self.copied = [torch.cuda.Event() for _ in range(2)]
        self.consumed = [torch.cuda.Event() for _ in range(2)]
        self.stream = torch.cuda.Stream(device=device)
        self.decoder = jpeg.JpegBatchDecoder(device)

    # The device buffers are written on self.stream, so they come from its pool.  Taken from the pool of the staging
    # thread's current stream (the compute stream) they could be blocks the embedder has freed while its kernels
    # that use them are still queued there, and the decode of the next batch would race with them.
    def u8(self, s):
        if self.host_u8[s] is None:
            self.host_u8[s] = torch.empty(self.batch, self.H, self.W, 3, dtype=torch.uint8).pin_memory()
            with torch.cuda.stream(self.stream):
                self.dev_u8[s] = torch.empty(self.batch, self.H, self.W, 3, dtype=torch.uint8, device=self.device)
        return self.host_u8[s], self.dev_u8[s]

    def f32(self, s):
        if self.dev_f32[s] is None:
            with torch.cuda.stream(self.stream):
                self.dev_f32[s] = torch.empty(self.batch, 3, self.H, self.W, dtype=torch.float32, device=self.device,
                                              memory_format=self.memory_format)
        return self.dev_f32[s]

    def check_status(self, s):
        """Raises if the last device decode of slot s reported a file it could not decode (call after its
        `copied` event has completed)."""
        names = self.status_names[s]
        if names is None:
            return
        self.status_names[s] = None
        st = self.status_host[s][:len(names)].numpy()
        if np.any(st != 0):
            from . import jpeg
            i = int(np.flatnonzero(st)[0])
            raise RuntimeError(f"JPEG decode of {names[i]} failed on the device: {jpeg.STATUS.get(int(st[i]), int(st[i]))}")


_STAGING = {}       # (device, batch, H, W, layout) -> _Staging: pinned + device buffers are reused from bag to bag


def _staging(batch, H, W, dev, fmt) -> "_Staging":
    key = (str(dev), batch, H, W, str(fmt))
    st = _STAGING.get(key)
    if st is None:
        if len(_STAGING) >= 2:                               # e.g. the two magnifications of tree mode; no unbounded growth
            old = _STAGING.pop(next(iter(_STAGING)))
            for e in old.consumed:                           # its buffers return to its stream's pool: the compute
                e.synchronize()                              # stream must have finished reading them
        st = _STAGING[key] = _Staging(batch, H, W, dev, fmt)
    st.status_names = [None, None]
    return st


def jpeg_route() -> str:
    r = os.environ.get("DSMIL_B200_JPEG", "auto")
    if r not in ("auto", "gpu", "host"):
        raise ValueError(f"DSMIL_B200_JPEG={r!r}: expected auto, gpu or host")
    return r


class _GraphedEmbedder:
    """The embedder forward of one full batch as a CUDA graph: ~70 launches (cuDNN convolutions, the fused norm kernels,
    the score kernel) become one replay, so the loop is paced by the GPU, not by the host thread that also stages the
    next batch.  The static input is this object's own buffer (one device copy per batch); outputs are cloned out."""

    def __init__(self, i_classifier, batch, H, W, dev, fmt):
        self.key = self.make_key(i_classifier, batch, H, W, dev, fmt)
        self.x = torch.zeros(batch, 3, H, W, dtype=torch.float32, device=dev).contiguous(memory_format=fmt)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(2):
                i_classifier(self.x)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.feats, self.classes = i_classifier(self.x)

    @staticmethod
    def make_key(i_classifier, batch, H, W, dev, fmt):
        # replaced parameter tensors (not in-place updates) invalidate a captured graph: key on their addresses
        return (batch, H, W, str(dev), str(fmt), tuple(p.data_ptr() for p in i_classifier.parameters()),
                tuple(b.data_ptr() for b in i_classifier.buffers()))

    def __call__(self, x):
        self.x.copy_(x)
        self.graph.replay()
        return self.feats.clone(), self.classes.clone()


_GRAPHS = weakref.WeakKeyDictionary()      # model -> (key, _GraphedEmbedder or None); kept off the module itself so that
                                            # deepcopy / pickling of the caller's model never meets a CUDA graph


def _graphed(i_classifier, batch, H, W, dev, fmt):
    """The cached graph of this (model, geometry), captured on first use; None when capture is not possible."""
    key = _GraphedEmbedder.make_key(i_classifier, batch, H, W, dev, fmt)
    cur = _GRAPHS.get(i_classifier)
    if cur is not None and cur[0] == key:
        return cur[1]
    try:
        g = _GraphedEmbedder(i_classifier, batch, H, W, dev, fmt)
    except Exception as e:                                   # a backbone with capture-hostile ops: run it eagerly
        sys.stderr.write(f"[dsmil_b200] embedder forward not captured as a CUDA graph ({type(e).__name__}: {e}); "
                         "running it eagerly\n")
        torch.cuda.synchronize(dev)
        g = None
    _GRAPHS[i_classifier] = (key, g)
    return g


@torch.no_grad()
def embed_bag(paths: Sequence[str], i_classifier, batch_size: int = 128, num_workers: int = 4,
              device: Optional[torch.device] = None):
    """Features [N, D] (device) and instance scores [N, C] (device) of one bag of patch files.

    Three things run concurrently per batch: a staging thread reads + parses the NEXT batch's files natively and
    enqueues its H2D copy and decode kernels on a side stream; the GPU decodes that batch under the backbone of the
    CURRENT one; the calling thread only replays the backbone's CUDA graph (DSMIL_B200_EMBED_GRAPH=0: launches it
    eagerly) and collects the features."""
    from . import jpeg
    dev = device or next(i_classifier.parameters()).device
    if dev.type != "cuda":
        raise RuntimeError("embed_bag needs the model on a CUDA device (no CPU path)")
    if not paths:
        return None, None
    i_classifier.eval()
    fe = getattr(i_classifier, "feature_extractor", None)
    if fe is not None and os.environ.get("DSMIL_B200_FUSE_IN", "1") != "0":
        from .embedder import fuse_instance_norm            # InstanceNorm + residual + ReLU of the backbone: one kernel each
        fuse_instance_norm(fe)                               # (idempotent; leaves parameters / state_dict untouched)
    fmt = torch.contiguous_format
    if fe is not None and os.environ.get("DSMIL_B200_NHWC", "1") != "0" and any(isinstance(m, torch.nn.Conv2d) for m in fe.modules()):
        # cuDNN's channels-last kernels run this backbone's convolutions 1.5x faster on B200; values and state_dict are
        # unchanged (only the strides of the 4-D weights), the decoded batch is produced in that layout directly
        fmt = torch.channels_last
        if not getattr(fe, "_dsmil_channels_last", False):
            fe.to(memory_format=torch.channels_last)
            fe._dsmil_channels_last = True
    route = jpeg_route()
    head = jpeg.parse_paths(paths[:1])                       # geometry of the bag from the first file's header
    if head.statuses[0] == 0:
        H, W = head.H, head.W
    else:                                                    # not a file the parser reads: let PIL say what it is
        H, W = _decode_u8(paths[0]).shape[:2]
    batches = [paths[i:i + batch_size] for i in range(0, len(paths), batch_size)]
    full_batches = sum(1 for b in batches if len(b) == batch_size)
    feats_out, cls_out = [], []
    with torch.cuda.device(dev):
        graphed = None
        if os.environ.get("DSMIL_B200_EMBED_GRAPH", "1") != "0" and full_batches >= 4:
            graphed = _graphed(i_classifier, batch_size, H, W, dev, fmt)     # before any other thread touches CUDA
        with ThreadPoolExecutor(max_workers=max(1, num_workers)) as pool, ThreadPoolExecutor(max_workers=1) as stager:
            st = _staging(batch_size, H, W, dev, fmt)
            compute = torch.cuda.current_stream()
            for s in range(2):
                st.consumed[s].record(compute)
                st.copied[s].record(st.stream)

            def stage(bi):                                  # runs on the staging thread
                s = bi % 2
                names = batches[bi]
                n = len(names)
                on_device = False
                pb = None
                with torch.cuda.device(dev):
                    if route != "host":
                        st.copied[s].synchronize()          # the pinned blob / headers of this slot are free again
                        st.check_status(s)
                        pb = jpeg.parse_paths(names, st.blob[s], st.hdr[s], pin=True, threads=max(1, num_workers))
                        on_device = pb.bad == 0 and (pb.H, pb.W) == (H, W)
                        if not on_device and route == "gpu":
                            raise RuntimeError(f"DSMIL_B200_JPEG=gpu, but {pb.bad} file(s) of the batch starting at {names[0]} "
                                               f"are not decodable on the device (statuses {pb.statuses.tolist()})")
                    st.consumed[s].synchronize()            # the previous user of this slot's device buffers has read them
                    if on_device:
                        out = st.f32(s)
                        status = st.decoder.decode(pb, out_f32=out[:n], stream=st.stream)
                        with torch.cuda.stream(st.stream):
                            st.status_host[s][:n].copy_(status, non_blocking=True)
                            st.copied[s].record(st.stream)
                        st.status_names[s] = names
                        return s, n, True
                    srcs = [pb.file_bytes(j) for j in range(n)] if pb is not None else names
                    imgs = list(pool.map(_decode_u8, srcs))
                    hb, db = st.u8(s)
                    st.copied[s].synchronize()
                    for j, im in enumerate(imgs):
                        if im.shape != (H, W, 3):
                            raise ValueError(f"patch {names[j]} is {im.shape}, expected {(H, W, 3)}")
                        hb[j].copy_(torch.from_numpy(im))
                    with torch.cuda.stream(st.stream):
                        db[:n].copy_(hb[:n], non_blocking=True)
                        st.copied[s].record(st.stream)
                    return s, n, False

            pending = stager.submit(stage, 0)
            for bi in range(len(batches)):
                s, n, on_device = pending.result()
                if bi + 1 < len(batches):
                    pending = stager.submit(stage, bi + 1)  # read / parse / copy / decode the next batch meanwhile
                compute.wait_event(st.copied[s])
                x = st.f32(s)[:n] if on_device else patches_to_float(st.dev_u8[s][:n]).contiguous(memory_format=fmt)
                if graphed is not None and n == batch_size:
                    feats, classes = graphed(x)             # copies x into the graph's input first
                else:
                    feats, classes = i_classifier(x)
                st.consumed[s].record(compute)              # the slot's device buffers have been read
                feats_out.append(feats)
                cls_out.append(classes)
            for s in range(2):
                st.copied[s].synchronize()
                st.check_status(s)
    return torch.cat(feats_out), torch.cat(cls_out)


def fuse_tree_feats(high: torch.Tensor, low: torch.Tensor, parent: torch.Tensor, mode: str) -> torch.Tensor:
    """Row m of the tree bag from high-magnification row m and its parent low-magnification row
    (compute_feats.py:111-116): 'fusion' -> high + 0.25 * low[parent] ([M, D]); 'cat' -> [high | low[parent]]
    ([M, 2D]).  Works on whatever device the operands live on; fp32 results equal the reference's numpy
    expression bit for bit (0.25 * x is exact, one rounding in the add)."""
    if mode not in ("fusion", "cat"):
        raise NotImplementedError(f"{mode} is not an excepted option for --tree_fusion. This argument accepts 2 "
                                  "options: 'fusion' and 'cat'.")          # wording of compute_feats.py:116
    if high.dim() != 2 or low.dim() != 2 or high.shape[1] != low.shape[1]:
        raise ValueError(f"high {tuple(high.shape)} and low {tuple(low.shape)} must be [M, D] and [L, D]")
    if parent.numel() != high.shape[0]:
        raise ValueError("one parent index per high-magnification row")
    par = low.index_select(0, parent.to(device=low.device, dtype=torch.int64))
    if mode == "fusion":
        return high + 0.25 * par
    return torch.cat((high, par), dim=-1)


def compute_tree_feats(args, bags_list, embedder_low, embedder_high, save_path=None,
                       sink: Optional[Callable[[str, torch.Tensor], None]] = None, wire: str = "csv", embed=None):
    """Mirror of compute_feats.compute_tree_feats (compute_feats.py:84-126); `args` needs batch_size,
    num_workers, tree_fusion.

    The reference embeds every high-magnification patch as its own batch of one (one PIL open, one H2D, ~60
    launches and one D2H per patch) and fuses in numpy on the host.  Here all high patches of a bag go through
    the same double-buffered uint8 staging loop as the low ones (`embed_bag`, full batches -- InstanceNorm is
    per-sample, so batch composition does not change a patch's features), the parent gather + fusion is one
    device op, and the bag leaves the device once.  Row order is the reference's: low patches in listing
    order, within each its high patches in listing order; low patches without a folder contribute nothing.
    `embed(paths, embedder, batch_size, num_workers) -> (feats, classes)` defaults to `embed_bag`."""
    if wire not in ("csv", "bin", "both"):
        raise ValueError(f"wire must be 'csv', 'bin' or 'both', got {wire!r}")
    mode = getattr(args, "tree_fusion", "cat")
    if mode not in ("fusion", "cat"):
        fuse_tree_feats(torch.empty(0, 1), torch.empty(0, 1), torch.empty(0, dtype=torch.int64), mode)   # raises
    embed = embed or embed_bag
    bs, nw = getattr(args, "batch_size", 128), getattr(args, "num_workers", 4)
    num_bags = len(bags_list)
    for i, bag_dir in enumerate(bags_list):
        low_paths, high_lists = list_tree_patches(bag_dir)
        high_paths = [p for hl in high_lists for p in hl]
        sys.stdout.write("\r Computed: {}/{} -- {}/{}".format(i + 1, num_bags, len(low_paths), len(low_paths)))
        if not high_paths:
            print("No valid patch extracted from: " + bag_dir)   # compute_feats.py:120-121
            continue
        low_feats, _ = embed(low_paths, embedder_low, bs, nw)
        high_feats, _ = embed(high_paths, embedder_high, bs, nw)
        parent = torch.tensor([j for j, hl in enumerate(high_lists) for _ in hl], dtype=torch.int64)
        feats = fuse_tree_feats(high_feats, low_feats, parent, mode)
        if sink is not None:
            sink(bag_dir, feats)
        if save_path is not None:
            host = feats.cpu().numpy()
            if wire in ("csv", "both"):
                write_bag_csv(host, save_path, bag_dir)
            if wire in ("bin", "both"):
                write_bag_container(host, save_path, bag_dir)


def write_bag_container(feats: np.ndarray, save_path: str, bag_dir: str) -> str:
    """Same naming as write_bag_csv, `.bin` container (formats.write_bag_bin): exact fp32, 4 B/value."""
    from .formats import write_bag_bin
    cls, name = bag_dir.split(os.path.sep)[-2], bag_dir.split(os.path.sep)[-1]
    os.makedirs(os.path.join(save_path, cls), exist_ok=True)
    out = os.path.join(save_path, cls, name + ".bin")
    write_bag_bin(out, feats)
    return out


def compute_feats(args, bags_list, i_classifier, save_path=None, magnification="single",
                  sink: Optional[Callable[[str, torch.Tensor, torch.Tensor], None]] = None, wire: str = "csv"):
    """Mirror of compute_feats.compute_feats (compute_feats.py:58-82).  `args` needs batch_size / num_workers.
    save_path: write one file per bag (None: skip) -- wire="csv" is the reference's `%.4f` text, "bin" the
    binary container, "both" writes the two.  sink(bag_dir, feats_dev, classes_dev): optional device-side
    hand-off (e.g. straight into the aggregator) that avoids any file round trip."""
    if wire not in ("csv", "bin", "both"):
        raise ValueError(f"wire must be 'csv', 'bin' or 'both', got {wire!r}")
    num_bags = len(bags_list)
    # the text of bag i is formatted and written (native code, GIL released) while bag i+1 is being embedded
    with ThreadPoolExecutor(max_workers=1) as writer:
        written = []
        for i, bag_dir in enumerate(bags_list):
            paths = list_patches(bag_dir, magnification)
            feats, classes = embed_bag(paths, i_classifier, getattr(args, "batch_size", 128), getattr(args, "num_workers", 4))
            sys.stdout.write("\r Computed: {}/{}".format(i + 1, num_bags))
            if feats is None:
                print("No valid patch extracted from: " + bag_dir)   # compute_feats.py:77-78
                continue
            if sink is not None:
                sink(bag_dir, feats, classes)
            if save_path is not None:
                host = feats.cpu().numpy()
                if wire in ("csv", "both"):
                    written.append(writer.submit(write_bag_csv, host, save_path, bag_dir))
                if wire in ("bin", "both"):
                    written.append(writer.submit(write_bag_container, host, save_path, bag_dir))
        for w in written:
            w.result()                                       # surfaces I/O errors; every file is on disk on return
