"""``ExtractResNet`` -- drop-in for the reference's models/resnet/extract_resnet.py on the B200 engine.

Same constructor / attributes / ``forward`` / ``extract`` surface (``forward`` returns None, or the per-video feature
dicts when ``--gather_features`` sets ``keep_features``); the output key is the feature type
(``resnet18`` ... ``resnet152``), a float64 ``(T, D)`` array (the reference builds it with ``.tolist()``), plus ``fps``
and ``timestamps_ms``, saved under ``{output_path}/{feature_type}``.  Every frame is read sequentially with OpenCV
(a failed FIRST read is skipped, extract_resnet.py:130-137); a reader thread fills pinned blocks of frames while the
engine runs the previous block, so at most a few blocks are held, never the whole video.  The BGR->RGB swap
(extract_resnet.py:142), Resize(256) / CenterCrop(224) / ToTensor / Normalize and the network run on the GPU.
"""
from __future__ import annotations

import glob
import os
import queue
import threading
from typing import Dict

import numpy as np
import torch
from tqdm import tqdm

from .. import synthetic_weights
from ..resnet_engine import ResNetEngine
from ..utils import AsyncSink, action_on_extraction, already_extracted, form_list_from_user_input

# attributes the reference's constructor copies from `args` unchanged (extract_resnet.py:26-41)
_ARG_ATTRS = ('feature_type', 'batch_size', 'extraction_fps', 'show_pred', 'keep_tmp_files', 'on_extraction')
_DEPTHS = {f'resnet{d}': d for d in (18, 34, 50, 101, 152)}


def load_resnet_state_dict(feature_type: str) -> Dict[str, torch.Tensor]:
    """``$VF_RESNET_CKPT``, then ``<torch.hub.get_dir()>/checkpoints/resnet{depth}-*.pth`` (where
    ``torchvision.models.resnet{depth}(pretrained=True)`` caches its download).  torchvision's key layout, unchanged;
    ``num_batches_tracked`` and ``fc.*`` are dropped.  ``VF_RESNET_SYNTHETIC=<seed>`` selects seeded synthetic weights
    instead (there is no network access to download the file)."""
    depth = _DEPTHS[feature_type]
    if os.environ.get("VF_RESNET_SYNTHETIC") is not None:
        sd = synthetic_weights.resnet_state_dict(depth, int(os.environ["VF_RESNET_SYNTHETIC"] or 0))
    else:
        hub = os.path.join(torch.hub.get_dir(), "checkpoints", f"resnet{depth}-*.pth")
        cands = [os.environ.get("VF_RESNET_CKPT")] + sorted(glob.glob(hub))
        path = next((p for p in cands if p and os.path.exists(p)), None)
        if path is None:
            looked = [c for c in [os.environ.get("VF_RESNET_CKPT"), hub] if c]
            raise FileNotFoundError(f"{feature_type} checkpoint not found (looked at {looked}); there is no network "
                                    "access -- set VF_RESNET_CKPT")
        sd = torch.load(path, map_location="cpu", weights_only=True)
    sd = {k: v for k, v in sd.items() if not (k.startswith("fc.") or k.endswith("num_batches_tracked"))}
    for conv, (co, ci, k) in synthetic_weights.resnet_conv_shapes(depth).items():
        bn = synthetic_weights.resnet_bn_name(conv)
        need = {conv + ".weight": (co, ci, k, k)}
        need.update({f"{bn}.{s}": (co,) for s in ("weight", "bias", "running_mean", "running_var")})
        for key, shape in need.items():
            if key not in sd:
                raise KeyError(f"{feature_type} checkpoint is missing '{key}'")
            if tuple(sd[key].shape) != shape:
                raise ValueError(f"{feature_type} checkpoint: '{key}' has shape {tuple(sd[key].shape)}, expected {shape}")
    return sd


class ExtractResNet(torch.nn.Module):

    def __init__(self, args):
        super().__init__()
        for name in _ARG_ATTRS:
            setattr(self, name, getattr(args, name))
        self.path_list = form_list_from_user_input(args)
        self.central_crop_size = 224
        # per-feature sub-folders of the scratch and output roots, as the reference lays them out
        self.tmp_path, self.output_path = (os.path.join(root, self.feature_type) for root in (args.tmp_path, args.output_path))
        self.progress = tqdm(total=len(self.path_list))
        if self.extraction_fps is not None:
            raise NotImplementedError("extraction_fps re-encodes with ffmpeg (outside the rebuilt path, SURVEY.md §2)")
        self._engines: Dict[int, ResNetEngine] = {}
        self.keep_features = False        # dispatch sets it when the features are all-gathered as well as saved
        # frames per engine call: frames are independent, so how many share a call does not change any value; the
        # reference's default of one frame per call (--batch_size 1) would leave the GPU idle between launches
        self.frames_per_call = max(self.batch_size, int(os.environ.get("VF_RESNET_FRAMES", "128")))

    def forward(self, indices: torch.LongTensor):
        device = indices.device
        if device.type != 'cuda':
            raise RuntimeError("the B200 engine has no CPU path: pass indices on a CUDA device")
        sink = AsyncSink() if os.environ.get("VF_ASYNC_SINK") == "1" else None     # opt-in extras, see ExtractCLIP.forward
        resume = os.environ.get("VF_RESUME") == "1"
        kept = []
        try:
            for idx in indices:
                video = self.path_list[idx]
                try:                                      # per-video catch-print-continue (extract_resnet.py:73-83)
                    if resume and already_extracted([self.feature_type], video, self.output_path, self.on_extraction):
                        self.progress.update()
                        continue
                    feats = self.extract(device, None, None, video)
                    if self.keep_features:
                        kept.append(feats)
                    if sink is not None:
                        sink.submit(feats, video, self.output_path, self.on_extraction)
                    else:
                        action_on_extraction(feats, video, self.output_path, self.on_extraction)
                except KeyboardInterrupt:
                    raise
                except Exception as err:
                    print(err)
                    print(f'Extraction failed at: {video} with error (↑). Continuing extraction')
                self.progress.update()
        finally:
            if sink is not None:
                sink.close()
        return kept if self.keep_features else None

    def _engine(self, device: torch.device) -> ResNetEngine:
        """One engine per device, created on first use (the constructor needs no GPU)."""
        idx = device.index if device.index is not None else torch.cuda.current_device()
        if idx not in self._engines:
            self._engines[idx] = ResNetEngine(load_resnet_state_dict(self.feature_type), _DEPTHS[self.feature_type], idx,
                                              max_frames=self.frames_per_call)
        return self._engines[idx]

    def extract(self, device, model=None, classifier=None, video_path=None) -> Dict[str, np.ndarray]:
        import cv2
        engine = self._engine(device)
        cap = cv2.VideoCapture(video_path)
        if not cap.isOpened():
            # the reference saves an empty array for a file OpenCV cannot open; here it is reported as a failed video
            # (a readable video without frames still gives the reference's empty array)
            raise RuntimeError(f"OpenCV cannot open {video_path}")
        fps = cap.get(cv2.CAP_PROP_FPS)
        stamps, feats = [], []
        blocks: "queue.Queue" = queue.Queue(maxsize=2)     # filled blocks waiting for the engine
        stop = threading.Event()
        F = self.frames_per_call

        def put(item):
            while not stop.is_set():
                try:
                    blocks.put(item, timeout=0.1)
                    return
                except queue.Full:
                    pass

        def reader():
            try:
                first, block, k = True, None, 0
                while cap.isOpened() and not stop.is_set():
                    ok, bgr = cap.read()
                    if first:                             # a failed FIRST read is skipped (extract_resnet.py:134-137)
                        first = False
                        if ok is False:
                            continue
                    if not ok:
                        break
                    stamps.append(cap.get(cv2.CAP_PROP_POS_MSEC))
                    if block is None:
                        block, k = torch.empty((F,) + bgr.shape, dtype=torch.uint8, pin_memory=True), 0
                    block[k].numpy()[...] = bgr           # BGR as decoded: the engine reads it as RGB
                    k += 1
                    if k == F:
                        put((block, k))
                        block = None
                if block is not None:
                    put((block, k))
                put(None)
            except Exception as err:                      # handed to the consumer, raised there
                put(err)
            finally:
                cap.release()

        t = threading.Thread(target=reader, daemon=True)
        t.start()
        try:
            while True:
                item = blocks.get()
                if item is None:
                    break
                if isinstance(item, Exception):
                    raise item
                block, k = item
                feats.append(engine.forward_frames_u8_host(block[:k], swap_rb=True, group=F))
        finally:
            stop.set()
            t.join()
        out = torch.cat(feats).numpy().astype(np.float64) if feats else np.array([])
        return {self.feature_type: out, 'fps': np.array(fps), 'timestamps_ms': np.array(stamps)}
