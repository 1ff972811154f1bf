"""Device data path of the training inputs (SURVEY.md section 8 f-3).

PyMIC feeds the step from 16 CPU workers that decode float64 NIfTI, normalise, pad, crop, flip and build an fp32 one-hot
per sample (io/nifty_dataset.py:171-218, transform/{normalize,pad,crop,flip,label_convert}.py); that pipeline cannot
feed a B200 at ~10^9 voxels/s.  Here the padded volumes of a domain live in HBM for the whole run and one gather kernel
per step (csrc/datapath.cu) cuts and flips the batch:

* ``RandomCrop`` with foreground focus (transform/crop.py:170-244) and ``RandomFlip`` (flip.py:14-62): the crop origin
  and the flip axes are drawn on the host with ``random.Random`` in the SAME order of draws as the reference transforms
  (per sample: one randint per axis with a non-zero margin, the foreground coin, the three bounding-box draws; then the
  width / height / depth coins), so a run seeded like the reference's workers makes the same decisions;
* ``NormalizeWithMeanStd`` (transform/normalize.py) either runs on the host per volume before the volumes are uploaded
  (where the transform list puts it before ``RandomCrop``), or, with ``normalize=``, per cut patch on the device (where
  it comes after ``RandomCrop``, as in the FPL+ configs): the volumes are then stored raw and a statistics kernel plus a
  normalising gather replace the plain gather;
* ``LabelToProbability`` (label_convert.py:82-88) and ``NiftyDataset.set_weight_`` (nifty_dataset.py:165-168) are NOT
  applied here: the batch carries the uint8 label map, the uint8 agreement code (0/1/2 = weight 0/0.5/1) and the
  per-sample image weight, and the loss kernels (fpl_dice_ce_*_ex) expand them per voxel.

The batch dicts it yields have the keys ``SegmentationAgent.train_step`` consumes: ``image`` fp32 [N,C,D,H,W], ``label``
uint8 [N,D,H,W], ``pixel_weight`` uint8 [N,1,D,H,W], ``image_weight`` fp32 [N] (device), ``names``.

``sampler_args_from_config`` and ``load_train_csv`` build the samplers of a training ``.cfg`` (``[dataset]
{1,2}_train_csv``, ``train_batch_size``, ``train_transform`` and its keys); ``SegmentationAgent`` uses them when no
training loaders were given.
"""
import random
import struct

import numpy as np
import torch

from .ops import call, ptr, stream_ptr


def normalize_with_mean_std(image, mask_nonzero=False, channels=None, mean=None, std=None):
    """NormalizeWithMeanStd (transform/normalize.py:36-62) per channel: (x - mean) / std; with ``mask_nonzero`` the
    statistics come from the voxels > 0 (the rest is left untouched apart from the affine map, as in the reference's
    default ``random_fill = False`` path).  ``channels`` (default all) are the channels normalised, the others are
    returned as they are; ``mean`` / ``std``, lists parallel to ``channels``, are fixed values that replace the
    statistics.  This is also the definition the per-patch device normalisation of ``DevicePatchSampler`` follows."""
    img = np.asarray(image, np.float32).copy()
    for i, c in enumerate(range(img.shape[0]) if channels is None else channels):
        ch = img[c]
        if mean is not None and mean[i] is not None:
            img[c] = (ch - np.float32(mean[i])) / np.float32(std[i])
            continue
        sel = ch[ch > 0] if mask_nonzero and (ch > 0).any() else ch
        img[c] = (ch - sel.mean()) / max(float(sel.std()), 1e-8)
    return img


def pad_to(volume, out_size, mode="reflect"):
    """Pad (transform/pad.py:60-90): centre-pad the trailing three axes up to ``out_size``."""
    shape = volume.shape[-3:]
    margin = [max(0, out_size[i] - shape[i]) for i in range(3)]
    if not any(margin):
        return volume
    lo = [m // 2 for m in margin]
    hi = [m - l for m, l in zip(margin, lo)]
    pad = [(0, 0)] * (volume.ndim - 3) + list(zip(lo, hi))
    return np.pad(volume, pad, mode if all(s > 1 for s in shape) else "edge")


def code_from_pixel_weight(w):
    """Agreement weight map {0, 0.5, 1} (data/get_pixel_weight.py:21-26) -> uint8 code {0, 1, 2}."""
    return np.rint(np.asarray(w, np.float32) * 2.0).astype(np.uint8)


class DevicePatchSampler(object):
    """Resident volumes of ONE domain + per-step RandomCrop / RandomFlip on the device.

    ``volumes``: list of dicts with ``image`` [C,D,H,W] fp32 (raw, or normalised on the host), optional ``label``
    [D,H,W] integer, optional ``pixel_weight`` [D,H,W] in {0, 0.5, 1} (or ``code`` uint8), optional ``image_weight``
    float, ``name``.  Iterating yields batch dicts forever (one epoch = a random permutation of the volumes, like a
    shuffling DataLoader with ``drop_last``).

    ``normalize``: None (default), or NormalizeWithMeanStd applied to every cut patch on the device, as a dict
    {channel: {"mean": m, "std": s, "mask": bool}} of the channels to normalise (at most 16 image channels; the
    others are copied raw).  ``mean`` / ``std`` (both or neither) are fixed values; without them the statistics are the
    patch's, over its voxels > 0 with ``mask`` (see ``normalize_with_mean_std``).  The crop / flip decisions do not
    depend on it."""

    def __init__(self, volumes, patch, batch_size, device, fg_focus=True, fg_ratio=0.5, mask_label=(1,),
                 flip=(False, True, True), seed=1, rank=0, world=1, normalize=None):
        self.patch = tuple(int(p) for p in patch)
        self.batch = int(batch_size)
        self.device = torch.device(device)
        self.fg_focus, self.fg_ratio, self.mask_label = fg_focus, fg_ratio, tuple(mask_label)
        self.flip_depth, self.flip_height, self.flip_width = flip
        self.rng = random.Random(int(seed) * 1000003 + rank)
        self.rank, self.world = rank, world
        self.vols = []
        for v in volumes:
            img = pad_to(np.asarray(v["image"], np.float32), self.patch)
            if img.ndim == 3:
                img = img[None]
            ent = {"name": v.get("name", "vol%d" % len(self.vols)), "shape": img.shape[1:],
                   "image": torch.from_numpy(np.ascontiguousarray(img)).to(self.device),
                   "label": None, "code": None, "bbox": None, "image_weight": float(v.get("image_weight", 1.0))}
            if v.get("label") is not None:
                lab = pad_to(np.asarray(v["label"]).astype(np.uint8), self.patch, "constant")
                ent["label"] = torch.from_numpy(np.ascontiguousarray(lab)).to(self.device)
                mask = np.isin(lab, self.mask_label)
                if mask.any():
                    idx = np.nonzero(mask)
                    # get_ND_bounding_box (util/image_process.py:8-35), margin 0: bb_max is max + 1
                    ent["bbox"] = ([int(i.min()) for i in idx], [int(i.max()) + 1 for i in idx])
            code = v.get("code")
            if code is None and v.get("pixel_weight") is not None:
                code = code_from_pixel_weight(v["pixel_weight"])
            if code is not None:
                code = pad_to(np.asarray(code, np.uint8), self.patch, "constant")
                ent["code"] = torch.from_numpy(np.ascontiguousarray(code)).to(self.device)
            self.vols.append(ent)
        if not self.vols:
            raise ValueError("DevicePatchSampler needs at least one volume")
        self.in_chns = int(self.vols[0]["image"].shape[0])
        self.has_label = all(v["label"] is not None for v in self.vols)
        self.has_code = any(v["code"] is not None for v in self.vols)
        self._order, self._pos = [], 0
        # double-buffered outputs + pinned parameter tables: the batch of step i+1 is gathered while step i trains
        n, (pd, ph, pw) = self.batch, self.patch
        self._out = [{"image": torch.empty((n, self.in_chns, pd, ph, pw), dtype=torch.float32, device=self.device),
                      "label": torch.empty((n, pd, ph, pw), dtype=torch.uint8, device=self.device) if self.has_label else None,
                      "code": torch.empty((n, 1, pd, ph, pw), dtype=torch.uint8, device=self.device) if self.has_code else None,
                      "iw": torch.empty(n, dtype=torch.float32, device=self.device),
                      "rows": torch.empty(64 * n, dtype=torch.uint8, device=self.device),
                      "rows_host": torch.empty(64 * n, dtype=torch.uint8).pin_memory() if self.device.type == "cuda" else None,
                      "iw_host": torch.empty(n, dtype=torch.float32).pin_memory() if self.device.type == "cuda" else None,
                      "copied": None}
                     for _ in range(2)]
        self._slot = 0
        self.last_params = None
        self._norm = None if normalize is None else self._norm_tables(normalize)

    def _norm_tables(self, normalize):
        """{channel: {mean, std, mask}} -> the per-channel (mode, mean, std) host arrays of fpl_gather_patches_norm and
        its statistics workspace (modes: 0 raw, 1 fixed, 2 patch statistics, 3 patch statistics of the voxels > 0)."""
        import ctypes
        c_num = self.in_chns
        if c_num > 16:
            raise ValueError("normalize: %d image channels, the device normalisation takes at most 16" % c_num)
        modes, means, stds = [0] * c_num, [0.0] * c_num, [1.0] * c_num
        for c, spec in dict(normalize).items():
            spec = dict(spec or {})
            unknown = set(spec) - {"mean", "std", "mask"}
            if unknown:
                raise ValueError("normalize[%r]: unknown keys %s" % (c, sorted(unknown)))
            if not (isinstance(c, int) and 0 <= c < c_num):
                raise ValueError("normalize: channel %r not in [0, %d)" % (c, c_num))
            m, s = spec.get("mean"), spec.get("std")
            if (m is None) != (s is None):
                raise ValueError("normalize[%d]: give both mean and std, or neither" % c)
            if m is not None:
                if not float(s) > 0.0:
                    raise ValueError("normalize[%d]: std %r must be > 0" % (c, s))
                modes[c], means[c], stds[c] = 1, float(m), float(s)
            else:
                modes[c] = 3 if spec.get("mask", False) else 2
        n, (pd, ph, pw) = self.batch, self.patch
        ws = None
        if self.device.type == "cuda" and any(m >= 2 for m in modes):
            from .lib import load
            nbytes = int(load().fpl_gather_patches_norm_workspace_bytes(n, c_num, pd, ph, pw))
            ws = torch.empty(nbytes // 8, dtype=torch.float64, device=self.device)
        return {"mode": (ctypes.c_int * c_num)(*modes), "mean": (ctypes.c_float * c_num)(*means),
                "std": (ctypes.c_float * c_num)(*stds), "ws": ws, "ws_bytes": 0 if ws is None else 8 * ws.numel()}

    # -- the reference's random decisions ------------------------------------------------------------------
    def _next_volume(self):
        if self._pos >= len(self._order):
            idx = list(range(self.rank, len(self.vols), self.world)) or list(range(len(self.vols)))
            self.rng.shuffle(idx)
            self._order, self._pos = idx, 0
        i = self._order[self._pos]
        self._pos += 1
        return i

    def draw(self, vol):
        """(crop origin, flip bits) of one sample: transform/crop.py:213-234 then flip.py:38-47."""
        shape, out = vol["shape"], self.patch
        margin = [shape[i] - out[i] for i in range(3)]
        crop_min = [0 if m == 0 else self.rng.randint(0, m) for m in margin]
        if self.fg_focus and self.rng.random() < self.fg_ratio:
            if vol["bbox"] is None:
                bb_min, bb_max = [0, 0, 0], list(shape)
            else:
                bb_min, bb_max = vol["bbox"]
            crop_min = [self.rng.randint(bb_min[i], bb_max[i]) - int(out[i] / 2) for i in range(3)]
            crop_min = [max(0, c) for c in crop_min]
            crop_min = [min(crop_min[i], shape[i] - out[i]) for i in range(3)]
        flip = 0
        if self.flip_width and self.rng.random() > 0.5:
            flip |= 4
        if self.flip_height and self.rng.random() > 0.5:
            flip |= 2
        if self.flip_depth and self.rng.random() > 0.5:
            flip |= 1
        return crop_min, flip

    # -- one batch ---------------------------------------------------------------------------------------------
    def next_batch(self):
        out = self._out[self._slot]
        self._slot ^= 1
        rows, names, params = bytearray(), [], []
        iw = []
        for _ in range(self.batch):
            v = self.vols[self._next_volume()]
            (d0, h0, w0), flip = self.draw(v)
            D, H, W = v["shape"]
            rows += struct.pack("<3Q7i3i", v["image"].data_ptr(), v["label"].data_ptr() if v["label"] is not None else 0,
                                v["code"].data_ptr() if v["code"] is not None else 0, D, H, W, d0, h0, w0, flip, 0, 0, 0)
            names.append(v["name"])
            iw.append(v["image_weight"])
            params.append((v["name"], (d0, h0, w0), flip))
        self.last_params = params
        if out["rows_host"] is not None:
            if out["copied"] is not None:
                out["copied"].synchronize()          # the pinned tables of this slot were last read two batches ago
            out["rows_host"].copy_(torch.frombuffer(rows, dtype=torch.uint8))
            out["rows"].copy_(out["rows_host"], non_blocking=True)
            out["iw_host"].copy_(torch.tensor(iw, dtype=torch.float32))
            out["iw"].copy_(out["iw_host"], non_blocking=True)
            out["copied"] = torch.cuda.Event()
            out["copied"].record()
        else:
            out["rows"].copy_(torch.frombuffer(rows, dtype=torch.uint8))
            out["iw"].copy_(torch.tensor(iw, dtype=torch.float32))
        pd, ph, pw = self.patch
        if self._norm is None:
            call("fpl_gather_patches", ptr(out["rows"]), self.batch, self.in_chns, pd, ph, pw, ptr(out["image"]),
                 ptr(out["label"]), ptr(out["code"]), stream_ptr())
        else:
            nt = self._norm
            call("fpl_gather_patches_norm", ptr(out["rows"]), self.batch, self.in_chns, pd, ph, pw, nt["mode"], nt["mean"],
                 nt["std"], ptr(nt["ws"]), nt["ws_bytes"], ptr(out["image"]), ptr(out["label"]), ptr(out["code"]),
                 stream_ptr())
        batch = {"image": out["image"], "names": names}
        if self.has_label:
            batch["label"] = out["label"]
        if self.has_code:
            batch["pixel_weight"] = out["code"]
            batch["image_weight"] = out["iw"]
        return batch

    def __iter__(self):
        return self

    def __next__(self):
        return self.next_batch()

    def __len__(self):
        return max(1, len(self.vols) // (self.batch * self.world))


# -- training samplers from a .cfg -------------------------------------------------------------------------------------
# keys (after the ``<Transform>_`` prefix, lower-cased as parse_config stores them) of the train transforms this path runs.
# NormalizeWithMeanStd's ``mask`` / ``random_fill`` follow PyMIC 0.3's transform/normalize.py; these two names have not
# been re-checked against the reference tree.
_TRANSFORM_KEYS = {
    "pad": ("output_size", "inverse"),
    "randomcrop": ("output_size", "foreground_focus", "foreground_ratio", "mask_label", "inverse"),
    "randomflip": ("flip_depth", "flip_height", "flip_width", "inverse"),
    "normalizewithmeanstd": ("channels", "mean", "std", "mask", "random_fill", "inverse"),
    "labeltoprobability": ("class_num", "inverse"),
}


def _normalize_spec(name, params):
    if params.get("random_fill", False):
        raise ValueError("%s_random_fill = True is not supported: NumPy's normal stream cannot be reproduced on the "
                         "device" % name)
    chans = params.get("channels")
    if chans is None:
        raise ValueError("%s needs %s_channels" % (name, name))
    chans = list(chans) if isinstance(chans, (list, tuple)) else [chans]
    mean, std = params.get("mean"), params.get("std")
    if (mean is None) != (std is None):
        raise ValueError("%s: give both %s_mean and %s_std, or neither" % (name, name, name))
    if mean is not None:
        mean = list(mean) if isinstance(mean, (list, tuple)) else [mean]
        std = list(std) if isinstance(std, (list, tuple)) else [std]
        if len(mean) != len(chans) or len(std) != len(chans):
            raise ValueError("%s: %s_mean / %s_std need one value per channel of %s_channels" % (name, name, name, name))
    mask = bool(params.get("mask", False))
    return {int(c): {"mean": None if mean is None else float(mean[i]), "std": None if std is None else float(std[i]),
                     "mask": mask} for i, c in enumerate(chans)}


def sampler_args_from_config(config, domain, rank=0, world=1):
    """The ``DevicePatchSampler`` of training domain ``domain`` (0 or 1) that a ``.cfg`` describes, without touching a
    device or a file: {"csv": [dataset] <domain+1>_train_csv, "root_dir", "host_transforms": [(name, params)] to apply
    per volume at load time (``load_train_csv``), "sampler": keyword arguments of ``DevicePatchSampler``}.

    ``train_transform`` is read in order, as PyMIC applies it:
    * ``Pad`` (``Pad_output_size``) pads at load time; it must come before ``RandomCrop``;
    * ``RandomCrop`` (``_output_size``, ``_foreground_focus``, ``_foreground_ratio``, ``_mask_label``) and ``RandomFlip``
      (``_flip_depth``, ``_flip_height``, ``_flip_width``) are the sampler's decisions; an absent key keeps the
      sampler's default, an absent ``RandomFlip`` flips nothing;
    * ``NormalizeWithMeanStd`` (``_channels``, ``_mean``, ``_std``, ``_mask``) after ``RandomCrop`` normalises every cut
      patch on the device (``normalize=``); before it, ``normalize_with_mean_std`` runs per volume at load time;
    * ``LabelToProbability`` is implied: the loss kernels build the one-hot from the uint8 label;
    * ``*_inverse`` keys only matter at test time and are ignored.
    Any other transform, any other key of these transforms, and ``NormalizeWithMeanStd_random_fill = True`` raise
    ``ValueError``.  The sampler draws from ``[training] random_seed`` + ``domain``, so the two domains do not repeat
    each other's decisions."""
    ds = config.get("dataset", {})
    csv_key = "%d_train_csv" % (domain + 1)
    if not ds.get(csv_key):
        raise ValueError("[dataset] %s is not set" % csv_key)
    seed = int(config.get("training", {}).get("random_seed", 1)) + int(domain)
    kwargs = {"batch_size": int(ds.get("train_batch_size", 1)), "flip": (False, False, False), "seed": seed,
              "rank": int(rank), "world": int(world)}
    host, cropped = [], False
    for name in ds.get("train_transform") or []:
        key = str(name).lower()
        if key not in _TRANSFORM_KEYS:
            raise ValueError("train_transform: %s is not supported by the device data path" % name)
        params = {k[len(key) + 1:]: v for k, v in ds.items() if k.startswith(key + "_")}
        bad = sorted(set(params) - set(_TRANSFORM_KEYS[key]))
        if bad:
            raise ValueError("%s: unsupported key(s) %s" % (name, ", ".join("%s_%s" % (name, b) for b in bad)))
        if key == "pad":
            if cropped:
                raise ValueError("train_transform: Pad must come before RandomCrop")
            if params.get("output_size") is not None:
                host.append(("Pad", {"output_size": [int(x) for x in params["output_size"]]}))
        elif key == "randomcrop":
            if params.get("output_size") is None:
                raise ValueError("RandomCrop needs RandomCrop_output_size")
            kwargs["patch"] = tuple(int(x) for x in params["output_size"])
            for k, arg in (("foreground_focus", "fg_focus"), ("foreground_ratio", "fg_ratio"), ("mask_label", "mask_label")):
                if params.get(k) is not None:
                    kwargs[arg] = params[k]
            if "mask_label" in kwargs and not isinstance(kwargs["mask_label"], (list, tuple)):
                kwargs["mask_label"] = [kwargs["mask_label"]]
            cropped = True
        elif key == "randomflip":
            kwargs["flip"] = tuple(bool(params.get("flip_" + a, dflt)) for a, dflt in
                                   (("depth", False), ("height", True), ("width", True)))
        elif key == "normalizewithmeanstd":
            spec = _normalize_spec(name, params)
            if cropped:
                kwargs["normalize"] = spec
            else:
                host.append(("NormalizeWithMeanStd", spec))
    if "patch" not in kwargs:
        raise ValueError("train_transform has no RandomCrop: the device data path trains on cut patches")
    return {"csv": ds[csv_key], "root_dir": ds.get("root_dir", "") or "", "host_transforms": host, "sampler": kwargs}


def _squeeze3(a):
    a = np.asarray(a)
    return a[0] if a.ndim == 4 and a.shape[0] == 1 else a


def load_train_csv(csv_path, root_dir="", host_transforms=()):
    """Volume dicts of ``DevicePatchSampler`` from a training CSV: a header row, then rows
    ``image,label[,pixel_weight,image_weight]`` (``artefacts.write_train_csv``) of ``.npy`` / ``.nii`` / ``.nii.gz``
    paths under ``root_dir``.  Labels become uint8, ``pixel_weight`` the agreement code, ``image_weight`` a float
    (1.0 when absent).  ``host_transforms`` (``sampler_args_from_config``) are applied to every volume in order."""
    import csv
    import os
    from .artefacts import load_volume
    with open(csv_path, newline="") as f:
        rows = [r for r in csv.reader(f)][1:]
    vols = []
    for row in rows:
        if not row or not row[0].strip():
            continue
        img = np.asarray(load_volume(os.path.join(root_dir, row[0])), np.float32)
        img = img[None] if img.ndim == 3 else img
        v = {"image": img, "name": row[0], "image_weight": 1.0}
        if len(row) > 1 and row[1].strip():
            v["label"] = _squeeze3(load_volume(os.path.join(root_dir, row[1]))).astype(np.uint8)
        if len(row) > 2 and row[2].strip():
            v["code"] = code_from_pixel_weight(_squeeze3(load_volume(os.path.join(root_dir, row[2]))))
        if len(row) > 3 and row[3].strip():
            v["image_weight"] = float(row[3])
        for name, params in host_transforms:
            if name == "Pad":
                v["image"] = pad_to(v["image"], params["output_size"])
                for k in ("label", "code"):
                    if k in v:
                        v[k] = pad_to(v[k], params["output_size"], "constant")
            else:
                for c, spec in sorted(params.items()):
                    v["image"] = normalize_with_mean_std(v["image"], spec["mask"], [c], [spec["mean"]], [spec["std"]])
        vols.append(v)
    return vols


def samplers_from_config(config, device, rank=0, world=1):
    """One ``DevicePatchSampler`` per training domain (``[network] num_domains``, at most 2) whose ``[dataset]
    <d>_train_csv`` is set; None for the others."""
    n_dom = min(2, int(config.get("network", {}).get("num_domains", 2)))
    out = []
    for d in range(2):
        if d >= n_dom or not config.get("dataset", {}).get("%d_train_csv" % (d + 1)):
            out.append(None)
            continue
        a = sampler_args_from_config(config, d, rank, world)
        vols = load_train_csv(a["csv"], a["root_dir"], a["host_transforms"])
        out.append(DevicePatchSampler(vols, device=device, **a["sampler"]))
    return out
